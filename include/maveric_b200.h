/* maveric_b200.h -- size-explicit and batched C ABI of libmaveric_b200.so.
 *
 * The legacy, reference-shaped symbols are declared in maveric_slam_compat.h.
 * This header adds what the reference's fixed-size signatures cannot express:
 * explicit grid sizes, device-resident batches of frame pairs, and the
 * Gauss-Newton PnP that the reference only sketches (include/tracking.h:45-52,
 * src/projection_factor.c:27-33).  Plain C: pointers and sizes only.
 *
 * Conventions
 *   - every function returns an mv_status (0 = MV_OK); nothing here calls exit()
 *   - "d_" pointers are device memory on the context's GPU, "h_" pointers are host
 *   - batched calls are asynchronous on the context's stream; mv_ctx_sync() waits
 *   - a frame is the reference's pair of int8 tensors (tracking_main.c:71-82):
 *       semi [cells][65], desc [cells][256], cell = col*rows + row (column-major,
 *       tracking_main.c:59-66); a batch is n_frames of them back to back
 *   - caller owns all buffers; the context owns only its scratch
 *
 * Device and thread contract
 *   - a context belongs to the GPU given to mv_ctx_create.  Every entry point that takes a
 *     context makes that GPU current for the duration of the call and restores the calling
 *     thread's current device before it returns (mv_ctx_create included), so contexts of
 *     different GPUs can be used from one thread and a context can be used from any thread
 *   - a context is not internally locked: one call at a time per context (one context per
 *     host thread or per GPU is the intended use); different contexts are independent.  The
 *     legacy void symbols share one process-global context on device 0 behind a mutex
 *   - batched calls take at most 65535 pairs / frames (MV_ERR_BAD_ARG beyond that; the
 *     host-buffer sequence calls chunk internally and have no such limit)
 *   - on any error return of mv_track_sequence_host or mv_track_sequence_landmarks_host the library has
 *     drained its streams: the caller's host buffers are no longer read when the call returns
 */
#ifndef MAVERIC_B200_H
#define MAVERIC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
  MV_OK = 0,
  MV_ERR_NO_DEVICE = 1,     /* no usable sm_100 device: there is no CPU fallback */
  MV_ERR_CUDA = 2,          /* a CUDA call failed; see mv_last_error() */
  MV_ERR_BAD_ARG = 3,
  MV_ERR_TOO_MANY_VALID = 4 /* top_N.c:91-94 condition (legacy symbol exits instead) */
} mv_status;

typedef struct mv_ctx mv_ctx;

mv_status   mv_ctx_create(int device, mv_ctx** out);
void        mv_ctx_destroy(mv_ctx* ctx);
/* Run subsequent batched calls on an existing CUDA stream (cudaStream_t as void*). */
mv_status   mv_ctx_set_stream(mv_ctx* ctx, void* cuda_stream);
mv_status   mv_ctx_sync(mv_ctx* ctx);
const char* mv_last_error(mv_ctx* ctx);
const char* mv_status_str(mv_status s);
/* Number of kernels this context has launched so far (bench.py's gpu_launches). */
unsigned long long mv_ctx_launch_count(mv_ctx* ctx);
/* Average device time in ms of the launches recorded under `tag` since the last reset
 * (CUDA events on the context's stream); tags: "detect","topn","norms","match",
 * "gather","pnp","ransac".  Enabled with mv_ctx_profile(ctx, 1). */
mv_status   mv_ctx_profile(mv_ctx* ctx, int enable);
mv_status   mv_ctx_profile_read(mv_ctx* ctx, const char* tag, double* avg_ms, int* launches);
/* Profile mode only: correspondence-passes the Gauss-Newton PnP kernel accepted (and therefore
 * accumulated into normal equations) in the launches since the last read; the executed-work
 * figure of bench.py's roofline.  Reading resets the counter. */
mv_status   mv_ctx_pnp_work(mv_ctx* ctx, unsigned long long* accepted);
/* Executed work of the last tensor-core matcher launch: tiles of 128 queries that held a query, and the
 * 128 x 256 x 64 int8 chunks the tensor pipe ran for them (blocks the call; bench.py's tensor roofline). */
mv_status   mv_ctx_match_work(mv_ctx* ctx, unsigned long long* tiles, unsigned long long* chunks);

/* ------------------------------------------------------------------------- */
/* Detector post-processing: src/top_N.c                                      */
/* ------------------------------------------------------------------------- */

/* compute_softmax (top_N.c:136-165) over n_frames frames.
 *   d_semi        int8  [n_frames][cells][65]
 *   d_semi_scale  float [n_frames]
 *   d_max_idx     int32 [n_frames][cells]   argmax channel 0..63, or 64
 *   d_prob        float [n_frames][cells]   prob, or -1 when max_idx == 64
 *   d_num_valid   int32 [n_frames]          may be NULL */
mv_status mv_softmax_batch(mv_ctx* ctx, int n_frames, int cells,
                           const int8_t* d_semi, const float* d_semi_scale,
                           int32_t* d_max_idx, float* d_prob, int32_t* d_num_valid);

/* compute_top_N (top_N.c:53-134) from the per-cell (max_idx, prob) above.
 *   top_n       the reference's N;  max_valid  the reference's MAX_VALID_FEATURES
 *   d_q_patch/d_q_idx int32 [n_frames][top_n], d_q_prob float [n_frames][top_n]
 *   d_q_count   int32 [n_frames]  (*num_selected)
 *   d_overflow  int32 [n_frames]  1 where the reference would exit(1); may be NULL */
mv_status mv_top_n_batch(mv_ctx* ctx, int n_frames, int cells, int top_n, int max_valid,
                         const int32_t* d_max_idx, const float* d_prob,
                         int32_t* d_q_patch, int32_t* d_q_idx, float* d_q_prob,
                         int32_t* d_q_count, int32_t* d_overflow);

/* Host-pointer, synchronous, single-frame forms with explicit sizes. */
mv_status compute_softmax_ex(mv_ctx* ctx, float scale, const int8_t* h_semi, int cells,
                             int* num_valid, int* max_indices, float* probs);
mv_status compute_top_N_ex(mv_ctx* ctx, float scale, const int8_t* h_semi, int cells,
                           int N, int max_valid, int* num_selected,
                           int* N_patches, int* N_indices, float* N_probs);

/* ------------------------------------------------------------------------- */
/* Windowed int8 descriptor search: src/tracking_main.c:18-43,103-194         */
/* ------------------------------------------------------------------------- */

typedef struct {
  int rows, cols;          /* feature grid of both frames */
  int shift_x, shift_y;    /* tracking_main.c:104-105 */
  int radius;              /* tracking_main.c:106 */
  int max_matches;         /* MAX_NUM_MATCH (150 in the reference) */
  double match_threshold;  /* MATCH_THRESHOLD (0.9); compared squared, in double */
  double min_prob0;        /* candidate gate, 0.2 at tracking_main.c:146 */
  int use_tensor_cores;    /* 0: dp4a warp-per-query kernel, 1: tcgen05 tile kernel, 2 (default): tcgen05
                            * where its limits hold (rows <= 256), else dp4a.  Same results either way. */
} mv_match_params;

void mv_match_params_default(mv_match_params* p, int rows, int cols);

/* Match n_pairs frame pairs.  Pair p searches frame f0[p] (candidates) for the
 * queries of frame f1[p]; d_f0/d_f1 NULL means the sequence (p, p+1).
 *   d_desc      int8  [n_frames][cells][256]
 *   d_max_idx/d_prob  per-cell detector output of every frame (mv_softmax_batch)
 *   d_q_patch/d_q_idx/d_q_count  query lists of every frame (mv_top_n_batch), stride top_n
 * Outputs, per pair, in query order, capped at max_matches (tracking_main.c:167-192):
 *   d_match_pts   float [n_pairs][max_matches][4]  (x0,y0,x1,y1) pixels
 *   d_match_count int32 [n_pairs]
 *   d_match_cell0 int32 [n_pairs][max_matches]  winning frame-0 cell   (may be NULL)
 *   d_match_query int32 [n_pairs][max_matches]  query ordinal i        (may be NULL)
 *   d_match_score float [n_pairs][max_matches]  best dist_squared      (may be NULL) */
mv_status mv_match_batch(mv_ctx* ctx, const mv_match_params* p,
                         int n_frames, int n_pairs, int top_n,
                         const int32_t* d_f0, const int32_t* d_f1,
                         const int8_t* d_desc,
                         const int32_t* d_max_idx, const float* d_prob,
                         const int32_t* d_q_patch, const int32_t* d_q_idx,
                         const int32_t* d_q_count,
                         float* d_match_pts, int32_t* d_match_count,
                         int32_t* d_match_cell0, int32_t* d_match_query,
                         float* d_match_score);

/* Host-pointer, synchronous, one pair; inputs as tracking_main.c has them after setup. */
mv_status mv_match_pair_host(mv_ctx* ctx, const mv_match_params* p,
                             const int8_t* h_desc0, const int8_t* h_desc1,
                             const int* max_indices0, const float* probs0,
                             int num_queries, const int* patches1, const int* indices1,
                             float* points1 /*[max][2] frame0*/, float* points2 /*[max][2] frame1*/,
                             int* num_matches, int* cell0 /*nullable*/, float* score /*nullable*/);

/* ------------------------------------------------------------------------- */
/* Pose: src/pnp_solver.c (legacy RANSAC-E) and the Gauss-Newton PnP          */
/* ------------------------------------------------------------------------- */

/* ransac_essential_matrix (pnp_solver.c:110-165) over a batch; E is the
 * identity the reference forces (pnp_solver.c:81-85), so an iteration is an inlier
 * count of ||p1 - p2||^2 < threshold.  The 8 rand() draws per iteration do not
 * influence any output and are not reproduced.
 *   d_pts        float [n_pairs][stride_pts][4]   (x0,y0,x1,y1)
 *   d_count      int32 [n_pairs]
 *   d_num_inliers int32 [n_pairs]   0 when no iteration finds an inlier (the
 *                                   reference leaves it uninitialised there)
 *   d_inliers    int32 [n_pairs][stride_pts]  indices of the winning iteration (nullable)
 *   d_pose       float [n_pairs][12]  R1 (row-major 3x3) then t, from
 *                recover_pose_from_essential_matrix (pnp_solver.c:168-194)        */
mv_status mv_ransac_identity_batch(mv_ctx* ctx, int n_pairs, int stride_pts,
                                   const float* d_pts, const int32_t* d_count,
                                   int num_iterations, float inlier_threshold,
                                   int32_t* d_num_inliers, int32_t* d_inliers,
                                   float* d_pose);

typedef struct {
  float fx, fy, cx, cy;     /* Camera, types.h:21-23 */
  int   hypotheses;         /* H: RANSAC hypotheses per frame pair */
  int   sample_size;        /* minimal sample, 8 as in pnp_solver.c:121-124 */
  int   sample_iters;       /* GN iterations on the minimal sample */
  int   refine_iters;       /* GN iterations over all correspondences (gated) */
  float gate_sq;            /* squared-pixel inlier gate */
  float min_depth;          /* cheirality guard on the camera-frame z */
  float damping;            /* relative Levenberg damping added to diag(JtJ) */
  uint64_t seed;            /* counter-based sampling: splitmix64(seed, pair, h, i) */
  int   lanes_per_hypothesis; /* threads cooperating on one hypothesis: 1 (one thread each) ..
                               32 (one warp each), a power of two */
  int   first_pair;         /* global index of pair 0 of this call: the sampler is keyed on the
                               global pair index, so results do not depend on chunking/sharding */
} mv_pnp_params;

void mv_pnp_params_default(mv_pnp_params* p);

/* Gauss-Newton PnP RANSAC.  Residual = cam_project(q*X*q^-1 + t) - z
 * (projection_factor.c:27-33), left-multiplicative pose update, normal equations
 * accumulated as the upper triangle of [J|r]^T[J|r] (local_bundle_adjustment.c:171-176).
 *   d_corr      float [n_pairs][5][stride]  SoA planes X,Y,Z (frame-0 camera), u,v (frame-1 px)
 *   d_count     int32 [n_pairs]
 *   d_init_pose float [n_pairs][7] (qw,qx,qy,qz,tx,ty,tz) or NULL for identity
 *   d_pose      float [n_pairs][7]  best hypothesis
 *   d_stats     float [n_pairs][4]  {inliers, cost, best_h, valid}
 *   d_hyp_pose  float [n_pairs][H][8] every hypothesis {q,t,inliers} (nullable) */
/* lanes_per_hypothesis: 1 = one thread per hypothesis (throughput form), 32 = one warp per hypothesis
 * (latency form).  2, 4, 8, 16 are superseded A/B forms that exist only in a library built with
 * -DMV_PNP_AB (mv_pnp_has_ab_forms() == 1); the product library answers MV_ERR_BAD_ARG for them. */
int mv_pnp_has_ab_forms(void);
mv_status mv_pnp_gn_batch(mv_ctx* ctx, const mv_pnp_params* p, int n_pairs, int stride,
                          const float* d_corr, const int32_t* d_count,
                          const float* d_init_pose,
                          float* d_pose, float* d_stats, float* d_hyp_pose);

/* Matches + per-cell depth of frame 0 -> PnP correspondences (stands in for the
 * landmark lookup local_feature_pool.h:16-22 `coords_3D` would provide).
 *   d_depth float [n_frames][cells]; X = depth * K^-1 (x0,y0,1) */
mv_status mv_build_corr_batch(mv_ctx* ctx, int n_pairs, int cells, int rows, int stride,
                              const int32_t* d_f0, const float* d_depth,
                              float fx, float fy, float cx, float cy,
                              const float* d_match_pts, const int32_t* d_match_count,
                              const int32_t* d_match_cell0,
                              float* d_corr);

/* ------------------------------------------------------------------------- */
/* BoW word assignment and the landmark table (SURVEY §8f rank 3)             */
/* ------------------------------------------------------------------------- */

/* Vocabulary of src/bow_main.c (include/data/LCD/vocabulary.h:5-272): base node descriptors int8 [256][n_base]
 * with their scale / bias, leaf descriptors int32 [n_base][words_per_base][4].  Host pointers, copied. */
mv_status mv_bow_set_vocabulary(mv_ctx* ctx, int n_base, int words_per_base, const int8_t* h_base_desc,
                                const float* h_scale, const float* h_bias, const int32_t* h_leaves);
/* Word of every query of every frame (bow_main.c:62-125 under the definition stated in csrc/bow.cu -- the
 * reference program has no defined result, PARITY UNPINNED; its helpers get_binary_descriptor and
 * count_matching_bits are reproduced bit for bit).
 *   d_desc int8 [n_frames][cells][256], d_desc_scale float [n_frames], d_q_patch / d_q_count as mv_top_n_batch
 *   d_word int32 [n_frames][top_n]  base * words_per_base + leaf, -1 beyond the frame's query count
 *   d_base int32 [n_frames][top_n]  the selected base node (nullable)                                        */
mv_status mv_bow_assign_batch(mv_ctx* ctx, int n_frames, int cells, int top_n, const int8_t* d_desc,
                              const float* d_desc_scale, const int32_t* d_q_patch, const int32_t* d_q_count,
                              int32_t* d_word, int32_t* d_base);

/* The reference's LocalFeature (include/local_feature_pool.h:16-22), field for field. */
typedef struct {
  int word_id;        /* -1: empty */
  int frame_ptr;
  int num_frames;
  int frames[8];      /* MAX_LOCAL_FRAMES ring */
  float coords[3];    /* coords_3D */
} mv_landmark;
/* Device-side contents of the reference's local feature pool: a direct map word id -> LocalFeature (the host
 * pool's hash-slot layout depends on insertion order and is not part of its contents).  d_table is caller-owned
 * device memory of n_words records.
 *   init        every record empty
 *   observe     local_feature_matching.c:153-161 for one frame: insert (coords of the word's first occurrence
 *               in the list) or update_local_feature, once per occurrence; ids outside [0, n_words) are skipped
 *   remove_old  local_feature_pool_remove_old (:268-279): one frame older than current_frame - 7 leaves every
 *               record, records without frames are emptied
 *   lookup      coords_3D of a list of words (0,0,0 and found = 0 where the word is not in the table): what
 *               supplies the 3-D side of PnP correspondences                                              */
mv_status mv_landmarks_init(mv_ctx* ctx, int n_words, mv_landmark* d_table);
mv_status mv_landmarks_observe(mv_ctx* ctx, int n_words, mv_landmark* d_table, int frame, int n,
                               const int32_t* d_word_ids, const float* d_coords);
mv_status mv_landmarks_remove_old(mv_ctx* ctx, int n_words, mv_landmark* d_table, int current_frame);
mv_status mv_landmarks_lookup(mv_ctx* ctx, int n_words, const mv_landmark* d_table, int n,
                              const int32_t* d_word_ids, float* d_coords, int32_t* d_found);
/* Matches -> PnP correspondences with the 3-D side from the landmark table instead of a depth map (the
 * lookup local_feature_pool.h:16-22 `coords_3D` exists for): match j of pair p -> its frame-0 cell -> that
 * cell's place in frame 0's query list -> its word (mv_bow_assign_batch) -> table[word].coords.  A match
 * without a landmark gets NaN coordinates (never accepted by the Gauss-Newton gate); lists keep order and
 * length.  Same d_corr layout as mv_build_corr_batch; d_n_with_landmark int32 [n_pairs] (nullable). */
mv_status mv_build_corr_landmarks_batch(mv_ctx* ctx, int n_pairs, int top_n, int stride, int n_words,
                                        const mv_landmark* d_table, const int32_t* d_f0,
                                        const int32_t* d_q_patch, const int32_t* d_q_count,
                                        const int32_t* d_word, const float* d_match_pts,
                                        const int32_t* d_match_count, const int32_t* d_match_cell0,
                                        float* d_corr, int32_t* d_n_with_landmark);

/* The whole sequence's table update in one call: frames 0 .. n_steps-1 with global frame numbers
 * first_frame + f.  Step f is exactly
 *     mv_landmarks_observe(first_frame + f, d_word[f][0 .. q_count), d_coords_in[f])
 *     mv_landmarks_remove_old(first_frame + f)
 * with q_count = min(d_q_count[f], top_n).  d_table is read at entry as the initial state and left in its final
 * state, byte for byte the table of that per-frame loop (stale frames[] / coords of deleted records included).
 * d_coords_out[f][q] receives what mv_landmarks_lookup of d_word[f][q] returns right after step f (0,0,0 where
 * the word is outside [0, n_words) or q >= q_count).  A record keeps the coordinates of the occurrence that
 * inserted it: update_local_feature never touches coords_3D, so a landmark older than frame f is expressed in the
 * camera frame of the frame that inserted it, not in frame f's.
 * Calls chain: [0, k) then [k, n) (first_frame advanced by k) equals one call over [0, n).
 *   d_word int32 [n_steps][top_n], d_q_count int32 [n_steps], d_coords_in / d_coords_out float [n_steps][top_n][3]
 * n_steps <= 65535, n_steps * top_n < 2^31. */
mv_status mv_landmarks_sequence(mv_ctx* ctx, int n_words, mv_landmark* d_table, int first_frame, int n_steps,
                                int top_n, const int32_t* d_word, const int32_t* d_q_count,
                                const float* d_coords_in, float* d_coords_out);

/* ------------------------------------------------------------------------- */
/* Whole path over a sequence of frames (pair p = frames p, p+1)              */
/* ------------------------------------------------------------------------- */

typedef struct {
  mv_match_params match;
  mv_pnp_params   pnp;
  int top_n;               /* queries per frame */
  int max_valid;           /* MAX_VALID_FEATURES analogue */
  int ransac_iterations;   /* legacy RANSAC-E iterations (10); 0 skips it */
  float ransac_threshold;  /* 1.1 */
} mv_track_params;

void mv_track_params_default(mv_track_params* p, int rows, int cols);

/* Result record per frame pair (64 bytes: one row of the multi-GPU pose gather). */
typedef struct {
  float q[4];              /* GN-PnP pose (w,x,y,z) */
  float t[3];
  float pnp_inliers;
  float pnp_cost;
  int32_t num_matches;
  int32_t ransac_inliers;
  int32_t best_hypothesis;
  int32_t status;          /* 0 ok; MV_ERR_TOO_MANY_VALID if a frame overflowed max_valid */
  int32_t pad[3];
} mv_pair_result;

/* Device-resident inputs: d_semi, d_semi_scale, d_desc, d_depth for n_frames; writes
 * n_frames-1 results to d_results.  All intermediates live in context scratch. */
mv_status mv_track_sequence(mv_ctx* ctx, const mv_track_params* p, int n_frames,
                            const int8_t* d_semi, const float* d_semi_scale,
                            const int8_t* d_desc, const float* d_depth,
                            mv_pair_result* d_results);

/* Host (ideally pinned) inputs: stages frames to the GPU in chunks on a copy stream
 * overlapped with compute, and copies the results back; returns when they are in
 * h_results.  h2d/d2h byte counts of the call are returned for bench.py's e2e. */
mv_status mv_track_sequence_host(mv_ctx* ctx, const mv_track_params* p, int n_frames,
                                 const int8_t* h_semi, const float* h_semi_scale,
                                 const int8_t* h_desc, const float* h_depth,
                                 mv_pair_result* h_results,
                                 unsigned long long* h2d_bytes, unsigned long long* d2h_bytes);

/* mv_track_sequence with the 3-D side of pair p's correspondences from the landmark table instead of depth
 * (the reference's data flow, local_feature_matching.c:153-163 and local_feature_pool.h:16-22):
 *   - the words of frames 0 .. n_frames-2 are mv_bow_assign_batch's with d_desc_scale (vocabulary set first);
 *   - a query keypoint of frame f, pixel x = (cell / rows) * 8 + idx % 8, y = (cell % rows) * 8 + idx / 8, is
 *     back-projected with frame f's depth at its cell by the fp32 operations of mv_build_corr_batch; those are
 *     the coordinates its occurrence hands to observe;
 *   - the table steps over frames 0 .. n_frames-2 exactly as mv_landmarks_sequence(first_frame, n_frames - 1)
 *     (frame n_frames-1 is only the query side of the last pair): d_table in/out;
 *   - pair p uses the table right after step p: match j -> its frame-0 cell -> that cell's place in frame p's
 *     query list -> the coordinates of that query's word, mv_build_corr_landmarks_batch against that snapshot
 *     (NaN without a landmark, lists keep order and length); d_n_with_landmark int32 [n_frames-1] (nullable)
 *     receives the count per pair;
 *   - match, RANSAC-E, the Gauss-Newton PnP (sampler keyed on pnp.first_pair + p) and the records are those of
 *     mv_track_sequence.
 * Landmark coordinates are in the camera frame of the frame that inserted the record (see mv_landmarks_sequence);
 * a world-frame map would need solved poses fed back, which serialises the pairs, and is not done here.
 * Two calls over frames [0, k] and [k, n-1] (one halo frame; first_frame and pnp.first_pair advanced by k) equal
 * one call over [0, n-1]. */
mv_status mv_track_sequence_landmarks(mv_ctx* ctx, const mv_track_params* p, int n_frames, int first_frame,
                                      const int8_t* d_semi, const float* d_semi_scale,
                                      const int8_t* d_desc, const float* d_desc_scale, const float* d_depth,
                                      int n_words, mv_landmark* d_table,
                                      mv_pair_result* d_results, int32_t* d_n_with_landmark);

/* mv_track_sequence_landmarks from host (ideally pinned) frames: the staging pipeline of mv_track_sequence_host
 * (chunks of pairs sharing one halo frame, the pair index of the PnP sampler global) with the table carried
 * from chunk to chunk on the device.  Returns when the results are in h_results.
 *   - results, h_n_with_landmark (int32 [n_frames-1], nullable) and the final d_table are byte for byte those of
 *     mv_track_sequence_landmarks on the same frames, whatever the chunk size, pinned or pageable buffers, and
 *     selective staging on or off;
 *   - d_table is caller-owned device memory of n_words records (it is the map, and small), read at entry and left
 *     in its final state;
 *   - two calls over frames [0, k] and [k, n-1] (first_frame and pnp.first_pair advanced by k) equal one call;
 *     there is no limit on n_frames;
 *   - h2d_bytes: those of mv_track_sequence_host (logits, semi scales, depth planes, the descriptor rows the
 *     matcher reads -- the word assignment reads only query rows, which are among them) plus the desc scales;
 *     d2h_bytes: the records, plus h_n_with_landmark when given;
 *   - argument errors (no vocabulary, NULL table, n_words <= 0, non-positive sizes, n_frames < 2) are
 *     MV_ERR_BAD_ARG before anything is enqueued: the table is untouched.  After a CUDA error the streams are
 *     drained and the host buffers no longer read, but the table's state is unspecified.
 * Not sharded over GPUs: a rank's initial table would depend on every earlier frame. */
mv_status mv_track_sequence_landmarks_host(mv_ctx* ctx, const mv_track_params* p, int n_frames, int first_frame,
                                           const int8_t* h_semi, const float* h_semi_scale,
                                           const int8_t* h_desc, const float* h_desc_scale, const float* h_depth,
                                           int n_words, mv_landmark* d_table,
                                           mv_pair_result* h_results, int32_t* h_n_with_landmark /* nullable */,
                                           unsigned long long* h2d_bytes, unsigned long long* d2h_bytes);

/* ------------------------------------------------------------------------- */
/* NMS between the detector and the matcher (src/run_nms.c)                     */
/* ------------------------------------------------------------------------- */

/* The 2x2-quadrant, 4-pixel non-maximum suppression of src/run_nms.c:65-156 on the per-cell
 * detector output of every frame, in place: a suppressed cell gets max_idx = 64 and
 * prob = 64.0f (:138-139).  The reference walks the cell corners sequentially (x outer, y
 * inner) and later corners see earlier suppressions; the kernel keeps exactly that order with a
 * wavefront over t = 2x + y (corners of one wavefront never share a cell), one warp per frame.
 *   d_max_idx int32 [n_frames][rows*cols]   d_prob float [n_frames][rows*cols] */
mv_status mv_nms_batch(mv_ctx* ctx, int n_frames, int rows, int cols, int32_t* d_max_idx, float* d_prob);

/* Host-pointer, synchronous, one frame (the arrays run_nms.c's main() keeps on its stack). */
mv_status run_nms_ex(mv_ctx* ctx, int rows, int cols, int* max_indices, float* probs);

/* ------------------------------------------------------------------------- */
/* Trajectory: chaining the pairwise poses (python/compute_trajectory.py)        */
/* ------------------------------------------------------------------------- */

/* The step after the pose gather.  The reference chains 3x4 [R|t] relative transforms
 * (float64, row-major, transform_XXXXXX_YYYYYY.npy) into frame poses with
 *     R_cur <- R_t R_cur,   t_cur <- t_t + t_cur        (compute_trajectory.py:76-77)
 * starting from the identity (:51).  mv_chain_transforms does the same for n transforms as a
 * parallel scan in float64: d_traj receives n+1 poses [R|t], pose 0 = identity.  The scan
 * regroups the products, so poses agree with the sequential reference to ~1e-13, not bit for bit.
 *   d_transforms double [n][12]      d_traj double [n+1][12] */
mv_status mv_chain_transforms(mv_ctx* ctx, int n, const double* d_transforms, double* d_traj);

/* The hot path's result records (unit quaternion + translation, float) as 3x4 float64
 * transforms, the reference's interchange format (python/pairwise_pnp.py:690-694). */
mv_status mv_results_to_transforms(mv_ctx* ctx, int n, const mv_pair_result* d_results, double* d_transforms);

/* ------------------------------------------------------------------------- */
/* Synthetic KITTI-shaped frames (counter-based, identical to oracle/ and numpy) */
/* ------------------------------------------------------------------------- */
typedef struct {
  uint64_t seed;
  int rows, cols;
  int keypoint_permille;   /* expected keypoints per 1000 world cells */
  int noise_amp;           /* descriptor noise is uniform in [-amp, amp] */
} mv_synth_params;

/* d_off int32 [n_frames][2]: world-cell offset (x, y) of every frame. */
mv_status mv_synth_frames(mv_ctx* ctx, const mv_synth_params* p, int first_frame, int n_frames,
                          const int32_t* d_off, int8_t* d_semi, int8_t* d_desc, float* d_depth);

/* ------------------------------------------------------------------------- */
/* Local bundle adjustment: src/local_bundle_adjustment.c (SURVEY 8f rank 4)   */
/* ------------------------------------------------------------------------- */

/* The Schur complement of the landmarks of `n_windows` independent windows, as main() of
 * local_bundle_adjustment.c:133-246 computes it for one: per (landmark, pose) factor the
 * 10 x 10 product [J|r]^T [J|r] scattered into the landmark / pose-landmark / pose blocks
 * (:152-224), 3 x 3 block inversion (:227), C -= B A^-1 B^T per chunk of landmarks (:229-245),
 * every fp32 sum in the reference's order.
 *   d_J  float [n_windows][n_ldmks][n_poses][20]  factor blocks as the reference stores them:
 *        2 x 10 column-major, columns dLandmark(3) | dPose(6) | residual(1)
 *   d_C  float [n_windows][(6 n_poses + 1)^2]     reduced camera matrix, column-major, last row
 *        = J^T r of the poses (what the reference hands to its unimplemented cholesky(), :247)
 * n_ldmks must be a multiple of chunk (the reference: 1000 landmarks, 8 poses, chunks of 4). */
mv_status mv_lba_schur_batch(mv_ctx* ctx, int n_windows, int n_ldmks, int n_poses, int chunk,
                             const float* d_J, float* d_C);

/* The Gauss-Newton step of the reduced camera systems mv_lba_schur_batch returns: S d = -g with S
 * the 6 n_poses square pose block (only its lower triangle C[j*SH + i], i >= j, is read) and g the
 * last row.  This is the cholesky(C, ...) call the reference leaves as a stub
 * (local_bundle_adjustment.c:88-90,247), so the arithmetic is this library's definition (parity
 * unpinned; stated by oracle/mv_oracle.c:orc_lba_solve): diagonal s + damping * s + 1e-12, L L^T,
 * two triangular sweeps, every sum an fmaf chain in a fixed order -- the 6 x 6 solve of the PnP
 * kernel at n = 6 n_poses.
 *   d_C     float [n_windows][(6 n_poses + 1)^2]   as written by mv_lba_schur_batch
 *   d_delta float [n_windows][6 n_poses]           the step; 0 where d_ok is 0
 *   d_ok    int32 [n_windows]                      1 = solved, 0 = a pivot was not positive (NaN included)
 * n_poses <= 16. */
mv_status mv_lba_solve_batch(mv_ctx* ctx, int n_windows, int n_poses, float damping,
                             const float* d_C, float* d_delta, int32_t* d_ok);

#ifdef __cplusplus
}
#endif
#endif /* MAVERIC_B200_H */
