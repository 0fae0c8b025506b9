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
  float min_depth;          /* cheirality guard on the camera-frame z: a correspondence counts only
                               where min_depth < z < 1e30.  At least FLT_MIN (a smaller value or
                               NaN is MV_ERR_BAD_ARG): the GPU reciprocal flushes a subnormal z to 0 */
  float damping;            /* relative Levenberg damping added to diag(JtJ) */
  uint64_t seed;            /* counter-based sampling: splitmix64(seed, pair, h, i) */
  int   lanes_per_hypothesis; /* threads cooperating on one hypothesis: 1 (one thread each) or
                               32 (one warp each) */
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
 * (latency form); any other value is MV_ERR_BAD_ARG.  mv_pnp_has_ab_forms() always returns 0: the
 * library has no other kernel forms, and the symbol is kept so that existing callers still link. */
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

/* mv_landmarks_sequence split at the point where the entry table is needed, so that a block of frames can be walked
 * before the table it starts from exists (the table relay of tracking.track_sequence_landmarks_sharded).
 *   speculate  walks the block's steps first_frame .. first_frame+n_steps-1 from a GUESSED entry table: the table
 *              that the n_warm steps before it (global frames first_frame-n_warm ..) produce from an empty table.
 *              Reads no caller table.  d_word int32 [n_warm + n_steps][top_n], d_q_count int32 [n_warm + n_steps],
 *              d_coords_in float [n_steps][top_n][3] (warm-up frames need words only); d_coords_in must stay valid
 *              until the resolve has run.  n_warm >= 0, n_steps >= 1, n_warm + n_steps <= 65535,
 *              (n_warm + n_steps) * top_n < 2^31.  *out owns its device memory (stream-ordered on the context's
 *              stream) until mv_lm_spec_release.
 *   resolve    d_table in/out, d_coords_out float [n_steps][top_n][3]: byte for byte
 *              mv_landmarks_sequence(first_frame, n_steps) on the same table, for every n_warm >= 0.  A word whose
 *              true entry record has the guess's shape (word_id; if alive, num_frames and the live frames in ring
 *              order) is patched, any other is walked again from the true record, so a wrong guess costs time and
 *              never changes a byte.  d_n_rewalked int32 [1] (nullable): the number of words walked again.  Refused
 *              (MV_ERR_BAD_ARG, nothing enqueued): a speculation of another context, a second resolve, a NULL table.
 *   release    frees the speculation (after its context's stream work; resolved or not).  Call it before the context
 *              is destroyed. */
typedef struct mv_lm_spec mv_lm_spec;
mv_status mv_landmarks_speculate(mv_ctx* ctx, int n_words, int first_frame, int n_warm, int n_steps, int top_n,
                                 const int32_t* d_word, const int32_t* d_q_count, const float* d_coords_in,
                                 mv_lm_spec** out);
mv_status mv_landmarks_resolve(mv_ctx* ctx, mv_lm_spec* spec, mv_landmark* d_table, float* d_coords_out,
                               int32_t* d_n_rewalked);
void mv_lm_spec_release(mv_lm_spec* spec);

/* ------------------------------------------------------------------------- */
/* Whole path over a sequence of frames (pair p = frames p, p+1)              */
/* ------------------------------------------------------------------------- */

/* Argument errors of the four sequence calls (mv_track_sequence, mv_track_sequence_host,
 * mv_track_sequence_landmarks, mv_track_sequence_landmarks_host) are MV_ERR_BAD_ARG before anything is
 * allocated or enqueued, so a landmark table is untouched.  They cover every refusal of the batched calls the
 * path is made of: NULL inputs, n_frames < 2, non-positive rows / cols / top_n / max_valid / max_matches,
 * match.radius < 0, max_matches > 65535, the PnP limits of mv_pnp_gn_batch (hypotheses, sample_size,
 * lanes_per_hypothesis), use_tensor_cores = 1 on a shape the tensor-core matcher does not take (for the host
 * calls: their largest chunk), more than 65535 frames in the device calls, a d_desc that is not 16-byte aligned
 * in the device calls; in landmark mode also no vocabulary, a vocabulary larger than the word assignment's
 * shared memory, n_words <= 0, a NULL table and (n_frames - 1) * top_n >= 2^31 in the device call. */

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
 *   - argument errors are MV_ERR_BAD_ARG before anything is enqueued (see above): the table is untouched.  After
 *     a CUDA error the streams are drained and the host buffers no longer read, but the table's state is
 *     unspecified.
 * It steps the table chunk by chunk while it stages, so it runs on one GPU; over several, each rank stages its block
 * with mv_track_landmarks_prepare_host (below) before the table arrives. */
mv_status mv_track_sequence_landmarks_host(mv_ctx* ctx, const mv_track_params* p, int n_frames, int first_frame,
                                           const int8_t* h_semi, const float* h_semi_scale,
                                           const int8_t* h_desc, const float* h_desc_scale, const float* h_depth,
                                           int n_words, mv_landmark* d_table,
                                           mv_pair_result* h_results, int32_t* h_n_with_landmark /* nullable */,
                                           unsigned long long* h2d_bytes, unsigned long long* d2h_bytes);

/* mv_track_sequence_landmarks split at the table, so that blocks of a sequence can run on several GPUs with only
 * the table passed from block to block (tracking.track_sequence_landmarks_sharded):
 *   prepare     frames: n_warm warm-up frames (global first_frame-n_warm ..) then the block's n_frames frames
 *               (pair p = block frames p, p+1; d_semi .. d_depth hold all n_warm + n_frames frames).  Enqueues the
 *               detector, the word assignment (with the back-projection), mv_landmarks_speculate, the matcher and
 *               RANSAC-E.  Reads no table.  Allocates everything the three calls need (stream-ordered, owned by *out).
 *   step_table  resolves the speculation against d_table (in/out), which is stepped over the block's frames
 *               0 .. n_frames-2 as mv_track_sequence_landmarks steps it; d_n_rewalked int32 [1] (nullable) as
 *               mv_landmarks_resolve.  Its first launch is the first read of d_table.
 *   solve       correspondences from the resolved coordinates, K3, records: d_results [n_frames-1],
 *               d_n_with_landmark int32 [n_frames-1] (nullable).
 *   release     frees the block (after its context's stream work), in any phase; before the context is destroyed.
 * Equivalence: prepare, step_table, solve on frames [0, n) equal mv_track_sequence_landmarks on them byte for byte --
 * records, counts and final table -- for every n_warm.  Chaining: blocks [0, k] and [k, n-1] (first_frame and
 * pnp.first_pair advanced by k, n_warm frames before each) may be prepared in either order, on one context or on
 * two; stepped in frame order they equal one call.  Other calls on the same context between prepare and solve do
 * not disturb a block.
 * Errors: prepare refuses what mv_track_sequence_landmarks refuses (bar the table, which it does not take) and
 * n_warm < 0 or more than 65535 frames in all, before any allocation or enqueue.  step_table and solve allocate
 * nothing and refuse, with nothing enqueued: a NULL block, a block of another context, a call out of phase (step
 * once after prepare, solve once after step_table) and a NULL table. */
typedef struct mv_lm_block mv_lm_block;
mv_status mv_track_landmarks_prepare(mv_ctx* ctx, const mv_track_params* p, int n_warm, int n_frames, int first_frame,
                                     const int8_t* d_semi, const float* d_semi_scale, const int8_t* d_desc,
                                     const float* d_desc_scale, const float* d_depth, int n_words, mv_lm_block** out);
/* mv_track_landmarks_prepare from host (ideally pinned) buffers laid out the same way (n_warm warm-up frames, then
 * the block's n_frames), over the staging pipeline of mv_track_sequence_landmarks_host
 * (tracking.track_sequence_landmarks_host_sharded).  It returns the same kind of block: step_table, solve and
 * release take it unchanged.
 *   - equivalence: prepare_host, step_table, solve give records, counts and a final table byte for byte those of
 *     mv_track_landmarks_prepare on the same frames (so of mv_track_sequence_landmarks and
 *     mv_track_sequence_landmarks_host), for every n_warm, chunk size, pinned or pageable buffers and selective
 *     staging on or off.  Blocks of either prepare chain with each other under the rule above;
 *   - returns when the host buffers are no longer read (the staging streams are drained); the block's last device
 *     work (the last chunk's matcher, the speculation) may still be queued on the context stream, ahead of anything
 *     enqueued after it.  The block owns only what step_table and solve read: the detector planes stay in the
 *     staging chunks;
 *   - h2d_bytes (nullable, filled at return): for the block's frames exactly what mv_track_sequence_landmarks_host
 *     moves for them; for each warm-up frame its logits, both scales and its query rows only (no depth: warm-up
 *     words need no coordinates; no candidate rows: no matcher runs on them);
 *   - errors: MV_ERR_BAD_ARG, before any allocation, enqueue or host read, for what mv_track_landmarks_prepare
 *     refuses (more than 65535 frames in all included: the speculation's limit) and NULL host pointers.  After a CUDA
 *     error the streams are drained, nothing is kept and *out is NULL. */
mv_status mv_track_landmarks_prepare_host(mv_ctx* ctx, const mv_track_params* p, int n_warm, int n_frames,
                                          int first_frame, const int8_t* h_semi, const float* h_semi_scale,
                                          const int8_t* h_desc, const float* h_desc_scale, const float* h_depth,
                                          int n_words, mv_lm_block** out, unsigned long long* h2d_bytes /* nullable */);
mv_status mv_track_landmarks_step_table(mv_ctx* ctx, mv_lm_block* block, mv_landmark* d_table,
                                        int32_t* d_n_rewalked);
mv_status mv_track_landmarks_solve(mv_ctx* ctx, mv_lm_block* block, mv_pair_result* d_results,
                                   int32_t* d_n_with_landmark);
void mv_track_landmarks_release(mv_lm_block* block);

/* ------------------------------------------------------------------------- */
/* Loop closure: BoW candidates (src/lcd_main.c), verified by match + PnP      */
/* ------------------------------------------------------------------------- */

/* The reference's lcd_main.c intersects the sorted BoW id lists of two frames.  The score below is this library's
 * definition (PARITY UNPINNED: the reference program cannot be run here); with unit weights it is the number of
 * distinct shared words, which is what a sorted-list intersection counts on duplicate-free lists.  All integer,
 * so exact:
 *   P[f][w]       1 where word w in [0, n_words) occurs among frame f's first min(q_count[f], top_n) words
 *                 (duplicates count once; ids outside the range, -1 included, are skipped), else 0
 *   score(i, j)   sum_w weight[w] * P[i][w] * P[j][w], int32; weights in [0, 127] (d_weight NULL: all 1)
 *   candidates    of frame i: the frames j <= i - min_gap of the same call (indices within the call) with
 *                 score >= min_score, the best k by score, descending, the smaller j first on equal scores;
 *                 reported as global frame numbers first_frame + j
 * Each call stands alone: a frame is scored against the earlier frames of its own call only.
 *   d_word int32 [n_frames][top_n], d_q_count int32 [n_frames]   as mv_bow_assign_batch writes them
 *   d_weight int8 [n_words] (nullable)
 *   d_cand int32 [n_frames][k]    candidate frames, -1 in unused slots
 *   d_score int32 [n_frames][k]   their scores, 0 in unused slots
 * With first_frame < 0 a candidate's global number can itself be -1 (j = -1 - first_frame), which reads like an
 * unused slot; a caller with negative frame numbers that must tell them apart passes first_frame 0 and adds its
 * offset to the non-negative entries (mv_detect_loops does so).
 * The similarity is an int8 GEMM on the tensor cores over the lower triangle of 128 x 128 frame tiles; the score
 * matrix is never stored.  Context scratch: the presence matrix, n_frames (rounded up to 128) x n_words (rounded up
 * to 64) bytes, twice with weights, and the per-tile lists, 8 * k bytes per frame and 128-frame column tile
 * (n_frames^2 * k / 16 bytes: 5 MB at 4 541 frames and k = 4, 2.1 GB at 65 535 frames and k = 8).  MV_ERR_BAD_ARG, with no kernel launched: n_frames outside [1, 65535], top_n <= 0, n_words
 * outside [1, 2^24], k outside [1, 8], min_gap < 0, first_frame + n_frames - 1 beyond int32, a NULL buffer, and a
 * negative weight (d_weight is copied to the host to check it, so a call with weights synchronises the context's
 * stream). */
mv_status mv_loop_candidates(mv_ctx* ctx, int n_frames, int first_frame, int top_n, int n_words,
                             const int32_t* d_word, const int32_t* d_q_count, const int8_t* d_weight,
                             int min_gap, int k, int min_score, int32_t* d_cand, int32_t* d_score);

/* idf weights for mv_loop_candidates from the frames given:
 *   weight[w] = df ? rint(127 * ln(n_frames / df) / ln(n_frames)) : 0,   computed in double,
 * df = the number of the n_frames frames whose first min(q_count, top_n) words hold w.  The one exact tie,
 * df * df == n_frames (63.5), is decided in integers and weighs 64.  A word in every frame weighs
 * 0, a word in one frame 127.  n_frames in [2, 65535]; d_weight int8 [n_words] (device). */
mv_status mv_lcd_word_weights(mv_ctx* ctx, int n_frames, int top_n, int n_words, const int32_t* d_word,
                              const int32_t* d_q_count, int8_t* d_weight);

typedef struct {
  mv_match_params match;   /* default: shift 0 and a radius that covers the grid (a revisit's offset is unknown) */
  mv_pnp_params   pnp;     /* the sampler of candidate r of frame i is keyed on pnp.first_pair + i * k + r */
  int top_n;               /* queries per frame (words per frame) */
  int max_valid;           /* MAX_VALID_FEATURES analogue */
  int min_gap;             /* candidates of frame i are frames j <= i - min_gap (default 30) */
  int k;                   /* candidates verified per frame, 1..8 (default 4) */
  int min_score;           /* least BoW score of a candidate (default 1) */
  int min_inliers;         /* least PnP inliers of an accepted loop (default 30) */
} mv_loop_params;

void mv_loop_params_default(mv_loop_params* p, int rows, int cols);

/* One record per frame (64 bytes). */
typedef struct {
  int32_t frame;           /* the accepted earlier frame j (global number: first_frame + its index in the call), -1
                            * if none; with first_frame < 0 an accepted frame can be -1 too: test bow_rank */
  int32_t bow_score;       /* its score and its rank (0 = best) in the frame's candidate list; 0 / -1 if none, */
  int32_t bow_rank;        /* so bow_rank >= 0 exactly where a loop was accepted */
  int32_t num_matches;     /* matches of pair (f0 = j, f1 = i) */
  float pnp_inliers;       /* Gauss-Newton PnP inliers and cost of that pair */
  float pnp_cost;
  float q[4];              /* the pose that takes frame j's camera points into frame i's (w,x,y,z), the */
  float t[3];              /* convention of mv_pair_result with f0 = j and f1 = i; zero if none */
  int32_t status;          /* 0 ok; MV_ERR_TOO_MANY_VALID if frame i, or the accepted j, overflowed max_valid */
  int32_t pad[2];
} mv_loop_result;

/* Loop closures of n_frames device-resident frames (inputs as mv_track_sequence, plus mv_bow_assign_batch's desc
 * scales), in context scratch:
 *   1. the detector and top-N of every frame;  2. their words (the context's vocabulary, n_words of it);
 *   3. mv_loop_candidates(p->min_gap, p->k, p->min_score, d_weight) with first_frame 0, so that a slot's -1 is
 *      unambiguous (first_frame is added to the accepted frame's index in the record);
 *   4. ONE mv_match_batch launch over the pairs (f0 = j, f1 = i) of every candidate slot;
 *   5. mv_build_corr_batch from frame j's depth;  6. ONE mv_pnp_gn_batch launch, slot r of frame i being pair
 *      i * k + r (so the sampler key is pnp.first_pair + i * k + r whatever the candidates are);
 *   7. per frame the candidate with the most PnP inliers, the better BoW rank on equal inliers, accepted where it
 *      has at least min_inliers.
 * Slots without a candidate run as pairs (i, i) and their matches are discarded before step 5.  Each record equals
 * what those calls give when made one by one.  d_results mv_loop_result [n_frames].
 * MV_ERR_BAD_ARG with no kernel launched: what mv_track_sequence refuses (bar n_frames >= 2: one frame is
 * allowed), what mv_loop_candidates refuses, no vocabulary, n_frames * k > 65535 (one batched matcher / PnP call),
 * and a NULL d_desc_scale or d_results. */
mv_status mv_detect_loops(mv_ctx* ctx, const mv_loop_params* p, int n_frames, int first_frame,
                          const int8_t* d_semi, const float* d_semi_scale,
                          const int8_t* d_desc, const float* d_desc_scale, const float* d_depth,
                          const int8_t* d_weight, mv_loop_result* d_results);

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
