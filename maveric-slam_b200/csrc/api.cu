// api.cu -- the C ABI of libmaveric_b200.so: context management, the legacy
// reference-shaped symbols (include/maveric_slam_compat.h), the host-pointer `_ex`
// forms and the whole-path sequence calls (include/maveric_b200.h).
//
// There is no CPU implementation of the hot path in this library: every compute entry
// point needs a CUDA device and reports MV_ERR_NO_DEVICE (new API) or aborts with a
// message on stderr (legacy void symbols) when there is none.
#include "mv_common.cuh"
#include "sm100_ptx.cuh"
#include "svd3.cuh"

#include <math.h>
#include <stdlib.h>

#include <algorithm>
#include <mutex>

#include "../../include/maveric_slam_compat.h"

void mv_host_recover_pose(const float E[3][3], float R1[3][3], float R2[3][3], float t[3]);

// ------------------------------------------------------------------------------------
// context
// ------------------------------------------------------------------------------------
extern "C" const char* mv_status_str(mv_status s) {
  switch (s) {
    case MV_OK: return "ok";
    case MV_ERR_NO_DEVICE: return "no usable CUDA device (this library has no CPU fallback)";
    case MV_ERR_CUDA: return "CUDA error";
    case MV_ERR_BAD_ARG: return "bad argument";
    case MV_ERR_TOO_MANY_VALID: return "valid cells reached max_valid (top_N.c:91-94)";
  }
  return "unknown";
}

extern "C" mv_status mv_ctx_create(int device, mv_ctx** out) {
  if (!out) return MV_ERR_BAD_ARG;
  *out = nullptr;
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0 || device < 0 || device >= n) {
    cudaGetLastError();
    return MV_ERR_NO_DEVICE;
  }
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess || prop.major < 10) {
    cudaGetLastError();
    return MV_ERR_NO_DEVICE;  // kernels are sm_100a only
  }
  mv_device_guard guard(device);   // the caller's current device is restored on return
  int cur = -1;
  if (cudaGetDevice(&cur) != cudaSuccess || cur != device) { cudaGetLastError(); return MV_ERR_NO_DEVICE; }
  mv_ctx* c = new mv_ctx();
  c->device = device;
  c->sm_count = prop.multiProcessorCount;
  int prio_lo = 0, prio_hi = 0;
  cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
  // the staging stream (copies + detector + row gather) outranks the compute stream so its
  // short kernels slot in between the CTAs of a long-running PnP launch
  if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaStreamCreateWithPriority(&c->copy_stream, cudaStreamNonBlocking, prio_hi) != cudaSuccess ||
      cudaStreamCreateWithPriority(&c->gather_stream, cudaStreamNonBlocking, prio_hi) != cudaSuccess) {
    if (c->stream) cudaStreamDestroy(c->stream);
    if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
    if (c->gather_stream) cudaStreamDestroy(c->gather_stream);
    cudaGetLastError();
    delete c;
    return MV_ERR_CUDA;
  }
  *out = c;
  return MV_OK;
}

extern "C" void mv_ctx_destroy(mv_ctx* c) {
  if (!c) return;
  mv_device_guard guard(c->device);
  cudaStreamSynchronize(c->stream);
  cudaStreamSynchronize(c->copy_stream);
  cudaStreamSynchronize(c->gather_stream);
  for (auto& ev : c->pending) { cudaEventDestroy(ev.beg); cudaEventDestroy(ev.end); }
  for (auto& kv : c->scratch) cudaFree(kv.second.first);
  if (c->block_pool) cudaMemPoolDestroy(c->block_pool);
  if (c->pinned) cudaFreeHost(c->pinned);
  if (c->abort_host) cudaFreeHost(c->abort_host);
  if (c->own_stream) cudaStreamDestroy(c->stream);
  cudaStreamDestroy(c->copy_stream);
  cudaStreamDestroy(c->gather_stream);
  delete c;
}

extern "C" mv_status mv_ctx_set_stream(mv_ctx* c, void* s) {
  MV_ENTER(c);
  if (c->own_stream && c->stream) { cudaStreamSynchronize(c->stream); cudaStreamDestroy(c->stream); }
  c->stream = (cudaStream_t)s;
  c->own_stream = false;
  return MV_OK;
}

extern "C" mv_status mv_ctx_sync(mv_ctx* c) {
  MV_ENTER(c);
  MV_CUDA(c, cudaStreamSynchronize(c->stream));
  return MV_OK;
}

extern "C" const char* mv_last_error(mv_ctx* c) { return c ? c->err : "null context"; }
extern "C" unsigned long long mv_ctx_launch_count(mv_ctx* c) { return c ? c->launches : 0; }

extern "C" mv_status mv_ctx_profile(mv_ctx* c, int enable) {
  MV_ENTER(c);
  c->profile = enable != 0;
  for (auto& ev : c->pending) { cudaEventDestroy(ev.beg); cudaEventDestroy(ev.end); }
  c->pending.clear();
  c->prof.clear();
  return MV_OK;
}

extern "C" mv_status mv_ctx_profile_read(mv_ctx* c, const char* tag, double* avg_ms, int* launches) {
  if (!tag) return MV_ERR_BAD_ARG;
  MV_ENTER(c);
  MV_CUDA(c, cudaStreamSynchronize(c->stream));
  for (auto& ev : c->pending) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, ev.beg, ev.end) == cudaSuccess) {
      c->prof[ev.tag].ms += ms;
      c->prof[ev.tag].launches += 1;
    }
    cudaEventDestroy(ev.beg);
    cudaEventDestroy(ev.end);
  }
  c->pending.clear();
  auto it = c->prof.find(tag);
  if (avg_ms) *avg_ms = (it == c->prof.end() || it->second.launches == 0) ? 0.0 : it->second.ms / it->second.launches;
  if (launches) *launches = it == c->prof.end() ? 0 : it->second.launches;
  return MV_OK;
}

mv_status mv_scratch(mv_ctx* c, const char* name, size_t bytes, void** out) {
  auto& slot = c->scratch[name];
  if (slot.second < bytes) {
    if (slot.first) {
      MV_CUDA(c, cudaStreamSynchronize(c->stream));
      MV_CUDA(c, cudaFree(slot.first));
      slot.first = nullptr;
      slot.second = 0;
    }
    size_t want = bytes + bytes / 8 + 256;
    MV_CUDA(c, cudaMalloc(&slot.first, want));
    slot.second = want;
  }
  *out = slot.first;
  return MV_OK;
}

mv_status mv_block_alloc(mv_ctx* c, size_t bytes, void** out) {
  if (!c->block_pool) {
    cudaMemPoolProps props = {};
    props.allocType = cudaMemAllocationTypePinned;
    props.location.type = cudaMemLocationTypeDevice;
    props.location.id = c->device;
    MV_CUDA(c, cudaMemPoolCreate(&c->block_pool, &props));
    uint64_t keep = ~0ull;
    MV_CUDA(c, cudaMemPoolSetAttribute(c->block_pool, cudaMemPoolAttrReleaseThreshold, &keep));
  }
  MV_CUDA(c, cudaMallocFromPoolAsync(out, bytes, c->block_pool, c->stream));
  return MV_OK;
}

mv_status mv_abort_flag(mv_ctx* c, int** out) {
  if (!c->abort_host) {
    MV_CUDA(c, cudaHostAlloc((void**)&c->abort_host, 64, cudaHostAllocMapped | cudaHostAllocPortable));
    *c->abort_host = 0;
  }
  *out = c->abort_host;   // unified addressing: the same pointer is valid on the device
  return MV_OK;
}

mv_status mv_pinned(mv_ctx* c, size_t bytes, void** out) {
  if (c->pinned_bytes < bytes) {
    if (c->pinned) { MV_CUDA(c, cudaFreeHost(c->pinned)); c->pinned = nullptr; c->pinned_bytes = 0; }
    MV_CUDA(c, cudaMallocHost(&c->pinned, bytes + 4096));
    c->pinned_bytes = bytes + 4096;
  }
  *out = c->pinned;
  return MV_OK;
}

// process-global context behind the legacy void symbols
static std::mutex g_mu;
static mv_ctx* g_ctx = nullptr;

static mv_ctx* legacy_ctx() {
  if (!g_ctx) {
    mv_status st = mv_ctx_create(0, &g_ctx);
    if (st != MV_OK) {
      fprintf(stderr, "libmaveric_b200: %s\n", mv_status_str(st));
      abort();
    }
  }
  return g_ctx;
}

static void legacy_check(mv_ctx* c, mv_status st, const char* what) {
  if (st != MV_OK) {
    fprintf(stderr, "libmaveric_b200: %s failed: %s (%s)\n", what, mv_status_str(st), mv_last_error(c));
    abort();
  }
}

#define H2D(ctx, dst, src, bytes) MV_CUDA(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, (ctx)->stream))
#define D2H(ctx, dst, src, bytes) MV_CUDA(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, (ctx)->stream))

// ------------------------------------------------------------------------------------
// detector: host-pointer forms
// ------------------------------------------------------------------------------------
static mv_status detect_one(mv_ctx* c, float scale, const int8_t* h_semi, int cells, int32_t** d_idx,
                            float** d_prob, int32_t** d_nv) {
  void *ds, *dsc, *di, *dp, *dn;
  mv_status st;
  if ((st = mv_scratch(c, "ex.semi", (size_t)cells * 65 + 16, &ds))) return st;
  if ((st = mv_scratch(c, "ex.scale", 16, &dsc))) return st;
  if ((st = mv_scratch(c, "ex.idx", sizeof(int32_t) * cells, &di))) return st;
  if ((st = mv_scratch(c, "ex.prob", sizeof(float) * cells, &dp))) return st;
  if ((st = mv_scratch(c, "ex.nv", 16, &dn))) return st;
  H2D(c, ds, h_semi, (size_t)cells * 65);
  H2D(c, dsc, &scale, sizeof(float));
  if ((st = mv_softmax_batch(c, 1, cells, (const int8_t*)ds, (const float*)dsc, (int32_t*)di, (float*)dp,
                             (int32_t*)dn)))
    return st;
  *d_idx = (int32_t*)di; *d_prob = (float*)dp; *d_nv = (int32_t*)dn;
  return MV_OK;
}

extern "C" mv_status compute_softmax_ex(mv_ctx* c, float scale, const int8_t* h_semi, int cells,
                                        int* num_valid, int* max_indices, float* probs) {
  MV_ENTER(c);
  if (!h_semi || cells <= 0 || !max_indices || !probs) MV_BAD_ARG(c, "compute_softmax_ex");
  int32_t *di, *dn; float* dp;
  mv_status st = detect_one(c, scale, h_semi, cells, &di, &dp, &dn);
  if (st) return st;
  int nv = 0;
  D2H(c, max_indices, di, sizeof(int32_t) * cells);
  D2H(c, probs, dp, sizeof(float) * cells);
  D2H(c, &nv, dn, sizeof(int));
  MV_CUDA(c, cudaStreamSynchronize(c->stream));
  if (num_valid) *num_valid += nv;  // top_N.c:159: accumulates into the caller's counter
  return MV_OK;
}

extern "C" mv_status compute_top_N_ex(mv_ctx* c, float scale, const int8_t* h_semi, int cells, int N,
                                      int max_valid, int* num_selected, int* N_patches, int* N_indices,
                                      float* N_probs) {
  MV_ENTER(c);
  if (!h_semi || cells <= 0 || N <= 0 || max_valid <= 0 || !num_selected || !N_patches || !N_indices || !N_probs)
    MV_BAD_ARG(c, "compute_top_N_ex");
  int32_t *di, *dn; float* dp;
  mv_status st = detect_one(c, scale, h_semi, cells, &di, &dp, &dn);
  if (st) return st;
  void *qp, *qi, *qpr, *qc;
  if ((st = mv_scratch(c, "ex.qp", sizeof(int32_t) * N, &qp))) return st;
  if ((st = mv_scratch(c, "ex.qi", sizeof(int32_t) * N, &qi))) return st;
  if ((st = mv_scratch(c, "ex.qpr", sizeof(float) * N, &qpr))) return st;
  if ((st = mv_scratch(c, "ex.qc", 16, &qc))) return st;
  int32_t* ov = (int32_t*)qc + 1;
  if ((st = mv_top_n_batch(c, 1, cells, N, max_valid, di, dp, (int32_t*)qp, (int32_t*)qi, (float*)qpr,
                           (int32_t*)qc, ov)))
    return st;
  int meta[2] = {0, 0};
  D2H(c, meta, qc, sizeof(meta));
  MV_CUDA(c, cudaStreamSynchronize(c->stream));
  *num_selected = 0;
  if (meta[1]) return MV_ERR_TOO_MANY_VALID;
  *num_selected = meta[0];
  if (meta[0] > 0) {
    D2H(c, N_patches, qp, sizeof(int32_t) * meta[0]);
    D2H(c, N_indices, qi, sizeof(int32_t) * meta[0]);
    D2H(c, N_probs, qpr, sizeof(float) * meta[0]);
    MV_CUDA(c, cudaStreamSynchronize(c->stream));
  }
  return MV_OK;
}

// legacy shape: 1920 cells, 1000 valid (top_N.c:51,73,151)
extern "C" void compute_softmax(float scale, int8_t semi[2400][65], int* num_valid, int* max_indices,
                                float* probs) {
  std::lock_guard<std::mutex> lk(g_mu);
  mv_ctx* c = legacy_ctx();
  legacy_check(c, compute_softmax_ex(c, scale, &semi[0][0], 1920, num_valid, max_indices, probs),
               "compute_softmax");
}

extern "C" void compute_top_N(float scale, int8_t semi[2400][65], int N, int* num_selected, int* N_patches,
                              int* N_indices, float* N_probs) {
  std::lock_guard<std::mutex> lk(g_mu);
  mv_ctx* c = legacy_ctx();
  mv_status st = compute_top_N_ex(c, scale, &semi[0][0], 1920, N, 1000, num_selected, N_patches, N_indices,
                                  N_probs);
  if (st == MV_ERR_TOO_MANY_VALID) {  // top_N.c:91-94
    printf("Exceed max number of features!\n");
    exit(1);
  }
  legacy_check(c, st, "compute_top_N");
}

// ------------------------------------------------------------------------------------
// matcher: host-pointer form
// ------------------------------------------------------------------------------------
extern "C" mv_status mv_match_pair_host(mv_ctx* c, const mv_match_params* p, const int8_t* h_desc0,
                                        const int8_t* h_desc1, const int* max_indices0, const float* probs0,
                                        int num_queries, const int* patches1, const int* indices1,
                                        float* points1, float* points2, int* num_matches, int* cell0,
                                        float* score) {
  MV_ENTER(c);
  if (!p || !h_desc0 || !h_desc1 || !max_indices0 || !probs0 || num_queries < 0 || !points1 || !points2 ||
      !num_matches)
    MV_BAD_ARG(c, "mv_match_pair_host");
  if (p->rows <= 0 || p->cols <= 0 || p->max_matches <= 0)
    MV_BAD_ARG(c, "mv_match_pair_host: rows, cols and max_matches must be positive");
  const int cells = p->rows * p->cols;
  const int top_n = num_queries > 0 ? num_queries : 1;
  const int M = p->max_matches;
  void *dd, *di, *dp, *qp, *qi, *qc, *mp, *mc, *mcell, *msc;
  mv_status st;
  if ((st = mv_scratch(c, "mp.desc", (size_t)2 * cells * 256, &dd))) return st;
  if ((st = mv_scratch(c, "mp.idx", sizeof(int32_t) * 2 * cells, &di))) return st;
  if ((st = mv_scratch(c, "mp.prob", sizeof(float) * 2 * cells, &dp))) return st;
  if ((st = mv_scratch(c, "mp.qp", sizeof(int32_t) * 2 * top_n, &qp))) return st;
  if ((st = mv_scratch(c, "mp.qi", sizeof(int32_t) * 2 * top_n, &qi))) return st;
  if ((st = mv_scratch(c, "mp.qc", 16, &qc))) return st;
  if ((st = mv_scratch(c, "mp.pts", sizeof(float) * 4 * M, &mp))) return st;
  if ((st = mv_scratch(c, "mp.cnt", 16, &mc))) return st;
  if ((st = mv_scratch(c, "mp.cell", sizeof(int32_t) * M, &mcell))) return st;
  if ((st = mv_scratch(c, "mp.score", sizeof(float) * M, &msc))) return st;
  H2D(c, dd, h_desc0, (size_t)cells * 256);
  H2D(c, (int8_t*)dd + (size_t)cells * 256, h_desc1, (size_t)cells * 256);
  H2D(c, di, max_indices0, sizeof(int32_t) * cells);
  H2D(c, dp, probs0, sizeof(float) * cells);
  if (num_queries > 0) {
    H2D(c, (int32_t*)qp + top_n, patches1, sizeof(int32_t) * num_queries);
    H2D(c, (int32_t*)qi + top_n, indices1, sizeof(int32_t) * num_queries);
  }
  const int counts[2] = {0, num_queries};
  H2D(c, qc, counts, sizeof(counts));
  if ((st = mv_match_batch(c, p, 2, 1, top_n, nullptr, nullptr, (const int8_t*)dd, (const int32_t*)di,
                           (const float*)dp, (const int32_t*)qp, (const int32_t*)qi, (const int32_t*)qc,
                           (float*)mp, (int32_t*)mc, (int32_t*)mcell, nullptr, (float*)msc)))
    return st;
  int n = 0;
  D2H(c, &n, mc, sizeof(int));
  MV_CUDA(c, cudaStreamSynchronize(c->stream));
  *num_matches = n;
  if (n > 0) {
    void* hp;
    if ((st = mv_pinned(c, sizeof(float) * 4 * n, &hp))) return st;
    D2H(c, hp, mp, sizeof(float) * 4 * n);
    if (cell0) D2H(c, cell0, mcell, sizeof(int32_t) * n);
    if (score) D2H(c, score, msc, sizeof(float) * n);
    MV_CUDA(c, cudaStreamSynchronize(c->stream));
    const float* v = (const float*)hp;
    for (int i = 0; i < n; i++) {  // tracking_main.c:182-185: points1 = frame 0, points2 = frame 1
      points1[2 * i] = v[4 * i]; points1[2 * i + 1] = v[4 * i + 1];
      points2[2 * i] = v[4 * i + 2]; points2[2 * i + 1] = v[4 * i + 3];
    }
  }
  return MV_OK;
}

// ------------------------------------------------------------------------------------
// legacy pose symbols (pnp_solver.h)
// ------------------------------------------------------------------------------------
extern "C" void normalize_points(const int num_points, const float points[][2], const float K[3][3],
                                 float normalized_points[][2]) {
  for (int i = 0; i < num_points; ++i) {  // pnp_solver.c:28-34
    normalized_points[i][0] = mvsvd::fdiv(mvsvd::fsub(points[i][0], K[0][2]), K[0][0]);
    normalized_points[i][1] = mvsvd::fdiv(mvsvd::fsub(points[i][1], K[1][2]), K[1][1]);
  }
}

extern "C" void compute_essential_matrix(const int, const float[][2], const float[][2], float E[3][3]) {
  // pnp_solver.c:36-86: the 8-point system is built and ignored; the result is I.
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) E[i][j] = i == j ? 1.0f : 0.0f;
}

extern "C" float compute_reprojection_error(const float p1[2], const float p2[2], const float E[3][3]) {
  return mvsvd::reproj_error(p1[0], p1[1], p2[0], p2[1], E);
}

extern "C" void recover_pose_from_essential_matrix(float E[3][3], float R1[3][3], float R2[3][3], float t[3]) {
  mv_host_recover_pose(E, R1, R2, t);
}

extern "C" void ransac_essential_matrix(const int num_points, const float points1[][2],
                                        const float points2[][2], const float K[3][3],
                                        const int num_iterations, const float inlier_threshold,
                                        float best_E[3][3], int* best_inliers, int* num_inliers) {
  (void)K;
  std::lock_guard<std::mutex> lk(g_mu);
  mv_ctx* c = legacy_ctx();
  mv_device_guard guard(c->device);
  // Defined result where the reference has none (no match / no inlier, SURVEY App. B-5).
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) best_E[i][j] = i == j ? 1.0f : 0.0f;
  *num_inliers = 0;
  if (num_points <= 0) return;
  void *hp, *dp, *dc, *dn, *di;
  legacy_check(c, mv_pinned(c, sizeof(float) * 4 * num_points, &hp), "ransac");
  float* v = (float*)hp;
  for (int i = 0; i < num_points; i++) {
    v[4 * i] = points1[i][0]; v[4 * i + 1] = points1[i][1];
    v[4 * i + 2] = points2[i][0]; v[4 * i + 3] = points2[i][1];
  }
  legacy_check(c, mv_scratch(c, "rs.pts", sizeof(float) * 4 * num_points, &dp), "ransac");
  legacy_check(c, mv_scratch(c, "rs.cnt", 16, &dc), "ransac");
  legacy_check(c, mv_scratch(c, "rs.ninl", 16, &dn), "ransac");
  legacy_check(c, mv_scratch(c, "rs.inl", sizeof(int32_t) * num_points, &di), "ransac");
  auto run = [&]() -> mv_status {
    H2D(c, dp, hp, sizeof(float) * 4 * num_points);
    H2D(c, dc, &num_points, sizeof(int));
    mv_status st = mv_ransac_identity_batch(c, 1, num_points, (const float*)dp, (const int32_t*)dc,
                                            num_iterations, inlier_threshold, (int32_t*)dn, (int32_t*)di,
                                            nullptr);
    if (st) return st;
    int n = 0;
    D2H(c, &n, dn, sizeof(int));
    MV_CUDA(c, cudaStreamSynchronize(c->stream));
    *num_inliers = n;
    if (n > 0 && best_inliers) {
      D2H(c, best_inliers, di, sizeof(int32_t) * n);
      MV_CUDA(c, cudaStreamSynchronize(c->stream));
    }
    return MV_OK;
  };
  legacy_check(c, run(), "ransac_essential_matrix");
}

// ------------------------------------------------------------------------------------
// geometry PODs / projection factor (types.c, projection_factor.c): scalar helpers
// ------------------------------------------------------------------------------------
using mvsvd::fadd; using mvsvd::fmul; using mvsvd::fsub; using mvsvd::fdiv;

extern "C" Vector2f add_Vector2f(Vector2f a, Vector2f b, float s) {
  Vector2f v; v.x = fadd(a.x, fmul(s, b.x)); v.y = fadd(a.y, fmul(s, b.y)); return v;
}
extern "C" Vector3f add_Vector3f(Vector3f a, Vector3f b, float s) {
  Vector3f v; v.x = fadd(a.x, fmul(s, b.x)); v.y = fadd(a.y, fmul(s, b.y)); v.z = fadd(a.z, fmul(s, b.z)); return v;
}
extern "C" Quaternionf mult_Quaternionf(Quaternionf a, Quaternionf b) {
  Quaternionf q;  // types.c:18-25, left-to-right sums
  q.w = fsub(fsub(fsub(fmul(a.w, b.w), fmul(a.x, b.x)), fmul(a.y, b.y)), fmul(a.z, b.z));
  q.x = fsub(fadd(fadd(fmul(a.w, b.x), fmul(a.x, b.w)), fmul(a.y, b.z)), fmul(a.z, b.y));
  q.y = fadd(fadd(fsub(fmul(a.w, b.y), fmul(a.x, b.z)), fmul(a.y, b.w)), fmul(a.z, b.x));
  q.z = fadd(fsub(fadd(fmul(a.w, b.z), fmul(a.x, b.y)), fmul(a.y, b.x)), fmul(a.z, b.w));
  return q;
}
extern "C" Quaternionf create_Quaternionf(float w, float x, float y, float z) {
  Quaternionf q; q.w = w; q.x = x; q.y = y; q.z = z; return q;
}
extern "C" Quaternionf Quaternionf_from_Vector3f(Vector3f v) { return create_Quaternionf(0.0f, v.x, v.y, v.z); }
extern "C" Quaternionf conjugate_Quaternionf(Quaternionf q) { return create_Quaternionf(q.w, -q.x, -q.y, -q.z); }
extern "C" Vector3f Vector3f_from_Quaternionf(Quaternionf q) { Vector3f v; v.x = q.x; v.y = q.y; v.z = q.z; return v; }
extern "C" Vector3f apply_rotation(Quaternionf q, Vector3f v) {
  return Vector3f_from_Quaternionf(
      mult_Quaternionf(mult_Quaternionf(q, Quaternionf_from_Vector3f(v)), conjugate_Quaternionf(q)));
}
extern "C" Vector3f apply_transform(SE3 T, Vector3f v) { return add_Vector3f(apply_rotation(T.q, v), T.t, 1.0f); }

extern "C" ProjectionFactor* create_ProjectionFactor(Vector3f* landmark, SE3* pose, Vector2f measurement,
                                                     Camera camera) {
  ProjectionFactor* f = (ProjectionFactor*)malloc(sizeof(ProjectionFactor));  // caller frees
  f->landmark = landmark; f->pose = pose; f->measurement = measurement; f->camera = camera;
  return f;
}
extern "C" Vector2f project2d(const Vector3f p) { Vector2f r; r.x = fdiv(p.x, p.z); r.y = fdiv(p.y, p.z); return r; }
extern "C" Vector2f cam_project(const Vector3f p, const Camera cam) {
  Vector2f n = project2d(p), r;
  r.x = fadd(fmul(n.x, cam.fx), cam.cx);
  r.y = fadd(fmul(n.y, cam.fy), cam.cy);
  return r;
}
extern "C" void compute_error_ProjectionFactor(ProjectionFactor* f) {
  f->error = add_Vector2f(cam_project(apply_transform(*f->pose, *f->landmark), f->camera), f->measurement, -1.0f);
}

extern "C" void frame_create(const int rows, const int cols, const int channels, const char* data,
                             const int feature_rows, const int feature_cols, const float semi_scale,
                             const int8_t* semi, const float desc_scale, const int8_t* desc, Frame* frame) {
  frame->rows = rows; frame->cols = cols; frame->channels = channels; frame->data = data;
  frame->feature_rows = feature_rows; frame->feature_cols = feature_cols;
  frame->semi_scale = semi_scale; frame->semi = semi;
  frame->desc_scale = desc_scale; frame->desc = desc;
}

// ------------------------------------------------------------------------------------
// matmul shim (gemmini_functions_cpu.h): one thread per C element, k sequential, in the
// reference's operation order  c += ((sA*a)*sB)*b  (gemmini_functions_cpu.h:48,110)
// ------------------------------------------------------------------------------------
__global__ void matmul_shim_kernel(size_t I, size_t J, size_t K, const float* A, const float* B,
                                   const float* D, float* C, size_t a_i, size_t a_k, size_t b_k, size_t b_j,
                                   size_t sD, size_t sC, float as, float bs, float ds, int use_d) {
  const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= I * J) return;
  const size_t i = idx / J, j = idx % J;
  float c = use_d ? __fmul_rn(ds, D[i * sD + j]) : C[i * sC + j];
  for (size_t k = 0; k < K; k++)
    c = __fadd_rn(c, __fmul_rn(__fmul_rn(__fmul_rn(as, A[i * a_i + k * a_k]), bs), B[k * b_k + j * b_j]));
  C[i * sC + j] = c;
}

static mv_status matmul_host(mv_ctx* c, size_t I, size_t J, size_t K, const float* A, const float* B,
                             const float* D, float* C, size_t sA, size_t sB, size_t sD, size_t sC, float as,
                             float bs, float ds, bool tA, bool tB) {
  if (I == 0 || J == 0) return MV_OK;
  mv_device_guard guard(c->device);
  const size_t nA = K == 0 ? 0 : (tA ? (K - 1) * sA + I : (I - 1) * sA + K);
  const size_t nB = K == 0 ? 0 : (tB ? (J - 1) * sB + K : (K - 1) * sB + J);
  const size_t nC = (I - 1) * sC + J;
  const size_t nD = D ? (I - 1) * sD + J : 0;
  void *dA, *dB, *dC, *dD = nullptr;
  mv_status st;
  if ((st = mv_scratch(c, "mm.A", sizeof(float) * (nA + 1), &dA))) return st;
  if ((st = mv_scratch(c, "mm.B", sizeof(float) * (nB + 1), &dB))) return st;
  if ((st = mv_scratch(c, "mm.C", sizeof(float) * nC, &dC))) return st;
  if (nA) H2D(c, dA, A, sizeof(float) * nA);
  if (nB) H2D(c, dB, B, sizeof(float) * nB);
  H2D(c, dC, C, sizeof(float) * nC);
  if (D) {
    if (D == C && sD == sC) {
      dD = dC;  // in-place form used by local_bundle_adjustment.c:232-245
    } else {
      if ((st = mv_scratch(c, "mm.D", sizeof(float) * nD, &dD))) return st;
      H2D(c, dD, D, sizeof(float) * nD);
    }
  }
  const size_t total = I * J;
  matmul_shim_kernel<<<(unsigned)((total + 127) / 128), 128, 0, c->stream>>>(
      I, J, K, (const float*)dA, (const float*)dB, (const float*)dD, (float*)dC, tA ? 1 : sA, tA ? sA : 1,
      tB ? 1 : sB, tB ? sB : 1, sD, sC, as, bs, ds, D ? 1 : 0);
  MV_CHECK_LAUNCH(c);
  D2H(c, C, dC, sizeof(float) * nC);
  MV_CUDA(c, cudaStreamSynchronize(c->stream));
  return MV_OK;
}

extern "C" void matmul(size_t dim_I, size_t dim_J, size_t dim_K, const elem_t* A, const elem_t* B, elem_t* C,
                       size_t stride_A, size_t stride_B, size_t stride_C, scale_t A_scale_factor,
                       scale_t B_scale_factor, bool transpose_A, bool transpose_B) {
  std::lock_guard<std::mutex> lk(g_mu);
  mv_ctx* c = legacy_ctx();
  legacy_check(c, matmul_host(c, dim_I, dim_J, dim_K, A, B, nullptr, C, stride_A, stride_B, 0, stride_C,
                              A_scale_factor, B_scale_factor, 0.0f, transpose_A, transpose_B), "matmul");
}

extern "C" void matmul2(size_t dim_I, size_t dim_J, size_t dim_K, const elem_t* A, const elem_t* B,
                        const elem_t* D, elem_t* C, size_t stride_A, size_t stride_B, size_t stride_D,
                        size_t stride_C, scale_t A_scale_factor, scale_t B_scale_factor,
                        scale_t D_scale_factor, bool transpose_A, bool transpose_B) {
  std::lock_guard<std::mutex> lk(g_mu);
  mv_ctx* c = legacy_ctx();
  legacy_check(c, matmul_host(c, dim_I, dim_J, dim_K, A, B, D, C, stride_A, stride_B, stride_D, stride_C,
                              A_scale_factor, B_scale_factor, D_scale_factor, transpose_A, transpose_B),
               "matmul2");
}

// ------------------------------------------------------------------------------------
// whole path over a sequence
// ------------------------------------------------------------------------------------
extern "C" void mv_track_params_default(mv_track_params* p, int rows, int cols) {
  memset(p, 0, sizeof(*p));
  mv_match_params_default(&p->match, rows, cols);
  mv_pnp_params_default(&p->pnp);
  p->top_n = 100;            // tracking_main.c:14
  p->max_valid = 1000;       // top_N.c:51
  p->ransac_iterations = 10; // tracking_main.c:210
  p->ransac_threshold = 1.1f;
}

__global__ void pack_results_kernel(int n_pairs, const float* __restrict__ pose, const float* __restrict__ stats,
                                    const int32_t* __restrict__ match_count,
                                    const int32_t* __restrict__ ransac_inliers,
                                    const int32_t* __restrict__ overflow, mv_pair_result* __restrict__ out) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n_pairs) return;
  mv_pair_result r;
  for (int i = 0; i < 4; i++) r.q[i] = pose[(size_t)p * 7 + i];
  for (int i = 0; i < 3; i++) r.t[i] = pose[(size_t)p * 7 + 4 + i];
  r.pnp_inliers = stats[(size_t)p * 4 + 0];
  r.pnp_cost = stats[(size_t)p * 4 + 1];
  r.best_hypothesis = (int)stats[(size_t)p * 4 + 2];
  r.num_matches = match_count[p];
  r.ransac_inliers = ransac_inliers ? ransac_inliers[p] : 0;
  r.status = (overflow[p] || overflow[p + 1]) ? (int)MV_ERR_TOO_MANY_VALID : 0;
  r.pad[0] = r.pad[1] = r.pad[2] = 0;
  out[p] = r;
}

// Landmark mode of one batch of frames: the 3-D side of pair p's correspondences comes from the caller's table right
// after step p instead of depth.  Device pointers of that batch only.
struct SeqLandmarks {
  int first_frame;            // the table's frame number of the batch's frame 0
  int n_words;
  mv_landmark* table;         // NULL where the batch steps no table (a block's prepare and solve)
  const float* desc_scale;    // one per frame
  int32_t* n_with_landmark;   // one per pair, nullable
};

// Scratch of one in-flight batch of frames ("ns" = arena namespace, so two batches can be
// in flight in the double-buffered host path).
struct SeqScratch {
  int32_t *idx, *qp, *qi, *qc, *ov, *mc, *mcell, *rin;
  float *prob, *qpr, *mp, *corr, *pose, *stats;
  uint8_t* flags;
  int32_t* word;              // landmark mode: [n_frames - 1][top_n]
  float *coords_in, *coords_out;   // landmark mode: [n_frames - 1][top_n][3]
};

// "bad argument: fn: why", or "bad argument: fn" without a reason
static mv_status bad_arg(mv_ctx* c, const char* fn, const char* why) {
  snprintf(c->err, sizeof(c->err), "bad argument: %s%s%s", fn, why ? ": " : "", why ? why : "");
  return MV_ERR_BAD_ARG;
}

// Every refusal seq_detect and the parts of a batch could make from the arguments, so that a sequence call refuses
// before it allocates or enqueues anything.  n_frames: the largest batch the call runs (the whole sequence for the
// device-resident calls, the largest chunk for the host ones); d_desc: the caller's descriptors, or NULL when they
// are staged into scratch; landmarks: the batches assign words of an n_words vocabulary (the calls that step a table
// refuse a NULL one themselves).
static mv_status seq_check(mv_ctx* c, const char* fn, const mv_track_params* p, int n_frames, const int8_t* d_desc,
                           bool landmarks, int n_words = 0) {
  auto refuse = [&](const char* why) { return bad_arg(c, fn, why); };
  const mv_match_params& m = p->match;
  if (m.rows <= 0 || m.cols <= 0 || p->top_n <= 0 || p->max_valid <= 0 || m.max_matches <= 0 ||
      (long long)m.rows * m.cols > 0x7fffffffLL)
    return refuse("rows, cols, top_n, max_valid and max_matches must be positive");
  if (m.radius < 0) return refuse("match.radius must be >= 0");
  if (!mv_pnp_params_ok(&p->pnp, m.max_matches))
    return refuse("max_matches <= 65535, pnp.hypotheses in [1,65536], pnp.sample_size in [1,255], "
                  "pnp.lanes_per_hypothesis 1 or 32, pnp.min_depth >= FLT_MIN");
  if (n_frames > 65535)
    return refuse("at most 65535 frames per call (grid y dimension); mv_track_sequence_host chunks longer sequences");
  if (m.use_tensor_cores != 0 && m.use_tensor_cores != 2 && !mv_match_tc_feasible(&m, n_frames, n_frames - 1, p->top_n))
    return refuse("use_tensor_cores = 1 on a shape the tensor-core matcher does not take (2 picks the matcher)");
  if (d_desc && (reinterpret_cast<uintptr_t>(d_desc) & 15)) return refuse("d_desc must be 16-byte aligned");
  if (!landmarks) return MV_OK;
  if (c->bow_n_base <= 0) return refuse("no vocabulary (mv_bow_set_vocabulary first)");
  if (!mv_bow_vocab_fits(c)) return refuse("vocabulary larger than an SM's shared memory");
  if (n_words <= 0) return refuse("n_words must be positive");
  if ((long long)(n_frames - 1) * p->top_n > 0x7fffffffLL) return refuse("(n_frames - 1) * top_n must be below 2^31");
  return MV_OK;
}

// own: allocate on the compute stream into this list instead of the context's arena (a block's scratch).
// planes = false leaves out the per-frame detector planes (idx, prob, qi, qpr, flags), which only the detector, the
// row marking and the matcher read: a block prepared from host buffers keeps them in the staging chunks.
static mv_status seq_scratch(mv_ctx* c, const mv_track_params* p, int n_frames, const char* ns, bool landmarks,
                             SeqScratch* o, std::vector<void*>* own = nullptr, bool planes = true) {
  const int cells = p->match.rows * p->match.cols;
  const int n_pairs = n_frames - 1;
  const int N = p->top_n, M = p->match.max_matches;
  std::string s(ns);
  mv_status st;
  void* v;
#define SCR(field, type, name, bytes)                                        \
  if (own) {                                                                 \
    if ((st = mv_block_alloc(c, (bytes), &v))) return st;                   \
    own->push_back(v);                                                       \
  } else if ((st = mv_scratch(c, (s + name).c_str(), (bytes), &v))) {        \
    return st;                                                               \
  }                                                                          \
  o->field = (type*)v
  if (planes) {
    SCR(idx, int32_t, ".idx", sizeof(int32_t) * (size_t)n_frames * cells);
    SCR(prob, float, ".prob", sizeof(float) * (size_t)n_frames * cells);
  }
  SCR(qp, int32_t, ".qp", sizeof(int32_t) * (size_t)n_frames * N);
  if (planes) {
    SCR(qi, int32_t, ".qi", sizeof(int32_t) * (size_t)n_frames * N);
    SCR(qpr, float, ".qpr", sizeof(float) * (size_t)n_frames * N);
  }
  SCR(qc, int32_t, ".qc", sizeof(int32_t) * (size_t)n_frames);
  SCR(ov, int32_t, ".ov", sizeof(int32_t) * (size_t)n_frames);
  if (planes) {
    SCR(flags, uint8_t, ".flags", (size_t)n_frames * cells + 64);
  }
  SCR(mp, float, ".mp", sizeof(float) * 4 * (size_t)n_pairs * M);
  SCR(mc, int32_t, ".mc", sizeof(int32_t) * (size_t)n_pairs);
  SCR(mcell, int32_t, ".mcell", sizeof(int32_t) * (size_t)n_pairs * M);
  SCR(rin, int32_t, ".rin", sizeof(int32_t) * (size_t)n_pairs);
  SCR(corr, float, ".corr", sizeof(float) * 5 * (size_t)n_pairs * M);
  SCR(pose, float, ".pose", sizeof(float) * 7 * (size_t)n_pairs);
  SCR(stats, float, ".stats", sizeof(float) * 4 * (size_t)n_pairs);
  if (landmarks) {
    SCR(word, int32_t, ".word", sizeof(int32_t) * (size_t)n_pairs * N);
    SCR(coords_in, float, ".coords_in", sizeof(float) * 3 * (size_t)n_pairs * N);
    SCR(coords_out, float, ".coords_out", sizeof(float) * 3 * (size_t)n_pairs * N);
  }
#undef SCR
  return MV_OK;
}

// Detector half: needs only the logits.
static mv_status seq_detect(mv_ctx* c, const mv_track_params* p, int n_frames, const int8_t* d_semi,
                            const float* d_semi_scale, const SeqScratch& w) {
  const int cells = p->match.rows * p->match.cols;
  mv_status st;
  if ((st = mv_softmax_batch(c, n_frames, cells, d_semi, d_semi_scale, w.idx, w.prob, nullptr))) return st;
  return mv_top_n_batch(c, n_frames, cells, p->top_n, p->max_valid, w.idx, w.prob, w.qp, w.qi, w.qpr, w.qc, w.ov);
}

// The rest of a batch whose detector has run, in the parts seq_step chains; the host pipeline and the landmark block
// call them apart.  seq_words: the word assignment of frames 0..n_word_frames-1 (all but the last of a batch; every
// frame of a warm-up chunk) with their query keypoints back-projected in the same launch (none where w.coords_in is
// NULL).
static mv_status seq_words(mv_ctx* c, const mv_track_params* p, int n_word_frames, const int8_t* d_desc,
                           const float* d_depth, const SeqScratch& w, const SeqLandmarks* lm) {
  MvBackProject bp;
  bp.q_idx = w.qi; bp.depth = d_depth; bp.rows = p->match.rows;
  bp.fx = p->pnp.fx; bp.fy = p->pnp.fy; bp.cx = p->pnp.cx; bp.cy = p->pnp.cy;
  bp.coords = w.coords_in;
  return mv_bow_assign_impl(c, n_word_frames, p->match.rows * p->match.cols, p->top_n, d_desc, lm->desc_scale, w.qp,
                            w.qc, w.word, nullptr, bp);
}

static mv_status seq_match(mv_ctx* c, const mv_track_params* p, int n_frames, const int8_t* d_desc,
                           const SeqScratch& w) {
  return mv_match_batch(c, &p->match, n_frames, n_frames - 1, p->top_n, nullptr, nullptr, d_desc, w.idx, w.prob, w.qp,
                        w.qi, w.qc, w.mp, w.mc, w.mcell, nullptr, nullptr);
}

static mv_status seq_ransac(mv_ctx* c, const mv_track_params* p, int n_frames, const SeqScratch& w) {
  if (p->ransac_iterations <= 0) return MV_OK;
  return mv_ransac_identity_batch(c, n_frames - 1, p->match.max_matches, w.mp, w.mc, p->ransac_iterations,
                                  p->ransac_threshold, w.rin, nullptr, nullptr);
}

// Correspondences: with `lm` from w.coords_out, each query's record right after its frame's step; else from depth.
static mv_status seq_corr(mv_ctx* c, const mv_track_params* p, int n_frames, const float* d_depth,
                          const SeqScratch& w, const SeqLandmarks* lm) {
  const int n_pairs = n_frames - 1, M = p->match.max_matches;
  if (lm)
    return mv_build_corr_landmarks_seq(c, n_pairs, p->top_n, M, lm->n_words, w.qp, w.qc, w.word, w.coords_out, w.mp,
                                       w.mc, w.mcell, w.corr, lm->n_with_landmark);
  return mv_build_corr_batch(c, n_pairs, p->match.rows * p->match.cols, p->match.rows, M, nullptr, d_depth, p->pnp.fx,
                             p->pnp.fy, p->pnp.cx, p->pnp.cy, w.mp, w.mc, w.mcell, w.corr);
}

// K3 and the records; first_pair: the batch's first pair in the call (the PnP sampler is keyed on it);
// max_ctas_per_sm: K3's residency cap (0: none).
static mv_status seq_pose(mv_ctx* c, const mv_track_params* p, int n_frames, const SeqScratch& w,
                          mv_pair_result* d_results, int first_pair, int max_ctas_per_sm) {
  const int n_pairs = n_frames - 1;
  mv_pnp_params pnp = p->pnp;
  pnp.first_pair += first_pair;
  mv_status st;
  if ((st = mv_pnp_gn_batch_impl(c, &pnp, n_pairs, p->match.max_matches, w.corr, w.mc, nullptr, w.pose, w.stats,
                                 nullptr, max_ctas_per_sm)))
    return st;
  pack_results_kernel<<<(n_pairs + 127) / 128, 128, 0, c->stream>>>(
      n_pairs, w.pose, w.stats, w.mc, p->ransac_iterations > 0 ? w.rin : nullptr, w.ov, d_results);
  MV_CHECK_LAUNCH(c);
  return MV_OK;
}

// The whole rest of a batch: with `lm` the words, then the table walked over frames 0..n-2 from lm->first_frame;
// then match / RANSAC-E / correspondences / K3 / pack.  Only descriptor rows of candidate / query cells are read,
// and depth only at matched frame-0 cells (or, with `lm`, at query cells).
static mv_status seq_step(mv_ctx* c, const mv_track_params* p, int n_frames, const int8_t* d_desc,
                          const float* d_depth, const SeqScratch& w, mv_pair_result* d_results,
                          const SeqLandmarks* lm) {
  mv_status st;
  if (lm && ((st = seq_words(c, p, n_frames - 1, d_desc, d_depth, w, lm)) ||
             (st = mv_landmarks_sequence_impl(c, lm->n_words, lm->table, lm->first_frame, n_frames - 1, p->top_n,
                                              w.word, w.qc, w.coords_in, w.coords_out))))
    return st;
  if ((st = seq_match(c, p, n_frames, d_desc, w)) || (st = seq_ransac(c, p, n_frames, w)) ||
      (st = seq_corr(c, p, n_frames, d_depth, w, lm)))
    return st;
  return seq_pose(c, p, n_frames, w, d_results, 0, 0);
}

extern "C" mv_status mv_track_sequence(mv_ctx* c, const mv_track_params* p, int n_frames, const int8_t* d_semi,
                                       const float* d_semi_scale, const int8_t* d_desc, const float* d_depth,
                                       mv_pair_result* d_results) {
  MV_ENTER(c);
  if (!p || n_frames < 2 || !d_semi || !d_semi_scale || !d_desc || !d_depth || !d_results)
    MV_BAD_ARG(c, "mv_track_sequence");
  SeqScratch w;
  mv_status st;
  if ((st = seq_check(c, "mv_track_sequence", p, n_frames, d_desc, false)) ||
      (st = seq_scratch(c, p, n_frames, "seq", false, &w)) || (st = seq_detect(c, p, n_frames, d_semi, d_semi_scale, w)))
    return st;
  return seq_step(c, p, n_frames, d_desc, d_depth, w, d_results, nullptr);
}

// Pair p = frames (p, p+1) with the 3-D side from the landmark table right after step p: detector, then seq_step in
// landmark mode over the whole sequence.
extern "C" mv_status mv_track_sequence_landmarks(mv_ctx* c, const mv_track_params* p, int n_frames, int first_frame,
                                                 const int8_t* d_semi, const float* d_semi_scale, const int8_t* d_desc,
                                                 const float* d_desc_scale, const float* d_depth, int n_words,
                                                 mv_landmark* d_table, mv_pair_result* d_results,
                                                 int32_t* d_n_with_landmark) {
  MV_ENTER(c);
  if (!p || n_frames < 2 || !d_semi || !d_semi_scale || !d_desc || !d_desc_scale || !d_depth || !d_results)
    MV_BAD_ARG(c, "mv_track_sequence_landmarks");
  const SeqLandmarks lm = {first_frame, n_words, d_table, d_desc_scale, d_n_with_landmark};
  SeqScratch w;
  mv_status st;
  if ((st = seq_check(c, "mv_track_sequence_landmarks", p, n_frames, d_desc, true, n_words))) return st;
  if (!d_table) MV_BAD_ARG(c, "mv_track_sequence_landmarks: NULL landmark table");
  if ((st = seq_scratch(c, p, n_frames, "lmseq", true, &w)) || (st = seq_detect(c, p, n_frames, d_semi, d_semi_scale, w)))
    return st;
  return seq_step(c, p, n_frames, d_desc, d_depth, w, d_results, &lm);
}

// ------------------------------------------------------------------------------------
// loop closure: BoW candidates (lcd.cu), then one matcher launch, depth correspondences and one K3 launch over
// every candidate slot
// ------------------------------------------------------------------------------------
extern "C" void mv_loop_params_default(mv_loop_params* p, int rows, int cols) {
  memset(p, 0, sizeof(*p));
  mv_match_params_default(&p->match, rows, cols);
  p->match.shift_x = p->match.shift_y = 0;   // a revisit's offset is unknown: search the whole grid
  p->match.radius = std::max(rows, cols);
  mv_pnp_params_default(&p->pnp);
  p->top_n = 100;
  p->max_valid = 1000;
  p->min_gap = 30;
  p->k = 4;
  p->min_score = 1;
  p->min_inliers = 30;
}

// The candidate stage of mv_detect_loops runs with first_frame 0: cand holds indices within the call, so -1 marks an
// empty slot whatever the caller's first_frame (a global frame number may itself be -1).
// slot s = i * k + r: pair (f0 = j, f1 = i) of candidate r of frame i, or (i, i) where the slot has no candidate
__global__ void loop_pairs_kernel(int n_slots, int k, const int32_t* __restrict__ cand, int32_t* __restrict__ f0,
                                  int32_t* __restrict__ f1) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_slots) return;
  const int i = s / k, c = cand[s];
  f0[s] = c >= 0 ? c : i;
  f1[s] = i;
}

// the matches of slots without a candidate are dropped before the correspondences
__global__ void loop_drop_empty_kernel(int n_slots, const int32_t* __restrict__ cand, int32_t* __restrict__ match_count) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s < n_slots && cand[s] < 0) match_count[s] = 0;
}

// per frame: the candidate with the most PnP inliers (the earlier slot, i.e. the better BoW rank, on equal inliers),
// accepted where it has at least min_inliers
__global__ void loop_select_kernel(int n_frames, int k, int first_frame, int min_inliers, const int32_t* __restrict__ cand,
                                   const int32_t* __restrict__ score, const int32_t* __restrict__ match_count,
                                   const float* __restrict__ pose, const float* __restrict__ stats,
                                   const int32_t* __restrict__ overflow, mv_loop_result* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_frames) return;
  int best = -1;
  float best_inl = 0.0f;
  for (int r = 0; r < k; r++) {
    const size_t s = (size_t)i * k + r;
    if (cand[s] < 0) continue;
    const float inl = stats[s * 4];
    if (best < 0 || inl > best_inl) { best = r; best_inl = inl; }
  }
  mv_loop_result res;
  memset(&res, 0, sizeof(res));
  res.frame = -1;
  res.bow_rank = -1;
  if (best >= 0 && best_inl >= (float)min_inliers) {
    const size_t s = (size_t)i * k + best;
    res.frame = first_frame + cand[s];
    res.bow_score = score[s];
    res.bow_rank = best;
    res.num_matches = match_count[s];
    res.pnp_inliers = stats[s * 4];
    res.pnp_cost = stats[s * 4 + 1];
    for (int c = 0; c < 4; c++) res.q[c] = pose[s * 7 + c];
    for (int c = 0; c < 3; c++) res.t[c] = pose[s * 7 + 4 + c];
  }
  res.status = (overflow[i] || (res.bow_rank >= 0 && overflow[res.frame - first_frame])) ? (int)MV_ERR_TOO_MANY_VALID : 0;
  out[i] = res;
}

extern "C" mv_status mv_detect_loops(mv_ctx* c, const mv_loop_params* p, int n_frames, int first_frame,
                                     const int8_t* d_semi, const float* d_semi_scale, const int8_t* d_desc,
                                     const float* d_desc_scale, const float* d_depth, const int8_t* d_weight,
                                     mv_loop_result* d_results) {
  MV_ENTER(c);
  const char* fn = "mv_detect_loops";
  if (!p || n_frames < 1 || !d_semi || !d_semi_scale || !d_desc || !d_desc_scale || !d_depth || !d_results)
    MV_BAD_ARG(c, "mv_detect_loops");
  // the detector, matcher and K3 refusals of the sequence calls; the matcher's tensor-core shape is checked below
  // for the call's real pair count
  mv_track_params tp;
  memset(&tp, 0, sizeof(tp));
  tp.match = p->match;
  tp.match.use_tensor_cores = 2;
  tp.pnp = p->pnp;
  tp.top_n = p->top_n;
  tp.max_valid = p->max_valid;
  const int n_words = c->bow_n_base * c->bow_wpb;
  mv_status st;
  if ((st = seq_check(c, fn, &tp, n_frames, d_desc, true, n_words))) return st;
  if (p->k < 1 || p->k > 8 || (long long)n_frames * p->k > 65535)
    return bad_arg(c, fn, "k in [1, 8] and n_frames * k <= 65535 (one batched matcher and PnP call)");
  const int n = n_frames, K = p->k, n_slots = n * K, N = p->top_n, M = p->match.max_matches;
  if (p->match.use_tensor_cores != 0 && p->match.use_tensor_cores != 2 && !mv_match_tc_feasible(&p->match, n, n_slots, N))
    return bad_arg(c, fn, "use_tensor_cores = 1 on a shape the tensor-core matcher does not take (2 picks the matcher)");
  if ((st = mv_loop_candidates_check(c, fn, n, first_frame, N, n_words, d_weight, p->min_gap, K))) return st;

  const int cells = p->match.rows * p->match.cols;
  SeqScratch w;
  memset(&w, 0, sizeof(w));
  int32_t *word, *cand, *score, *f0, *f1;
  void* v;
#define SCR(ptr, type, name, bytes)                                   \
  if ((st = mv_scratch(c, "loop." name, (bytes), &v))) return st;     \
  ptr = (type*)v
  SCR(w.idx, int32_t, "idx", sizeof(int32_t) * (size_t)n * cells);
  SCR(w.prob, float, "prob", sizeof(float) * (size_t)n * cells);
  SCR(w.qp, int32_t, "qp", sizeof(int32_t) * (size_t)n * N);
  SCR(w.qi, int32_t, "qi", sizeof(int32_t) * (size_t)n * N);
  SCR(w.qpr, float, "qpr", sizeof(float) * (size_t)n * N);
  SCR(w.qc, int32_t, "qc", sizeof(int32_t) * (size_t)n);
  SCR(w.ov, int32_t, "ov", sizeof(int32_t) * (size_t)n);
  SCR(word, int32_t, "word", sizeof(int32_t) * (size_t)n * N);
  SCR(cand, int32_t, "cand", sizeof(int32_t) * (size_t)n_slots);
  SCR(score, int32_t, "score", sizeof(int32_t) * (size_t)n_slots);
  SCR(f0, int32_t, "f0", sizeof(int32_t) * (size_t)n_slots);
  SCR(f1, int32_t, "f1", sizeof(int32_t) * (size_t)n_slots);
  SCR(w.mp, float, "mp", sizeof(float) * 4 * (size_t)n_slots * M);
  SCR(w.mc, int32_t, "mc", sizeof(int32_t) * (size_t)n_slots);
  SCR(w.mcell, int32_t, "mcell", sizeof(int32_t) * (size_t)n_slots * M);
  SCR(w.corr, float, "corr", sizeof(float) * 5 * (size_t)n_slots * M);
  SCR(w.pose, float, "pose", sizeof(float) * 7 * (size_t)n_slots);
  SCR(w.stats, float, "stats", sizeof(float) * 4 * (size_t)n_slots);
#undef SCR

  if ((st = seq_detect(c, &tp, n, d_semi, d_semi_scale, w)) ||
      (st = mv_bow_assign_impl(c, n, cells, N, d_desc, d_desc_scale, w.qp, w.qc, word, nullptr, MvBackProject())) ||
      (st = mv_loop_candidates_impl(c, n, 0, N, n_words, word, w.qc, d_weight, p->min_gap, K, p->min_score,
                                    cand, score)))
    return st;
  const unsigned slot_blocks = (unsigned)((n_slots + 255) / 256);
  loop_pairs_kernel<<<slot_blocks, 256, 0, c->stream>>>(n_slots, K, cand, f0, f1);
  MV_CHECK_LAUNCH(c);
  if ((st = mv_match_batch(c, &p->match, n, n_slots, N, f0, f1, d_desc, w.idx, w.prob, w.qp, w.qi, w.qc, w.mp, w.mc,
                           w.mcell, nullptr, nullptr)))
    return st;
  loop_drop_empty_kernel<<<slot_blocks, 256, 0, c->stream>>>(n_slots, cand, w.mc);
  MV_CHECK_LAUNCH(c);
  if ((st = mv_build_corr_batch(c, n_slots, cells, p->match.rows, M, f0, d_depth, p->pnp.fx, p->pnp.fy, p->pnp.cx,
                                p->pnp.cy, w.mp, w.mc, w.mcell, w.corr)) ||
      (st = mv_pnp_gn_batch(c, &p->pnp, n_slots, M, w.corr, w.mc, nullptr, w.pose, w.stats, nullptr)))
    return st;
  loop_select_kernel<<<(n + 127) / 128, 128, 0, c->stream>>>(n, K, first_frame, p->min_inliers, cand, score, w.mc,
                                                             w.pose, w.stats, w.ov, d_results);
  MV_CHECK_LAUNCH(c);
  return MV_OK;
}

// ---- chunks of the host staging pipeline (track_sequence_host_impl below)
// A call's host frames in chunks of `pairs` pairs: first the n_warm warm-up frames of a block being prepared, at most
// `pairs` frames per chunk and no halo, then the n_pairs pairs, each chunk sharing its first frame with the last
// frame of the chunk before.
struct HostPlan {
  int pairs, n_warm_chunks, n_chunks, n_warm, n_pairs;
  bool warm(int k) const { return k < n_warm_chunks; }                                // words only, no matcher
  int first_pair(int k) const { return (k - n_warm_chunks) * pairs; }                 // of a pairs' chunk
  int frame0(int k) const { return warm(k) ? k * pairs : n_warm + first_pair(k); }   // in the host buffers
  int frames(int k) const {
    return warm(k) ? std::min(pairs, n_warm - k * pairs) : std::min(pairs, n_pairs - first_pair(k)) + 1;
  }
};

// K3's CTAs per SM while the pipeline stages: the PnP kernel (37 KB of shared memory per CTA) would otherwise fill an
// SM's shared memory with 6 CTAs and starve the one-warp row-gather kernel (17 KB) that must run beside it.
constexpr int kStagingPnpCtasPerSm = 5;

static HostPlan host_plan(const mv_ctx* c, const mv_track_params* p, int n_warm, int n_pairs, bool landmarks) {
  // chunk = two full waves of the PnP kernel at its staging residency
  const int pnp_ctas_per_pair = mv_pnp_ctas_per_pair(&p->pnp);
  int chunk_pairs = 2 * (kStagingPnpCtasPerSm * c->sm_count) / (pnp_ctas_per_pair > 0 ? pnp_ctas_per_pair : 1);
  if (chunk_pairs < 8) chunk_pairs = 8;
  // short sequences (a rank's shard of a multi-GPU run): at least ~8 chunks, so that the staging
  // pipeline has something to overlap with instead of one long fill and drain
  if (chunk_pairs > (n_pairs + 7) / 8) chunk_pairs = (n_pairs + 7) / 8 > 32 ? (n_pairs + 7) / 8 : 32;
  if (const char* e = getenv("MV_HOST_CHUNK_PAIRS")) {  // test hook: force small chunks
    const int v = atoi(e);
    if (v > 0) chunk_pairs = v;
  }
  if (chunk_pairs > n_pairs) chunk_pairs = n_pairs;
  if (landmarks) {  // one table step per pair: mv_landmarks_sequence's limits on one call (top_n > 0 is checked)
    const int most = (int)std::min<long long>(65535, 0x7fffffffLL / std::max(p->top_n, 1));
    if (chunk_pairs > most) chunk_pairs = most;
  }
  const int n_warm_chunks = (n_warm + chunk_pairs - 1) / chunk_pairs;
  return {chunk_pairs, n_warm_chunks, n_warm_chunks + (n_pairs + chunk_pairs - 1) / chunk_pairs, n_warm, n_pairs};
}

// ---- the landmark path split at the table (mv_track_landmarks_prepare / step_table / solve)
// A block owns a SeqScratch over its n_warm + n_frames frames and a speculation; `b` is the view of the scratch
// that starts at the block's first frame, the scratch seq_step would have had for the block alone.
struct mv_lm_block {
  mv_ctx* ctx;
  mv_track_params p;
  int n_warm, n_frames, n_words;
  int first_frame;   // the table's frame number of the block's first frame (after the warm-up)
  SeqScratch w, b;
  std::vector<void*> mem;
  mv_lm_spec* spec = nullptr;
  int phase = 0;   // 1 prepared, 2 table stepped, 3 solved
};

static void lm_block_free(mv_lm_block* k) {
  mv_device_guard guard(k->ctx->device);
  mv_lm_spec_free(k->spec);
  for (void* v : k->mem) cudaFreeAsync(v, k->ctx->stream);
  delete k;
}

// Both prepare forms: checks the arguments (inputs: every input pointer is non-NULL), then allocates the block and
// its scratch.  `plan`, the host form only: filled with the staging plan, whose chunks are checked too; that form
// leaves the detector planes in the chunk buffers.  seq_check's tensor-core check over all n_warm + n_frames frames
// also covers the matcher's n_frames: mv_match_tc_feasible only takes fewer shapes as the frames grow.
static mv_status lm_block_new(mv_ctx* c, const char* fn, const mv_track_params* p, int n_warm, int n_frames,
                              int first_frame, int n_words, bool inputs, const int8_t* d_desc, HostPlan* plan,
                              mv_lm_block** out, mv_lm_block** block) {
  if (!out) return bad_arg(c, fn, "NULL out");
  *out = nullptr;
  if (!p || n_frames < 2 || n_warm < 0 || !inputs) return bad_arg(c, fn, nullptr);
  if ((long long)n_warm + n_frames > 65535) return bad_arg(c, fn, "at most 65535 frames in all");
  const int T = n_warm + n_frames;
  mv_status st;
  if ((st = seq_check(c, fn, p, T, d_desc, true, n_words))) return st;
  if (plan) {
    *plan = host_plan(c, p, n_warm, n_frames - 1, true);
    if ((st = seq_check(c, fn, p, plan->pairs + 1, nullptr, true, n_words))) return st;
  }
  mv_lm_block* k = new mv_lm_block{c, *p, n_warm, n_frames, n_words, first_frame};
  if ((st = seq_scratch(c, p, T, "", true, &k->w, &k->mem, !plan))) {
    lm_block_free(k);
    return st;
  }
  // k->b = the view of k->w at the block's first frame (coords_out aside: the speculation's)
  const size_t W = n_warm, N = p->top_n, cells = (size_t)p->match.rows * p->match.cols;
  SeqScratch& b = k->b = k->w;
  if (b.idx) {
    b.idx += W * cells; b.prob += W * cells;
    b.qi += W * N; b.qpr += W * N;
  }
  b.qp += W * N; b.qc += W; b.ov += W;
  b.word += W * N; b.coords_in += 3 * W * N;
  *block = k;
  return MV_OK;
}

extern "C" mv_status mv_track_landmarks_prepare(mv_ctx* c, const mv_track_params* p, int n_warm, int n_frames,
                                                int first_frame, const int8_t* d_semi, const float* d_semi_scale,
                                                const int8_t* d_desc, const float* d_desc_scale, const float* d_depth,
                                                int n_words, mv_lm_block** out) {
  MV_ENTER(c);
  mv_lm_block* k;
  mv_status st = lm_block_new(c, "mv_track_landmarks_prepare", p, n_warm, n_frames, first_frame, n_words,
                              d_semi && d_semi_scale && d_desc && d_desc_scale && d_depth, d_desc, nullptr, out, &k);
  if (st) return st;
  const int T = n_warm + n_frames;
  const SeqLandmarks lm = {first_frame - n_warm, n_words, nullptr, d_desc_scale, nullptr};
  const int8_t* b_desc = d_desc + (size_t)n_warm * p->match.rows * p->match.cols * 256;
  if ((st = seq_detect(c, p, T, d_semi, d_semi_scale, k->w)) || (st = seq_words(c, p, T - 1, d_desc, d_depth, k->w, &lm)) ||
      (st = mv_landmarks_speculate_impl(c, n_words, first_frame, n_warm, n_frames - 1, p->top_n, k->w.word, k->w.qc,
                                        k->b.coords_in, &k->spec)) ||
      (st = seq_match(c, p, n_frames, b_desc, k->b)) || (st = seq_ransac(c, p, n_frames, k->b))) {
    lm_block_free(k);
    return st;
  }
  k->b.coords_out = mv_lm_spec_coords(k->spec);   // the matcher and RANSAC-E do not read it
  k->phase = 1;
  *out = k;
  return MV_OK;
}

static mv_status lm_block_check(mv_ctx* c, mv_lm_block* k, int phase, const char* fn) {
  if (!k) return bad_arg(c, fn, "NULL block");
  if (k->ctx != c) return bad_arg(c, fn, "block of another context");
  if (k->phase != phase) return bad_arg(c, fn, "out of phase (prepare, step_table, solve, each once)");
  return MV_OK;
}

extern "C" mv_status mv_track_landmarks_step_table(mv_ctx* c, mv_lm_block* k, mv_landmark* d_table,
                                                   int32_t* d_n_rewalked) {
  MV_ENTER(c);
  mv_status st;
  if ((st = lm_block_check(c, k, 1, "mv_track_landmarks_step_table"))) return st;
  if (!d_table) MV_BAD_ARG(c, "mv_track_landmarks_step_table: NULL landmark table");
  k->phase = 2;
  return mv_landmarks_resolve_impl(c, k->spec, d_table, k->b.coords_out, d_n_rewalked);
}

extern "C" mv_status mv_track_landmarks_solve(mv_ctx* c, mv_lm_block* k, mv_pair_result* d_results,
                                              int32_t* d_n_with_landmark) {
  MV_ENTER(c);
  mv_status st;
  if ((st = lm_block_check(c, k, 2, "mv_track_landmarks_solve"))) return st;
  if (!d_results) MV_BAD_ARG(c, "mv_track_landmarks_solve: NULL results");
  k->phase = 3;
  const SeqLandmarks lm = {k->first_frame, k->n_words, nullptr, nullptr, d_n_with_landmark};
  if ((st = seq_corr(c, &k->p, k->n_frames, nullptr, k->b, &lm))) return st;
  return seq_pose(c, &k->p, k->n_frames, k->b, d_results, 0, 0);
}

extern "C" void mv_track_landmarks_release(mv_lm_block* k) {
  if (k) lm_block_free(k);
}

// ---- selective staging of descriptors from pinned host memory ------------------------
// After the detector has run, the matcher will only ever read the descriptor rows of
//   - frame-0 candidates: argmax != dustbin and !(prob < min_prob0)   (tracking_main.c:142-148)
//   - frame-1 queries: the cells compute_top_N selected               (tracking_main.c:115-119)
// and depth only at candidate cells.  So instead of copying every frame's 1.86 MB of
// descriptors, a kernel pulls just those 256-byte rows straight out of the caller's pinned
// buffer over PCIe (zero-copy reads) into the same [frame][cell] layout on the device.
__global__ void mark_needed_rows_kernel(int n_frames, int cells, int top_n, float prob_lt,
                                        const int32_t* __restrict__ max_idx, const float* __restrict__ prob,
                                        const int32_t* __restrict__ q_patch, const int32_t* __restrict__ q_count,
                                        uint8_t* __restrict__ flags) {
  const int f = blockIdx.y;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < cells; i += gridDim.x * blockDim.x) {
    const size_t g = (size_t)f * cells + i;
    flags[g] = (max_idx[g] != 64 && !(prob[g] < prob_lt)) ? 1 : 0;
  }
}
__global__ void mark_query_rows_kernel(int cells, int top_n, const int32_t* __restrict__ q_patch,
                                       const int32_t* __restrict__ q_count, uint8_t* __restrict__ flags) {
  const int f = blockIdx.y;
  const int n = min(q_count[f], top_n);
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    flags[(size_t)f * cells + q_patch[(size_t)f * top_n + i]] |= 2;
}

// One warp per SM.  Rows move host -> shared -> device through the TMA unit (cp.async.bulk ->
// UBLKCP): flagged cells are queued 32 at a time, each lane issues the 256-byte bulk load of one
// row into a shared-memory slot (completion on an mbarrier) and, one stage later, the bulk
// store of that slot to the device row.  Nothing passes through the SM's load/store pipeline,
// whose in-order return queue would otherwise hold every device load of the co-resident
// kernels behind multi-microsecond PCIe reads (measured: the tensor-core matcher ran 12x
// slower beside an LDG-based gather).  Two 8 KB stages keep ~2.4 MB in flight chip-wide.
constexpr int kGatherStages = 2;
__global__ void __launch_bounds__(32)
gather_rows_kernel(long long total_cells, const uint8_t* __restrict__ flags, const int8_t* __restrict__ h_desc,
                   int8_t* __restrict__ d_desc, unsigned long long* __restrict__ rows_moved, int* abort_flag) {
  __shared__ __align__(128) uint8_t slots[kGatherStages][32][256];
  __shared__ uint64_t bar[kGatherStages];
  __shared__ long long queue[64];
  const int lane = threadIdx.x;
  if (lane == 0) {
    for (int i = 0; i < kGatherStages; i++) sm100::mbar_init(sm100::smem_u32(&bar[i]), 1);
    sm100::mbar_fence_init();
  }
  __syncwarp();
  const long long groups = (total_cells + 31) >> 5;
  int queued = 0;                    // flagged cells waiting in queue[]
  unsigned long long moved = 0;
  int stage = 0;
  unsigned used[kGatherStages] = {0, 0};   // times each stage's barrier has been armed
  long long pend_cell = -1;          // this lane's row in the stage whose load is in flight
  int pend_stage = -1;

  auto flush_pending = [&]() {       // wait for the in-flight stage, then store its rows
    if (pend_stage < 0) return;
    sm100::mbar_wait(sm100::smem_u32(&bar[pend_stage]), (used[pend_stage] - 1) & 1, abort_flag, 9);
    if (pend_cell >= 0)
      asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], 256;"
                   ::"l"(reinterpret_cast<uint64_t>(d_desc + pend_cell * 256)),
                     "r"(sm100::smem_u32(&slots[pend_stage][lane][0]))
                   : "memory");
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    pend_stage = -1;
    pend_cell = -1;
  };
  auto issue = [&](int n) {          // load the first n (<= 32) queued rows into `stage`
    // the store that last read this stage's slots (the most recent bulk group) must have
    // finished reading them; the other stage's PCIe load stays in flight meanwhile
    asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    __syncwarp();
    if (lane == 0) sm100::mbar_expect_tx(sm100::smem_u32(&bar[stage]), (uint32_t)n * 256u);
    __syncwarp();
    const long long cell = lane < n ? queue[lane] : -1;
    if (cell >= 0) {
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], 256, [%2];"
                   ::"r"(sm100::smem_u32(&slots[stage][lane][0])),
                     "l"(reinterpret_cast<uint64_t>(h_desc + cell * 256)), "r"(sm100::smem_u32(&bar[stage]))
                   : "memory");
    }
    used[stage]++;
    const int this_stage = stage;
    stage ^= 1;
    flush_pending();                 // the other stage: its load overlapped this issue
    pend_stage = this_stage;
    pend_cell = cell;
    // shift the queue
    __syncwarp();
    const long long rest = (lane + n < queued) ? queue[lane + n] : -1;
    __syncwarp();
    if (lane + n < queued) queue[lane] = rest;
    queued -= n;
    moved += n;
    __syncwarp();
  };

  for (long long g = blockIdx.x; g < groups; g += gridDim.x) {
    const long long cell = (g << 5) + lane;
    const int flag = cell < total_cells ? flags[cell] : 0;
    const unsigned votes = __ballot_sync(0xffffffffu, flag != 0);
    if (flag) queue[queued + __popc(votes & ((1u << lane) - 1))] = cell;
    queued += __popc(votes);
    __syncwarp();
    if (queued >= 32) issue(32);
  }
  if (queued > 0) issue(queued);
  flush_pending();
  asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  if (lane == 0 && moved) atomicAdd(rows_moved, moved);
}

// The call that stages host buffers through track_sequence_host_impl: mv_track_sequence_host,
// mv_track_sequence_landmarks_host or mv_track_landmarks_prepare_host.
enum class HostCall { depth, landmarks, prepare };

// Host inputs.  The chunks of `plan` are double-buffered: on the staging stream the logits are copied and the detector
// runs, then descriptors arrive (selectively when the host buffers are pinned, else as a plain copy); the compute
// stream runs the previous chunk's compute meanwhile.  Consecutive chunks share one halo frame.  HostCall::landmarks
// also steps the caller's table over the chunk's frames but its halo before matching; chunks run in order on that
// stream, so the table chains from chunk to chunk.  With HostCall::prepare the host buffers start with the block's
// warm-up frames, staged first in chunks of their own without a halo (logits and query rows; words only), and each
// chunk of the block's frames runs the words and the matcher into the block's memory; the speculation follows the
// last chunk.  first_frame: the table's frame number of the first pair's frame.  Returns once the host buffers are no
// longer read: a prepared block's work may still be queued on the compute stream.
static mv_status track_sequence_host_impl(mv_ctx* c, HostCall call, const HostPlan& plan, const mv_track_params* p,
                                          const int8_t* h_semi, const float* h_semi_scale, const int8_t* h_desc,
                                          const float* h_desc_scale, const float* h_depth, int first_frame,
                                          int n_words, mv_landmark* d_table, mv_pair_result* h_results,
                                          int32_t* h_n_with_landmark, mv_lm_block* blk,
                                          unsigned long long* h2d_bytes, unsigned long long* d2h_bytes) {
  const int cells = p->match.rows * p->match.cols;
  const int n_pairs = plan.n_pairs, n_warm = plan.n_warm, cf = plan.pairs + 1;
  const int N = p->top_n;
  const bool landmarks = call != HostCall::depth;
  mv_status st;

  // zero-copy gather needs device-visible (pinned) descriptor and depth buffers
  bool gather = true;
  const int8_t* hd_desc = nullptr;
  cudaPointerAttributes a1;
  if (cudaPointerGetAttributes(&a1, h_desc) == cudaSuccess && a1.type == cudaMemoryTypeHost && a1.devicePointer &&
      (reinterpret_cast<uintptr_t>(a1.devicePointer) & 15) == 0) {
    hd_desc = (const int8_t*)a1.devicePointer;
  } else {
    cudaGetLastError();
    gather = false;  // pageable memory: plain staged copies
  }

  constexpr int NB = 3;  // chunks in flight: staging DMA / row gather / compute
  void *bs[NB], *bd[NB], *bz[NB], *bsc[NB], *dres, *dmoved;
  void *bdsc[NB] = {}, *dnwl = nullptr;   // landmark mode
  SeqScratch w[NB];
  const size_t semi_pad = ((size_t)cf * cells * 65 + 255) & ~(size_t)255;
  for (int b = 0; b < NB; b++) {
    const std::string n = "host.buf" + std::to_string(b);
    if ((st = mv_scratch(c, (n + ".semi").c_str(), semi_pad, &bs[b]))) return st;
    if ((st = mv_scratch(c, (n + ".desc").c_str(), (size_t)cf * cells * 256, &bd[b]))) return st;
    if ((st = mv_scratch(c, (n + ".depth").c_str(), sizeof(float) * (size_t)cf * cells, &bz[b]))) return st;
    if ((st = mv_scratch(c, (n + ".scale").c_str(), sizeof(float) * (size_t)cf, &bsc[b]))) return st;
    if ((st = seq_scratch(c, p, cf, n.c_str(), landmarks, &w[b]))) return st;
    if (landmarks && (st = mv_scratch(c, (n + ".dscale").c_str(), sizeof(float) * (size_t)cf, &bdsc[b]))) return st;
  }
  if (call == HostCall::landmarks) {
    // the table update's shared sort scratch, for the full chunk and the last one: growing it between
    // enqueues would free memory (cudaFree) while the three streams run
    if ((st = mv_landmarks_sequence_reserve(c, n_words, plan.pairs, N))) return st;
    if ((st = mv_landmarks_sequence_reserve(c, n_words, plan.frames(plan.n_chunks - 1) - 1, N))) return st;
    if (h_n_with_landmark &&
        (st = mv_scratch(c, "host.n_with_landmark", sizeof(int32_t) * (size_t)n_pairs, &dnwl)))
      return st;
  }
  if ((st = mv_scratch(c, "host.results", sizeof(mv_pair_result) * (size_t)n_pairs, &dres))) return st;
  if ((st = mv_scratch(c, "host.moved", 16, &dmoved))) return st;
  int* abort_flag = nullptr;
  if ((st = mv_abort_flag(c, &abort_flag))) return st;
  // every event of this call lives in `events` and is destroyed on any return path
  struct EventBag {
    std::vector<cudaEvent_t> v;
    ~EventBag() { for (cudaEvent_t e : v) cudaEventDestroy(e); }
  } events;
  // On every return path -- errors included -- the three streams are drained before the events die and
  // before the caller gets its buffers back: the DMA engine and the row-gather kernel read the caller's
  // pinned h_semi / h_desc / h_depth asynchronously.
  struct Drain {
    mv_ctx* c;
    bool compute = true;   // cleared once a prepared block's work may stay queued (the host buffers are read by then)
    ~Drain() {
      if (compute) cudaStreamSynchronize(c->stream);
      cudaStreamSynchronize(c->copy_stream);
      cudaStreamSynchronize(c->gather_stream);
    }
  } drain{c};
  auto new_event = [&](cudaEvent_t* e) -> mv_status {
    MV_CUDA(c, cudaEventCreateWithFlags(e, cudaEventDisableTiming));
    events.v.push_back(*e);
    return MV_OK;
  };
  cudaEvent_t ready[NB], consumed[NB], detected[NB], copied[NB];
  for (int b = 0; b < NB; b++) {
    if ((st = new_event(&ready[b])) || (st = new_event(&consumed[b])) || (st = new_event(&detected[b])) ||
        (st = new_event(&copied[b])))
      return st;
  }
  // NB chunks in flight on three engines:
  //   copy_stream    DMA of a chunk's logits (and descriptors/depth when not gathering)
  //   stream         in order: detector + row marking of chunk k+1, then match + pose of chunk k
  //   gather_stream  zero-copy pull of chunk k+1's marked descriptor rows, concurrent with the
  //                  PnP launch of chunk k.  That launch is capped at kStagingPnpCtasPerSm, which
  //                  leaves registers and 38 KB of shared memory free; the gather kernel is a
  //                  one-warp CTA that fits in them, so it is resident alongside.
  // whatever the caller queued on the compute stream must be ordered before the staging
  cudaEvent_t start;
  if ((st = new_event(&start))) return st;
  MV_CUDA(c, cudaEventRecord(start, c->stream));
  MV_CUDA(c, cudaStreamWaitEvent(c->copy_stream, start, 0));
  MV_CUDA(c, cudaStreamWaitEvent(c->gather_stream, start, 0));
  MV_CUDA(c, cudaMemsetAsync(dmoved, 0, 8, c->gather_stream));

  unsigned long long up = 0;
  // The scratch of chunk k: its buffer set, but a block being prepared keeps what step_table and solve read at the
  // chunk's frames and pairs in its own memory.  The detector of chunk k+1 writes the halo frame's qp / qc / ov there
  // again before the compute of chunk k reads them: the same bytes (the same frame, the same kernels), in the same
  // stream order as the chunk-local copies of the host calls.
  auto chunk_scratch = [&](int k) {
    SeqScratch v = w[k % NB];
    if (call != HostCall::prepare) return v;
    const size_t f0 = plan.frame0(k), M = p->match.max_matches;
    const SeqScratch& a = blk->w;
    v.qp = a.qp + f0 * N; v.qc = a.qc + f0; v.ov = a.ov + f0;
    v.word = a.word + f0 * N;
    v.coords_in = plan.warm(k) ? nullptr : a.coords_in + 3 * f0 * N;   // warm-up words need no coordinates
    if (!plan.warm(k)) {
      const size_t p0 = plan.first_pair(k);
      v.mp = a.mp + 4 * p0 * M; v.mc = a.mc + p0; v.mcell = a.mcell + p0 * M; v.rin = a.rin + p0;
    }
    return v;
  };

  auto stage_dma = [&](int k) -> mv_status {
    const int b = k % NB, p0 = plan.frame0(k), nf = plan.frames(k);
    cudaStream_t cs = c->copy_stream;
    // buffer set b may be refilled only after the compute that read it is done
    MV_CUDA(c, cudaStreamWaitEvent(cs, consumed[b], 0));
    MV_CUDA(c, cudaMemcpyAsync(bs[b], h_semi + (size_t)p0 * cells * 65, (size_t)nf * cells * 65,
                               cudaMemcpyHostToDevice, cs));
    MV_CUDA(c, cudaMemcpyAsync(bsc[b], h_semi_scale + p0, sizeof(float) * (size_t)nf, cudaMemcpyHostToDevice, cs));
    up += (unsigned long long)nf * ((size_t)cells * 65 + 4);
    if (!plan.warm(k)) {
      MV_CUDA(c, cudaMemcpyAsync(bz[b], h_depth + (size_t)p0 * cells, sizeof(float) * (size_t)nf * cells,
                                 cudaMemcpyHostToDevice, cs));
      up += (unsigned long long)nf * cells * 4;
    }
    if (landmarks) {
      MV_CUDA(c, cudaMemcpyAsync(bdsc[b], h_desc_scale + p0, sizeof(float) * (size_t)nf, cudaMemcpyHostToDevice, cs));
      up += (unsigned long long)nf * 4;
    }
    if (!gather) {
      MV_CUDA(c, cudaMemcpyAsync(bd[b], h_desc + (size_t)p0 * cells * 256, (size_t)nf * cells * 256,
                                 cudaMemcpyHostToDevice, cs));
      up += (unsigned long long)nf * (size_t)cells * 256;
    }
    MV_CUDA(c, cudaEventRecord(copied[b], cs));
    return MV_OK;
  };
  // The row gather of chunk k+1 runs beside the pose kernels of chunk k, not beside its matcher:
  // the tensor-core matcher is one latency-sensitive CTA per SM, and zero-copy host reads
  // queued on the same SM stretch its global loads; the pose kernel (FP32-bound, its inputs in
  // shared memory) does not care.
  int pending_gather = -1;
  cudaEvent_t matched;
  if ((st = new_event(&matched))) return st;
  auto launch_gather = [&](int k, cudaEvent_t after) -> mv_status {
    const int b = k % NB, p0 = plan.frame0(k), nf = plan.frames(k);
    cudaStream_t gs = c->gather_stream;
    MV_CUDA(c, cudaStreamWaitEvent(gs, detected[b], 0));
    if (after) MV_CUDA(c, cudaStreamWaitEvent(gs, after, 0));
    // An SM's L1/shared split is per-SM state: a kernel that asks for no shared memory
    // configures "all L1", and the PnP CTAs (5 x 37 KB shared) then cannot join that SM until
    // it drains.  Ask for the max-shared carveout so both kernels agree on the split.
    // The attribute belongs to the device: each context sets it on its own, so every GPU of the process gets it.
    if (!c->gather_carveout_set) {
      cudaFuncSetAttribute(gather_rows_kernel, cudaFuncAttributePreferredSharedMemoryCarveout,
                           cudaSharedmemCarveoutMaxShared);
      c->gather_carveout_set = true;
    }
    gather_rows_kernel<<<c->sm_count, 32, 0, gs>>>((long long)nf * cells, w[b].flags,
                                                   hd_desc + (size_t)p0 * cells * 256, (int8_t*)bd[b],
                                                   (unsigned long long*)dmoved, abort_flag);
    MV_CHECK_LAUNCH(c);
    MV_CUDA(c, cudaEventRecord(ready[b], gs));
    return MV_OK;
  };
  auto stage_detect = [&](int k) -> mv_status {
    const int b = k % NB, nf = plan.frames(k);
    const SeqScratch v = chunk_scratch(k);
    mv_status s2;
    MV_CUDA(c, cudaStreamWaitEvent(c->stream, copied[b], 0));
    if ((s2 = seq_detect(c, p, nf, (const int8_t*)bs[b], (const float*)bsc[b], v))) return s2;
    if (gather) {
      dim3 g1((cells + 255) / 256, nf), g2((p->top_n + 255) / 256, nf);
      if (plan.warm(k)) {   // no matcher runs on a warm-up frame: its query rows only
        MV_CUDA(c, cudaMemsetAsync(v.flags, 0, (size_t)nf * cells, c->stream));
      } else {
        mark_needed_rows_kernel<<<g1, 256, 0, c->stream>>>(nf, cells, p->top_n, mv_round_up(p->match.min_prob0),
                                                           v.idx, v.prob, v.qp, v.qc, v.flags);
        MV_CHECK_LAUNCH(c);
      }
      mark_query_rows_kernel<<<g2, 256, 0, c->stream>>>(cells, p->top_n, v.qp, v.qc, v.flags);
      MV_CHECK_LAUNCH(c);
    }
    MV_CUDA(c, cudaEventRecord(detected[b], c->stream));
    if (!gather) {
      MV_CUDA(c, cudaEventRecord(ready[b], c->stream));
    } else if (k == 0) {
      return launch_gather(k, nullptr);
    } else {
      pending_gather = k;   // released by chunk k-1's compute, see stage_compute
    }
    return MV_OK;
  };
  auto release_gather = [&](int k) -> mv_status {
    if (pending_gather != k + 1) return MV_OK;
    pending_gather = -1;
    MV_CUDA(c, cudaEventRecord(matched, c->stream));
    return launch_gather(k + 1, matched);
  };
  // The word assignment (a persistent CTA per SM with the vocabulary in shared memory) runs after the chunk's `ready`
  // and before its matcher, so it never runs beside a row gather.  Chunk k+1's gather is released once chunk k's
  // matcher is enqueued, so that it runs beside K3.  A block being prepared runs no K3: there it is released after
  // the chunk's whole compute (words, matcher, RANSAC-E; the words only for a warm-up chunk), which measured the
  // same as after the matcher (profiles/r07).
  auto stage_compute = [&](int k) -> mv_status {
    const int b = k % NB, nf = plan.frames(k), p0 = plan.first_pair(k);
    const bool warm = plan.warm(k), prepare = call == HostCall::prepare;
    const int8_t* desc = (const int8_t*)bd[b];
    const float* depth = warm ? nullptr : (const float*)bz[b];
    const SeqScratch v = chunk_scratch(k);
    const SeqLandmarks lm = {first_frame - n_warm + plan.frame0(k), n_words, d_table, (const float*)bdsc[b],
                             dnwl ? (int32_t*)dnwl + p0 : nullptr};
    mv_status s2;
    MV_CUDA(c, cudaStreamWaitEvent(c->stream, ready[b], 0));
    if (landmarks && (s2 = seq_words(c, p, warm ? nf : nf - 1, desc, depth, v, &lm))) return s2;
    if (call == HostCall::landmarks &&
        (s2 = mv_landmarks_sequence_impl(c, n_words, d_table, lm.first_frame, nf - 1, N, v.word, v.qc, v.coords_in,
                                         v.coords_out)))
      return s2;
    if (!warm) {
      if ((s2 = seq_match(c, p, nf, desc, v))) return s2;
      if ((!prepare && (s2 = release_gather(k))) || (s2 = seq_ransac(c, p, nf, v))) return s2;
    }
    if (prepare && (s2 = release_gather(k))) return s2;
    if (!prepare) {
      if ((s2 = seq_corr(c, p, nf, depth, v, landmarks ? &lm : nullptr))) return s2;
      if ((s2 = seq_pose(c, p, nf, v, (mv_pair_result*)dres + p0, p0, kStagingPnpCtasPerSm))) return s2;
    }
    MV_CUDA(c, cudaEventRecord(consumed[b], c->stream));
    return MV_OK;
  };

  if ((st = stage_dma(0))) return st;
  if (plan.n_chunks > 1 && (st = stage_dma(1))) return st;
  if ((st = stage_detect(0))) return st;
  for (int k = 0; k < plan.n_chunks; k++) {
    if (k + 2 < plan.n_chunks && (st = stage_dma(k + 2))) return st;
    if (k + 1 < plan.n_chunks && (st = stage_detect(k + 1))) return st;
    if ((st = stage_compute(k))) return st;
  }
  unsigned long long moved = 0;
  unsigned long long down = 0;
  if (call == HostCall::prepare) {
    // one speculation over the warm-up and block words; the block's remaining work stays queued
    if ((st = mv_landmarks_speculate_impl(c, n_words, first_frame, n_warm, n_pairs, p->top_n, blk->w.word, blk->w.qc,
                                          blk->b.coords_in, &blk->spec)))
      return st;
    blk->b.coords_out = mv_lm_spec_coords(blk->spec);
    drain.compute = false;
  } else {
    down = sizeof(mv_pair_result) * (unsigned long long)n_pairs;
    MV_CUDA(c, cudaMemcpyAsync(h_results, dres, sizeof(mv_pair_result) * (size_t)n_pairs, cudaMemcpyDeviceToHost,
                               c->stream));
    if (dnwl) {
      MV_CUDA(c, cudaMemcpyAsync(h_n_with_landmark, dnwl, sizeof(int32_t) * (size_t)n_pairs, cudaMemcpyDeviceToHost,
                                 c->stream));
      down += sizeof(int32_t) * (unsigned long long)n_pairs;
    }
    MV_CUDA(c, cudaStreamSynchronize(c->stream));
  }
  MV_CUDA(c, cudaStreamSynchronize(c->copy_stream));
  MV_CUDA(c, cudaMemcpyAsync(&moved, dmoved, 8, cudaMemcpyDeviceToHost, c->gather_stream));
  MV_CUDA(c, cudaStreamSynchronize(c->gather_stream));
  if (gather) up += moved * 256ull;  // one 256 B descriptor row per staged cell
  if (h2d_bytes) *h2d_bytes = up;
  if (d2h_bytes) *d2h_bytes = down;
  return MV_OK;
}

extern "C" mv_status mv_track_sequence_host(mv_ctx* c, const mv_track_params* p, int n_frames,
                                            const int8_t* h_semi, const float* h_semi_scale,
                                            const int8_t* h_desc, const float* h_depth,
                                            mv_pair_result* h_results, unsigned long long* h2d_bytes,
                                            unsigned long long* d2h_bytes) {
  MV_ENTER(c);
  if (!p || n_frames < 2 || !h_semi || !h_semi_scale || !h_desc || !h_depth || !h_results)
    MV_BAD_ARG(c, "mv_track_sequence_host");
  const HostPlan plan = host_plan(c, p, 0, n_frames - 1, false);
  if (mv_status st = seq_check(c, "mv_track_sequence_host", p, plan.pairs + 1, nullptr, false)) return st;
  return track_sequence_host_impl(c, HostCall::depth, plan, p, h_semi, h_semi_scale, h_desc, nullptr, h_depth, 0, 0,
                                  nullptr, h_results, nullptr, nullptr, h2d_bytes, d2h_bytes);
}

extern "C" mv_status mv_track_sequence_landmarks_host(mv_ctx* c, const mv_track_params* p, int n_frames,
                                                      int first_frame, const int8_t* h_semi, const float* h_semi_scale,
                                                      const int8_t* h_desc, const float* h_desc_scale,
                                                      const float* h_depth, int n_words, mv_landmark* d_table,
                                                      mv_pair_result* h_results, int32_t* h_n_with_landmark,
                                                      unsigned long long* h2d_bytes, unsigned long long* d2h_bytes) {
  MV_ENTER(c);
  if (!p || n_frames < 2 || !h_semi || !h_semi_scale || !h_desc || !h_desc_scale || !h_depth || !h_results)
    MV_BAD_ARG(c, "mv_track_sequence_landmarks_host");
  const HostPlan plan = host_plan(c, p, 0, n_frames - 1, true);
  if (mv_status st = seq_check(c, "mv_track_sequence_landmarks_host", p, plan.pairs + 1, nullptr, true, n_words))
    return st;
  if (!d_table) MV_BAD_ARG(c, "mv_track_sequence_landmarks_host: NULL landmark table");
  return track_sequence_host_impl(c, HostCall::landmarks, plan, p, h_semi, h_semi_scale, h_desc, h_desc_scale, h_depth,
                                  first_frame, n_words, d_table, h_results, h_n_with_landmark, nullptr, h2d_bytes,
                                  d2h_bytes);
}

extern "C" mv_status mv_track_landmarks_prepare_host(mv_ctx* c, const mv_track_params* p, int n_warm, int n_frames,
                                                     int first_frame, const int8_t* h_semi, const float* h_semi_scale,
                                                     const int8_t* h_desc, const float* h_desc_scale,
                                                     const float* h_depth, int n_words, mv_lm_block** out,
                                                     unsigned long long* h2d_bytes) {
  MV_ENTER(c);
  HostPlan plan;
  mv_lm_block* k;
  mv_status st = lm_block_new(c, "mv_track_landmarks_prepare_host", p, n_warm, n_frames, first_frame, n_words,
                              h_semi && h_semi_scale && h_desc && h_desc_scale && h_depth, nullptr, &plan, out, &k);
  if (st) return st;
  if ((st = track_sequence_host_impl(c, HostCall::prepare, plan, p, h_semi, h_semi_scale, h_desc, h_desc_scale, h_depth,
                                     first_frame, n_words, nullptr, nullptr, nullptr, k, h2d_bytes, nullptr))) {
    lm_block_free(k);
    return st;
  }
  k->phase = 1;
  *out = k;
  return MV_OK;
}

// ------------------------------------------------------------------------------------
// track() (tracking.h:3) with the semantics of tracking_main.c:84-218
// ------------------------------------------------------------------------------------
static void rot_to_quat(const float R[3][3], Quaternionf* q) {
  const float tr = R[0][0] + R[1][1] + R[2][2];
  if (tr > 0.0f) {
    float s = sqrtf(tr + 1.0f) * 2.0f;
    q->w = 0.25f * s; q->x = (R[2][1] - R[1][2]) / s; q->y = (R[0][2] - R[2][0]) / s; q->z = (R[1][0] - R[0][1]) / s;
  } else if (R[0][0] > R[1][1] && R[0][0] > R[2][2]) {
    float s = sqrtf(1.0f + R[0][0] - R[1][1] - R[2][2]) * 2.0f;
    q->w = (R[2][1] - R[1][2]) / s; q->x = 0.25f * s; q->y = (R[0][1] + R[1][0]) / s; q->z = (R[0][2] + R[2][0]) / s;
  } else if (R[1][1] > R[2][2]) {
    float s = sqrtf(1.0f + R[1][1] - R[0][0] - R[2][2]) * 2.0f;
    q->w = (R[0][2] - R[2][0]) / s; q->x = (R[0][1] + R[1][0]) / s; q->y = 0.25f * s; q->z = (R[1][2] + R[2][1]) / s;
  } else {
    float s = sqrtf(1.0f + R[2][2] - R[0][0] - R[1][1]) * 2.0f;
    q->w = (R[1][0] - R[0][1]) / s; q->x = (R[0][2] + R[2][0]) / s; q->y = (R[1][2] + R[2][1]) / s; q->z = 0.25f * s;
  }
}

extern "C" void track(const Frame* last_frame, const Frame* current_frame, const int x_shift,
                      const int y_shift, const int window_size, const float threshold, SE3* transform) {
  transform->q = create_Quaternionf(1.0f, 0.0f, 0.0f, 0.0f);
  transform->t.x = transform->t.y = transform->t.z = 0.0f;
  if (last_frame == NULL || current_frame == NULL) return;  // tracking.h:4-7
  const int rows = current_frame->feature_rows, cols = current_frame->feature_cols;
  const int cells = rows * cols;
  const int N = 100, MAXM = 150;
  mv_ctx* c;
  {
    std::lock_guard<std::mutex> lk(g_mu);
    c = legacy_ctx();
  }
  int* idx0 = (int*)malloc(sizeof(int) * cells);
  float* pr0 = (float*)malloc(sizeof(float) * cells);
  int qp[N], qi[N]; float qpr[N];
  int nv = 0, nq = 0;
  {
    std::lock_guard<std::mutex> lk(g_mu);
    legacy_check(c, compute_softmax_ex(c, last_frame->semi_scale, last_frame->semi, cells, &nv, idx0, pr0), "track");
    mv_status st = compute_top_N_ex(c, current_frame->semi_scale, current_frame->semi, cells, N, 1000, &nq, qp, qi, qpr);
    if (st == MV_ERR_TOO_MANY_VALID) { printf("Exceed max number of features!\n"); exit(1); }
    legacy_check(c, st, "track");
  }
  mv_match_params mp;
  mv_match_params_default(&mp, rows, cols);
  mp.shift_x = x_shift; mp.shift_y = y_shift; mp.radius = (window_size - 1) / 2;  // tracking.h:20
  mp.match_threshold = (double)threshold; mp.max_matches = MAXM;
  float p1[MAXM][2], p2[MAXM][2];
  int nm = 0;
  {
    std::lock_guard<std::mutex> lk(g_mu);
    legacy_check(c, mv_match_pair_host(c, &mp, last_frame->desc, current_frame->desc, idx0, pr0, nq, qp, qi,
                                       &p1[0][0], &p2[0][0], &nm, nullptr, nullptr), "track");
  }
  free(idx0); free(pr0);
  float E[3][3], K[3][3] = {{1, 0, 0}, {0, 1, 0}, {0, 0, 1}};
  int inl[MAXM], ninl = 0;
  ransac_essential_matrix(nm, p1, p2, K, 10, 1.1f, E, inl, &ninl);  // tracking_main.c:210-214
  float R1[3][3], R2[3][3], t[3];
  recover_pose_from_essential_matrix(E, R1, R2, t);                  // :218
  rot_to_quat(R1, &transform->q);
  transform->t.x = t[0]; transform->t.y = t[1]; transform->t.z = t[2];
}
