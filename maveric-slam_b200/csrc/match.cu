// match.cu -- windowed int8 descriptor search (reference: src/tracking_main.c:18-43,
// 103-194), the dp4a form: one warp per query keypoint.
//
// Reference semantics that the kernels reproduce bit for bit (SURVEY App. A/B):
//   * candidates of a query are the cells of the clamped window, scanned x-outer /
//     y-inner (tracking_main.c:127-136), skipping cells whose detector argmax is the
//     dustbin or whose prob < 0.2 (:142,:146);
//   * squared_dist (:18-43) uses all 256 dims only while its sticky candidate norm is
//     0 -- i.e. for the leading candidates up to and including the first one with a
//     non-zero norm ("F") -- and afterwards 64 dims, F's stale 256-d norm and a 64-d
//     query norm;
//   * the score (:154) is int32-wrapped dot^2 over int32-wrapped norm product,
//     int->float RN, IEEE divide;  accepted iff (double)score > thr^2 (:155), best
//     is the first maximum in scan order (:156);
//   * matches are emitted in query order, capped at max_matches (:167-192).
//
//   K1a match_queries_kernel : per query best candidate  (HBM/L2-bound gather + dp4a)
//   K1b emit_matches_kernel  : ordered compaction to (x0,y0,x1,y1) pixel pairs
#include "mv_common.cuh"

namespace {

constexpr int kWarpsPerCta = 8;

__device__ __forceinline__ int dp4a_ss(int a, int b, int c) { return __dp4a(a, b, c); }

// tracking_main.c:154 with defined (two's complement) wrap
__device__ __forceinline__ float wrapped_cos2(int dot, int n_cand, int n_query) {
  const int num = (int)((unsigned)dot * (unsigned)dot);
  const int den = (int)((unsigned)n_cand * (unsigned)n_query);
  return __fdiv_rn(__int2float_rn(num), __int2float_rn(den));
}

__device__ __forceinline__ int warp_sum(int v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

struct MatchGeom {
  int rows, cols, shift_x, shift_y, radius;
  float accept_gt;   // round_down(thr*thr): (double)s > thr^2  <=>  s > accept_gt
  float prob_lt;     // round_up(min_prob0): (double)p < 0.2    <=>  p < prob_lt
};

__global__ void __launch_bounds__(kWarpsPerCta * 32)
match_queries_kernel(MatchGeom g, int cells, int top_n, int n_pairs,
                     const int32_t* __restrict__ f0_of, const int32_t* __restrict__ f1_of,
                     const int8_t* __restrict__ desc,
                     const int32_t* __restrict__ max_idx, const float* __restrict__ prob,
                     const int32_t* __restrict__ q_patch, const int32_t* __restrict__ q_count,
                     int32_t* __restrict__ best_cell, float* __restrict__ best_score) {
  const int lane = threadIdx.x & 31;
  const int pair = blockIdx.y;
  const int qi = blockIdx.x * kWarpsPerCta + (threadIdx.x >> 5);
  if (qi >= top_n) return;
  const int f0 = f0_of ? f0_of[pair] : pair;
  const int f1 = f1_of ? f1_of[pair] : pair + 1;
  const size_t out = (size_t)pair * top_n + qi;
  if (qi >= q_count[f1]) {
    if (lane == 0) best_cell[out] = -1;
    return;
  }
  const int cell1 = q_patch[(size_t)f1 * top_n + qi];
  const int qx = cell1 / g.rows, qy = cell1 - qx * g.rows;
  const int x_lo = max(qx + g.shift_x - g.radius, 0), x_hi = min(qx + g.shift_x + g.radius, g.cols - 1);
  const int y_lo = max(qy + g.shift_y - g.radius, 0), y_hi = min(qy + g.shift_y + g.radius, g.rows - 1);
  const int wh = y_hi - y_lo + 1;
  const int total = (x_hi >= x_lo && wh > 0) ? (x_hi - x_lo + 1) * wh : 0;

  const int8_t* dq = desc + ((size_t)f1 * cells + cell1) * 256;
  const int8_t* d0 = desc + (size_t)f0 * cells * 256;
  const int32_t* mi0 = max_idx + (size_t)f0 * cells;
  const float* pr0 = prob + (size_t)f0 * cells;

  // query descriptor: this lane's 8 bytes (for the 256-d pass) and the first 64
  // bytes in every lane (for the per-lane 64-d pass)
  const int2 q8 = __ldg(reinterpret_cast<const int2*>(dq) + lane);
  int4 q64[4];
#pragma unroll
  for (int k = 0; k < 4; k++) q64[k] = __ldg(reinterpret_cast<const int4*>(dq) + k);
  const int nq256 = warp_sum(dp4a_ss(q8.y, q8.y, dp4a_ss(q8.x, q8.x, 0)));
  int nq64 = 0;
#pragma unroll
  for (int k = 0; k < 4; k++) {
    nq64 = dp4a_ss(q64[k].x, q64[k].x, nq64);
    nq64 = dp4a_ss(q64[k].y, q64[k].y, nq64);
    nq64 = dp4a_ss(q64[k].z, q64[k].z, nq64);
    nq64 = dp4a_ss(q64[k].w, q64[k].w, nq64);
  }

  int n_cand = 0;        // sticky candidate norm (norm1_squared, :133)
  bool have = false;     // lane-local best
  float bs = 0.0f;
  int bw = 0x7fffffff;   // scan rank of the lane-local best

  for (int w0 = 0; w0 < total; w0 += 32) {
    const int w = w0 + lane;
    int c = -1;
    bool valid = false;
    if (w < total) {
      const int dx = w / wh;
      c = (x_lo + dx) * g.rows + y_lo + (w - dx * wh);
      valid = (mi0[c] != 64) && !(pr0[c] < g.prob_lt);
    }
    unsigned todo = __ballot_sync(0xffffffffu, valid);

    // leading candidates: full 256-d, cooperatively, in scan order
    while (n_cand == 0 && todo) {
      const int src = __ffs(todo) - 1;
      todo &= todo - 1;
      const int cc = __shfl_sync(0xffffffffu, c, src);
      const int2 c8 = __ldg(reinterpret_cast<const int2*>(d0 + (size_t)cc * 256) + lane);
      const int dot = warp_sum(dp4a_ss(c8.y, q8.y, dp4a_ss(c8.x, q8.x, 0)));
      const int nc = warp_sum(dp4a_ss(c8.y, c8.y, dp4a_ss(c8.x, c8.x, 0)));
      n_cand = nc;
      const float s = wrapped_cos2(dot, nc, nq256);
      if (lane == src && s > g.accept_gt && (!have || s > bs)) {
        have = true; bs = s; bw = w;
      }
    }
    // the rest of this chunk: one candidate per lane, 64-d, stale candidate norm
    if ((todo >> lane) & 1u) {
      const int4* cp = reinterpret_cast<const int4*>(d0 + (size_t)c * 256);
      int dot = 0;
#pragma unroll
      for (int k = 0; k < 4; k++) {
        const int4 v = __ldg(cp + k);
        dot = dp4a_ss(v.x, q64[k].x, dot);
        dot = dp4a_ss(v.y, q64[k].y, dot);
        dot = dp4a_ss(v.z, q64[k].z, dot);
        dot = dp4a_ss(v.w, q64[k].w, dot);
      }
      const float s = wrapped_cos2(dot, n_cand, nq64);
      if (s > g.accept_gt && (!have || s > bs)) {
        have = true; bs = s; bw = w;
      }
    }
  }

  // first maximum in scan order: max score, ties to the smaller scan rank (:156)
#pragma unroll
  for (int o = 16; o; o >>= 1) {
    const bool oh = __shfl_xor_sync(0xffffffffu, have, o);
    const float os = __shfl_xor_sync(0xffffffffu, bs, o);
    const int ow = __shfl_xor_sync(0xffffffffu, bw, o);
    if (oh && (!have || os > bs || (os == bs && ow < bw))) {
      have = true; bs = os; bw = ow;
    }
  }
  if (lane == 0) {
    int cell = -1;
    if (have) {
      const int dx = bw / wh;
      cell = (x_lo + dx) * g.rows + y_lo + (bw - dx * wh);
    }
    best_cell[out] = cell;
    best_score[out] = bs;
  }
}

constexpr int kEmitThreads = 256;

// One CTA per pair: ordered compaction of the per-query winners (:167-192).
__global__ void __launch_bounds__(kEmitThreads)
emit_matches_kernel(int rows, int cells, int top_n, int max_matches,
                    const int32_t* __restrict__ f0_of, const int32_t* __restrict__ f1_of,
                    const int32_t* __restrict__ max_idx,
                    const int32_t* __restrict__ q_patch, const int32_t* __restrict__ q_idx,
                    const int32_t* __restrict__ q_count,
                    const int32_t* __restrict__ best_cell, const float* __restrict__ best_score,
                    int n_parts, size_t part_stride, const int32_t* __restrict__ rank_to_cell, int rank_stride,
                    float* __restrict__ match_pts, int32_t* __restrict__ match_count,
                    int32_t* __restrict__ match_cell0, int32_t* __restrict__ match_query,
                    float* __restrict__ match_score) {
  __shared__ int s_warp[kEmitThreads / 32];
  __shared__ int s_base;
  const int pair = blockIdx.x;
  const int f0 = f0_of ? f0_of[pair] : pair;
  const int f1 = f1_of ? f1_of[pair] : pair + 1;
  const int nq = min(q_count[f1], top_n);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (threadIdx.x == 0) s_base = 0;
  __syncthreads();
  for (int i0 = 0; i0 < nq; i0 += kEmitThreads) {
    const int i = i0 + threadIdx.x;
    // the matcher reports one candidate per part (the tcgen05 kernel: one per epilogue thread of
    // the query's row); the winner is the larger score, ties to the earlier cell.  The tcgen05 kernel
    // reports candidates by their rank in frame 0's compacted candidate list, which is in cell order, so
    // the tie rule is the same on ranks; rank_to_cell turns the winner back into a cell.
    int cell = -1;
    float score = 0.0f;
    if (i < nq) {
      for (int part = 0; part < n_parts; part++) {
        const int oc = best_cell[part * part_stride + (size_t)pair * top_n + i];
        const float os = best_score[part * part_stride + (size_t)pair * top_n + i];
        if (oc >= 0 && (cell < 0 || os > score || (os == score && oc < cell))) { score = os; cell = oc; }
      }
      if (rank_to_cell && cell >= 0) cell = rank_to_cell[(size_t)f0 * rank_stride + cell];
    }
    const unsigned votes = __ballot_sync(0xffffffffu, cell >= 0);
    if (lane == 0) s_warp[wid] = __popc(votes);
    __syncthreads();
    int before = s_base;
    for (int w = 0; w < wid; w++) before += s_warp[w];
    const int pos = before + __popc(votes & ((1u << lane) - 1));
    if (cell >= 0 && pos < max_matches) {
      const int ch0 = max_idx[(size_t)f0 * cells + cell];
      const int ch1 = q_idx[(size_t)f1 * top_n + i];
      const int cell1 = q_patch[(size_t)f1 * top_n + i];
      const int bx = cell / rows, by = cell - bx * rows;
      const int qx = cell1 / rows, qy = cell1 - qx * rows;
      const size_t o = (size_t)pair * max_matches + pos;
      float4 v;
      v.x = (float)(bx * 8 + ch0 % 8);
      v.y = (float)(by * 8 + ch0 / 8);
      v.z = (float)(qx * 8 + ch1 % 8);
      v.w = (float)(qy * 8 + ch1 / 8);
      reinterpret_cast<float4*>(match_pts)[o] = v;
      if (match_cell0) match_cell0[o] = cell;
      if (match_query) match_query[o] = i;
      if (match_score) match_score[o] = score;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      int t = 0;
      for (int w = 0; w < kEmitThreads / 32; w++) t += s_warp[w];
      s_base += t;
    }
    __syncthreads();
    if (s_base >= max_matches) break;
  }
  if (threadIdx.x == 0) match_count[pair] = min(s_base, max_matches);
}

}  // namespace

extern "C" void mv_match_params_default(mv_match_params* p, int rows, int cols) {
  memset(p, 0, sizeof(*p));
  p->rows = rows; p->cols = cols;
  p->shift_x = 4; p->shift_y = 4; p->radius = 4;   // tracking_main.c:104-106
  p->max_matches = 150;                            // :13
  p->match_threshold = 0.9;                        // :12
  p->min_prob0 = 0.2;                              // :146
  p->use_tensor_cores = 2;                         // auto: tcgen05 tile kernel where its shape limits hold
}

int mv_match_tc_parts();
mv_status mv_match_tc_launch(mv_ctx* ctx, const mv_match_params* p, int n_frames, int n_pairs, int top_n,
                             const int32_t* d_f0, const int32_t* d_f1, const int8_t* d_desc,
                             const int32_t* d_max_idx, const float* d_prob, const int32_t* d_q_patch,
                             const int32_t* d_q_count, int32_t* d_best_rank, float* d_best_score,
                             const int32_t** d_rank_to_cell, int* rank_stride);

extern "C" mv_status mv_match_batch(mv_ctx* ctx, const mv_match_params* p, int n_frames, int n_pairs,
                                    int top_n, const int32_t* d_f0, const int32_t* d_f1,
                                    const int8_t* d_desc, const int32_t* d_max_idx, const float* d_prob,
                                    const int32_t* d_q_patch, const int32_t* d_q_idx,
                                    const int32_t* d_q_count, float* d_match_pts, int32_t* d_match_count,
                                    int32_t* d_match_cell0, int32_t* d_match_query, float* d_match_score) {
  MV_ENTER(ctx);
  if (!p || n_pairs <= 0 || top_n <= 0 || !d_desc || !d_max_idx || !d_prob || !d_q_patch || !d_q_idx ||
      !d_q_count || !d_match_pts || !d_match_count || p->rows <= 0 || p->cols <= 0 || p->radius < 0 ||
      p->max_matches <= 0)
    MV_BAD_ARG(ctx, "mv_match_batch");
  if ((reinterpret_cast<uintptr_t>(d_desc) & 15) || (reinterpret_cast<uintptr_t>(d_match_pts) & 15))
    MV_BAD_ARG(ctx, "mv_match_batch: d_desc and d_match_pts must be 16-byte aligned");
  if (n_pairs > 65535 || n_frames > 65535)
    MV_BAD_ARG(ctx, "mv_match_batch: at most 65535 pairs / frames per call (grid y dimension); split the batch");
  const int cells = p->rows * p->cols;
  int use_tc = p->use_tensor_cores;
  if (use_tc == 2) use_tc = mv_match_tc_feasible(p, n_frames, n_pairs, top_n) ? 1 : 0;
  const int n_parts = use_tc ? mv_match_tc_parts() : 1;
  const size_t part_stride = (size_t)n_pairs * top_n;
  void* bc = nullptr; void* bsc = nullptr;
  mv_status st = mv_scratch(ctx, "match.best_cell", sizeof(int32_t) * part_stride * n_parts, &bc);
  if (st) return st;
  st = mv_scratch(ctx, "match.best_score", sizeof(float) * part_stride * n_parts, &bsc);
  if (st) return st;

  // 0: dp4a warp-per-query kernel; 1: tcgen05 tile kernel (MV_ERR_BAD_ARG if the shape is outside its
  // limits); 2: the tcgen05 kernel wherever mv_match_tc_feasible() says it can run (rows <= 256, a
  // threshold that is a number, shared memory, a driver with tensor maps), else dp4a.
  // Both produce the same bytes (tests/test_gpu_parity.py); tools/match_sweep.py times them.
  const int32_t* rank_to_cell = nullptr;
  int rank_stride = 0;
  if (use_tc) {
    st = mv_match_tc_launch(ctx, p, n_frames, n_pairs, top_n, d_f0, d_f1, d_desc, d_max_idx, d_prob,
                            d_q_patch, d_q_count, (int32_t*)bc, (float*)bsc, &rank_to_cell, &rank_stride);
    if (st) return st;
  } else {
    MatchGeom g;
    g.rows = p->rows; g.cols = p->cols; g.shift_x = p->shift_x; g.shift_y = p->shift_y; g.radius = p->radius;
    g.accept_gt = mv_round_down(p->match_threshold * p->match_threshold);
    g.prob_lt = mv_round_up(p->min_prob0);
    dim3 grid((top_n + kWarpsPerCta - 1) / kWarpsPerCta, n_pairs);
    mv_prof_scope ps(ctx, "match");
    match_queries_kernel<<<grid, kWarpsPerCta * 32, 0, ctx->stream>>>(
        g, cells, top_n, n_pairs, d_f0, d_f1, d_desc, d_max_idx, d_prob, d_q_patch, d_q_count,
        (int32_t*)bc, (float*)bsc);
    MV_CHECK_LAUNCH(ctx);
  }
  {
    mv_prof_scope ps(ctx, "emit");
    emit_matches_kernel<<<n_pairs, kEmitThreads, 0, ctx->stream>>>(
        p->rows, cells, top_n, p->max_matches, d_f0, d_f1, d_max_idx, d_q_patch, d_q_idx, d_q_count,
        (const int32_t*)bc, (const float*)bsc, n_parts, part_stride, rank_to_cell, rank_stride, d_match_pts,
        d_match_count, d_match_cell0, d_match_query, d_match_score);
    MV_CHECK_LAUNCH(ctx);
  }
  return MV_OK;
}
