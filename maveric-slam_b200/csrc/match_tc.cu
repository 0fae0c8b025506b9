// match_tc.cu -- windowed int8 descriptor search on the 5th-generation tensor cores
// (reference: src/tracking_main.c:18-43,103-194; same results as match.cu, bit for bit).
//
// The reference evaluates a 64-dimension dot product for every candidate of a query but the
// first one (squared_dist, tracking_main.c:33-41), so the bulk of the search is an int8 GEMM
//     D[query][candidate] = sum_{k<64} desc1[query][k] * desc0[candidate][k]
// Only ~14 % of a KITTI frame's cells are candidates at all (argmax != dustbin and prob >= 0.2,
// tracking_main.c:142,146), and the reference scans a window x-outer / y-inner, i.e. in ascending
// cell index.  So the candidates of a frame are first COMPACTED in cell order -- which is scan
// order, so ties keep their meaning -- and the GEMM runs over candidates only:
//
//   K1p compact_candidates_kernel  (per frame)  validity bits, candidate list c_cell[rank], first rank of
//        every cell column c_col[x], the first 64 bytes of every candidate descriptor c_desc[rank][64]
//        (the B operand, rank-major), and per block of 32 ranks a table "which of them have y >= t"
//        for every row t (the y half of a window mask is then GE[y_lo] & ~GE[y_hi + 1]).
//   K1q lead_kernel  (per tile of 128 queries, four lanes per query)  the query's window as a rank
//        range, its LEADING candidate -- squared_dist's first call (tracking_main.c:21-32) scores the
//        first candidate with a non-zero norm over all 256 dimensions; zero descriptors before it
//        score NaN and can never match -- with dp4a, the per-query constants of every later score,
//        the first 64 bytes of the query descriptor (the A operand) and the tile's rank span.
//   K1  match_tc_kernel  (persistent, one CTA per SM, no global loads outside TMA / bulk copies)
//        warp 0      producer: per tile one TMA box [64 B][128 queries] + its 4 KB of row state, per
//                    chunk one TMA box [64 B][256 candidates] + the chunk's y tables (SWIZZLE_64B)
//        warp 1      MMA issuer: per chunk two tcgen05.mma.kind::i8 (M=128, N=256, K=32) into one of
//                    two 256-column TMEM accumulator stages
//        warps 2-17  epilogue, thread <-> query row (TMEM lane), four threads per row taking every
//                    fourth block of 32 candidates: window mask from the row's rank range and the y
//                    table, tcgen05.ld, then a BRANCH-FREE pass that squares each accumulator and
//                    collects the few that beat the row's running key in a bitmask; only those take
//                    the reference's exact float path (see "filter").
//
// The distance matrix never leaves TMEM.  Compared with a tile over the cell grid (the first form of
// this kernel) the tensor pipe, the tcgen05.ld traffic and the filter touch candidates only: a KITTI
// tile is one chunk of ~190 candidates instead of six chunks of 235 cells.
//
// Filter.  For the non-leading candidates of a query the score (tracking_main.c:154) is
//     s = float(int32(dot*dot)) / float(int32(norm_F * norm_q64))
// with a denominator that is constant per query.  int->float and IEEE division are monotone,
// so s is non-decreasing in key = n (denominator >= 0) or key = ~n (denominator < 0), n the
// wrapped int32 square.  A candidate whose key does not exceed the largest key seen so far can
// neither pass the threshold nor beat the current best (strict '>' at :155-156), so the exact
// float path runs only on strict prefix maxima of the key, which start above a conservative
// bound derived from the acceptance threshold.  Ties keep the smaller rank = the earlier
// candidate in the reference's x-outer / y-inner scan.
#include "mv_common.cuh"
#include "sm100_ptx.cuh"

namespace {

using namespace sm100;

constexpr int kTileQ = 128;
constexpr int kChunkN = 256;                    // candidates per chunk = UMMA N = TMEM columns per stage
constexpr int kBStages = 6;
constexpr int kBStageBytes = kChunkN * 64;
constexpr int kAStages = 4;
constexpr int kAStageBytes = kTileQ * 64;
constexpr int kRowBytes = kTileQ * 32;          // row state of a tile
constexpr int kAccStages = 2;
constexpr int kTmemCols = kAccStages * kChunkN;
constexpr int kEpiWarp0 = 2;
#ifndef MV_TC_EPI_WARPS
#define MV_TC_EPI_WARPS 16
#endif
constexpr int kEpiWarps = MV_TC_EPI_WARPS;   // 4 quadrants x kParts
constexpr int kParts = kEpiWarps / 4;           // threads per query row, each takes every kParts-th block of 32
constexpr int kThreads = 32 * (kEpiWarp0 + kEpiWarps);
#ifndef MV_LEAD_Q
#define MV_LEAD_Q 32                             // queries per lead_kernel CTA (a divisor of the tile's 128; measured 0.509 / 0.512 / 0.530 ms at 32 / 64 / 128)
#endif
#ifndef MV_LEAD_CTAS
#define MV_LEAD_CTAS (3 * 128 / MV_LEAD_Q)
#endif
constexpr int kLeadQ = MV_LEAD_Q;
constexpr int kLeadParts = kTileQ / kLeadQ;     // CTAs per tile
constexpr int kLeadThreads = 4 * kLeadQ;        // lead_kernel: four lanes per query
constexpr int kMaxCols = 4096;

struct TcGeom {
  int rows, cols, cells, shift_x, shift_y, radius, top_n;
  int qstride;        // query rows per pair in the A operand / row state: tiles_per_pair * 128
  int cstride;        // candidate rows per frame in c_desc / c_cell (cells rounded up to 32)
  int nblk;           // blocks of 32 ranks per frame (cstride / 32)
  int ystride;        // words per block in the y table: rows + 1 rounded up to 4
  int vwords;         // validity words per frame
  int tiles_per_pair, n_items;
  float accept_gt;    // (double)s > thr^2  <=>  s > accept_gt
  float prob_lt;      // (double)p < min    <=>  p < prob_lt
};

// tracking_main.c:154 with defined (two's complement) wrap
__device__ __forceinline__ float wrapped_cos2(int dot, int n_cand, int n_query) {
  const int num = (int)((unsigned)dot * (unsigned)dot);
  const int den = (int)((unsigned)n_cand * (unsigned)n_query);
  return __fdiv_rn(__int2float_rn(num), __int2float_rn(den));
}

__device__ __forceinline__ int dp4a4(const int4& a, const int4& b, int acc) {
  acc = __dp4a(a.x, b.x, acc);
  acc = __dp4a(a.y, b.y, acc);
  acc = __dp4a(a.z, b.z, acc);
  return __dp4a(a.w, b.w, acc);
}

// ---------------------------------------------------------------------------------------------
// K1p: candidates of a frame in cell (= scan) order
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
compact_candidates_kernel(TcGeom g, const int32_t* __restrict__ max_idx, const float* __restrict__ prob,
                          const int8_t* __restrict__ desc, uint32_t* __restrict__ vbits,
                          int32_t* __restrict__ c_cell, int32_t* __restrict__ c_col, int8_t* __restrict__ c_desc,
                          uint32_t* __restrict__ c_ytab) {
  extern __shared__ int s_dyn[];   // [cols + 1] candidates per column, then [vwords] validity words
  __shared__ int s_warp[8];
  int* s_col = s_dyn;
  uint32_t* s_vb = reinterpret_cast<uint32_t*>(s_dyn + g.cols + 1);
  const int f = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  for (int i = tid; i <= g.cols; i += 256) s_col[i] = 0;
  for (int i = tid; i < g.vwords; i += 256) s_vb[i] = 0;
  __syncthreads();
  const int32_t* mi = max_idx + (size_t)f * g.cells;
  const float* pr = prob + (size_t)f * g.cells;
  int32_t* cc = c_cell + (size_t)f * g.cstride;
  // every thread owns a contiguous run of cells, so ranks in cell order are one block scan of the runs'
  // counts: two passes over the run (the second one hits L1), three barriers in all
  const int per = (g.cells + 255) >> 8;
  const int c_lo = min(g.cells, tid * per), c_hi = min(g.cells, c_lo + per);
  int mine = 0;
  unsigned flags = 0;   // the run's verdicts, kept when the run fits a word (no second read of idx / prob)
#pragma unroll 8
  for (int c = c_lo; c < c_hi; c++) {
    const bool v = mi[c] != 64 && !(pr[c] < g.prob_lt);   // tracking_main.c:142,146
    mine += v ? 1 : 0;
    flags |= (v ? 1u : 0u) << ((c - c_lo) & 31);
  }
  int incl = mine;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int u = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += u;
  }
  if (lane == 31) s_warp[wid] = incl;
  __syncthreads();
  int rank = incl - mine, count = 0;
  for (int w = 0; w < 8; w++) {
    if (w < wid) rank += s_warp[w];
    count += s_warp[w];
  }
  for (int c = c_lo; c < c_hi; c++) {
    const bool v = per <= 32 ? ((flags >> (c - c_lo)) & 1u) != 0 : (mi[c] != 64 && !(pr[c] < g.prob_lt));
    if (v) {
      cc[rank++] = c;
      atomicAdd(&s_col[c / g.rows], 1);
      atomicOr(&s_vb[c >> 5], 1u << (c & 31));
    }
  }
  __syncthreads();
  {
    uint32_t* vb = vbits + (size_t)f * g.vwords;
    for (int i = tid; i < g.vwords; i += 256) vb[i] = s_vb[i];
  }
  // exclusive prefix of the column counts (one warp, carried)
  if (wid == 0) {
    int carry = 0;
    for (int x0 = 0; x0 <= g.cols; x0 += 32) {
      const int x = x0 + lane;
      const int v = x < g.cols ? s_col[x] : 0;
      int in2 = v;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int u = __shfl_up_sync(0xffffffffu, in2, o);
        if (lane >= o) in2 += u;
      }
      if (x <= g.cols) c_col[(size_t)f * (g.cols + 1) + x] = carry + in2 - v;
      carry += __shfl_sync(0xffffffffu, in2, 31);
    }
  }
  __syncthreads();   // the candidate list written above is read back below
  // B operand: the first 64 bytes of every candidate's descriptor, rank-major (four threads per row)
  {
    const int4* src = reinterpret_cast<const int4*>(desc + (size_t)f * g.cells * 256);
    int4* dst = reinterpret_cast<int4*>(c_desc + (size_t)f * g.cstride * 64);
    // eight rows in flight per thread (the row's cell is a dependent load in front of the row itself)
    const int total = count * 4;
    for (int i0 = tid; i0 < total; i0 += 256 * 8) {
      int cellv[8];
#pragma unroll
      for (int u = 0; u < 8; u++) cellv[u] = (i0 + 256 * u < total) ? cc[(i0 + 256 * u) >> 2] : 0;
      int4 val[8];
#pragma unroll
      for (int u = 0; u < 8; u++) val[u] = __ldg(src + (size_t)cellv[u] * 16 + (tid & 3));
#pragma unroll
      for (int u = 0; u < 8; u++)
        if (i0 + 256 * u < total) dst[i0 + 256 * u] = val[u];
    }
  }
  // y table: for block b of 32 ranks and every t in [0, rows], the ranks whose cell row is >= t
  const int nb = (count + 31) >> 5;
  for (int b = wid; b < nb; b += 8) {
    const int r = b * 32 + lane;
    const int y = r < count ? cc[r] % g.rows : -1;
    uint32_t* dst = c_ytab + ((size_t)f * g.nblk + b) * g.ystride;
    for (int t0 = 0; t0 < g.ystride; t0 += 32) {
      uint32_t mine = 0;
#pragma unroll 8
      for (int j = 0; j < 32; j++) {
        const uint32_t m = __ballot_sync(0xffffffffu, y >= t0 + j);
        if (lane == j) mine = m;
      }
      if (t0 + lane < g.ystride) dst[t0 + lane] = (t0 + lane <= g.rows) ? mine : 0u;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// K1q: per query the window as a rank range, the leading candidate, the later scores' constants
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ int first_set_in_range(const uint32_t* vb, int lo, int hi) {
  int p = lo;
  while (p <= hi) {
    const uint32_t w = vb[p >> 5] >> (p & 31);
    if (w) {
      const int q = p + __ffs(w) - 1;
      return q <= hi ? q : -1;
    }
    p = (p | 31) + 1;
  }
  return -1;
}
// set bits in [lo, hi)
__device__ __forceinline__ int popc_range(const uint32_t* vb, int lo, int hi) {
  int n = 0;
  for (int w = lo >> 5; (w << 5) < hi; w++) {
    uint32_t v = vb[w];
    const int b0 = w << 5;
    if (lo > b0) v &= 0xffffffffu << (lo - b0);
    if (hi < b0 + 32) v &= (1u << (hi - b0)) - 1u;
    n += __popc(v);
  }
  return n;
}

// Row state the lead kernel hands to the epilogue (32 bytes).  Ranks are relative to the frame.
//   w0: rlo   first rank after the leading candidate (0 when the window holds no candidate)
//   w1: rhi   one past the last rank of the window's columns (rlo >= rhi: nothing to scan)
//   w2: y_lo | y_hi << 16
//   w3: brank best so far as a rank (-1: none)      w4: its score
//   w5: den_f  float(int32(norm_F * norm_q64)), the denominator of every later score
//   w6: curmax start of the key filter             w7: flip  0 / -1: key = n ^ flip
__global__ void __launch_bounds__(kLeadThreads, MV_LEAD_CTAS)
lead_kernel(TcGeom g, const int32_t* __restrict__ f0_of, const int32_t* __restrict__ f1_of,
            const int8_t* __restrict__ desc, const uint32_t* __restrict__ vbits, const int32_t* __restrict__ c_col,
            const int32_t* __restrict__ q_patch, const int32_t* __restrict__ q_count, int8_t* __restrict__ qa,
            int4* __restrict__ rowinfo, int4* __restrict__ spans) {
  // frame 0's validity bits and column prefix, staged once per CTA: the search below is then shared-memory
  // lookups, and a query's chain of dependent global loads is cell -> descriptors, nothing else
  extern __shared__ uint32_t s_tab[];            // [vwords] validity words, then [cols + 1] column prefix
  const int item = blockIdx.x / kLeadParts, part = blockIdx.x - item * kLeadParts;
  const int pair = item / g.tiles_per_pair;
  const int q0 = (item - pair * g.tiles_per_pair) * kTileQ;
  const int f0 = f0_of ? f0_of[pair] : pair;
  const int f1 = f1_of ? f1_of[pair] : pair + 1;
  const int nq = min(q_count[f1], g.top_n);
  const int n_rows = max(0, min(kTileQ, nq - q0));
  const int tid = threadIdx.x, lane = tid & 31, sub = tid & 3, row = part * kLeadQ + (tid >> 2);
  const int quad0 = lane & ~3;
  const bool active = row < n_rows;
  // this thread's query: issue its loads before the tables are staged
  int cell1 = 0;
  if (active) cell1 = __ldg(q_patch + (size_t)f1 * g.top_n + q0 + row);
  {
    const uint32_t* gv = vbits + (size_t)f0 * g.vwords;
    const int32_t* gc = c_col + (size_t)f0 * (g.cols + 1);
    for (int i = tid; i < g.vwords; i += kLeadThreads) s_tab[i] = __ldg(gv + i);
    for (int i = tid; i <= g.cols; i += kLeadThreads) s_tab[g.vwords + i] = (uint32_t)__ldg(gc + i);
  }
  const uint32_t* vb = s_tab;
  const int32_t* col0 = reinterpret_cast<const int32_t*>(s_tab + g.vwords);
  const int8_t* d0 = desc + (size_t)f0 * g.cells * 256;

  int x_lo = 0, x_hi = -1, y_lo = 0, y_hi = -1;
  int4 q4[4] = {make_int4(0, 0, 0, 0), make_int4(0, 0, 0, 0), make_int4(0, 0, 0, 0), make_int4(0, 0, 0, 0)};
  if (active) {
    const int qx = cell1 / g.rows, qy = cell1 - qx * g.rows;
    x_lo = max(qx + g.shift_x - g.radius, 0);
    x_hi = min(qx + g.shift_x + g.radius, g.cols - 1);
    y_lo = max(qy + g.shift_y - g.radius, 0);
    y_hi = min(qy + g.shift_y + g.radius, g.rows - 1);
    if (y_hi < y_lo) { x_lo = 0; x_hi = -1; }
    // the four lanes of a query hold the 16-byte pieces sub, sub + 4, sub + 8, sub + 12 of a descriptor:
    // each load instruction of the quad reads 64 contiguous bytes (whole sectors)
    const int4* qp = reinterpret_cast<const int4*>(desc + ((size_t)f1 * g.cells + cell1) * 256) + sub;
#pragma unroll
    for (int c = 0; c < 4; c++) q4[c] = __ldg(qp + 4 * c);
  }
  __syncthreads();   // the staged tables

  // Leading candidates (tracking_main.c:21-32): every candidate of the window, in scan order, is scored
  // over 256 dims until one has a non-zero norm.  The four lanes of a query look at four columns at a
  // time; the evaluation is warp-convergent, each lane on its quarter of the two descriptors.  Nothing
  // before the first candidate's loads are issued depends on the query descriptor, so the two
  // descriptors' loads are in flight together; the query norms are taken after the loop.
  bool searching = active && x_hi >= x_lo;
  int cx = x_lo, cy = y_lo;
  int lead_cell = -1, n_cand = 0, lead_dot = 0;
  while (__any_sync(0xffffffffu, searching)) {
    int c = -1;
    if (searching) {
      const int x = cx + sub;
      if (x <= x_hi) c = first_set_in_range(vb, x * g.rows + (sub == 0 ? cy : y_lo), x * g.rows + y_hi);
    }
    const unsigned found = (__ballot_sync(0xffffffffu, c >= 0) >> quad0) & 0xfu;
    int csel = __shfl_sync(0xffffffffu, c, quad0 + (found ? __ffs(found) - 1 : 0));
    if (!found) csel = -1;
    if (searching && csel < 0) {
      cx += 4; cy = y_lo;
      searching = cx <= x_hi;
    }
    int dot = 0, nc = 0;
    if (csel >= 0) {
      const int4* cp = reinterpret_cast<const int4*>(d0 + (size_t)csel * 256) + sub;
      int4 cv[4];
#pragma unroll
      for (int k = 0; k < 4; k++) cv[k] = __ldg(cp + 4 * k);
#pragma unroll
      for (int k = 0; k < 4; k++) { dot = dp4a4(cv[k], q4[k], dot); nc = dp4a4(cv[k], cv[k], nc); }
    }
    dot += __shfl_xor_sync(0xffffffffu, dot, 1); nc += __shfl_xor_sync(0xffffffffu, nc, 1);
    dot += __shfl_xor_sync(0xffffffffu, dot, 2); nc += __shfl_xor_sync(0xffffffffu, nc, 2);
    if (csel >= 0) {
      if (nc != 0) {
        lead_cell = csel; n_cand = nc; lead_dot = dot;
        searching = false;
      } else {   // a zero descriptor scores NaN (0/0), never matches, and leaves the norm sticky
        const int xs = csel / g.rows, ys = csel - xs * g.rows;
        cx = xs; cy = ys + 1;
        if (cy > y_hi) { cx = xs + 1; cy = y_lo; }
        searching = cx <= x_hi;
      }
    }
  }
  // first use of the query descriptor: the A operand row (its first 64 bytes = piece 0 of every lane) and
  // the two query norms (64 and 256 dims)
  if (active)
    reinterpret_cast<int4*>(qa + ((size_t)pair * g.qstride + q0 + row) * 64)[sub] = q4[0];
  int nq64 = dp4a4(q4[0], q4[0], 0);
  int nq256 = nq64;
#pragma unroll
  for (int c = 1; c < 4; c++) nq256 = dp4a4(q4[c], q4[c], nq256);
  nq64 += __shfl_xor_sync(0xffffffffu, nq64, 1); nq256 += __shfl_xor_sync(0xffffffffu, nq256, 1);
  nq64 += __shfl_xor_sync(0xffffffffu, nq64, 2); nq256 += __shfl_xor_sync(0xffffffffu, nq256, 2);

  if (sub == 0) {
    int rlo = 0, rhi = 0, curmax = 0x7fffffff, flip = 0, brank = -1;
    float den_f = 1.0f, bs = 0.0f;
    if (lead_cell >= 0) {
      const int xs = lead_cell / g.rows;
      const int lead_rank = col0[xs] + popc_range(vb, xs * g.rows, lead_cell);
      rlo = lead_rank + 1;
      rhi = col0[x_hi + 1];
      const float s = wrapped_cos2(lead_dot, n_cand, nq256);
      if (s > g.accept_gt) { bs = s; brank = lead_rank; }
      const int den_i = (int)((unsigned)n_cand * (unsigned)nq64);
      den_f = __int2float_rn(den_i);
      // conservative start of the key filter: every key <= curmax has s <= accept_gt
      if (den_i > 0) {
        const double b = floor((double)g.accept_gt * (double)den_f) - 256.0;
        curmax = b < -2147483648.0 ? (int)0x80000000 : (b > 2147483647.0 ? 0x7fffffff : (int)b);
      } else if (den_i < 0) {
        flip = -1;
        const double b = -ceil((double)g.accept_gt * (double)den_f) - 257.0;
        curmax = b < -2147483648.0 ? (int)0x80000000 : (b > 2147483647.0 ? 0x7fffffff : (int)b);
      } else {
        curmax = 0;   // s = +inf only for n > 0
      }
      // the tile's rank span, straight into its (zeroed) span record: y = max of (INT_MAX - rlo), z = max of rhi
      if (rlo < rhi) {
        atomicMax(&reinterpret_cast<int*>(spans + item)[1], 0x7fffffff - rlo);
        atomicMax(&reinterpret_cast<int*>(spans + item)[2], rhi);
      }
    }
    int4* rdst = rowinfo + ((size_t)pair * g.qstride + q0 + row) * 2;
    rdst[0] = make_int4(rlo, rhi, (y_lo & 0xffff) | (y_hi << 16), brank);
    rdst[1] = make_int4(__float_as_int(bs), __float_as_int(den_f), curmax, flip);
  }
  if (tid == 0 && part == 0) reinterpret_cast<int*>(spans + item)[0] = n_rows;
}

// ---------------------------------------------------------------------------------------------
// K1: the tile GEMM and its exact-score epilogue
// ---------------------------------------------------------------------------------------------
struct TileSpan {
  int pair, f0, q0, n_rows;   // n_rows == 0: nothing to do
  int r0a, n_chunks;          // first candidate rank (a multiple of 32), chunks of 256 ranks
};

// A role's walk over its CTA's tiles with the NEXT tile's span already in flight: the span is a global
// load, and a role that waited for it at the top of every tile would add its latency to every tile.
struct TileIter {
  int item, stride, n_items;
  int4 sp;
  int f0;
  __device__ __forceinline__ void fetch(const TcGeom& g, const int32_t* __restrict__ f0_of,
                                        const int4* __restrict__ spans) {
    sp = make_int4(0, 0, 0, 0);
    f0 = 0;
    if (item < n_items) {
      sp = __ldg(spans + item);
      const int pair = item / g.tiles_per_pair;
      f0 = f0_of ? __ldg(f0_of + pair) : pair;
    }
  }
  __device__ __forceinline__ TileSpan take(const TcGeom& g) const {
    TileSpan t;
    t.pair = item / g.tiles_per_pair;
    t.q0 = (item - t.pair * g.tiles_per_pair) * kTileQ;
    t.f0 = f0;
    t.n_rows = sp.x;
    const int lo = 0x7fffffff - sp.y, hi = sp.z;   // min rlo, max rhi over the tile's rows (lead_kernel)
    t.r0a = 0; t.n_chunks = 0;
    if (hi > lo) {
      t.r0a = lo & ~31;
      t.n_chunks = (hi - t.r0a + kChunkN - 1) / kChunkN;
    }
    return t;
  }
};
#define MV_TILE_LOOP(T)                                                          \
  TileIter it_;                                                                  \
  it_.item = blockIdx.x; it_.stride = gridDim.x; it_.n_items = g.n_items;        \
  it_.fetch(g, f0_of, spans);                                                    \
  for (; it_.item < it_.n_items;)                                                \
    if (TileSpan T = it_.take(g); true)                                          \
      if (it_.item += it_.stride, it_.fetch(g, f0_of, spans), true)

__global__ void __launch_bounds__(kThreads, 1)
match_tc_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b, TcGeom g,
                const int32_t* __restrict__ f0_of, const int4* __restrict__ rowinfo,
                const uint32_t* __restrict__ c_ytab, const int4* __restrict__ spans,
                int32_t* __restrict__ best_rank, float* __restrict__ best_score, size_t part_stride,
                int* abort_flag) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sB = smem;
  uint8_t* sA = sB + kBStages * kBStageBytes;
  uint8_t* sR = sA + kAStages * kAStageBytes;                        // [kAStages][kTileQ][32 B]
  const uint32_t ybytes = 32u * (uint32_t)g.ystride;                 // 8 blocks x ystride words
  uint32_t* sY = reinterpret_cast<uint32_t*>(sR + kAStages * kRowBytes);   // [kBStages][8][ystride]

  __shared__ uint64_t bar_full_b[kBStages], bar_empty_b[kBStages];
  __shared__ uint64_t bar_full_a[kAStages], bar_empty_a[kAStages];
  __shared__ uint64_t bar_acc_full[kAccStages], bar_acc_empty[kAccStages];
  __shared__ uint32_t s_tmem_base;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int i = 0; i < kBStages; i++) { mbar_init(smem_u32(&bar_full_b[i]), 1); mbar_init(smem_u32(&bar_empty_b[i]), 1 + kEpiWarps); }
    for (int i = 0; i < kAStages; i++) { mbar_init(smem_u32(&bar_full_a[i]), 1); mbar_init(smem_u32(&bar_empty_a[i]), 1 + kEpiWarps); }
    for (int i = 0; i < kAccStages; i++) { mbar_init(smem_u32(&bar_acc_full[i]), 1); mbar_init(smem_u32(&bar_acc_empty[i]), kEpiWarps); }
    mbar_fence_init();
    tma_prefetch_desc(&tmap_a);
    tma_prefetch_desc(&tmap_b);
  }
  if (warp == 1) {
    tmem_alloc(smem_u32(&s_tmem_base), kTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = s_tmem_base;

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer
    uint32_t chunk = 0, tile = 0;
    MV_TILE_LOOP(t) {
      if (t.n_rows == 0) continue;
      if (lane == 0) {
        const uint32_t a = tile % kAStages, aph = (tile / kAStages) & 1;
        mbar_wait(smem_u32(&bar_empty_a[a]), aph ^ 1, abort_flag, 1, 256);
        mbar_expect_tx(smem_u32(&bar_full_a[a]), kAStageBytes + kRowBytes);
        const int qrow = t.pair * g.qstride + t.q0;
        tma_load_2d(smem_u32(sA + a * kAStageBytes), &tmap_a, smem_u32(&bar_full_a[a]), 0, qrow);
        bulk_load(smem_u32(sR + a * kRowBytes), rowinfo + (size_t)qrow * 2, kRowBytes, smem_u32(&bar_full_a[a]));
        for (int c = 0; c < t.n_chunks; c++, chunk++) {
          const uint32_t s = chunk % kBStages, ph = (chunk / kBStages) & 1;
          mbar_wait(smem_u32(&bar_empty_b[s]), ph ^ 1, abort_flag, 2, 256);
          mbar_expect_tx(smem_u32(&bar_full_b[s]), kBStageBytes + ybytes);
          tma_load_2d(smem_u32(sB + s * kBStageBytes), &tmap_b, smem_u32(&bar_full_b[s]), 0,
                      t.f0 * g.cstride + t.r0a + c * kChunkN);
          bulk_load(smem_u32(sY) + s * ybytes,
                    c_ytab + ((size_t)t.f0 * g.nblk + (t.r0a >> 5) + 8 * c) * g.ystride, ybytes,
                    smem_u32(&bar_full_b[s]));
        }
      }
      __syncwarp();
      tile++;
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer
    const uint32_t idesc = umma_idesc_s8(kTileQ, kChunkN);
    uint32_t chunk = 0, tile = 0;
    MV_TILE_LOOP(t) {
      if (t.n_rows == 0) continue;
      if (lane == 0) {
        const uint32_t a = tile % kAStages, aph = (tile / kAStages) & 1;
        mbar_wait(smem_u32(&bar_full_a[a]), aph, abort_flag, 3, 64);
        const uint32_t a_addr = smem_u32(sA + a * kAStageBytes);
        for (int c = 0; c < t.n_chunks; c++, chunk++) {
          const uint32_t s = chunk % kBStages, ph = (chunk / kBStages) & 1;
          const uint32_t acc = chunk % kAccStages, accph = (chunk / kAccStages) & 1;
          mbar_wait(smem_u32(&bar_acc_empty[acc]), accph ^ 1, abort_flag, 4, 64);
          mbar_wait(smem_u32(&bar_full_b[s]), ph, abort_flag, 5);
          tc_fence_after();
          const uint32_t b_addr = smem_u32(sB + s * kBStageBytes);
          const uint32_t d_addr = tmem_base + acc * (uint32_t)kChunkN;
          umma_s8(d_addr, umma_desc_k_sw64(a_addr), umma_desc_k_sw64(b_addr), idesc, 0);
          umma_s8(d_addr, umma_desc_k_sw64(a_addr + 32), umma_desc_k_sw64(b_addr + 32), idesc, 1);
          umma_commit(smem_u32(&bar_empty_b[s]));      // one of the 1 + kEpiWarps arrivals that free the stage
          umma_commit(smem_u32(&bar_acc_full[acc]));
        }
        if (t.n_chunks > 0) umma_commit(smem_u32(&bar_empty_a[a]));
        else mbar_arrive(smem_u32(&bar_empty_a[a]));
      }
      __syncwarp();
      tile++;
    }
  } else {
    // ------------------------------------------------------------ epilogue
    const int ew = warp - kEpiWarp0;
    const int qd = warp & 3;          // TMEM lane quadrant this warp may read
    const int part = ew >> 2;         // which of the row's kParts threads
    const int row = qd * 32 + lane;
    uint32_t chunk = 0, tile = 0;
    MV_TILE_LOOP(t) {
      if (t.n_rows == 0) continue;
      const uint32_t a = tile % kAStages, aph = (tile / kAStages) & 1;
      mbar_wait(smem_u32(&bar_full_a[a]), aph, abort_flag, 6);
      const int4 r0 = reinterpret_cast<const int4*>(sR + a * kRowBytes)[row * 2];
      const int4 r1 = reinterpret_cast<const int4*>(sR + a * kRowBytes)[row * 2 + 1];
      const bool active = row < t.n_rows;
      const int rlo = active ? r0.x : 0, rhi = active ? r0.y : 0;
      const int y_lo = r0.z & 0xffff, y_hi = r0.z >> 16;
      int brank = r0.w;
      float bs = __int_as_float(r1.x);
      const float den_f = __int_as_float(r1.y);
      int curmax = r1.z;
      const int flip = r1.w;
      // warp-uniform rank range of this warp's windows (blocks outside it are skipped outright)
      int w_lo = rhi > rlo ? rlo : 0x7fffffff;
      int w_hi = rhi > rlo ? rhi : 0;
#pragma unroll
      for (int o = 16; o; o >>= 1) {
        w_lo = min(w_lo, __shfl_xor_sync(0xffffffffu, w_lo, o));
        w_hi = max(w_hi, __shfl_xor_sync(0xffffffffu, w_hi, o));
      }

      for (int c = 0; c < t.n_chunks; c++, chunk++) {
        const uint32_t s = chunk % kBStages, ph = (chunk / kBStages) & 1;
        const uint32_t acc = chunk % kAccStages, accph = (chunk / kAccStages) & 1;
        const int rb0 = t.r0a + c * kChunkN;          // frame rank of the chunk's column 0
        // Every warp observes every phase of both barriers, needed or not: a parity wait can only tell
        // the current phase from the previous one, so a warp must never run two phases ahead.
        mbar_wait(smem_u32(&bar_full_b[s]), ph, abort_flag, 7);      // the chunk's y tables (complete long ago)
        mbar_wait(smem_u32(&bar_acc_full[acc]), accph, abort_flag, 8);
        if (w_hi > rb0 && w_lo < rb0 + kChunkN) {
          tc_fence_after();
          const uint32_t* yt = sY + s * (ybytes >> 2);
          const uint32_t t_row = tmem_base + ((uint32_t)(qd * 32) << 16) + acc * (uint32_t)kChunkN;
          // this thread's blocks: part, part + kParts, ... restricted to the warp's range
          const int b_lo = max(0, (w_lo - rb0) >> 5), b_hi = min(kChunkN / 32 - 1, (w_hi - 1 - rb0) >> 5);
          for (int b = b_lo + ((part - b_lo) & (kParts - 1)); b <= b_hi; b += kParts) {
            const int rb = rb0 + 32 * b;
            // the row's window inside the block: ranks [rlo, rhi) and rows [y_lo, y_hi]
            const int lo = max(rlo - rb, 0), hi = min(rhi - rb, 32);
            uint32_t m = 0;
            if (hi > lo) {
              m = (0xffffffffu >> (32 - (hi - lo))) << lo;
              m &= yt[b * g.ystride + y_lo] & ~yt[b * g.ystride + y_hi + 1];
            }
            if (__any_sync(0xffffffffu, m != 0)) {
              int v[32];
              tmem_ld_32x32(t_row + 32 * b, v);
              tmem_ld_wait();
              // branch-free: which in-window columns exceed the key filter?
              // key > curmax  <=>  n > curmax (flip = 0)  /  n < ~curmax (flip = -1); the flipped
              // lanes test n <= ~curmax, a superset the exact path re-checks: one compare with the
              // lane's flip folded in as a predicate, no per-column xor.
              const bool flipb = flip != 0;
              const int cm = flipb ? ~curmax : curmax;
              uint32_t trig = 0;
#pragma unroll
              for (int j = 0; j < 32; j++) {
                const int n = (int)((unsigned)v[j] * (unsigned)v[j]);
                trig |= ((n > cm) != flipb) ? (1u << j) : 0u;
              }
              trig &= m;
              // Survivors: exact score, in rank order.  With candidates only in a block, most rows meet
              // their true match somewhere, so a warp-block holds a handful of survivors in different
              // columns; each lane picks ITS next column out of its 32 registers with a five-level select
              // tree (31 SEL for the whole warp per round, one round unless a row has several prefix maxima).
              uint32_t rem = trig;
              while (__any_sync(0xffffffffu, rem != 0)) {
                const int j = rem ? __ffs(rem) - 1 : 0;
                int s16[16], s8[8], s4[4];
#pragma unroll
                for (int i = 0; i < 16; i++) s16[i] = (j & 1) ? v[2 * i + 1] : v[2 * i];
#pragma unroll
                for (int i = 0; i < 8; i++) s8[i] = (j & 2) ? s16[2 * i + 1] : s16[2 * i];
#pragma unroll
                for (int i = 0; i < 4; i++) s4[i] = (j & 4) ? s8[2 * i + 1] : s8[2 * i];
                const int s2a = (j & 8) ? s4[1] : s4[0], s2b = (j & 8) ? s4[3] : s4[2];
                const int vj = (j & 16) ? s2b : s2a;
                if (rem) {
                  rem &= rem - 1;
                  const int n = (int)((unsigned)vj * (unsigned)vj);
                  const int key = n ^ flip;
                  if (key > curmax) {
                    curmax = key;
                    const float sc = __fdiv_rn(__int2float_rn(n), den_f);
                    if (sc > g.accept_gt && (brank < 0 || sc > bs)) { bs = sc; brank = rb + j; }
                  }
                }
              }
            }
          }
          tc_fence_before();
        }
        __syncwarp();
        if (lane == 0) {
          mbar_arrive(smem_u32(&bar_acc_empty[acc]));
          mbar_arrive(smem_u32(&bar_empty_b[s]));
        }
      }

      // every one of the row's kParts threads reports its own best candidate; the emit kernel
      // merges them (larger score, ties to the earlier rank) and turns the rank into a cell
      if (active) {
        const size_t out = (size_t)part * part_stride + (size_t)t.pair * g.top_n + t.q0 + row;
        best_rank[out] = brank;
        best_score[out] = bs;
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&bar_empty_a[a]));
      tile++;
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, kTmemCols);
}

static void tc_geom(const mv_match_params* p, int n_pairs, int top_n, TcGeom* g) {
  g->rows = p->rows; g->cols = p->cols; g->cells = p->rows * p->cols;
  g->shift_x = p->shift_x; g->shift_y = p->shift_y; g->radius = p->radius; g->top_n = top_n;
  g->tiles_per_pair = (top_n + kTileQ - 1) / kTileQ;
  g->qstride = g->tiles_per_pair * kTileQ;
  g->cstride = (g->cells + 31) & ~31;
  g->nblk = g->cstride / 32;
  g->ystride = (p->rows + 1 + 3) & ~3;
  g->vwords = ((g->cells + 31) >> 5) + 4;
  g->n_items = n_pairs * g->tiles_per_pair;
  const double thr2 = p->match_threshold * p->match_threshold;
  g->accept_gt = mv_round_down(thr2);
  g->prob_lt = mv_round_up(p->min_prob0);
}

static constexpr size_t tc_smem_of(int ystride) {
  return 1024 + (size_t)kBStages * kBStageBytes + (size_t)kAStages * (kAStageBytes + kRowBytes) +
         (size_t)kBStages * 32u * ystride;
}
static size_t tc_smem(const TcGeom& g) { return tc_smem_of(g.ystride); }
// The most any launch needs, 198 400 B: mv_match_tc_feasible takes at most 256 rows, so ystride <= 260.  The
// kernel's static shared memory (its mbarriers) counts against the same 227 KB a block may opt in to, so the
// limit cannot be 227 KB itself.
constexpr size_t kTcSmemMax = tc_smem_of((256 + 1 + 3) & ~3);
static_assert(kTcSmemMax + 1024 <= 227 * 1024, "the largest matcher launch must fit beside the static shared memory");

}  // namespace

int mv_match_tc_parts() { return kParts; }

// Shapes the tensor-core matcher takes; everything else goes to the dp4a kernel (same bytes).
bool mv_match_tc_feasible(const mv_match_params* p, int n_frames, int n_pairs, int top_n) {
  if (n_frames <= 0 || n_pairs <= 0 || top_n <= 0 || p->rows <= 0 || p->cols <= 0) return false;
  if (p->rows > 256 || p->cols >= kMaxCols) return false;
  if ((long long)p->rows * p->cols >= (1ll << 24)) return false;
  const double thr2 = p->match_threshold * p->match_threshold;
  if (!(thr2 >= 0.0)) return false;
  TcGeom g;
  tc_geom(p, n_pairs, top_n, &g);
  if ((long long)n_frames * g.cstride >= (1ll << 31) - 512 || (long long)n_pairs * g.qstride >= (1ll << 31)) return false;
  return tc_smem(g) <= 227 * 1024 && mv_get_tmap_encode() != nullptr;
}

mv_status mv_match_tc_launch(mv_ctx* ctx, const mv_match_params* p, int n_frames, int n_pairs, int top_n,
                             const int32_t* d_f0, const int32_t* d_f1, const int8_t* d_desc,
                             const int32_t* d_max_idx, const float* d_prob, const int32_t* d_q_patch,
                             const int32_t* d_q_count, int32_t* d_best_rank, float* d_best_score,
                             const int32_t** d_rank_to_cell, int* rank_stride) {
  // d_best_rank / d_best_score: [mv_match_tc_parts()][n_pairs][top_n], one candidate per epilogue part, as a
  // frame-0 candidate RANK; *d_rank_to_cell [n_frames][*rank_stride] turns it into a cell (emit kernel)
  if (!mv_match_tc_feasible(p, n_frames, n_pairs, top_n))
    MV_BAD_ARG(ctx, "tensor-core matcher: rows <= 256, cols < 4096, match_threshold^2 >= 0 and a driver with "
                    "cuTensorMapEncodeTiled (use_tensor_cores = 2 falls back to the dp4a kernel by itself)");
  mv_tmap_encode_fn encode = mv_get_tmap_encode();
  TcGeom g;
  tc_geom(p, n_pairs, top_n, &g);

  void *vb, *ccell, *ccol, *cdesc, *cytab, *qa, *rinfo, *spans;
  int* flag = nullptr;
  mv_status st;
  const size_t cdesc_rows = (size_t)n_frames * g.cstride + kChunkN;
  const size_t qa_rows = (size_t)n_pairs * g.qstride;
  if ((st = mv_scratch(ctx, "match.vbits", sizeof(uint32_t) * (size_t)n_frames * g.vwords, &vb))) return st;
  if ((st = mv_scratch(ctx, "match.c_cell", sizeof(int32_t) * (size_t)n_frames * g.cstride, &ccell))) return st;
  if ((st = mv_scratch(ctx, "match.c_col", sizeof(int32_t) * (size_t)n_frames * (g.cols + 1), &ccol))) return st;
  if ((st = mv_scratch(ctx, "match.c_desc", cdesc_rows * 64, &cdesc))) return st;
  if ((st = mv_scratch(ctx, "match.c_ytab", sizeof(uint32_t) * ((size_t)n_frames * g.nblk + 16) * g.ystride, &cytab))) return st;
  if ((st = mv_scratch(ctx, "match.qa", qa_rows * 64, &qa))) return st;
  if ((st = mv_scratch(ctx, "match.rowinfo", qa_rows * 32, &rinfo))) return st;
  if ((st = mv_scratch(ctx, "match.tc_spans", sizeof(int4) * (size_t)g.n_items, &spans))) return st;
  if ((st = mv_abort_flag(ctx, &flag))) return st;

  CUtensorMap tmap_a, tmap_b;
  {
    const cuuint32_t es[2] = {1, 1};
    const cuuint64_t dims_a[2] = {64, (cuuint64_t)qa_rows}, dims_b[2] = {64, (cuuint64_t)cdesc_rows};
    const cuuint64_t strides[1] = {64};
    const cuuint32_t box_a[2] = {64, kTileQ}, box_b[2] = {64, kChunkN};
    CUresult cr = encode(&tmap_a, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, qa, dims_a, strides, box_a, es,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (cr == CUDA_SUCCESS)
      cr = encode(&tmap_b, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, cdesc, dims_b, strides, box_b, es,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (cr != CUDA_SUCCESS) {
      snprintf(ctx->err, sizeof(ctx->err), "cuTensorMapEncodeTiled failed (%d)", (int)cr);
      return MV_ERR_CUDA;
    }
  }

  mv_prof_scope ps(ctx, "match");
  {
    mv_prof_scope p1(ctx, "match_compact");
    compact_candidates_kernel<<<n_frames, 256, sizeof(int) * (size_t)(g.cols + 1 + g.vwords), ctx->stream>>>(
        g, d_max_idx, d_prob, d_desc, (uint32_t*)vb, (int32_t*)ccell, (int32_t*)ccol, (int8_t*)cdesc, (uint32_t*)cytab);
    MV_CHECK_LAUNCH(ctx);
  }
  MV_CUDA(ctx, cudaMemsetAsync(spans, 0, sizeof(int4) * (size_t)g.n_items, ctx->stream));
  {
    mv_prof_scope p2(ctx, "match_lead");
    lead_kernel<<<g.n_items * kLeadParts, kLeadThreads, sizeof(uint32_t) * (size_t)(g.vwords + g.cols + 1), ctx->stream>>>(g, d_f0, d_f1, d_desc, (const uint32_t*)vb,
                                                           (const int32_t*)ccol, d_q_patch, d_q_count, (int8_t*)qa,
                                                           (int4*)rinfo, (int4*)spans);
    MV_CHECK_LAUNCH(ctx);
  }
  {
    mv_prof_scope p3(ctx, "match_gemm");
    const size_t smem = tc_smem(g);
    // The limit is an attribute of the kernel in the device's primary context, which every mv_ctx on that device
    // shares: set to this call's size, it could drop under the size another thread's context is about to launch
    // with.  So every context sets the same bound, the most any launch needs, once.
    if (!ctx->tc_smem_attr_set) {
      MV_CUDA(ctx, cudaFuncSetAttribute(match_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTcSmemMax));
      ctx->tc_smem_attr_set = true;
    }
    const int grid = g.n_items < ctx->sm_count ? g.n_items : ctx->sm_count;
    match_tc_kernel<<<grid, kThreads, smem, ctx->stream>>>(tmap_a, tmap_b, g, d_f0, (const int4*)rinfo,
                                                          (const uint32_t*)cytab, (const int4*)spans, d_best_rank,
                                                          d_best_score, (size_t)n_pairs * (size_t)top_n, flag);
    MV_CHECK_LAUNCH(ctx);
  }
  *d_rank_to_cell = (const int32_t*)ccell;
  *rank_stride = g.cstride;
  ctx->match_items = g.n_items;
  return MV_OK;
}

// Executed work of the last tensor-core matcher launch on this context: tiles with at least one query and the
// 128 x 256 x 64 chunks the tensor pipe ran for them (bench.py's `bound: tensor` roofline entry).
extern "C" mv_status mv_ctx_match_work(mv_ctx* ctx, unsigned long long* tiles, unsigned long long* chunks) {
  if (!tiles || !chunks) return MV_ERR_BAD_ARG;
  MV_ENTER(ctx);
  *tiles = *chunks = 0;
  if (ctx->match_items <= 0) return MV_OK;
  void* spans = nullptr;
  mv_status st = mv_scratch(ctx, "match.tc_spans", sizeof(int4) * (size_t)ctx->match_items, &spans);
  if (st) return st;
  std::vector<int4> h((size_t)ctx->match_items);
  MV_CUDA(ctx, cudaMemcpyAsync(h.data(), spans, sizeof(int4) * h.size(), cudaMemcpyDeviceToHost, ctx->stream));
  MV_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  for (const int4& sp : h) {
    if (sp.x <= 0) continue;
    *tiles += 1;
    const int lo = 0x7fffffff - sp.y, hi = sp.z;
    if (hi > lo) *chunks += (unsigned long long)((hi - (lo & ~31) + kChunkN - 1) / kChunkN);
  }
  return MV_OK;
}
