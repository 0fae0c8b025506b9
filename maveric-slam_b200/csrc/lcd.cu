// lcd.cu -- loop-closure candidates: the BoW similarity of every frame of a call against every earlier frame of
// that call on the 5th-generation tensor cores, per-frame top-k selection, and the idf word weights.
//
// Definition (this library's; the reference's lcd_main.c intersects sorted BoW id lists, which this equals with
// unit weights on duplicate-free lists -- PARITY UNPINNED beyond that):
//   P[f][w] = 1 where word w in [0, n_words) occurs among frame f's first min(q_count, top_n) queries
//   score(i, j) = sum_w weight[w] * P[i][w] * P[j][w]           int32, weight in [0, 127]
//   candidates of i: j <= i - min_gap with score >= min_score, best k by score, ties to the smaller j
//
// Kernels
//   presence_kernel   scatter of the word lists into P (int8, [frames padded to 128][n_words padded to 64],
//                     K-major) and, with weights, into PW = P * weight; both are exact in int8 (without weights
//                     PW is P itself)
//   lcd_tile_kernel   one CTA per 128 x 128 tile of the allowed lower triangle: TMA boxes [64 B][128 frames] of PW
//                     (A, rows i) and P (B, columns j), SWIZZLE_64B, two tcgen05.mma.kind::i8 (K = 32) per box into
//                     one 128-column int32 TMEM accumulator; the epilogue (thread = row i) masks j > i - min_gap and
//                     keeps the row's best 8 of the tile's 128 columns
//   lcd_merge_kernel  per row, the tiles' lists merged into the row's best k
// The score matrix never leaves TMEM: the only global output of the tile kernel is 8 entries per row and tile.
#include "mv_common.cuh"
#include "sm100_ptx.cuh"

#include <math.h>

namespace {

using namespace sm100;

constexpr int kTile = 128;                        // frames per tile side: UMMA M = N = 128
constexpr int kKBlock = 64;                       // words per TMA box row (64 bytes, two K = 32 MMAs)
constexpr int kStages = 4;
constexpr int kOpBytes = kTile * kKBlock;         // one operand's box
constexpr int kStageBytes = 2 * kOpBytes;
constexpr int kThreads = 128;                     // four warps: TMEM lane quadrants 0..3
constexpr int kSlots = 8;                         // the most candidates per frame
constexpr size_t kTileSmem = 1024 + (size_t)kStages * kStageBytes;

struct LcdGeom {
  int n, kpad, min_gap, k, min_score, n_col_tiles;
};

// column tiles of row tile ti that hold an allowed pair (j <= i - min_gap for some row i < n of the tile)
__host__ __device__ __forceinline__ int lcd_col_tiles(int ti, int n, int min_gap) {
  const int max_i = min(ti * kTile + kTile - 1, n - 1);
  return max_i >= min_gap ? (max_i - min_gap) / kTile + 1 : 0;
}

// A sorted list of the best kSlots (score descending, j ascending), j = -1 marks an empty slot.  Entries arrive in
// ascending j, so a strict '>' leaves an equal score behind the entries already there.
struct TopList {
  int s[kSlots], j[kSlots];
  __device__ __forceinline__ void clear() {
#pragma unroll
    for (int r = 0; r < kSlots; r++) { s[r] = 0; j[r] = -1; }
  }
  __device__ __forceinline__ void insert(int sc, int jj) {
#pragma unroll
    for (int r = kSlots - 1; r >= 0; r--) {
      const bool before_r = j[r] < 0 || sc > s[r];
      const bool before_prev = r > 0 && (j[r - 1] < 0 || sc > s[r - 1]);
      if (before_r) {
        s[r] = before_prev ? s[r - 1] : sc;
        j[r] = before_prev ? j[r - 1] : jj;
      }
    }
  }
};

__global__ void presence_kernel(int n, int top_n, int n_words, int kpad, const int32_t* __restrict__ word,
                                const int32_t* __restrict__ q_count, const int8_t* __restrict__ weight,
                                int8_t* __restrict__ P, int8_t* __restrict__ PW) {
  const int f = blockIdx.y;
  const int nq = min(max(q_count[f], 0), top_n);
  for (int q = blockIdx.x * blockDim.x + threadIdx.x; q < nq; q += gridDim.x * blockDim.x) {
    const int w = word[(size_t)f * top_n + q];
    if (w < 0 || w >= n_words) continue;
    const size_t o = (size_t)f * kpad + w;
    P[o] = 1;   // duplicates write the same byte
    if (PW) PW[o] = weight[w];
  }
}

// weight[w] = df ? rint(127 ln(n / df) / ln(n)) : 0 in double, df = frames whose presence row holds w
__global__ void word_weights_kernel(int n, int n_words, int kpad, const int8_t* __restrict__ P,
                                    int8_t* __restrict__ weight) {
  const int w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= n_words) return;
  int df = 0;
  for (int f = 0; f < n; f++) df += P[(size_t)f * kpad + w];
  weight[w] = df ? (int8_t)rint(127.0 * log((double)n / (double)df) / log((double)n)) : (int8_t)0;
}

__global__ void __launch_bounds__(kThreads)
lcd_tile_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b, LcdGeom g,
                int2* __restrict__ part, int* abort_flag) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  __shared__ uint64_t bar_full[kStages], bar_empty[kStages], bar_done;
  __shared__ uint32_t s_tmem_base;

  // this CTA's tile: the allowed tiles listed row tile by row tile
  int t = blockIdx.x, ti = 0;
  for (;; ti++) {
    const int c = lcd_col_tiles(ti, g.n, g.min_gap);
    if (t < c) break;
    t -= c;
  }
  const int tj = t;
  const int kblocks = g.kpad / kKBlock;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int s = 0; s < kStages; s++) { mbar_init(smem_u32(&bar_full[s]), 1); mbar_init(smem_u32(&bar_empty[s]), 1); }
    mbar_init(smem_u32(&bar_done), 1);
    mbar_fence_init();
    tma_prefetch_desc(&tmap_a);
    tma_prefetch_desc(&tmap_b);
  }
  if (warp == 1) {
    tmem_alloc(smem_u32(&s_tmem_base), kTile);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = s_tmem_base;

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer
    if (lane == 0) {
      for (int kb = 0; kb < kblocks; kb++) {
        const uint32_t s = kb % kStages, ph = (kb / kStages) & 1;
        mbar_wait(smem_u32(&bar_empty[s]), ph ^ 1, abort_flag, 1, 64);
        mbar_expect_tx(smem_u32(&bar_full[s]), kStageBytes);
        uint8_t* st = smem + s * kStageBytes;
        tma_load_2d(smem_u32(st), &tmap_a, smem_u32(&bar_full[s]), kb * kKBlock, ti * kTile);
        tma_load_2d(smem_u32(st + kOpBytes), &tmap_b, smem_u32(&bar_full[s]), kb * kKBlock, tj * kTile);
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer
    if (lane == 0) {
      const uint32_t idesc = umma_idesc_s8(kTile, kTile);
      for (int kb = 0; kb < kblocks; kb++) {
        const uint32_t s = kb % kStages, ph = (kb / kStages) & 1;
        mbar_wait(smem_u32(&bar_full[s]), ph, abort_flag, 2);
        tc_fence_after();
        const uint32_t a = smem_u32(smem + s * kStageBytes), b = a + kOpBytes;
        umma_s8(tmem_base, umma_desc_k_sw64(a), umma_desc_k_sw64(b), idesc, kb > 0 ? 1u : 0u);
        umma_s8(tmem_base, umma_desc_k_sw64(a + 32), umma_desc_k_sw64(b + 32), idesc, 1u);
        umma_commit(smem_u32(&bar_empty[s]));
      }
      umma_commit(smem_u32(&bar_done));
    }
    __syncwarp();
  }

  // ------------------------------------------------------------ epilogue: thread = row i of the tile
  mbar_wait(smem_u32(&bar_done), 0, abort_flag, 3);
  tc_fence_after();
  const int i = ti * kTile + warp * 32 + lane;
  TopList top;
  top.clear();
  const uint32_t t_row = tmem_base + ((uint32_t)(warp * 32) << 16);
  for (int b = 0; b < kTile / 32; b++) {
    int v[32];
    tmem_ld_32x32(t_row + 32 * b, v);
    tmem_ld_wait();
    const int j0 = tj * kTile + 32 * b;
#pragma unroll
    for (int c = 0; c < 32; c++)
      if (i < g.n && i - (j0 + c) >= g.min_gap && v[c] >= g.min_score) top.insert(v[c], j0 + c);
  }
  if (i < g.n) {
    int2* out = part + ((size_t)i * g.n_col_tiles + tj) * g.k;
#pragma unroll
    for (int r = 0; r < kSlots; r++)
      if (r < g.k) out[r] = make_int2(top.s[r], top.j[r]);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, kTile);
}

__global__ void lcd_merge_kernel(LcdGeom g, int first_frame, const int2* __restrict__ part, int32_t* __restrict__ cand,
                                 int32_t* __restrict__ score) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= g.n) return;
  TopList top;
  top.clear();
  const int nct = lcd_col_tiles(i / kTile, g.n, g.min_gap);
  for (int tj = 0; tj < nct; tj++) {
    const int2* in = part + ((size_t)i * g.n_col_tiles + tj) * g.k;
    for (int r = 0; r < g.k; r++) {
      const int2 e = in[r];
      if (e.y < 0) break;
      top.insert(e.x, e.y);
    }
  }
#pragma unroll
  for (int r = 0; r < kSlots; r++)
    if (r < g.k) {
      cand[(size_t)i * g.k + r] = top.j[r] >= 0 ? first_frame + top.j[r] : -1;
      score[(size_t)i * g.k + r] = top.j[r] >= 0 ? top.s[r] : 0;
    }
}

// P of the call's frames, and PW = P * weight where d_weight is given (else *PW = NULL: PW would equal P), zero-padded
// to [rows_pad][kpad]
mv_status lcd_presence(mv_ctx* ctx, int n, int rows_pad, int kpad, int top_n, int n_words, const int32_t* d_word,
                       const int32_t* d_q_count, const int8_t* d_weight, int8_t** P, int8_t** PW) {
  void *vp, *vw = nullptr;
  mv_status st;
  const size_t bytes = (size_t)rows_pad * kpad;
  if ((st = mv_scratch(ctx, "lcd.P", bytes, &vp))) return st;
  if (d_weight && (st = mv_scratch(ctx, "lcd.PW", bytes, &vw))) return st;
  MV_CUDA(ctx, cudaMemsetAsync(vp, 0, bytes, ctx->stream));
  if (vw) MV_CUDA(ctx, cudaMemsetAsync(vw, 0, bytes, ctx->stream));
  dim3 grid((top_n + 255) / 256 < 8 ? (top_n + 255) / 256 : 8, n);
  presence_kernel<<<grid, 256, 0, ctx->stream>>>(n, top_n, n_words, kpad, d_word, d_q_count, d_weight, (int8_t*)vp,
                                                 (int8_t*)vw);
  MV_CHECK_LAUNCH(ctx);
  *P = (int8_t*)vp;
  *PW = (int8_t*)vw;
  return MV_OK;
}

int lcd_kpad(int n_words) { return (n_words + kKBlock - 1) / kKBlock * kKBlock; }

}  // namespace

// Refusals of mv_loop_candidates (and of the candidate stage of mv_detect_loops), before anything is enqueued.
// A device weight vector is read back once to check its sign: weights are data, and a negative one would make
// P * weight signed, which the definition excludes.
mv_status mv_loop_candidates_check(mv_ctx* ctx, const char* fn, int n_frames, int first_frame, int top_n, int n_words,
                                   const int8_t* d_weight, int min_gap, int k) {
  auto refuse = [&](const char* why) {
    snprintf(ctx->err, sizeof(ctx->err), "bad argument: %s: %s", fn, why);
    return MV_ERR_BAD_ARG;
  };
  if (n_frames < 1 || n_frames > 65535) return refuse("n_frames in [1, 65535]");
  if (top_n <= 0) return refuse("top_n must be positive");
  if (n_words <= 0 || n_words > (1 << 24)) return refuse("n_words in [1, 2^24] (an int32 score of weights <= 127)");
  if (k < 1 || k > kSlots) return refuse("k in [1, 8]");
  if (min_gap < 0) return refuse("min_gap must be >= 0");
  if ((long long)first_frame + n_frames - 1 > 0x7fffffffLL) return refuse("first_frame + n_frames - 1 must fit an int32");
  if ((long long)n_frames * top_n >= (1ll << 31)) return refuse("n_frames * top_n must be below 2^31");
  if (!mv_get_tmap_encode()) return refuse("the driver has no cuTensorMapEncodeTiled");
  if (d_weight) {
    void* h;
    mv_status st;
    if ((st = mv_pinned(ctx, (size_t)n_words, &h))) return st;
    MV_CUDA(ctx, cudaMemcpyAsync(h, d_weight, (size_t)n_words, cudaMemcpyDeviceToHost, ctx->stream));
    MV_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    const int8_t* w = (const int8_t*)h;
    for (int i = 0; i < n_words; i++)
      if (w[i] < 0) return refuse("a negative word weight (weights are in [0, 127])");
  }
  return MV_OK;
}

// The candidate stage after mv_loop_candidates_check: presence, tiles, merge.
mv_status mv_loop_candidates_impl(mv_ctx* ctx, int n_frames, int first_frame, int top_n, int n_words,
                                  const int32_t* d_word, const int32_t* d_q_count, const int8_t* d_weight, int min_gap,
                                  int k, int min_score, int32_t* d_cand, int32_t* d_score) {
  LcdGeom g;
  g.n = n_frames; g.kpad = lcd_kpad(n_words); g.min_gap = min_gap; g.k = k; g.min_score = min_score;
  g.n_col_tiles = (n_frames + kTile - 1) / kTile;
  const int rows_pad = g.n_col_tiles * kTile;
  long long n_tiles = 0;
  for (int ti = 0; ti < g.n_col_tiles; ti++) n_tiles += lcd_col_tiles(ti, n_frames, min_gap);

  mv_prof_scope ps(ctx, "lcd");
  int8_t *P = nullptr, *PW = nullptr;
  void* part = nullptr;
  int* flag = nullptr;
  mv_status st;
  if ((st = lcd_presence(ctx, n_frames, rows_pad, g.kpad, top_n, n_words, d_word, d_q_count, d_weight, &P, &PW)))
    return st;
  if ((st = mv_scratch(ctx, "lcd.part", sizeof(int2) * (size_t)n_frames * g.n_col_tiles * k, &part))) return st;
  if ((st = mv_abort_flag(ctx, &flag))) return st;
  if (n_tiles > 0) {
    mv_tmap_encode_fn encode = mv_get_tmap_encode();
    CUtensorMap tmap_a, tmap_b;
    const cuuint32_t es[2] = {1, 1};
    const cuuint64_t dims[2] = {(cuuint64_t)g.kpad, (cuuint64_t)rows_pad};
    const cuuint64_t strides[1] = {(cuuint64_t)g.kpad};
    const cuuint32_t box[2] = {kKBlock, kTile};
    CUresult cr = encode(&tmap_a, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, PW ? PW : P, dims, strides, box, es,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (cr == CUDA_SUCCESS)
      cr = encode(&tmap_b, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, P, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (cr != CUDA_SUCCESS) {
      snprintf(ctx->err, sizeof(ctx->err), "cuTensorMapEncodeTiled failed (%d)", (int)cr);
      return MV_ERR_CUDA;
    }
    // every context sets the same bound, once (the attribute is shared by all contexts of the device)
    if (!ctx->lcd_smem_attr_set) {
      MV_CUDA(ctx, cudaFuncSetAttribute(lcd_tile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTileSmem));
      ctx->lcd_smem_attr_set = true;
    }
    mv_prof_scope pt(ctx, "lcd_tiles");
    lcd_tile_kernel<<<(unsigned)n_tiles, kThreads, kTileSmem, ctx->stream>>>(tmap_a, tmap_b, g, (int2*)part, flag);
    MV_CHECK_LAUNCH(ctx);
  }
  lcd_merge_kernel<<<(n_frames + 127) / 128, 128, 0, ctx->stream>>>(g, first_frame, (const int2*)part, d_cand, d_score);
  MV_CHECK_LAUNCH(ctx);
  return MV_OK;
}

extern "C" mv_status mv_loop_candidates(mv_ctx* ctx, int n_frames, int first_frame, int top_n, int n_words,
                                        const int32_t* d_word, const int32_t* d_q_count, const int8_t* d_weight,
                                        int min_gap, int k, int min_score, int32_t* d_cand, int32_t* d_score) {
  MV_ENTER(ctx);
  if (!d_word || !d_q_count || !d_cand || !d_score) MV_BAD_ARG(ctx, "mv_loop_candidates: NULL buffer");
  mv_status st = mv_loop_candidates_check(ctx, "mv_loop_candidates", n_frames, first_frame, top_n, n_words, d_weight,
                                          min_gap, k);
  if (st) return st;
  return mv_loop_candidates_impl(ctx, n_frames, first_frame, top_n, n_words, d_word, d_q_count, d_weight, min_gap, k,
                                 min_score, d_cand, d_score);
}

extern "C" mv_status mv_lcd_word_weights(mv_ctx* ctx, int n_frames, int top_n, int n_words, const int32_t* d_word,
                                         const int32_t* d_q_count, int8_t* d_weight) {
  MV_ENTER(ctx);
  if (!d_word || !d_q_count || !d_weight) MV_BAD_ARG(ctx, "mv_lcd_word_weights: NULL buffer");
  if (n_frames < 2 || n_frames > 65535 || top_n <= 0 || n_words <= 0 || n_words > (1 << 24) ||
      (long long)n_frames * top_n >= (1ll << 31))
    MV_BAD_ARG(ctx, "mv_lcd_word_weights: n_frames in [2, 65535], top_n > 0, n_words in [1, 2^24]");
  const int kpad = lcd_kpad(n_words);
  int8_t *P = nullptr, *PW = nullptr;
  mv_status st;
  if ((st = lcd_presence(ctx, n_frames, n_frames, kpad, top_n, n_words, d_word, d_q_count, nullptr, &P, &PW)))
    return st;
  word_weights_kernel<<<(n_words + 255) / 256, 256, 0, ctx->stream>>>(n_frames, n_words, kpad, P, d_weight);
  MV_CHECK_LAUNCH(ctx);
  return MV_OK;
}
