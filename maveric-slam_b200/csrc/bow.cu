// bow.cu -- SURVEY §8f rank 3: bag-of-words word assignment of the query descriptors (src/bow_main.c:62-125)
// and the landmark table it feeds, the device-side contents of the reference's local feature pool
// (include/local_feature_pool.h:16-62, driven as in src/local_feature_matching.c:153-163).
//
// Word assignment.  bow_main.c has no defined result as shipped (it crashes; every stage reads memory as
// the wrong type: int8 arrays through the float matmul shim :81-86, an int8 row as int* :105, 8 ints of a
// 4-int leaf :115), so the arithmetic is the definition STATED HERE (DESIGN.md 4.6) -- PARITY
// UNPINNED as a whole; its two helpers (get_binary_descriptor :13-41, count_matching_bits :43-55) are
// pinned to the reference's own functions:
//     raw_j   = sum_k desc[k] * base[k][j]                  int32 (dp4a)
//     m_j     = sat_int8(rint(desc_scale * raw_j / 256))
//     score_j = scale[j] * m_j + 256 * bias[j]              fp32, unfused
//     base    = first j whose score exceeds 0 and every earlier score
//     bits    = one bit per descriptor element (> 0, or <= 0 for a non-positive scale), 8 words, MSB first
//     wid     = first leaf of `base` with the most matching bits over 8 words of the FLAT leaf array
// Bound: HBM -- 256 B read per query, 10 + 1000 x 8 word operations on it: ten output columns are no
// tensor-core shape, and the Hamming search is 32 bit-products per XOR/POPC, 30x cheaper than an int8
// GEMM of the same comparison.  One persistent CTA per SM holds the whole vocabulary (160 KB of leaves)
// in shared memory; eight lanes per query, lane l <-> bytes 32l..32l+31 <-> bit word l <-> leaves l, l+8, ...
//
// Landmark table.  The reference's pool is an open-addressing hash table whose slot layout depends on the
// insertion order; its CONTENTS are a map word id -> LocalFeature.  Word ids are bounded (base x leaf), so
// on the device the map is direct: table[word id], 56-byte records of the reference's layout.  A frame's
// observations are one launch (insert-or-update per word, duplicates of a word applied as often as they
// occur, coordinates taken from the first), ageing is one launch over the table.
#include "mv_common.cuh"

#include <algorithm>

namespace {

constexpr int kBowThreads = 1024;   // 32 warps: the leaf search is POPC-bound (a quarter-rate pipe); one CTA per SM holds the vocabulary
constexpr int kBowLanes = 8;     // lanes per query

struct BowVocabDev {
  int n_base, wpb;
  const int8_t* base_t;     // [n_base][256]  (transposed: a column of vocabulary.h:11 contiguous)
  const float* scale;       // [n_base]
  const float* bias;        // [n_base]
  const int32_t* leaves;    // [n_base * wpb * 4 + 4], the last 4 zero
};

__global__ void __launch_bounds__(kBowThreads, 1)
bow_assign_kernel(BowVocabDev v, int n_frames, int cells, int top_n, const int8_t* __restrict__ desc,
                  const float* __restrict__ desc_scale, const int32_t* __restrict__ q_patch,
                  const int32_t* __restrict__ q_count, int32_t* __restrict__ word, int32_t* __restrict__ base_out,
                  MvBackProject bp) {
  extern __shared__ __align__(16) uint8_t s_raw[];
  int32_t* s_leaves = reinterpret_cast<int32_t*>(s_raw);
  const int n_leaf_ints = v.n_base * v.wpb * 4 + 4;
  int8_t* s_base = reinterpret_cast<int8_t*>(s_leaves + ((n_leaf_ints + 3) & ~3));
  float* s_scale = reinterpret_cast<float*>(s_base + v.n_base * 256);
  float* s_bias = s_scale + v.n_base;
  for (int i = threadIdx.x; i < n_leaf_ints; i += kBowThreads) s_leaves[i] = v.leaves[i];
  for (int i = threadIdx.x; i < v.n_base * 64; i += kBowThreads)
    reinterpret_cast<int32_t*>(s_base)[i] = reinterpret_cast<const int32_t*>(v.base_t)[i];
  for (int i = threadIdx.x; i < v.n_base; i += kBowThreads) { s_scale[i] = v.scale[i]; s_bias[i] = v.bias[i]; }
  __syncthreads();

  const int lane = threadIdx.x & 31, sub = threadIdx.x & 7, q0 = lane & ~7;
  const long long total = (long long)n_frames * top_n;
  const int per_cta = kBowThreads / kBowLanes;
  for (long long g0 = (long long)blockIdx.x * per_cta; g0 < total; g0 += (long long)gridDim.x * per_cta) {
    const long long g = g0 + (threadIdx.x >> 3);
    const bool in = g < total;
    const int f = in ? (int)(g / top_n) : 0, q = in ? (int)(g - (long long)f * top_n) : 0;
    const bool active = in && q < min(q_count[f], top_n);
    int4 d[2] = {make_int4(0, 0, 0, 0), make_int4(0, 0, 0, 0)};
    float ds = 1.0f;
    const int cell = active ? q_patch[(size_t)f * top_n + q] : 0;
    if (active) {
      const int4* p = reinterpret_cast<const int4*>(desc + ((size_t)f * cells + cell) * 256 + sub * 32);
      d[0] = __ldg(p); d[1] = __ldg(p + 1);
      ds = desc_scale[f];
    }
    const int dw[8] = {d[0].x, d[0].y, d[0].z, d[0].w, d[1].x, d[1].y, d[1].z, d[1].w};
    // ---- base node (bow_main.c:81-101)
    int sel = 0;
    float max_score = 0.0f;
    for (int j = 0; j < v.n_base; j++) {
      const int32_t* bj = reinterpret_cast<const int32_t*>(s_base + j * 256 + sub * 32);
      int raw = 0;
#pragma unroll
      for (int k = 0; k < 8; k++) raw = __dp4a(dw[k], bj[k], raw);
      raw += __shfl_xor_sync(0xffffffffu, raw, 1);
      raw += __shfl_xor_sync(0xffffffffu, raw, 2);
      raw += __shfl_xor_sync(0xffffffffu, raw, 4);
      float m = rintf(__fmul_rn(__fmul_rn(ds, __int2float_rn(raw)), 1.0f / 256.0f));
      m = m > 127.0f ? 127.0f : m;
      m = m < -128.0f ? -128.0f : m;
      if (m != m) m = 0.0f;
      const float score = __fadd_rn(__fmul_rn(s_scale[j], m), __fmul_rn(256.0f, s_bias[j]));
      if (score > max_score) { max_score = score; sel = j; }
    }
    // ---- binary descriptor (bow_main.c:13-41): this lane's 32 elements are word `sub`, MSB first
    unsigned mine = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) {
#pragma unroll
      for (int b = 0; b < 4; b++) {
        const int e = (int)(int8_t)(dw[k] >> (8 * b));
        const bool bit = ds > 0.0f ? (e > 0) : (e <= 0);
        mine = (mine << 1) | (bit ? 1u : 0u);
      }
    }
    unsigned bits[8];
#pragma unroll
    for (int i = 0; i < 8; i++) bits[i] = __shfl_sync(0xffffffffu, mine, q0 + i);
    // ---- leaves of the base node (bow_main.c:106-120): 8 words of the flat array per leaf
    int best_d = 0x7fffffff, best_w = 0;
    const int4* lf = reinterpret_cast<const int4*>(s_leaves) + (size_t)sel * v.wpb;
    for (int w = sub; w < v.wpb; w += kBowLanes) {
      const int4 a = lf[w], b = lf[w + 1];
      // Hamming distance over 8 words with 4 POPC instead of 8 (POPC runs at a quarter of the integer rate and
      // bounds this loop): a carry-save adder tree (Harley-Seal) leaves the bit counts' ones / twos / fours /
      // eights planes, each a LOP3
      const unsigned x0 = bits[0] ^ (unsigned)a.x, x1 = bits[1] ^ (unsigned)a.y, x2 = bits[2] ^ (unsigned)a.z,
                     x3 = bits[3] ^ (unsigned)a.w, x4 = bits[4] ^ (unsigned)b.x, x5 = bits[5] ^ (unsigned)b.y,
                     x6 = bits[6] ^ (unsigned)b.z, x7 = bits[7] ^ (unsigned)b.w;
      const unsigned s1 = x0 ^ x1 ^ x2, c1 = (x0 & x1) | (x2 & (x0 ^ x1));
      const unsigned s2 = x3 ^ x4 ^ x5, c2 = (x3 & x4) | (x5 & (x3 ^ x4));
      const unsigned s3 = s1 ^ s2 ^ x6, c3 = (s1 & s2) | (x6 & (s1 ^ s2));
      const unsigned ones = s3 ^ x7, c4 = s3 & x7;
      const unsigned t1 = c1 ^ c2 ^ c3, d1 = (c1 & c2) | (c3 & (c1 ^ c2));
      const unsigned twos = t1 ^ c4, d2 = t1 & c4;
      const unsigned fours = d1 ^ d2, eights = d1 & d2;
      const int dist = __popc(ones) + 2 * __popc(twos) + 4 * __popc(fours) + 8 * __popc(eights);
      if (dist < best_d) { best_d = dist; best_w = w; }   // matching bits = 256 - dist; strict >: the first one
    }
#pragma unroll
    for (int o = 1; o < 8; o <<= 1) {
      const int od = __shfl_xor_sync(0xffffffffu, best_d, o), ow = __shfl_xor_sync(0xffffffffu, best_w, o);
      if (od < best_d || (od == best_d && ow < best_w)) { best_d = od; best_w = ow; }
    }
    if (best_d >= 256) best_w = 0;   // no matching bit at all: best_match stays 0 and best_wid 0 (:108-109)
    if (in && sub == 0) {
      word[g] = active ? sel * v.wpb + best_w : -1;
      if (base_out) base_out[g] = active ? sel : -1;
    }
    if (bp.coords && in && sub == 1) {   // the query keypoint back-projected as build_corr_kernel does (pnp_gn.cu)
      float X = 0.0f, Y = 0.0f, Z = 0.0f;
      if (active) {
        const int idx = bp.q_idx[g];
        const float x = (float)((cell / bp.rows) * 8 + idx % 8), y = (float)((cell % bp.rows) * 8 + idx / 8);
        Z = bp.depth[(size_t)f * cells + cell];
        X = __fmul_rn(__fdiv_rn(__fsub_rn(x, bp.cx), bp.fx), Z);
        Y = __fmul_rn(__fdiv_rn(__fsub_rn(y, bp.cy), bp.fy), Z);
      }
      bp.coords[3 * g] = X; bp.coords[3 * g + 1] = Y; bp.coords[3 * g + 2] = Z;
    }
  }
}

// ------------------------------------------------------------------------------------ landmark table
__global__ void landmarks_init_kernel(int n_words, mv_landmark* __restrict__ table, int32_t* __restrict__ first,
                                      int32_t* __restrict__ cnt) {
  const int w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= n_words) return;
  if (table) {
    mv_landmark z;
    z.word_id = -1; z.frame_ptr = 0; z.num_frames = 0;
    for (int i = 0; i < 8; i++) z.frames[i] = 0;
    z.coords[0] = z.coords[1] = z.coords[2] = 0.0f;
    table[w] = z;
  }
  if (first) { first[w] = 0x7fffffff; cnt[w] = 0; }
}

__global__ void landmarks_mark_kernel(int n_words, int n, const int32_t* __restrict__ ids, int32_t* __restrict__ first,
                                      int32_t* __restrict__ cnt) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int w = ids[i];
  if (w < 0 || w >= n_words) return;
  atomicMin(&first[w], i);
  atomicAdd(&cnt[w], 1);
}

// local_feature_matching.c:153-161 for one word that occurs k >= 1 times in a frame's list: insert
// (init_local_feature_with_id, local_feature_pool.h:31-36, coordinates of the first occurrence) or update
// (update_local_feature, :38-48), once per occurrence.  Shared by the per-frame kernel and the sequence walk.
__device__ __forceinline__ void landmark_observe(mv_landmark& f, int w, int frame, int k, const float* coords) {
  if (f.word_id == -1) {
    f.word_id = w; f.frame_ptr = 0; f.num_frames = 1; f.frames[0] = frame;
    for (int c = 0; c < 3; c++) f.coords[c] = coords ? coords[c] : 0.0f;
    k--;
  }
  for (; k > 0 && f.num_frames < 8; k--) {
    f.frames[(f.frame_ptr + f.num_frames) % 8] = frame;
    f.num_frames++;
  }
  // a full ring: each further update overwrites the oldest slot and advances frame_ptr, so after 8 of them every
  // slot holds `frame` and the rest only advance frame_ptr
  for (int i = 0; i < k && i < 8; i++) f.frames[(f.frame_ptr + i) % 8] = frame;
  if (k > 0) f.frame_ptr = (f.frame_ptr + k) % 8;
}

// local_feature_pool_remove_old (local_feature_pool.h:268-279) with remove_old_frame (:50-62) on one record: one
// frame older than `keep` leaves, a record without frames is deleted (stale frames[] / coords stay in place)
__device__ __forceinline__ void landmark_remove_old(mv_landmark& f, int keep) {
  if (f.word_id == -1) return;
  int fp = f.frame_ptr, nf = f.num_frames;
  if (f.frames[fp] < keep) { fp = (fp + 1) % 8; nf--; }
  if (nf == 0) { f.word_id = -1; fp = 0; }
  f.frame_ptr = fp; f.num_frames = nf;
}

__global__ void landmarks_apply_kernel(int n_words, mv_landmark* __restrict__ table, int frame, int n,
                                       const int32_t* __restrict__ ids, const float* __restrict__ coords,
                                       int32_t* __restrict__ first, int32_t* __restrict__ cnt) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int w = ids[i];
  if (w < 0 || w >= n_words || first[w] != i) return;
  mv_landmark f = table[w];
  landmark_observe(f, w, frame, cnt[w], coords ? coords + 3 * (size_t)i : nullptr);
  table[w] = f;
  first[w] = 0x7fffffff;   // scratch left clean for the next frame
  cnt[w] = 0;
}

__global__ void landmarks_remove_old_kernel(int n_words, mv_landmark* __restrict__ table, int keep) {
  const int w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= n_words) return;
  landmark_remove_old(table[w], keep);
}

// ---------------------------------------------------------------- the whole sequence's table update
// The table is a direct map word -> record and words never interact, so a sequence of per-frame steps
// (observe frame f, then remove_old(f)) is one independent state machine per word, run over that word's
// occurrences in frame order.  The occurrences are grouped by word with a counting sort whose tiles are blocks of
// `fb` consecutive frames: cnt[t][w] counts word w in tile t, a column scan turns the counts into each tile's
// place inside the word's list, and the scatter walks a tile's frames in order.  Inside one frame the order of
// a word's occurrences is not kept (atomics): it does not matter, one frame's occurrences of a word are one
// observe whose coordinates are those of the smallest query index, and the walk takes that minimum.
__global__ void lmseq_count_kernel(int n_steps, int top_n, int n_words, int fb, const int32_t* __restrict__ word,
                                   const int32_t* __restrict__ q_count, int32_t* __restrict__ cnt,
                                   float* __restrict__ coords_out) {
  const long long total = (long long)n_steps * top_n;
  const int lane = threadIdx.x & 31;
  for (long long b = (long long)blockIdx.x * blockDim.x; b < total; b += (long long)gridDim.x * blockDim.x) {
    const long long g = b + threadIdx.x;
    bool valid = false;
    unsigned long long key = ~0ull;
    if (g < total) {
      const int f = (int)(g / top_n), q = (int)(g - (long long)f * top_n);
      const int w = word[g];
      valid = q < min(q_count[f], top_n) && w >= 0 && w < n_words;
      if (valid) key = (unsigned long long)(f / fb) * n_words + w;
      else { coords_out[3 * g] = 0.0f; coords_out[3 * g + 1] = 0.0f; coords_out[3 * g + 2] = 0.0f; }   // lookup: not found
    }
    const unsigned peers = __match_any_sync(0xffffffffu, key);   // warp-aggregated: hot words are common
    if (valid && lane == __ffs(peers) - 1) atomicAdd(&cnt[key], __popc(peers));
  }
}

// cnt[t][w] -> number of w's occurrences in tiles before t; total[w]
__global__ void lmseq_colscan_kernel(int n_words, int n_tiles, int32_t* __restrict__ cnt, int32_t* __restrict__ total) {
  const int w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= n_words) return;
  int run = 0;
#pragma unroll 8
  for (int t = 0; t < n_tiles; t++) {
    int32_t* p = cnt + (size_t)t * n_words + w;
    const int c = *p;
    *p = run;
    run += c;
  }
  total[w] = run;
}

// exclusive scan of total[0, n) into start[0, n]: one CTA of 1024 threads, a contiguous slice per thread
__global__ void __launch_bounds__(1024) lmseq_wordscan_kernel(int n, const int32_t* __restrict__ total,
                                                              int32_t* __restrict__ start) {
  __shared__ int s_warp[32];
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int per = (n + 1023) / 1024, lo = min(n, tid * per), hi = min(n, lo + per);
  int sum = 0;
  for (int i = lo; i < hi; i++) sum += total[i];
  int incl = sum;
  for (int o = 1; o < 32; o <<= 1) {
    const int v = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += v;
  }
  if (lane == 31) s_warp[wid] = incl;
  __syncthreads();
  if (wid == 0) {
    int v = s_warp[lane];
    for (int o = 1; o < 32; o <<= 1) {
      const int u = __shfl_up_sync(0xffffffffu, v, o);
      if (lane >= o) v += u;
    }
    s_warp[lane] = v;
  }
  __syncthreads();
  int run = incl - sum + (wid > 0 ? s_warp[wid - 1] : 0);
  for (int i = lo; i < hi; i++) { start[i] = run; run += total[i]; }
  if (tid == 1023) start[n] = run;
}

// one CTA per tile: its frames in order, a frame's occurrences at once
__global__ void lmseq_scatter_kernel(int n_steps, int top_n, int n_words, int fb, const int32_t* __restrict__ word,
                                     const int32_t* __restrict__ q_count, int32_t* __restrict__ cnt,
                                     const int32_t* __restrict__ start, int32_t* __restrict__ sorted) {
  const int t = blockIdx.x, lane = threadIdx.x & 31;
  int32_t* row = cnt + (size_t)t * n_words;
  const int f_end = min(n_steps, (t + 1) * fb);
  for (int f = t * fb; f < f_end; f++) {
    const int n = min(q_count[f], top_n);
    for (int q0 = 0; q0 < n; q0 += blockDim.x) {
      const int q = q0 + threadIdx.x;
      const long long g = (long long)f * top_n + q;
      const int w = q < n ? word[g] : -1;
      const bool valid = w >= 0 && w < n_words;
      const unsigned peers = __match_any_sync(0xffffffffu, valid ? w : -1);
      const int leader = __ffs(peers) - 1;
      int base = 0;
      if (valid && lane == leader) base = atomicAdd(&row[w], __popc(peers));
      base = __shfl_sync(0xffffffffu, base, leader);
      if (valid) sorted[start[w] + base + __popc(peers & ((1u << lane) - 1))] = (int32_t)g;
    }
    __syncthreads();   // the next frame's occurrences go after this one's
  }
}

// remove_old(first_frame + k) for k in [from, to) on a record the word's list does not touch there; only a
// step with frames[frame_ptr] < first_frame + k - 7 changes it, so the walk jumps to those (at most 8: each
// removes a frame)
__device__ __forceinline__ void landmark_age(mv_landmark& r, int first_frame, int from, int to) {
  long long k = from;
  while (k < to && r.word_id != -1) {
    const long long need = (long long)r.frames[r.frame_ptr] - first_frame + 8;
    if (need > k) k = need;
    if (k >= to) break;
    landmark_remove_old(r, (int)(first_frame + k - 7));
    k++;
  }
}

// One warp per word, every word (records age while unseen): its list in frame order, one observe per frame, the
// ageing between its frames applied lazily; coords_out of each occurrence = the record's coordinates after that
// frame's step (what mv_landmarks_lookup would return then).  Lists are very uneven (on the bench sequence one
// word holds 95 k of 4.5 M occurrences), so the lanes read and write occurrences 32 at a time and only the
// per-frame state machine is serial: every lane holds the same record and applies the same steps.
constexpr int kWalkWarps = 4;
__global__ void __launch_bounds__(32 * kWalkWarps)
lmseq_walk_kernel(int n_words, mv_landmark* __restrict__ table, int first_frame, int n_steps, int top_n,
                  const int32_t* __restrict__ start, const int32_t* __restrict__ sorted,
                  const float* __restrict__ coords_in, float* __restrict__ coords_out) {
  const int w = blockIdx.x * kWalkWarps + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (w >= n_words) return;   // warp-uniform
  mv_landmark r = table[w];
  int aged = 0;     // steps before `aged` are applied, except the remove_old of the last observed frame
  int cur_f = -1;   // frame of the last observed occurrence
  const int beg = start[w], end = start[w + 1];
  for (int b = beg; b < end; b += 32) {
    const int i = b + lane;
    const bool in = i < end;
    const int g = in ? sorted[i] : 0;
    const int f = in ? g / top_n : 0x7fffffff;
    int prev = __shfl_up_sync(0xffffffffu, f, 1);
    if (lane == 0) prev = cur_f;
    const unsigned fresh = __ballot_sync(0xffffffffu, in && f != prev);   // lanes where a frame's run begins
    const unsigned live = __ballot_sync(0xffffffffu, in);
    float X = 0.0f, Y = 0.0f, Z = 0.0f;
    unsigned segs = (fresh | 1u) & live;   // lane 0 may continue the previous chunk's run
    while (segs) {
      const int s = __ffs(segs) - 1;
      segs &= segs - 1;
      const int e = segs ? __ffs(segs) - 1 : 32;
      const unsigned mask = live & (e == 32 ? 0xffffffffu : (1u << e) - 1) & ~((1u << s) - 1);
      const int fs = __shfl_sync(0xffffffffu, f, s);
      if ((fresh >> s) & 1) {
        landmark_age(r, first_frame, aged, fs);
        aged = cur_f = fs;   // this frame's remove_old comes with the next ageing: it never deletes a record just observed
      }
      const float* ins = nullptr;
      if (r.word_id == -1) {   // an insert takes the coordinates of the run's smallest query: the run may go on past this chunk
        int gm = 0x7fffffff;
        for (int j0 = b + s; j0 < end; j0 += 32) {
          const int j = j0 + lane;
          const int gj = j < end ? sorted[j] : 0;
          const bool same = j < end && gj / top_n == fs;
          if (same) gm = min(gm, gj);
          if (__ballot_sync(0xffffffffu, !same)) break;   // frames are non-decreasing: the run ends here
        }
        for (int o = 16; o > 0; o >>= 1) gm = min(gm, __shfl_xor_sync(0xffffffffu, gm, o));
        ins = coords_in + 3 * (size_t)gm;
      }
      landmark_observe(r, w, first_frame + fs, __popc(mask), ins);
      if ((mask >> lane) & 1) {
        const bool ok = r.word_id == w;
        X = ok ? r.coords[0] : 0.0f; Y = ok ? r.coords[1] : 0.0f; Z = ok ? r.coords[2] : 0.0f;
      }
    }
    if (in) { coords_out[3 * (size_t)g] = X; coords_out[3 * (size_t)g + 1] = Y; coords_out[3 * (size_t)g + 2] = Z; }
  }
  landmark_age(r, first_frame, aged, n_steps);
  if (lane == 0) table[w] = r;
}

__global__ void landmarks_lookup_kernel(int n_words, const mv_landmark* __restrict__ table, int n,
                                        const int32_t* __restrict__ ids, float* __restrict__ coords,
                                        int32_t* __restrict__ found) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int w = ids[i];
  const bool ok = w >= 0 && w < n_words && table[w].word_id == w;
  for (int c = 0; c < 3; c++) coords[3 * (size_t)i + c] = ok ? table[w].coords[c] : 0.0f;
  if (found) found[i] = ok ? 1 : 0;
}

// Matches -> PnP correspondences whose 3-D side comes from the landmark table (local_feature_pool.h:16-22
// `coords_3D`): the matched frame-0 cell is looked up in frame 0's query list (ascending cells: binary search),
// its word in the table.  A match whose cell is no query of frame 0, or whose word has no landmark, gets NaN
// coordinates: the Gauss-Newton gate never accepts it, the correspondence lists keep their order and length.
// With occ_coords (the sequence path) the table is not read: occ_coords [frame][query][3] already holds the
// coordinates of each query's record after its frame's step, and a query's word in range always has a record then.
__global__ void build_corr_landmarks_kernel(int n_words, const mv_landmark* __restrict__ table, int top_n, int stride,
                                            const int32_t* __restrict__ f0_of, const int32_t* __restrict__ q_patch,
                                            const int32_t* __restrict__ q_count, const int32_t* __restrict__ word,
                                            const float* __restrict__ match_pts, const int32_t* __restrict__ match_count,
                                            const int32_t* __restrict__ match_cell0, float* __restrict__ corr,
                                            int32_t* __restrict__ n_with_landmark, const float* __restrict__ occ_coords) {
  const int pair = blockIdx.y;
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= match_count[pair]) return;
  const int f0 = f0_of ? f0_of[pair] : pair;
  const int cell = match_cell0[(size_t)pair * stride + j];
  const int32_t* qp = q_patch + (size_t)f0 * top_n;
  int lo = 0, hi = min(q_count[f0], top_n);
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (qp[mid] < cell) lo = mid + 1; else hi = mid;
  }
  const float qnan = __int_as_float(0x7fc00000);
  float X = qnan, Y = qnan, Z = qnan;
  if (lo < min(q_count[f0], top_n) && qp[lo] == cell) {
    const size_t o = (size_t)f0 * top_n + lo;
    const int w = word[o];
    if (occ_coords) {
      if (w >= 0 && w < n_words) {
        X = occ_coords[3 * o]; Y = occ_coords[3 * o + 1]; Z = occ_coords[3 * o + 2];
        if (n_with_landmark) atomicAdd(&n_with_landmark[pair], 1);
      }
    } else if (w >= 0 && w < n_words && table[w].word_id == w) {
      X = table[w].coords[0]; Y = table[w].coords[1]; Z = table[w].coords[2];
      if (n_with_landmark) atomicAdd(&n_with_landmark[pair], 1);
    }
  }
  const float4 m = reinterpret_cast<const float4*>(match_pts)[(size_t)pair * stride + j];
  float* o = corr + (size_t)pair * 5 * stride;
  o[j] = X; o[stride + j] = Y; o[2 * stride + j] = Z;
  o[3 * stride + j] = m.z;
  o[4 * stride + j] = m.w;
}

}  // namespace

extern "C" mv_status mv_build_corr_landmarks_batch(mv_ctx* ctx, int n_pairs, int top_n, int stride, int n_words,
                                                   const mv_landmark* d_table, const int32_t* d_f0,
                                                   const int32_t* d_q_patch, const int32_t* d_q_count,
                                                   const int32_t* d_word, const float* d_match_pts,
                                                   const int32_t* d_match_count, const int32_t* d_match_cell0,
                                                   float* d_corr, int32_t* d_n_with_landmark) {
  MV_ENTER(ctx);
  if (n_pairs <= 0 || n_pairs > 65535 || top_n <= 0 || stride <= 0 || n_words <= 0 || !d_table || !d_q_patch || !d_q_count ||
      !d_word || !d_match_pts || !d_match_count || !d_match_cell0 || !d_corr)
    MV_BAD_ARG(ctx, "mv_build_corr_landmarks_batch");
  if (d_n_with_landmark) MV_CUDA(ctx, cudaMemsetAsync(d_n_with_landmark, 0, sizeof(int32_t) * (size_t)n_pairs, ctx->stream));
  mv_prof_scope ps(ctx, "gather");
  dim3 grid((stride + 127) / 128, n_pairs);
  build_corr_landmarks_kernel<<<grid, 128, 0, ctx->stream>>>(n_words, d_table, top_n, stride, d_f0, d_q_patch, d_q_count,
                                                            d_word, d_match_pts, d_match_count, d_match_cell0, d_corr,
                                                            d_n_with_landmark, nullptr);
  MV_CHECK_LAUNCH(ctx);
  return MV_OK;
}

mv_status mv_build_corr_landmarks_seq(mv_ctx* ctx, int n_pairs, int top_n, int stride, int n_words,
                                      const int32_t* d_q_patch, const int32_t* d_q_count, const int32_t* d_word,
                                      const float* d_coords_out, const float* d_match_pts, const int32_t* d_match_count,
                                      const int32_t* d_match_cell0, float* d_corr, int32_t* d_n_with_landmark) {
  if (d_n_with_landmark) MV_CUDA(ctx, cudaMemsetAsync(d_n_with_landmark, 0, sizeof(int32_t) * (size_t)n_pairs, ctx->stream));
  mv_prof_scope ps(ctx, "corr");
  dim3 grid((stride + 127) / 128, n_pairs);
  build_corr_landmarks_kernel<<<grid, 128, 0, ctx->stream>>>(n_words, nullptr, top_n, stride, nullptr, d_q_patch, d_q_count,
                                                            d_word, d_match_pts, d_match_count, d_match_cell0, d_corr,
                                                            d_n_with_landmark, d_coords_out);
  MV_CHECK_LAUNCH(ctx);
  return MV_OK;
}

extern "C" mv_status mv_bow_set_vocabulary(mv_ctx* ctx, int n_base, int words_per_base, const int8_t* h_base_desc,
                                           const float* h_scale, const float* h_bias, const int32_t* h_leaves) {
  MV_ENTER(ctx);
  if (n_base <= 0 || n_base > 64 || words_per_base <= 0 || !h_base_desc || !h_scale || !h_bias || !h_leaves)
    MV_BAD_ARG(ctx, "mv_bow_set_vocabulary");
  const size_t n_leaf = (size_t)n_base * words_per_base * 4 + 4;
  void *dl, *db, *ds;
  mv_status st;
  if ((st = mv_scratch(ctx, "bow.leaves", sizeof(int32_t) * n_leaf, &dl))) return st;
  if ((st = mv_scratch(ctx, "bow.base_t", (size_t)n_base * 256, &db))) return st;
  if ((st = mv_scratch(ctx, "bow.scale_bias", sizeof(float) * 2 * n_base, &ds))) return st;
  std::vector<int32_t> leaves(n_leaf, 0);
  memcpy(leaves.data(), h_leaves, sizeof(int32_t) * (n_leaf - 4));
  std::vector<int8_t> bt((size_t)n_base * 256);
  for (int k = 0; k < 256; k++)
    for (int j = 0; j < n_base; j++) bt[(size_t)j * 256 + k] = h_base_desc[(size_t)k * n_base + j];
  std::vector<float> sb(2 * (size_t)n_base);
  for (int j = 0; j < n_base; j++) { sb[j] = h_scale[j]; sb[n_base + j] = h_bias[j]; }
  MV_CUDA(ctx, cudaMemcpyAsync(dl, leaves.data(), sizeof(int32_t) * n_leaf, cudaMemcpyHostToDevice, ctx->stream));
  MV_CUDA(ctx, cudaMemcpyAsync(db, bt.data(), bt.size(), cudaMemcpyHostToDevice, ctx->stream));
  MV_CUDA(ctx, cudaMemcpyAsync(ds, sb.data(), sizeof(float) * sb.size(), cudaMemcpyHostToDevice, ctx->stream));
  MV_CUDA(ctx, cudaStreamSynchronize(ctx->stream));   // the host vectors die with this call
  ctx->bow_n_base = n_base;
  ctx->bow_wpb = words_per_base;
  return MV_OK;
}

extern "C" mv_status mv_bow_assign_batch(mv_ctx* ctx, int n_frames, int cells, int top_n, const int8_t* d_desc,
                                         const float* d_desc_scale, const int32_t* d_q_patch,
                                         const int32_t* d_q_count, int32_t* d_word, int32_t* d_base) {
  MV_ENTER(ctx);
  return mv_bow_assign_impl(ctx, n_frames, cells, top_n, d_desc, d_desc_scale, d_q_patch, d_q_count, d_word, d_base,
                            MvBackProject());
}

mv_status mv_bow_assign_impl(mv_ctx* ctx, int n_frames, int cells, int top_n, const int8_t* d_desc,
                             const float* d_desc_scale, const int32_t* d_q_patch, const int32_t* d_q_count,
                             int32_t* d_word, int32_t* d_base, const MvBackProject& bp) {
  if (n_frames <= 0 || cells <= 0 || top_n <= 0 || !d_desc || !d_desc_scale || !d_q_patch || !d_q_count || !d_word)
    MV_BAD_ARG(ctx, "mv_bow_assign_batch");
  if (ctx->bow_n_base <= 0) MV_BAD_ARG(ctx, "mv_bow_assign_batch: no vocabulary (mv_bow_set_vocabulary first)");
  if (reinterpret_cast<uintptr_t>(d_desc) & 15) MV_BAD_ARG(ctx, "mv_bow_assign_batch: d_desc must be 16-byte aligned");
  BowVocabDev v;
  v.n_base = ctx->bow_n_base; v.wpb = ctx->bow_wpb;
  void *dl, *db, *ds;
  mv_status st;
  const size_t n_leaf = (size_t)v.n_base * v.wpb * 4 + 4;
  if ((st = mv_scratch(ctx, "bow.leaves", sizeof(int32_t) * n_leaf, &dl))) return st;
  if ((st = mv_scratch(ctx, "bow.base_t", (size_t)v.n_base * 256, &db))) return st;
  if ((st = mv_scratch(ctx, "bow.scale_bias", sizeof(float) * 2 * v.n_base, &ds))) return st;
  v.leaves = (const int32_t*)dl; v.base_t = (const int8_t*)db;
  v.scale = (const float*)ds; v.bias = (const float*)ds + v.n_base;
  const size_t smem = sizeof(int32_t) * ((n_leaf + 3) & ~(size_t)3) + (size_t)v.n_base * 256 + sizeof(float) * 2 * v.n_base;
  if (smem > 227 * 1024) MV_BAD_ARG(ctx, "mv_bow_assign_batch: vocabulary larger than an SM's shared memory");
  if (smem > ctx->bow_smem_attr) {   // a function attribute of the context's device: set once per size
    MV_CUDA(ctx, cudaFuncSetAttribute(bow_assign_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    ctx->bow_smem_attr = smem;
  }
  const int per_cta = kBowThreads / kBowLanes;   // queries a CTA handles per trip
  const long long trips = ((long long)n_frames * top_n + per_cta - 1) / per_cta;
  const int grid = (int)(trips < ctx->sm_count ? trips : ctx->sm_count);
  mv_prof_scope ps(ctx, "bow");
  bow_assign_kernel<<<grid, kBowThreads, smem, ctx->stream>>>(v, n_frames, cells, top_n, d_desc, d_desc_scale, d_q_patch,
                                                            d_q_count, d_word, d_base, bp);
  MV_CHECK_LAUNCH(ctx);
  return MV_OK;
}

static mv_status landmark_scratch(mv_ctx* ctx, int n_words, int32_t** first, int32_t** cnt) {
  // per-word scratch of the observe call, kept clean between calls; (re)initialised when the table grows
  void* p = nullptr;
  const bool fresh = ctx->scratch.find("lm.scratch") == ctx->scratch.end() ||
                     ctx->scratch["lm.scratch"].second < sizeof(int32_t) * 2 * (size_t)n_words || ctx->lm_words != n_words;
  mv_status st = mv_scratch(ctx, "lm.scratch", sizeof(int32_t) * 2 * (size_t)n_words, &p);
  if (st) return st;
  *first = (int32_t*)p;
  *cnt = (int32_t*)p + n_words;
  if (fresh) {
    landmarks_init_kernel<<<(n_words + 255) / 256, 256, 0, ctx->stream>>>(n_words, nullptr, *first, *cnt);
    MV_CHECK_LAUNCH(ctx);
    ctx->lm_words = n_words;
  }
  return MV_OK;
}

extern "C" mv_status mv_landmarks_init(mv_ctx* ctx, int n_words, mv_landmark* d_table) {
  MV_ENTER(ctx);
  if (n_words <= 0 || !d_table) MV_BAD_ARG(ctx, "mv_landmarks_init");
  landmarks_init_kernel<<<(n_words + 255) / 256, 256, 0, ctx->stream>>>(n_words, d_table, nullptr, nullptr);
  MV_CHECK_LAUNCH(ctx);
  return MV_OK;
}

extern "C" mv_status mv_landmarks_observe(mv_ctx* ctx, int n_words, mv_landmark* d_table, int frame, int n,
                                          const int32_t* d_word_ids, const float* d_coords) {
  MV_ENTER(ctx);
  if (n_words <= 0 || !d_table || n < 0 || (n > 0 && !d_word_ids)) MV_BAD_ARG(ctx, "mv_landmarks_observe");
  if (n == 0) return MV_OK;
  int32_t *first, *cnt;
  mv_status st = landmark_scratch(ctx, n_words, &first, &cnt);
  if (st) return st;
  landmarks_mark_kernel<<<(n + 255) / 256, 256, 0, ctx->stream>>>(n_words, n, d_word_ids, first, cnt);
  MV_CHECK_LAUNCH(ctx);
  landmarks_apply_kernel<<<(n + 255) / 256, 256, 0, ctx->stream>>>(n_words, d_table, frame, n, d_word_ids, d_coords, first, cnt);
  MV_CHECK_LAUNCH(ctx);
  return MV_OK;
}

extern "C" mv_status mv_landmarks_remove_old(mv_ctx* ctx, int n_words, mv_landmark* d_table, int current_frame) {
  MV_ENTER(ctx);
  if (n_words <= 0 || !d_table) MV_BAD_ARG(ctx, "mv_landmarks_remove_old");
  landmarks_remove_old_kernel<<<(n_words + 255) / 256, 256, 0, ctx->stream>>>(n_words, d_table, current_frame - 8 + 1);
  MV_CHECK_LAUNCH(ctx);
  return MV_OK;
}

extern "C" mv_status mv_landmarks_lookup(mv_ctx* ctx, int n_words, const mv_landmark* d_table, int n,
                                         const int32_t* d_word_ids, float* d_coords, int32_t* d_found) {
  MV_ENTER(ctx);
  if (n_words <= 0 || !d_table || n < 0 || (n > 0 && (!d_word_ids || !d_coords))) MV_BAD_ARG(ctx, "mv_landmarks_lookup");
  if (n == 0) return MV_OK;
  landmarks_lookup_kernel<<<(n + 255) / 256, 256, 0, ctx->stream>>>(n_words, d_table, n, d_word_ids, d_coords, d_found);
  MV_CHECK_LAUNCH(ctx);
  return MV_OK;
}

// The counting sort's tiling (tiles of fb frames: at most 512 of them, the column scan's serial length, and 2^24
// counters) and its scratch, shared by the call and by mv_landmarks_sequence_reserve.
static void lmseq_tiles(int n_words, int n_steps, int* n_tiles, int* fb) {
  int t = (int)std::min<long long>(std::min<long long>(512, (1LL << 24) / n_words), n_steps);
  if (t < 1) t = 1;
  *fb = (n_steps + t - 1) / t;
  *n_tiles = (n_steps + *fb - 1) / *fb;
}

static mv_status lmseq_scratch(mv_ctx* ctx, int n_words, int n_steps, int top_n, void** cnt, void** tot, void** start,
                               void** sorted) {
  int n_tiles, fb;
  lmseq_tiles(n_words, n_steps, &n_tiles, &fb);
  mv_status st;
  if ((st = mv_scratch(ctx, "lms.cnt", sizeof(int32_t) * (size_t)n_tiles * n_words, cnt))) return st;
  if ((st = mv_scratch(ctx, "lms.total", sizeof(int32_t) * (size_t)n_words, tot))) return st;
  if ((st = mv_scratch(ctx, "lms.start", sizeof(int32_t) * ((size_t)n_words + 1), start))) return st;
  return mv_scratch(ctx, "lms.sorted", sizeof(int32_t) * (size_t)n_steps * top_n, sorted);
}

mv_status mv_landmarks_sequence_reserve(mv_ctx* ctx, int n_words, int n_steps, int top_n) {
  void *cnt, *tot, *start, *sorted;
  return lmseq_scratch(ctx, n_words, n_steps, top_n, &cnt, &tot, &start, &sorted);
}

mv_status mv_landmarks_sequence_impl(mv_ctx* ctx, int n_words, mv_landmark* d_table, int first_frame, int n_steps,
                                     int top_n, const int32_t* d_word, const int32_t* d_q_count,
                                     const float* d_coords_in, float* d_coords_out) {
  if (n_words <= 0) MV_BAD_ARG(ctx, "mv_landmarks_sequence: n_words must be positive");
  if (!d_table) MV_BAD_ARG(ctx, "mv_landmarks_sequence: NULL landmark table");
  if (n_steps < 0 || n_steps > 65535 || top_n <= 0 || (long long)n_steps * top_n > 0x7fffffffLL)
    MV_BAD_ARG(ctx, "mv_landmarks_sequence: 0..65535 steps of top_n > 0 queries, fewer than 2^31 in all");
  if (n_steps == 0) return MV_OK;
  if (!d_word || !d_q_count || !d_coords_in || !d_coords_out) MV_BAD_ARG(ctx, "mv_landmarks_sequence");
  int n_tiles, fb;
  lmseq_tiles(n_words, n_steps, &n_tiles, &fb);
  const long long total = (long long)n_steps * top_n;
  void *cnt, *tot, *start, *sorted;
  mv_status st;
  if ((st = lmseq_scratch(ctx, n_words, n_steps, top_n, &cnt, &tot, &start, &sorted))) return st;
  {
    mv_prof_scope ps(ctx, "sort");
    MV_CUDA(ctx, cudaMemsetAsync(cnt, 0, sizeof(int32_t) * (size_t)n_tiles * n_words, ctx->stream));
    const long long blocks = (total + 255) / 256;
    lmseq_count_kernel<<<(int)std::min<long long>(blocks, 8LL * ctx->sm_count), 256, 0, ctx->stream>>>(
        n_steps, top_n, n_words, fb, d_word, d_q_count, (int32_t*)cnt, d_coords_out);
    MV_CHECK_LAUNCH(ctx);
    lmseq_colscan_kernel<<<(n_words + 127) / 128, 128, 0, ctx->stream>>>(n_words, n_tiles, (int32_t*)cnt, (int32_t*)tot);
    MV_CHECK_LAUNCH(ctx);
    lmseq_wordscan_kernel<<<1, 1024, 0, ctx->stream>>>(n_words, (const int32_t*)tot, (int32_t*)start);
    MV_CHECK_LAUNCH(ctx);
    lmseq_scatter_kernel<<<n_tiles, 256, 0, ctx->stream>>>(n_steps, top_n, n_words, fb, d_word, d_q_count, (int32_t*)cnt,
                                                          (const int32_t*)start, (int32_t*)sorted);
    MV_CHECK_LAUNCH(ctx);
  }
  mv_prof_scope ps(ctx, "walk");
  lmseq_walk_kernel<<<(n_words + kWalkWarps - 1) / kWalkWarps, 32 * kWalkWarps, 0, ctx->stream>>>(
      n_words, d_table, first_frame, n_steps, top_n, (const int32_t*)start, (const int32_t*)sorted, d_coords_in,
      d_coords_out);
  MV_CHECK_LAUNCH(ctx);
  return MV_OK;
}

extern "C" mv_status mv_landmarks_sequence(mv_ctx* ctx, int n_words, mv_landmark* d_table, int first_frame, int n_steps,
                                           int top_n, const int32_t* d_word, const int32_t* d_q_count,
                                           const float* d_coords_in, float* d_coords_out) {
  MV_ENTER(ctx);
  return mv_landmarks_sequence_impl(ctx, n_words, d_table, first_frame, n_steps, top_n, d_word, d_q_count, d_coords_in,
                                    d_coords_out);
}
