// lba.cu -- local bundle adjustment: Schur complement of the landmarks, batched over windows
// (reference: src/local_bundle_adjustment.c:133-246; SURVEY §8f rank 4).
//
// The reference walks the landmarks of one window in chunks of 4: every (landmark, pose) factor's
// [J|r]^T [J|r] (10 x 10, from a 2 x 10 Jacobian block) is scattered into the landmark block
// diagonal A, the pose-landmark block B and the pose block C; A is inverted 3 x 3 block by block
// and C -= B A^-1 B^T.  All of it is fp32 whose result depends on the order of the additions
// (chunk after chunk into C, pose after pose into A, k innermost in the shim's matmul2), so the
// order is part of the contract.  Here one CTA owns one window and keeps C, A, B, B A^-1 and the
// chunk's factor products in shared memory; a chunk is five barrier-separated phases in which
// every thread owns whole output entries and adds their terms in the reference's order -- the
// parallelism is across entries (2 304 of C per chunk) and across windows, never inside a sum.
// Bit-identical to the reference program on its own input and on substituted inputs
// (tests/test_lba.py, oracle/ref_harness.c).
//
// Bound: FP32 issue.  A window reads 80 B per factor (640 KB for 1000 landmarks x 8 poses) and
// writes (6P+1)^2 floats, against 21.9 MFLOP of multiplies and adds that must be rounded one by one
// (no FMA, the reference has none): 34 flop/B, above the ridge of the non-fused rate (37 TFLOP/s /
// 6.5 TB/s = 5.7).  tools/lba_bench.py measures both.
#include "mv_common.cuh"

namespace {

constexpr int kLbaThreads = 256;

// local_bundle_adjustment.c:48-75, operation for operation (no FMA: the file is built -fmad=false)
__device__ __forceinline__ void invert_3x3(float* matrix, int stride) {
  float m[9], inv[9];
#pragma unroll
  for (int j = 0; j < 3; j++)
#pragma unroll
    for (int i = 0; i < 3; i++) m[j * 3 + i] = matrix[j * stride + i];
  const float det = __fadd_rn(__fsub_rn(__fmul_rn(m[0], __fsub_rn(__fmul_rn(m[4], m[8]), __fmul_rn(m[5], m[7]))),
                                        __fmul_rn(m[1], __fsub_rn(__fmul_rn(m[3], m[8]), __fmul_rn(m[5], m[6])))),
                              __fmul_rn(m[2], __fsub_rn(__fmul_rn(m[3], m[7]), __fmul_rn(m[4], m[6]))));
  inv[0] = __fdiv_rn(__fsub_rn(__fmul_rn(m[4], m[8]), __fmul_rn(m[5], m[7])), det);
  inv[1] = __fdiv_rn(__fsub_rn(__fmul_rn(m[2], m[7]), __fmul_rn(m[1], m[8])), det);
  inv[2] = __fdiv_rn(__fsub_rn(__fmul_rn(m[1], m[5]), __fmul_rn(m[2], m[4])), det);
  inv[3] = __fdiv_rn(__fsub_rn(__fmul_rn(m[5], m[6]), __fmul_rn(m[3], m[8])), det);
  inv[4] = __fdiv_rn(__fsub_rn(__fmul_rn(m[0], m[8]), __fmul_rn(m[2], m[6])), det);
  inv[5] = __fdiv_rn(__fsub_rn(__fmul_rn(m[2], m[3]), __fmul_rn(m[0], m[5])), det);
  inv[6] = __fdiv_rn(__fsub_rn(__fmul_rn(m[3], m[7]), __fmul_rn(m[4], m[6])), det);
  inv[7] = __fdiv_rn(__fsub_rn(__fmul_rn(m[1], m[6]), __fmul_rn(m[0], m[7])), det);
  inv[8] = __fdiv_rn(__fsub_rn(__fmul_rn(m[0], m[4]), __fmul_rn(m[1], m[3])), det);
#pragma unroll
  for (int j = 0; j < 3; j++)
#pragma unroll
    for (int i = 0; i < 3; i++) matrix[j * stride + i] = inv[j * 3 + i];
}

// One CTA per window.  Shared memory: Jc[nf*20] Hs[nf*100] C[SH*SH] A[LD*LD] B[SH*LD] BA[SH*LD]
__global__ void __launch_bounds__(kLbaThreads)
lba_schur_kernel(int n_ldmks, int n_poses, int chunk, const float* __restrict__ J_all, float* __restrict__ C_all) {
  extern __shared__ __align__(16) float lba_smem[];
  const int PD = 6 * n_poses, SH = PD + 1, LD = 3 * chunk, nf = chunk * n_poses;
  float* Jc = lba_smem;            // first: filled with 16-byte stores
  float* Hs = Jc + nf * 20;
  float* C = Hs + nf * 100;
  float* A = C + SH * SH;
  float* B = A + LD * LD;
  float* BA = B + SH * LD;
  const int tid = threadIdx.x;
  const float* J = J_all + (size_t)blockIdx.x * n_ldmks * n_poses * 20;

  for (int e = tid; e < SH * SH; e += kLbaThreads) C[e] = 0.0f;
  for (int e = tid; e < LD * LD; e += kLbaThreads) A[e] = 0.0f;
  for (int e = tid; e < SH * LD; e += kLbaThreads) BA[e] = 0.0f;
  float hprev = 0.0f;   // entry tid of the previous factor's product (the shim's 0 * D, :166-172)

  for (int c0 = 0; c0 < n_ldmks; c0 += chunk) {
    // ---- phase 0: the chunk's factors; A's diagonal blocks and B start at zero (:141-143)
    {
      const float4* src = reinterpret_cast<const float4*>(J + (size_t)c0 * n_poses * 20);
      float4* dst = reinterpret_cast<float4*>(Jc);
      for (int e = tid; e < nf * 5; e += kLbaThreads) dst[e] = __ldg(src + e);
      for (int e = tid; e < chunk * 9; e += kLbaThreads) {
        const int I = (e / 9) * 3, i = (e % 9) / 3, j = e % 3;
        A[(I + i) * LD + I + j] = 0.0f;
      }
      for (int e = tid; e < SH * LD; e += kLbaThreads) B[e] = 0.0f;
    }
    __syncthreads();
    // ---- phase 1: H = [J|r]^T [J|r] per factor, entry (i, j) by thread 10 i + j, factors in
    // the reference's order (landmark of the chunk outer, pose inner); each product starts as
    // 0 * (the previous factor's entry), so a non-finite entry sticks exactly as it does there
    if (tid < 100) {
      const int i = tid / 10, j = tid % 10;
      for (int f = 0; f < nf; f++) {
        const float* Jf = Jc + f * 20;
        float h = __fmul_rn(0.0f, hprev);
        h = __fadd_rn(h, __fmul_rn(Jf[i * 2], Jf[j * 2]));
        h = __fadd_rn(h, __fmul_rn(Jf[i * 2 + 1], Jf[j * 2 + 1]));
        Hs[f * 100 + tid] = h;
        hprev = h;
      }
    }
    __syncthreads();
    // ---- phase 2: scatter (:176-219).  H is addressed column-major with stride 10, as there.
    {
      const int nA = chunk * 9, nB = nf * 18, nBf = chunk * 3, nC = n_poses * 36, nCf = n_poses * 6;
      for (int e = tid; e < nA + nB + nBf + nC + nCf; e += kLbaThreads) {
        if (e < nA) {                                    // H_LL: sum over poses
          const int ci = e / 9, j = (e % 9) / 3, i = e % 3, li = ci * 3;
          float v = A[(li + j) * LD + li + i];
          for (int p = 0; p < n_poses; p++) v = __fadd_rn(Hs[(ci * n_poses + p) * 100 + j * 10 + i], v);
          A[(li + j) * LD + li + i] = v;
        } else if (e < nA + nB) {                        // H_PL: one factor each
          const int q = e - nA, f = q / 18, j = (q % 18) / 6, i = q % 6;
          const int ci = f / n_poses, p = f % n_poses;
          float* b = B + p * 6 + i + (ci * 3 + j) * SH;
          *b = __fadd_rn(Hs[f * 100 + j * 10 + 3 + i], *b);
        } else if (e < nA + nB + nBf) {                  // landmark gradient row: sum over poses
          const int q = e - nA - nB, ci = q / 3, j = q % 3;
          float* b = B + (ci * 3 + j) * SH + SH - 1;
          float v = *b;
          for (int p = 0; p < n_poses; p++) v = __fadd_rn(Hs[(ci * n_poses + p) * 100 + j * 10 + 9], v);
          *b = v;
        } else if (e < nA + nB + nBf + nC) {             // H_PP: sum over the chunk's landmarks
          const int q = e - nA - nB - nBf, p = q / 36, j = (q % 36) / 6, i = q % 6;
          float* c = C + (p * 6 + j) * SH + p * 6 + i;
          float v = *c;
          for (int ci = 0; ci < chunk; ci++) v = __fadd_rn(Hs[(ci * n_poses + p) * 100 + (3 + j) * 10 + 3 + i], v);
          *c = v;
        } else {                                         // pose gradient row
          const int q = e - nA - nB - nBf - nC, p = q / 6, j = q % 6;
          float* c = C + (p * 6 + j) * SH + SH - 1;
          float v = *c;
          for (int ci = 0; ci < chunk; ci++) v = __fadd_rn(Hs[(ci * n_poses + p) * 100 + (3 + j) * 10 + 9], v);
          *c = v;
        }
      }
    }
    __syncthreads();
    // ---- phase 3: A^-1, block by block (:227)
    if (tid < chunk) invert_3x3(A + (tid * 3) * LD + tid * 3, LD);
    __syncthreads();
    // ---- phase 4: (B A^-1)^T = A^-T B^T as the shim computes it (:230-235): 0 * old + sum over k
    for (int e = tid; e < LD * PD; e += kLbaThreads) {
      const int i = e / PD, j = e % PD;
      float v = __fmul_rn(0.0f, BA[i * SH + j]);
      for (int k = 0; k < LD; k++) v = __fadd_rn(v, __fmul_rn(A[i * LD + k], B[k * SH + j]));
      BA[i * SH + j] = v;
    }
    __syncthreads();
    // ---- phase 5: C -= B A^-1 B^T (:238-243): 1 * old, then (-1 * b) * ba for k ascending
    for (int e = tid; e < PD * PD; e += kLbaThreads) {
      const int i = e / PD, j = e % PD;
      float v = C[i * SH + j];
      for (int k = 0; k < LD; k++) v = __fadd_rn(v, __fmul_rn(-B[k * SH + i], BA[k * SH + j]));
      C[i * SH + j] = v;
    }
    __syncthreads();
  }
  float* out = C_all + (size_t)blockIdx.x * SH * SH;
  for (int e = tid; e < SH * SH; e += kLbaThreads) out[e] = C[e];
}

// The reference's shape (8 poses, chunks of 4) with everything a compile-time constant: the 48 x 48
// pose block of C never leaves registers -- 256 threads, one 3 x 3 tile each for the whole window,
// so a k-step of the update costs 6 shared loads for 9 multiply-adds -- and the index arithmetic of
// the scatter folds away.  Same sums in the same order as the generic kernel above.
constexpr int kP8 = 8, kC4 = 4;
__global__ void __launch_bounds__(256, 6)
lba_schur_p8c4_kernel(int n_ldmks, const float* __restrict__ J_all, float* __restrict__ C_all) {
  constexpr int P = kP8, CH = kC4, PD = 6 * P, SH = PD + 1, LD = 3 * CH, NF = CH * P;
  __shared__ __align__(16) float Jc[2][NF * 20];   // the chunk's factors, next chunk prefetched
  __shared__ float Hs[NF * 100];
  // A, A^-1, B, B A^-1 and the last row of C (pose gradient, column-major row SH-1) in one array, so
  // that a destination of the scatter phase is one 16-bit offset
  constexpr int oA = 0, oAi = LD * LD, oB = 2 * LD * LD, oBA = oB + SH * LD, oCrow = oBA + SH * LD;
  __shared__ __align__(16) float S[oCrow + PD];
  float* const A = S + oA; float* const Ai = S + oAi; float* const B = S + oB; float* const BA = S + oBA;
  float* const Crow = S + oCrow;
  // scatter phase as a table: entry e sums n entries of Hs (first, stride) onto +0 -- or onto the
  // destination's old value (the gradient row, which runs on across the chunks) -- and stores the sum
  constexpr int nA = CH * 9, nB = NF * 18, nBf = CH * 3, nCf = P * 6, nScatter = nA + nB + nBf + nCf;
  static_assert(CH == 4 && P == 8, "the scatter loop below is written for sums of 1, 4 or 8 terms");
  __shared__ uint2 tab[nScatter];   // .x = first | dst << 16, .y = n | stride << 8 | accumulate << 31
  const int tid = threadIdx.x;
  // Tile of the thread: rows 3ti.., columns 3tj.. of C[i*SH + j].  The 32 tiles inside the poses'
  // 6 x 6 diagonal blocks (they alone receive the H_PP terms) belong to warp 0, so that only one
  // warp executes that code; the other 224 tiles follow row by row.
  int ti, tj;
  if (tid < 32) {
    ti = 2 * (tid >> 2) + ((tid >> 1) & 1);
    tj = 2 * (tid >> 2) + (tid & 1);
  } else {
    const int m = tid - 32, r = m % 14;
    ti = m / 14;
    tj = r + (r >= 2 * (ti >> 1) ? 2 : 0);
  }
  const float* J = J_all + (size_t)blockIdx.x * n_ldmks * P * 20;
  for (int e = tid; e < nScatter; e += 256) {
    unsigned first, dst, n, stride, acc = 0;
    if (e < nA) {                      // landmark block: the 8 poses' H_LL entries (:176-183)
      const int ci = e / 9, j = (e % 9) / 3, i = e % 3, li = ci * 3;
      first = ci * P * 100 + j * 10 + i; stride = 100; n = P; dst = oA + (li + j) * LD + li + i;
    } else if (e < nA + nB) {          // pose-landmark block: one H_PL entry each (:185-192)
      const int q = e - nA, f = q / 18, j = (q % 18) / 6, i = q % 6;
      const int ci = f / P, p_ = f % P;
      first = f * 100 + j * 10 + 3 + i; stride = 0; n = 1; dst = oB + p_ * 6 + i + (ci * 3 + j) * SH;
    } else if (e < nA + nB + nBf) {    // landmark gradient row: the 8 poses' H_Lf entries (:194-201)
      const int q = e - nA - nB, ci = q / 3, j = q % 3;
      first = ci * P * 100 + j * 10 + 9; stride = 100; n = P; dst = oB + (ci * 3 + j) * SH + SH - 1;
    } else {                           // pose gradient row: the chunk's 4 landmarks' H_Pf entries (:212-219)
      const int q = e - nA - nB - nBf, p_ = q / 6, j = q % 6;
      first = p_ * 100 + (3 + j) * 10 + 9; stride = P * 100; n = CH; dst = oCrow + p_ * 6 + j; acc = 1;
    }
    tab[e] = make_uint2(first | (dst << 16), n | (stride << 8) | (acc << 31));
  }

  float c[3][3];
#pragma unroll
  for (int a = 0; a < 3; a++)
#pragma unroll
    for (int b = 0; b < 3; b++) c[a][b] = 0.0f;
  for (int e = tid; e < LD * LD; e += 256) { A[e] = 0.0f; Ai[e] = 0.0f; }
  for (int e = tid; e < SH * LD; e += 256) BA[e] = 0.0f;
  if (tid < PD) Crow[tid] = 0.0f;
  float hprev = 0.0f;
  const bool diag = tid < 32;                       // the tile lies in a pose's 6 x 6 diagonal block
  const int pose = ti >> 1, di = 3 * (ti & 1), dj = 3 * (tj & 1);

  bool serial = false;   // sticky: once a product needed the previous factor's entry, every later one does
  if (tid < NF * 5) reinterpret_cast<float4*>(Jc[0])[tid] = __ldg(reinterpret_cast<const float4*>(J) + tid);
  __syncthreads();

  for (int c0 = 0, buf = 0; c0 < n_ldmks; c0 += CH, buf ^= 1) {
    // ---- phase 1: H = [J|r]^T [J|r] per factor, from the staged factors (2.5 KB per chunk).
    // The shim computes entry (i, j) of factor f as (0 * h_prev + t0) + t1 with h_prev the same entry of
    // the previous factor: a serial chain that matters only if h_prev is not finite (the NaN sticks) or
    // t0 is a zero (whose sign then comes from h_prev).  Fast path: all 256 threads take the 3 200
    // entries of the chunk with h_prev = +0; if any thread met one of the two cases the chunk -- and
    // every later one -- is redone by 100 threads walking the factors in order, as the reference does.
    const float* Jch = Jc[buf];
    bool special = serial;
    if (!serial && (tid & 127) < 100) {
      // entry (i, j) = tid mod 128 (100 of every 128 threads), factors of the thread's parity: all
      // loads of the 16 factors are independent, so they overlap
      const int ij = tid & 127, i = ij / 10, j = ij - i * 10;
      const float* Ji = Jch + (tid >> 7) * 20 + i * 2;
      const float* Jj = Jch + (tid >> 7) * 20 + j * 2;
      float* Hd = Hs + (tid >> 7) * 100 + ij;
#pragma unroll
      for (int k = 0; k < NF / 2; k++) {
        const float2 a = *reinterpret_cast<const float2*>(Ji + k * 40);
        const float2 bb = *reinterpret_cast<const float2*>(Jj + k * 40);
        const float t0 = __fmul_rn(a.x, bb.x);
        const float h = __fadd_rn(__fadd_rn(0.0f, t0), __fmul_rn(a.y, bb.y));
        Hd[k * 200] = h;
        special = special || t0 == 0.0f || !(fabsf(h) <= 3.402823466e38f);
      }
    }
    serial = __syncthreads_or(special) != 0;
    if (serial) {
      if (tid < 100) {
        const int i = tid / 10, j = tid % 10;
        for (int f = 0; f < NF; f++) {
          const float* Jf = Jch + f * 20;
          float h = __fmul_rn(0.0f, hprev);
          h = __fadd_rn(h, __fmul_rn(Jf[i * 2], Jf[j * 2]));
          h = __fadd_rn(h, __fmul_rn(Jf[i * 2 + 1], Jf[j * 2 + 1]));
          Hs[f * 100 + tid] = h;
          hprev = h;
        }
      }
      __syncthreads();
    } else if (tid < 100) {
      hprev = Hs[(NF - 1) * 100 + tid];
    }
    // ---- phase 2: scatter into A, B and the gradient rows (the pose blocks are added in phase 5).
    // (The reference zeroes A's diagonal blocks and B before every chunk, :141-142: the sums start
    // from +0 here instead of from memory; every entry of B is written.)
    for (int e = tid; e < nScatter; e += 256) {
      const uint2 t = tab[e];
      const float* src = Hs + (t.x & 0xffffu);
      float* dst = S + (t.x >> 16);
      const int n = (int)(t.y & 0xffu), stride = (int)((t.y >> 8) & 0xffffu);
      float v = (t.y >> 31) ? *dst : 0.0f;
      v = __fadd_rn(src[0], v);
      if (n >= CH) {      // n is 1, CH (= 4) or P (= 8)
        v = __fadd_rn(src[stride], v); v = __fadd_rn(src[2 * stride], v); v = __fadd_rn(src[3 * stride], v);
        if (n == P) {
          v = __fadd_rn(src[4 * stride], v); v = __fadd_rn(src[5 * stride], v);
          v = __fadd_rn(src[6 * stride], v); v = __fadd_rn(src[7 * stride], v);
        }
      }
      *dst = v;
    }
    __syncthreads();
    // ---- phase 3: A^-1 into Ai; one thread per entry of a block's inverse (each recomputes the
    // determinant: same operations, same value).  Ai's off-diagonal blocks stay 0 like A's.
    if (tid < CH * 9) {
      const int blk = tid / 9, ent = tid % 9;
      const float* M = A + (blk * 3) * LD + blk * 3;
      float m[9];
#pragma unroll
      for (int j = 0; j < 3; j++)
#pragma unroll
        for (int i = 0; i < 3; i++) m[j * 3 + i] = M[j * LD + i];
      const float det = __fadd_rn(__fsub_rn(__fmul_rn(m[0], __fsub_rn(__fmul_rn(m[4], m[8]), __fmul_rn(m[5], m[7]))),
                                            __fmul_rn(m[1], __fsub_rn(__fmul_rn(m[3], m[8]), __fmul_rn(m[5], m[6])))),
                                  __fmul_rn(m[2], __fsub_rn(__fmul_rn(m[3], m[7]), __fmul_rn(m[4], m[6]))));
      // cofactor `ent` of local_bundle_adjustment.c:60-68: (m[p]*m[q] - m[r]*m[s]) / det, its four
      // operands read by index (entry e of the 3 x 3 copy is M[(e/3)*LD + e%3])
      const int sh = 4 * (8 - ent);   // tables packed one hex digit per entry, entry 0 first
      const int cp = (int)((0x421502310ull >> sh) & 15), cq = (int)((0x875683764ull >> sh) & 15);
      const int cr = (int)((0x512320401ull >> sh) & 15), cs = (int)((0x784865673ull >> sh) & 15);
      const float vp = M[(cp / 3) * LD + cp % 3], vq = M[(cq / 3) * LD + cq % 3];
      const float vr = M[(cr / 3) * LD + cr % 3], vs = M[(cs / 3) * LD + cs % 3];
      Ai[(blk * 3 + ent / 3) * LD + blk * 3 + ent % 3] = __fdiv_rn(__fsub_rn(__fmul_rn(vp, vq), __fmul_rn(vr, vs)), det);
    }
    __syncthreads();
    // ---- phase 4: B A^-1
    for (int e = tid; e < LD * PD; e += 256) {
      const int i = e / PD, j = e % PD;
      float v = __fmul_rn(0.0f, BA[i * SH + j]);
      float ai[LD];   // row i of A^-1: 48 bytes, 16-byte aligned
#pragma unroll
      for (int k = 0; k < LD; k += 4) *reinterpret_cast<float4*>(ai + k) = *reinterpret_cast<const float4*>(Ai + i * LD + k);
#pragma unroll
      for (int k = 0; k < LD; k++) v = __fadd_rn(v, __fmul_rn(ai[k], B[k * SH + j]));
      BA[i * SH + j] = v;
    }
    __syncthreads();
    // ---- phase 5: this chunk's H_PP terms (diagonal tiles, landmark by landmark), then C -= B A^-1 B^T;
    // the next chunk's factors arrive meanwhile (the barrier that ends the chunk publishes them)
    if (c0 + CH < n_ldmks && tid < NF * 5)
      reinterpret_cast<float4*>(Jc[buf ^ 1])[tid] = __ldg(reinterpret_cast<const float4*>(J + (size_t)(c0 + CH) * P * 20) + tid);
    if (diag) {
#pragma unroll
      for (int a = 0; a < 3; a++)
#pragma unroll
        for (int b = 0; b < 3; b++) {
          // C[i*SH + j], i = 6 pose + di + a, j = 6 pose + dj + b  <-  H[(3 + di + a)*10 + 3 + dj + b]
          float v = c[a][b];
#pragma unroll
          for (int ci = 0; ci < CH; ci++) v = __fadd_rn(Hs[(ci * P + pose) * 100 + (3 + di + a) * 10 + 3 + dj + b], v);
          c[a][b] = v;
        }
    }
#pragma unroll
    for (int k = 0; k < LD; k++) {
      const float b0 = -B[k * SH + 3 * ti], b1 = -B[k * SH + 3 * ti + 1], b2 = -B[k * SH + 3 * ti + 2];
      const float a0 = BA[k * SH + 3 * tj], a1 = BA[k * SH + 3 * tj + 1], a2 = BA[k * SH + 3 * tj + 2];
      c[0][0] = __fadd_rn(c[0][0], __fmul_rn(b0, a0)); c[0][1] = __fadd_rn(c[0][1], __fmul_rn(b0, a1)); c[0][2] = __fadd_rn(c[0][2], __fmul_rn(b0, a2));
      c[1][0] = __fadd_rn(c[1][0], __fmul_rn(b1, a0)); c[1][1] = __fadd_rn(c[1][1], __fmul_rn(b1, a1)); c[1][2] = __fadd_rn(c[1][2], __fmul_rn(b1, a2));
      c[2][0] = __fadd_rn(c[2][0], __fmul_rn(b2, a0)); c[2][1] = __fadd_rn(c[2][1], __fmul_rn(b2, a1)); c[2][2] = __fadd_rn(c[2][2], __fmul_rn(b2, a2));
    }
    __syncthreads();
  }
  float* out = C_all + (size_t)blockIdx.x * SH * SH;
#pragma unroll
  for (int a = 0; a < 3; a++)
#pragma unroll
    for (int b = 0; b < 3; b++) out[(3 * ti + a) * SH + 3 * tj + b] = c[a][b];
  if (tid < PD) out[tid * SH + SH - 1] = Crow[tid];
  if (tid < SH) out[PD * SH + tid] = 0.0f;          // the last column stays 0, as in the reference
}

// ---------------------------------------------------------------------------------------
// The step of the reduced camera system, S d = -g: what the reference would get from the
// cholesky() it leaves as a stub (local_bundle_adjustment.c:88-90,247).  This repository's
// definition (parity unpinned; the CPU restatement in the test tree states the same sums): the
// PnP kernel's damped 6 x 6 Cholesky solve at n = 6 n_poses.  One warp owns a window; lane l owns rows
// l, l+32, l+64 of L (shared memory, row stride n+1 -- odd, so a column is conflict-free and a
// row element is a broadcast).  Every sum is one thread's fmaf chain in the defined order
// (k ascending in the factorisation and the forward sweep, descending in the backward sweep),
// so the parallelism is across rows only and the result is the sequential one bit for bit.
constexpr int kSolveWarps = 4;

__device__ __forceinline__ float pick3(const float (&v)[3], int slot) {
  return slot == 0 ? v[0] : (slot == 1 ? v[1] : v[2]);
}

__global__ void __launch_bounds__(32 * kSolveWarps)
lba_solve_kernel(int n_windows, int n_poses, float damping, const float* __restrict__ C_all,
                 float* __restrict__ d_all, int32_t* __restrict__ ok_all) {
  extern __shared__ __align__(16) float solve_smem[];
  const int n = 6 * n_poses, SH = n + 1, ST = n + 1;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int w = blockIdx.x * kSolveWarps + warp;
  if (w >= n_windows) return;   // whole warps leave; there is no block-wide barrier below
  const unsigned full = 0xffffffffu;
  float* L = solve_smem + (size_t)warp * n * ST;
  const float* C = C_all + (size_t)w * SH * SH;
  // the lower triangle S[i][j] = C[j*SH + i], i >= j (a column of C is contiguous)
  for (int j = 0; j < n; j++)
    for (int i = j + lane; i < n; i += 32) L[i * ST + j] = __ldg(C + (size_t)j * SH + i);
  __syncwarp();

  float inv[3] = {0.0f, 0.0f, 0.0f}, s[3];
  bool ok = true;
  for (int j = 0; j < n; j++) {
    const float* Lj = L + j * ST;
    bool act[3];
#pragma unroll
    for (int r = 0; r < 3; r++) {
      const int i = lane + 32 * r;
      act[r] = i < n && i >= j;
      s[r] = act[r] ? L[i * ST + j] : 0.0f;
      if (i == j) s[r] = __fadd_rn(__fmaf_rn(damping, s[r], s[r]), 1e-12f);
    }
    for (int k = 0; k < j; k++) {
      const float ljk = Lj[k];
#pragma unroll
      for (int r = 0; r < 3; r++)
        if (act[r]) s[r] = __fmaf_rn(-L[(lane + 32 * r) * ST + k], ljk, s[r]);
    }
    const float sj = __shfl_sync(full, pick3(s, j >> 5), j & 31);
    if (!(sj > 0.0f)) {   // not positive definite (NaN included): uniform across the warp
      ok = false;
      break;
    }
    const float dj = __fsqrt_rn(sj), ij = __fdiv_rn(1.0f, dj);
#pragma unroll
    for (int r = 0; r < 3; r++) {
      const int i = lane + 32 * r;
      if (i == j) {
        inv[r] = ij;
        L[i * ST + j] = dj;
      } else if (act[r]) {
        L[i * ST + j] = __fmul_rn(s[r], ij);
      }
    }
    __syncwarp();
  }

  if (ok) {
    // L y = -g, column by column: row i meets its terms with k ascending
#pragma unroll
    for (int r = 0; r < 3; r++) {
      const int i = lane + 32 * r;
      s[r] = i < n ? -__ldg(C + (size_t)i * SH + n) : 0.0f;
    }
    for (int k = 0; k < n; k++) {
      const float yk = __shfl_sync(full, __fmul_rn(pick3(s, k >> 5), pick3(inv, k >> 5)), k & 31);
#pragma unroll
      for (int r = 0; r < 3; r++) {
        const int i = lane + 32 * r;
        if (i == k) s[r] = yk;
        else if (i > k && i < n) s[r] = __fmaf_rn(-L[i * ST + k], yk, s[r]);
      }
    }
    // L^T d = y, column by column from the last: row i meets its terms with k descending
    for (int k = n - 1; k >= 0; k--) {
      const float xk = __shfl_sync(full, __fmul_rn(pick3(s, k >> 5), pick3(inv, k >> 5)), k & 31);
#pragma unroll
      for (int r = 0; r < 3; r++) {
        const int i = lane + 32 * r;
        if (i == k) s[r] = xk;
        else if (i < k) s[r] = __fmaf_rn(-L[k * ST + i], xk, s[r]);
      }
    }
  }
#pragma unroll
  for (int r = 0; r < 3; r++) {
    const int i = lane + 32 * r;
    if (i < n) d_all[(size_t)w * n + i] = ok ? s[r] : 0.0f;
  }
  if (lane == 0) ok_all[w] = ok ? 1 : 0;
}

}  // namespace

extern "C" mv_status mv_lba_schur_batch(mv_ctx* ctx, int n_windows, int n_ldmks, int n_poses, int chunk,
                                        const float* d_J, float* d_C) {
  MV_ENTER(ctx);
  if (n_windows <= 0 || n_ldmks <= 0 || n_poses <= 0 || chunk <= 0 || !d_J || !d_C)
    MV_BAD_ARG(ctx, "mv_lba_schur_batch");
  if (n_ldmks % chunk != 0 || n_poses > 16 || chunk > 16)
    MV_BAD_ARG(ctx, "mv_lba_schur_batch: n_ldmks a multiple of chunk, n_poses <= 16, chunk <= 16");
  const int PD = 6 * n_poses, SH = PD + 1, LD = 3 * chunk, nf = chunk * n_poses;
  const size_t smem = sizeof(float) * ((size_t)SH * SH + (size_t)LD * LD + 2 * (size_t)SH * LD + (size_t)nf * 120);
  if (smem > 200 * 1024) MV_BAD_ARG(ctx, "mv_lba_schur_batch: window too large for shared memory");
  // The limit is shared by every mv_ctx on the device (see match_tc.cu): set once per context to the most this call
  // admits, never to this call's own size.
  if (smem > 48 * 1024 && !ctx->lba_schur_smem_attr_set) {
    MV_CUDA(ctx, cudaFuncSetAttribute(lba_schur_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    ctx->lba_schur_smem_attr_set = true;
  }
  mv_prof_scope ps(ctx, "lba");
  if (n_poses == kP8 && chunk == kC4)
    lba_schur_p8c4_kernel<<<n_windows, 256, 0, ctx->stream>>>(n_ldmks, d_J, d_C);
  else
    lba_schur_kernel<<<n_windows, kLbaThreads, smem, ctx->stream>>>(n_ldmks, n_poses, chunk, d_J, d_C);
  MV_CHECK_LAUNCH(ctx);
  return MV_OK;
}

extern "C" mv_status mv_lba_solve_batch(mv_ctx* ctx, int n_windows, int n_poses, float damping,
                                        const float* d_C, float* d_delta, int32_t* d_ok) {
  MV_ENTER(ctx);
  if (n_windows <= 0 || n_poses <= 0 || !d_C || !d_delta || !d_ok) MV_BAD_ARG(ctx, "mv_lba_solve_batch");
  if (n_poses > 16) MV_BAD_ARG(ctx, "mv_lba_solve_batch: n_poses <= 16");
  const int n = 6 * n_poses;
  const size_t smem = sizeof(float) * (size_t)kSolveWarps * n * (n + 1);
  // as in mv_lba_schur_batch: the bound of n_poses = 16, once per context
  if (smem > 48 * 1024 && !ctx->lba_solve_smem_attr_set) {
    MV_CUDA(ctx, cudaFuncSetAttribute(lba_solve_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)(sizeof(float) * kSolveWarps * 96 * 97)));
    ctx->lba_solve_smem_attr_set = true;
  }
  mv_prof_scope ps(ctx, "lba_solve");
  lba_solve_kernel<<<(n_windows + kSolveWarps - 1) / kSolveWarps, 32 * kSolveWarps, smem, ctx->stream>>>(
      n_windows, n_poses, damping, d_C, d_delta, d_ok);
  MV_CHECK_LAUNCH(ctx);
  return MV_OK;
}
