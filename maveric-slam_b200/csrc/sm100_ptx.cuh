// sm100_ptx.cuh -- the Blackwell (sm_100a) primitives the tensor-core matcher is built from:
// mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (alloc / mma / commit / ld) and the shared-memory
// and instruction descriptors of the UMMA unit.  Inline PTX only; no library templates.
//
// Every wait is bounded: a barrier that does not complete within MV_MBAR_TIMEOUT_NS (10 s by default;
// compile with -DMV_MBAR_TIMEOUT_NS=0 for unbounded waits under a debugger or sanitizer) writes its wait
// site into a flag in mapped host memory and traps, so a protocol bug surfaces as a launch failure that
// names the site (mv_last_error), never as a hung GPU.
#pragma once

#include <cuda.h>
#include <stdint.h>

namespace sm100 {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ------------------------------------------------------------------ mbarrier
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: polls, and every 256 probes checks the global nanosecond timer; a barrier
// that has not completed after MV_MBAR_TIMEOUT_NS flags *abort_flag (mapped host memory) and traps.
#ifndef MV_MBAR_TIMEOUT_NS
#define MV_MBAR_TIMEOUT_NS 10000000000ull
#endif
__device__ __forceinline__ uint64_t globaltimer_ns() {
  uint64_t t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
// `backoff_ns` > 0: sleep between probes -- for producer-side waits (a free slot), which are long
// and off the critical path; a spinning warp would otherwise take issue slots from the epilogue.
#ifdef MV_TC_TRACE
// debug build (-DMV_TC_TRACE): cycles spent in every wait site, summed over the grid
__device__ unsigned long long mv_tc_trace[16];
#define MV_TC_TRACE_ADD(who, c0) atomicAdd(&mv_tc_trace[(who)], (unsigned long long)(clock64() - (c0)))
#else
#define MV_TC_TRACE_ADD(who, c0)
#endif
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, int* abort_flag, int who,
                                          unsigned backoff_ns = 0) {
  uint64_t t0 = 0;
#ifdef MV_TC_TRACE
  const long long c0 = clock64();
#endif
  for (uint32_t i = 1;; i++) {
    if (mbar_try_wait(bar, parity)) { MV_TC_TRACE_ADD(who, c0); return; }
    if (backoff_ns) __nanosleep(backoff_ns);
    if (MV_MBAR_TIMEOUT_NS != 0 && (i & 255u) == 0) {
      const uint64_t t = globaltimer_ns();
      if (t0 == 0) t0 = t;
      else if (t - t0 > MV_MBAR_TIMEOUT_NS) break;
    }
  }
  if (abort_flag) {
    *reinterpret_cast<volatile int*>(abort_flag) = 0x1000 + who;
    __threadfence_system();
  }
  __trap();
}

// ------------------------------------------------------------------ proxies / fences
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// ------------------------------------------------------------------ TMA
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1,
                                            int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}

__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
// plain bulk copy global -> shared (16-byte aligned, size a multiple of 16), completion on an mbarrier
__device__ __forceinline__ void bulk_load(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(reinterpret_cast<uint64_t>(src)), "r"(bytes), "r"(bar)
               : "memory");
}

// ------------------------------------------------------------------ TMEM
__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(cols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// 32 lanes x 32 consecutive columns of 32-bit accumulators: thread l of the warp receives
// lane (base_lane + l), columns [col, col+32).  A warp may only touch lanes 32*(warpid%4)...
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, int (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
        "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
        "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}

// one column: thread l receives lane (base_lane + l), column col
__device__ __forceinline__ void tmem_ld_32x1(uint32_t taddr, int& v) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(v) : "r"(taddr) : "memory");
}

// ------------------------------------------------------------------ UMMA descriptors
// K-major operand, 64-byte rows, SWIZZLE_64B: 8 rows form a 512-byte atom in which the 16-byte
// chunk index is XORed with (row>>1)&3 -- what a TMA box with a 64-byte inner extent and
// CU_TENSOR_MAP_SWIZZLE_64B writes.  Field layout per the PTX ISA "shared memory descriptor":
// start>>4 [0,14), LBO>>4 [16,30), SBO>>4 [32,46), version=1 [46,48), layout [61,64).
constexpr uint32_t kSw64AtomBytes = 512;
__device__ __forceinline__ uint64_t umma_desc_k_sw64(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>(1) << 16;                       // LBO: unused for swizzled K-major
  d |= static_cast<uint64_t>(kSw64AtomBytes >> 4) << 32;     // SBO: next group of 8 rows
  d |= static_cast<uint64_t>(1) << 46;                       // descriptor version (Blackwell)
  d |= static_cast<uint64_t>(4) << 61;                       // SWIZZLE_64B
  return d;
}
// byte offset of 16-byte chunk `c` (0..3) of row `r` in that layout
__device__ __forceinline__ uint32_t sw64_offset(uint32_t r, uint32_t c) {
  return r * 64u + ((c ^ ((r >> 1) & 3u)) << 4);
}

// kind::i8, signed x signed -> s32, both operands K-major, dense.
//   c_format [4,6)=2 (S32), a_format [7,10)=1, b_format [10,13)=1 (INT8),
//   n>>3 [17,23), m>>4 [24,29)
__host__ __device__ constexpr uint32_t umma_idesc_s8(int m, int n) {
  return (2u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(n >> 3) << 17) |
         (static_cast<uint32_t>(m >> 4) << 24);
}

// D[tmem] (+)= A[smem] * B[smem]^T, one K=32 int8 step, issued by ONE thread.
__device__ __forceinline__ void umma_s8(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                        uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// mbarrier arrive once every MMA issued so far by this thread has completed (implies
// tcgen05.fence::before_thread_sync).
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar)
               : "memory");
}

__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

}  // namespace sm100

// ------------------------------------------------------------------ host: tensor maps
// The driver entry point is fetched through the runtime so the library needs no -lcuda.
#include <cuda_runtime.h>
typedef CUresult (*mv_tmap_encode_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                      const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                      CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                      CUtensorMapFloatOOBfill);
// Looked up on first use.  The initialiser of a function-local static is thread-safe, so contexts used from
// several threads at once may call this concurrently.
static inline mv_tmap_encode_fn mv_get_tmap_encode() {
  static const mv_tmap_encode_fn fn = []() -> mv_tmap_encode_fn {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      return reinterpret_cast<mv_tmap_encode_fn>(p);
    return nullptr;
  }();
  return fn;
}
