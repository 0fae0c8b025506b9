// mv_common.cuh -- context, error plumbing and launch helpers shared by the kernels
// of libmaveric_b200.so (sm_100a only; there is deliberately no host fallback).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <map>
#include <string>
#include <vector>

#include "../../include/maveric_b200.h"

struct mv_prof_slot {
  double ms = 0.0;
  int launches = 0;
};

struct mv_pending_event {
  std::string tag;
  cudaEvent_t beg, end;
};

struct mv_ctx {
  int device = 0;
  int sm_count = 148;
  cudaStream_t stream = nullptr;      // compute stream (owned unless set_stream)
  bool own_stream = true;
  cudaStream_t copy_stream = nullptr; // host-buffer sequence call: logits DMA + detector (high priority)
  cudaStream_t gather_stream = nullptr; // host-buffer sequence call: selective descriptor staging
  int pnp_max_ctas_per_sm = 0;        // >0: cap K3 residency so staging kernels can co-reside
  char err[512] = {0};
  unsigned long long launches = 0;
  bool profile = false;
  bool pnp_work_live = false;           // profile mode: the PnP work counter holds launches not yet read
  int match_items = 0;                  // tiles of the last tensor-core matcher launch (mv_ctx_match_work)
  int bow_n_base = 0, bow_wpb = 0;      // vocabulary on the device (mv_bow_set_vocabulary)
  size_t bow_smem_attr = 0;             // dynamic shared memory the word-assignment kernel is allowed so far
  int lm_words = 0;                     // size the landmark scratch was initialised for
  std::map<std::string, mv_prof_slot> prof;
  std::vector<mv_pending_event> pending;

  // scratch arena, grown on demand, never shrunk; owned by the context
  std::map<std::string, std::pair<void*, size_t>> scratch;
  // Wait-site diagnostic of the mbarrier pipelines (tcgen05 matcher, TMA row gather): one int in mapped
  // pinned host memory, written by a kernel just before it traps on a barrier that never completed.  Host
  // memory survives the sticky error a trap leaves behind, so MV_CUDA can still name the wait site.
  int* abort_host = nullptr;
  // pinned host mirror for small synchronous host-pointer calls
  void* pinned = nullptr;
  size_t pinned_bytes = 0;
};

#define MV_CUDA(ctx, call)                                                          \
  do {                                                                              \
    cudaError_t e__ = (call);                                                       \
    if (e__ != cudaSuccess) {                                                       \
      const int site__ = (ctx)->abort_host ? *(volatile int*)(ctx)->abort_host : 0; \
      snprintf((ctx)->err, sizeof((ctx)->err), "%s:%d %s -> %s%s%.0d", __FILE__, __LINE__, \
               #call, cudaGetErrorString(e__),                                      \
               site__ ? " (an mbarrier wait timed out in a pipeline kernel, wait site " : "", \
               site__ ? site__ - 0x1000 : 0);                                       \
      return MV_ERR_CUDA;                                                           \
    }                                                                               \
  } while (0)

mv_status mv_abort_flag(mv_ctx* ctx, int** out);

#define MV_CHECK_LAUNCH(ctx)                                                        \
  do {                                                                              \
    (ctx)->launches++;                                                              \
    cudaError_t e__ = cudaGetLastError();                                           \
    if (e__ != cudaSuccess) {                                                       \
      snprintf((ctx)->err, sizeof((ctx)->err), "%s:%d launch -> %s", __FILE__,      \
               __LINE__, cudaGetErrorString(e__));                                  \
      return MV_ERR_CUDA;                                                           \
    }                                                                               \
  } while (0)

#define MV_BAD_ARG(ctx, msg)                                              \
  do {                                                                    \
    snprintf((ctx)->err, sizeof((ctx)->err), "bad argument: %s", msg);    \
    return MV_ERR_BAD_ARG;                                                \
  } while (0)

// Scoped per-tag device timing (CUDA events on the compute stream), on when the
// context is in profile mode.  Results are folded in by mv_ctx_profile_read().
struct mv_prof_scope {
  mv_ctx* ctx;
  mv_pending_event ev;
  bool on;
  mv_prof_scope(mv_ctx* c, const char* tag) : ctx(c), on(c->profile) {
    if (!on) return;
    ev.tag = tag;
    cudaEventCreate(&ev.beg);
    cudaEventCreate(&ev.end);
    cudaEventRecord(ev.beg, ctx->stream);
  }
  ~mv_prof_scope() {
    if (!on) return;
    cudaEventRecord(ev.end, ctx->stream);
    ctx->pending.push_back(ev);
  }
};


// Device contract (include/maveric_b200.h): a context belongs to one GPU; every entry point that takes
// a context makes that GPU current for the duration of the call and restores the caller's device on
// return, so contexts of different GPUs may be used from one thread and a context from any thread.
struct mv_device_guard {
  int prev = -1;
  bool switched = false;
  explicit mv_device_guard(int device) {
    if (cudaGetDevice(&prev) != cudaSuccess) { cudaGetLastError(); prev = -1; }
    if (prev != device) switched = cudaSetDevice(device) == cudaSuccess;
  }
  ~mv_device_guard() {
    if (switched && prev >= 0) cudaSetDevice(prev);
  }
};
#define MV_ENTER(ctx)                       \
  if (!(ctx)) return MV_ERR_BAD_ARG;        \
  mv_device_guard mv_guard__((ctx)->device)

mv_status mv_scratch(mv_ctx* ctx, const char* name, size_t bytes, void** out);
mv_status mv_pinned(mv_ctx* ctx, size_t bytes, void** out);

// ---- landmark sequence path (bow.cu), called by mv_track_sequence_landmarks (api.cu)
// Back-projection of every query keypoint with its frame's depth, fused into the word assignment launch:
// coords [n_frames][top_n][3] (zeros beyond the query count); nothing is written when coords is NULL.
struct MvBackProject {
  const int32_t* q_idx = nullptr;
  const float* depth = nullptr;
  int rows = 0;
  float fx = 0.0f, fy = 0.0f, cx = 0.0f, cy = 0.0f;
  float* coords = nullptr;
};
mv_status mv_bow_assign_impl(mv_ctx* ctx, int n_frames, int cells, int top_n, const int8_t* d_desc,
                             const float* d_desc_scale, const int32_t* d_q_patch, const int32_t* d_q_count,
                             int32_t* d_word, int32_t* d_base, const MvBackProject& bp);
mv_status mv_landmarks_sequence_impl(mv_ctx* ctx, int n_words, mv_landmark* d_table, int first_frame, int n_steps,
                                     int top_n, const int32_t* d_word, const int32_t* d_q_count,
                                     const float* d_coords_in, float* d_coords_out);
// allocates the scratch mv_landmarks_sequence_impl needs for n_steps steps (callers that must not grow scratch
// while other streams run, i.e. the host-buffer pipeline, reserve it for their largest call up front)
mv_status mv_landmarks_sequence_reserve(mv_ctx* ctx, int n_words, int n_steps, int top_n);
// mv_build_corr_landmarks_batch for pairs (p, p+1) with the 3-D side from mv_landmarks_sequence's coords_out
mv_status mv_build_corr_landmarks_seq(mv_ctx* ctx, int n_pairs, int top_n, int stride, int n_words,
                                      const int32_t* d_q_patch, const int32_t* d_q_count, const int32_t* d_word,
                                      const float* d_coords_out, const float* d_match_pts, const int32_t* d_match_count,
                                      const int32_t* d_match_cell0, float* d_corr, int32_t* d_n_with_landmark);

// float bounds that make a float-vs-double comparison exact in fp32:
//   (double)s >  T  <=>  s >  mv_round_down(T)
//   (double)s <  T  <=>  s <  mv_round_up(T)
static inline float mv_round_down(double t) {
  float f = (float)t;
  if ((double)f > t) f = nextafterf(f, -INFINITY);
  return f;
}
static inline float mv_round_up(double t) {
  float f = (float)t;
  if ((double)f < t) f = nextafterf(f, INFINITY);
  return f;
}

// ---- counter-based random numbers (same as oracle/ and synth.py) ----
__host__ __device__ static inline uint64_t mv_sm64(uint64_t x) {
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}
__host__ __device__ static inline uint64_t mv_ctr(uint64_t mixed_seed, uint64_t tag, uint64_t a,
                                                  uint64_t b, uint64_t c) {
  return mv_sm64(mixed_seed + ((tag << 56) | ((a & 0xFFFFFFull) << 32) | ((b & 0xFFFFFFull) << 8) |
                               (c & 0xFFull)));
}

