// Shared helpers for the b200rl CUDA library (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <string>

#include "b200rl.h"

namespace b200rl {

void set_error(const char* fmt, ...);
void count_launch();
// gemm_simt.cu: index in [0, 64) of `s` for the per-stream last-CTA tickets of single-launch reductions (-1 once 64
// streams have been seen)
int ticket_for(cudaStream_t s);

#define B200RL_CUDA_OK(expr)                                                              \
  do {                                                                                    \
    cudaError_t _e = (expr);                                                              \
    if (_e != cudaSuccess) {                                                              \
      ::b200rl::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return B200RL_ECUDA;                                                                \
    }                                                                                     \
  } while (0)

#define B200RL_REQUIRE(cond, ...)          \
  do {                                     \
    if (!(cond)) {                         \
      ::b200rl::set_error(__VA_ARGS__);    \
      return B200RL_EINVAL;                \
    }                                      \
  } while (0)

#define B200RL_LAUNCH_OK()                                                                 \
  do {                                                                                     \
 ::b200rl::count_launch();                                                                \
    cudaError_t _e = cudaGetLastError();                                                   \
    if (_e != cudaSuccess) {                                                               \
      ::b200rl::set_error("kernel launch failed: %s (%s:%d)", cudaGetErrorString(_e), __FILE__, __LINE__); \
      return B200RL_ECUDA;                                                                 \
    }                                                                                      \
  } while (0)

constexpr int kFanout = 32;
constexpr int kMaxLevels = 8;
constexpr int kNumSMs = 148;

// Device view of the fan-out-32 sum tree: lvl[0] = root (1 float) .. lvl[L] = leaf weights (raw child
// values); pre[l] = sequential fp32 inclusive prefixes of every node's 32 children at level l.
struct TreeView {
  float* lvl[kMaxLevels];
  float* pre[kMaxLevels];
  int64_t width[kMaxLevels];
  int32_t L;
};

// Live key range of the item ring, kept in device memory so graph replays see fresh values.
struct ReplayState {
  unsigned long long item_head;  // next key to be issued
  unsigned long long item_tail;  // oldest live key
};

// Philox4x32-10 uniform in [0,1) for (element i, draw counter `step`) keyed by `seed`: the learner's device-side uniform
// stream (b200rl_uniform) and K1's built-in draws (b200rl_replay_sample_philox) are the same function.
#ifdef __CUDACC__
__device__ __forceinline__ float philox_uniform(unsigned int i, unsigned long long seed, unsigned long long step) {
  unsigned int c0 = i, c1 = 0u, c2 = (unsigned int)step, c3 = (unsigned int)(step >> 32);
  unsigned int k0 = (unsigned int)seed, k1 = (unsigned int)(seed >> 32);
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const unsigned int hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const unsigned int hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    const unsigned int n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  return (float)(c0 >> 8) * (1.0f / 16777216.0f);  // 24 bits -> [0,1), exact in fp32
}
#endif

static inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

// Programmatic dependent launch (B200RL_PDL=1).  A learner step is a chain of ~16 short kernels, each waiting for the
// one before it; with a programmatic edge the next kernel's CTAs are scheduled while the previous kernel drains and run
// their set-up (barrier init, TMEM allocation, tensor-map prefetch) up to `pdl_wait()`, which returns when every
// prerequisite grid has completed and its memory is visible.  Kernels call pdl_launch_dependents() first thing and
// pdl_wait() before their first access to global memory; both are no-ops in a launch without the attribute, so only
// kernels that contain pdl_wait() may be launched through launch_pdl().
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

#define B200RL_PDL_DEFAULT true    // measured on B200: 0.289 -> 0.269 ms per DQN step (gpurun_out/c3_*, c4_*)
#define B200RL_PDL_LATE_DEFAULT 1   // trigger at accumulator-ready: 0.276 -> 0.269 ms
bool pdl_enabled();   // replay.cu: B200RL_PDL (or b200rl_debug_set_pdl)
int pdl_late_mode();  // replay.cu: B200RL_PDL_LATE

// Two domains.  launch_pdl: the tensor-core GEMM / convolution kernels and the kernels between them on the DQN step's
// critical path (10-30 us each: scheduling the next grid during the previous one's epilogue pays; measured 0.291 -> 0.271
// ms per step).  launch_pdl_small: the FFMA GEMM and the element-wise / reduction kernels of a few microseconds that
// make up the D4PG step and the fp32 parity mode -- there the programmatic edges cost more than they hide (measured with
// them on: D4PG 0.267 -> 0.317 ms, fp32 DQN 2.41 -> 2.69 ms), so that domain is off unless B200RL_PDL_SMALL=1.
bool pdl_small_enabled();
template <typename... KArgs, typename... Args>
static inline cudaError_t launch_pdl_on(bool on, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                                        Args&&... args);
template <typename... KArgs, typename... Args>
static inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args&&... args) {
  return launch_pdl_on(pdl_enabled(), kernel, grid, block, smem, stream, static_cast<Args&&>(args)...);
}
template <typename... KArgs, typename... Args>
static inline cudaError_t launch_pdl_small(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                                           Args&&... args) {
  return launch_pdl_on(pdl_enabled() && pdl_small_enabled(), kernel, grid, block, smem, stream, static_cast<Args&&>(args)...);
}
template <typename... KArgs, typename... Args>
static inline cudaError_t launch_pdl_on(bool on, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                                        Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = on ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<Args&&>(args)...);
}
#endif

template <typename T>
static inline T ceil_div(T a, T b) {
  return (a + b - 1) / b;
}

}  // namespace b200rl
