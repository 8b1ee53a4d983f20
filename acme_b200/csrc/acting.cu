// Exploration for the batched actor: epsilon-greedy action selection over Q rows and clipped Gaussian action noise, both
// drawing from the device Philox stream (philox_uniform, the function b200rl_uniform evaluates) at a draw counter read
// from device memory, so a captured act step draws fresh numbers on every replay once the counter is advanced.
#include "common.cuh"

namespace b200rl {

// One warp per row.  Lane j holds q[j], q[j + 32], ...; the row maximum is a warp max, the tied actions are counted with
// ballots over the same 32-wide chunks, and the t-th tie (index order) is found chunk by chunk.
__global__ void epsilon_greedy_kernel(int N, int A, const float* __restrict__ q, long long ldq, float epsilon,
                                      unsigned long long seed, const long long* __restrict__ counter,
                                      int32_t* __restrict__ actions, float* __restrict__ u_out) {
  const int lane = threadIdx.x & 31;
  const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= N) return;
  const unsigned long long step = (unsigned long long)*counter;
  const float u0 = philox_uniform(2u * (unsigned)r, seed, step);
  const float u1 = philox_uniform(2u * (unsigned)r + 1u, seed, step);
  const float* row = q + (long long)r * ldq;
  int action;
  if (u0 < epsilon) {
    action = min((int)floorf(__fmul_rn(u1, (float)A)), A - 1);
  } else {
    float m = -INFINITY;
    for (int j = lane; j < A; j += 32) m = fmaxf(m, row[j]);
#pragma unroll
    for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    int k = 0;
    for (int j0 = 0; j0 < A; j0 += 32) {
      const int j = j0 + lane;
      k += __popc(__ballot_sync(0xffffffffu, j < A && row[j] == m));
    }
    int t = min((int)floorf(__fmul_rn(u1, (float)k)), k - 1);
    action = A - 1;   // kept only when no element equals the maximum (an all-NaN row): k = 0
    for (int j0 = 0; j0 < A && k > 0; j0 += 32) {
      const int j = j0 + lane;
      const unsigned ties = __ballot_sync(0xffffffffu, j < A && row[j] == m);
      const int c = __popc(ties);
      if (t < c) {
        unsigned b = ties;
        for (int s = 0; s < t; ++s) b &= b - 1;   // drop the t lowest set bits
        action = j0 + __ffs(b) - 1;
        break;
      }
      t -= c;
    }
  }
  if (lane == 0) {
    actions[r] = action;
    if (u_out) { u_out[2 * r] = u0; u_out[2 * r + 1] = u1; }
  }
}

// out = clip(fl(a + fl(z * sigma)), lo, hi), z = sqrtf(-2 logf(1 - u_2m)) cosf(2 pi u_2m+1), m = r * A + j.
__global__ void gaussian_explore_kernel(long long n, int A, const float* __restrict__ a, float sigma, const float* __restrict__ lo,
                                        const float* __restrict__ hi, unsigned long long seed,
                                        const long long* __restrict__ counter, float* __restrict__ out, float* __restrict__ z_out) {
  const long long m = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= n) return;
  const unsigned long long step = (unsigned long long)*counter;
  const float u0 = philox_uniform(2u * (unsigned)m, seed, step);
  const float u1 = philox_uniform(2u * (unsigned)m + 1u, seed, step);
  const float z = __fmul_rn(sqrtf(__fmul_rn(-2.0f, logf(__fsub_rn(1.0f, u0)))), cosf(__fmul_rn(6.283185307179586f, u1)));
  const int j = (int)(m % A);
  out[m] = fminf(fmaxf(__fadd_rn(a[m], __fmul_rn(z, sigma)), lo[j]), hi[j]);
  if (z_out) z_out[m] = z;
}

}  // namespace b200rl

using namespace b200rl;

extern "C" int b200rl_epsilon_greedy(int32_t N, int32_t A, const float* q, int64_t ldq, float epsilon, uint64_t seed,
                                     const int64_t* counter_dev, int32_t* actions_out, float* u_out, void* stream) {
  B200RL_REQUIRE(q && counter_dev && actions_out, "null argument");
  B200RL_REQUIRE(N >= 0 && A >= 1 && ldq >= A, "bad shape: N %d, A %d, ldq %lld", N, A, (long long)ldq);
  B200RL_REQUIRE(N <= (1 << 30), "N %d exceeds the Philox element range (2N draws)", N);
  if (N == 0) return B200RL_OK;
  constexpr int kRowsPerBlock = 8;
  epsilon_greedy_kernel<<<ceil_div(N, kRowsPerBlock), kRowsPerBlock * 32, 0, as_stream(stream)>>>(
      N, A, q, (long long)ldq, epsilon, (unsigned long long)seed, (const long long*)counter_dev, actions_out, u_out);
  B200RL_LAUNCH_OK();
  return B200RL_OK;
}

extern "C" int b200rl_gaussian_explore(int32_t N, int32_t A, const float* a, float sigma, const float* lo, const float* hi,
                                       uint64_t seed, const int64_t* counter_dev, float* out, float* z_out, void* stream) {
  B200RL_REQUIRE(a && lo && hi && counter_dev && out, "null argument");
  B200RL_REQUIRE(N >= 0 && A >= 1, "bad shape: N %d, A %d", N, A);
  const long long n = (long long)N * A;
  B200RL_REQUIRE(n <= (1ll << 30), "N * A = %lld exceeds the Philox element range (2 N A draws)", n);
  if (n == 0) return B200RL_OK;
  gaussian_explore_kernel<<<(int)ceil_div<long long>(n, 256), 256, 0, as_stream(stream)>>>(
      n, A, a, sigma, lo, hi, (unsigned long long)seed, (const long long*)counter_dev, out, z_out);
  B200RL_LAUNCH_OK();
  return B200RL_OK;
}
