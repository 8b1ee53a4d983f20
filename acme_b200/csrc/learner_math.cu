// K4 (double-Q TD / Huber / importance weights / priorities), K5 (C51 projection + cross-entropy),
// K7 (Adam, global-norm clip, target copy) and the small element-wise pieces of the networks.
// Each kernel cites the reference lines it restates; all are HBM-bound and deterministic
// (fixed-order reductions, no atomics).
#include <algorithm>

#include <cstdlib>
#include "common.cuh"

#include <cuda_bf16.h>

namespace b200rl {

// ------------------------------------------------------------------------------ Philox4x32-10 (common.cuh)
__global__ void uniform_kernel(float* __restrict__ out, int n, unsigned long long seed,
                               const long long* __restrict__ step_dev, long long step_offset) {
  pdl_launch_dependents();
  pdl_wait();
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const unsigned long long step = (unsigned long long)((step_dev ? *step_dev : 0) + step_offset);
  out[i] = philox_uniform((unsigned int)i, seed, step);
}

// ------------------------------------------------------------------------------ block reductions
template <typename T, typename Op>
__device__ __forceinline__ T block_reduce(T v, Op op, T identity, T* scratch /* >= 32 */) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) v = op(v, __shfl_xor_sync(0xffffffffu, v, d));
  __syncthreads();
  if (lane == 0) scratch[warp] = v;
  __syncthreads();
  v = (threadIdx.x < nw) ? scratch[threadIdx.x] : identity;
  if (warp == 0) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v = op(v, __shfl_xor_sync(0xffffffffu, v, d));
  }
  __syncthreads();
  if (threadIdx.x == 0) scratch[0] = v;
  __syncthreads();
  v = scratch[0];
  return v;
}

struct MaxD { __device__ double operator()(double a, double b) const { return a > b ? a : b; } };
struct SumF { __device__ float operator()(float a, float b) const { return a + b; } };
struct MaxF { __device__ float operator()(float a, float c) const { return fmaxf(a, c); } };
struct SumD { __device__ double operator()(double a, double b) const { return a + b; } };

// ------------------------------------------------------------------------------------------ K4
// acme/agents/tf/dqn/learning.py:127-154; trfl.double_qlearning; acme/tf/losses/huber.py:48-57.
// importance weight before normalisation: TF learner (f64, learning.py:138-139) or JAX learner (f32, jax learning.py:94-95)
__device__ __forceinline__ double is_weight_raw(float prob, double beta, int flags) {
  if (flags & B200RL_TD_IS_WEIGHTS_F32) return (double)powf((float)(1.0 / (double)prob), (float)beta);
  return pow(1.0 / (double)prob, beta);
}
__device__ __forceinline__ float is_weight_norm(double raw, double wmax, int flags) {
  if (flags & B200RL_TD_IS_WEIGHTS_F32) return __fdiv_rn((float)raw, (float)wmax);
  return (float)(raw / wmax);
}

__global__ void __launch_bounds__(1024)
is_weight_max_kernel(int B, const float* __restrict__ prob, double beta, double* __restrict__ out, int flags) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ double scratch[32];
  double m = 0.0;
  for (int b = threadIdx.x; b < B; b += blockDim.x) m = fmax(m, is_weight_raw(prob[b], beta, flags));
  m = block_reduce(m, MaxD(), 0.0, scratch);
  if (threadIdx.x == 0) *out = m;
}

__global__ void __launch_bounds__(1024)
dqn_td_kernel(int B, int A, const float* __restrict__ q_tm1, const float* __restrict__ q_tv,
              const float* __restrict__ q_ts, const int* __restrict__ a_tm1,
              const float* __restrict__ R, const float* __restrict__ D, const float* __restrict__ prob,
              float gamma, float delta, double beta, float max_abs_r, const double* __restrict__ wmax_dev,
              float grad_scale, float* __restrict__ td_out, float* __restrict__ loss_ps,
              float* __restrict__ weight, float* __restrict__ priority, float* __restrict__ dq,
              float* __restrict__ loss_mean, int flags) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ double scratch_d[32];
  __shared__ float scratch_f[32];
  double wmax = 0.0;
  for (int b = threadIdx.x; b < B; b += blockDim.x) wmax = fmax(wmax, is_weight_raw(prob[b], beta, flags));
  if (wmax_dev) wmax = *wmax_dev;                          // global max (data-parallel learners)
  else wmax = block_reduce(wmax, MaxD(), 0.0, scratch_d);  // tf.reduce_max, learning.py:140
  float lsum = 0.f;
  for (int b = threadIdx.x; b < B; b += blockDim.x) {
    const float* sel = q_ts + (size_t)b * A;
    int best = 0;
    float bv = sel[0];
    for (int a = 1; a < A; ++a) {
      float v = sel[a];
      if (v > bv) { bv = v; best = a; }   // first maximum wins
    }
    float r = fminf(fmaxf(R[b], -max_abs_r), max_abs_r);          // learning.py:129
    float d = __fmul_rn(D[b], gamma);                             // learning.py:130
    float target = __fadd_rn(r, __fmul_rn(d, q_tv[(size_t)b * A + best]));
    const int act = a_tm1[b];
    float td = __fsub_rn(target, q_tm1[(size_t)b * A + act]);
    float absx = fabsf(td);
    float quad = fminf(absx, delta);
    float lin = __fsub_rn(absx, quad);
    float hub = __fadd_rn(__fmul_rn(__fmul_rn(0.5f, quad), quad), __fmul_rn(delta, lin));
    float w = is_weight_norm(is_weight_raw(prob[b], beta, flags), wmax, flags);   // f64 then cast, learning.py:138-143
    float l = __fmul_rn(hub, w);
    td_out[b] = td;
    loss_ps[b] = l;
    weight[b] = w;
    priority[b] = absx;                                           // learning.py:152 (no epsilon)
    float g = -(w * grad_scale) * fminf(fmaxf(td, -delta), delta);
    for (int a = 0; a < A; ++a) dq[(size_t)b * A + a] = (a == act) ? g : 0.f;
    lsum += l;
  }
  lsum = block_reduce(lsum, SumF(), 0.f, scratch_f);
  if (threadIdx.x == 0 && loss_mean) *loss_mean = lsum / (float)B;
}

// ------------------------------------------------------------------------------------------ K5
// Prioritized form of the critic losses (b200rl_c51_loss_weighted / b200rl_td_learning_weighted): the kernels below are
// templated on W.  W = false is the uniform loss; W = true adds, per sample, the importance weight of b200rl_dqn_td
// (flags 0) against the precomputed batch maximum, the weighted loss, the priority and the weighted gradient, and the
// batch mean of the weighted losses in the same launch: every warp that has written its samples' losses counts them on a
// per-stream ticket, and the warp that brings the count to B adds loss_ps[0..B) in index order (lane l takes l, l + 32,
// ... sequentially, then a fixed butterfly) and resets the ticket, so the mean is bit-identical across launches, streams
// and graph replays.
struct IsWeighted {
  const float* prob;
  double beta;
  const double* wmax;
  float* weight;
  float* priority;
  float* loss_mean;
  int ticket;   // slot in g_loss_tickets
  int B;
};
__device__ unsigned int g_loss_tickets[64];

__device__ __forceinline__ float is_weight_of(const IsWeighted& iw, int b) {
  return is_weight_norm(is_weight_raw(iw.prob[b], iw.beta, 0), *iw.wmax, 0);   // learning.py:138-143
}

// called by all 32 lanes of a warp after its `n` samples' loss_ps have been written (by any of its lanes)
__device__ __forceinline__ void weighted_mean_tail(const IsWeighted& iw, const float* loss_ps, int n) {
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  if (!iw.loss_mean || n == 0) return;
  __threadfence();
  __syncwarp();
  unsigned int old = 0;
  if (lane == 0) old = atomicAdd(&g_loss_tickets[iw.ticket], (unsigned int)n);
  old = __shfl_sync(full, old, 0);
  if (old + (unsigned int)n != (unsigned int)iw.B) return;
  __threadfence();
  float s = 0.f;
  for (int i = lane; i < iw.B; i += 32) s = __fadd_rn(s, __ldcg(loss_ps + i));
  for (int o = 16; o; o >>= 1) s = __fadd_rn(s, __shfl_xor_sync(full, s, o));
  if (lane == 0) {
    *iw.loss_mean = s / (float)iw.B;
    g_loss_tickets[iw.ticket] = 0u;
  }
}

// acme/tf/losses/distributional.py:22-83.  One CTA per sample; thread i owns atom i and evaluates
// the dense projection row sum_j clip(1 - |clip(z'_j) - z_i| / delta_i, 0, 1) * p_j with p, z' in
// shared memory -- the reference's arithmetic without materialising [B,K,K].
__device__ __forceinline__ float atom_value(int i, int K, float vmin, float vmax) {
  if (i == K - 1) return vmax;
  double step = ((double)vmax - (double)vmin) / (double)(K - 1);
  return (float)((double)vmin + (double)i * step);   // np.linspace(..., dtype=float32)
}

template <bool W>
__global__ void c51_loss_kernel(int K, float vmin, float vmax, const float* __restrict__ logits_tm1,
                                const float* __restrict__ logits_t, const float* __restrict__ R,
                                const float* __restrict__ D, float gamma, float grad_scale,
                                float* __restrict__ target_out, float* __restrict__ loss_ps,
                                float* __restrict__ dlogits, IsWeighted iw) {
  pdl_launch_dependents();
  pdl_wait();
  extern __shared__ float sm[];
  float* p = sm;          // softmax(logits_t)          [K]
  float* zc = sm + K;     // clip(R + Dg * z_j)         [K]
  float* zq = sm + 2 * K; // support                    [K]
  __shared__ float scratch[32];
  const int b = blockIdx.x, i = threadIdx.x;
  const bool on = i < K;
  const float lt = on ? logits_t[(size_t)b * K + i] : -INFINITY;
  float mx = block_reduce(lt, MaxF(), -INFINITY, scratch);
  float e = on ? expf(lt - mx) : 0.f;
  float se = block_reduce(e, SumF(), 0.f, scratch);
  const float zi = on ? atom_value(i, K, vmin, vmax) : 0.f;
  if (on) {
    p[i] = e / se;
    float dg = __fmul_rn(gamma, D[b]);                            // discount * d_t, learning.py:202
    float z = __fadd_rn(R[b], __fmul_rn(dg, zi));                 // distributional.py:27
    zc[i] = fminf(fmaxf(z, vmin), vmax);
    zq[i] = zi;
  }
  __syncthreads();
  float tgt = 0.f;
  if (on) {
    // distributional.py:66-76: d_pos = z_{i+1}-z_i (vmin-z_i at the top), d_neg = z_i-z_{i-1} (z_0-vmax at 0)
    const float d_pos = (i + 1 < K ? zq[i + 1] : vmin) - zi;
    const float d_neg = zi - (i > 0 ? zq[i - 1] : vmax);
    for (int j = 0; j < K; ++j) {
      float delta = zc[j] - zi;
      float dh = (delta >= 0.f) ? (delta / d_pos) : -(delta / d_neg);
      float wgt = fminf(fmaxf(1.f - dh, 0.f), 1.f);
      tgt = __fadd_rn(tgt, __fmul_rn(wgt, p[j]));
    }
    if (target_out) target_out[(size_t)b * K + i] = tgt;
  }
  // softmax cross-entropy of logits_tm1 against the (stop-gradient) target
  const float l1 = on ? logits_tm1[(size_t)b * K + i] : -INFINITY;
  float m1 = block_reduce(l1, MaxF(), -INFINITY, scratch);
  float e1 = on ? expf(l1 - m1) : 0.f;
  float s1 = block_reduce(e1, SumF(), 0.f, scratch);
  float lse = m1 + logf(s1);
  float contrib = on ? -tgt * (l1 - lse) : 0.f;
  float loss = block_reduce(contrib, SumF(), 0.f, scratch);
  float tsum = block_reduce(tgt, SumF(), 0.f, scratch);
  if constexpr (W) {
    const float w = is_weight_of(iw, b);
    const float gs = __fmul_rn(w, grad_scale);
    if (on && dlogits) dlogits[(size_t)b * K + i] = ((e1 / s1) * tsum - tgt) * gs;
    if (i == 0) {
      loss_ps[b] = __fmul_rn(loss, w);
      iw.weight[b] = w;
      iw.priority[b] = loss;
    }
    if (threadIdx.x < 32) weighted_mean_tail(iw, loss_ps, 1);
  } else {
    if (on && dlogits) dlogits[(size_t)b * K + i] = ((e1 / s1) * tsum - tgt) * grad_scale;
    if (i == 0 && loss_ps) loss_ps[b] = loss;
  }
}

// K5, K <= 64: ONE WARP per sample (lane owns atoms lane and lane + 32), no block barriers, and the projection row of
// atom i only visits the source atoms that can reach it.  clip(R + dg * z_j) is non-decreasing in j for dg >= 0, so the
// sources with a non-zero triangular weight for atom i are the contiguous range z_{i-1} < z'_j < z_{i+1}, found by two
// binary searches in shared memory; every term outside it is an exact +0 in the dense sum above (weight clamped to 0,
// p_j >= 0), so visiting only the range in ascending j gives the SAME bits as the dense O(K^2) loop at O(K) cost
// (dg < 0 -- never produced by the learners -- takes the dense loop).  At B = 65,536 the dense one-CTA-per-sample kernel
// ran at 3 % of the HBM roofline, bound by 2,601 IEEE divisions per sample.
constexpr int kC51WarpsPerCta = 8;
template <bool W>
__global__ void __launch_bounds__(32 * kC51WarpsPerCta)
c51_loss_warp_kernel(int B, int K, float vmin, float vmax, const float* __restrict__ logits_tm1,
                     const float* __restrict__ logits_t, const float* __restrict__ R, const float* __restrict__ D,
                     float gamma, float grad_scale, float* __restrict__ target_out, float* __restrict__ loss_ps,
                     float* __restrict__ dlogits, IsWeighted iw) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ float s_p[kC51WarpsPerCta][64], s_zc[kC51WarpsPerCta][64];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x * kC51WarpsPerCta + w;
  if (b >= B) return;   // whole warps leave together; no block-level barrier below
  float* p = s_p[w];
  float* zc = s_zc[w];
  const unsigned full = 0xffffffffu;
  auto wmax = [&](float x) { for (int o = 16; o; o >>= 1) x = fmaxf(x, __shfl_xor_sync(full, x, o)); return x; };
  auto wsum = [&](float x) { for (int o = 16; o; o >>= 1) x += __shfl_xor_sync(full, x, o); return x; };
  const int i0 = lane, i1 = lane + 32;
  const bool on0 = i0 < K, on1 = i1 < K;
  const size_t row = (size_t)b * K;
  // softmax(logits_t)
  const float lt0 = on0 ? logits_t[row + i0] : -INFINITY, lt1 = on1 ? logits_t[row + i1] : -INFINITY;
  const float mx = wmax(fmaxf(lt0, lt1));
  const float e0 = on0 ? expf(lt0 - mx) : 0.f, e1 = on1 ? expf(lt1 - mx) : 0.f;
  const float se = wsum(e0 + e1);
  const float z0 = on0 ? atom_value(i0, K, vmin, vmax) : 0.f, z1 = on1 ? atom_value(i1, K, vmin, vmax) : 0.f;
  const float dg = __fmul_rn(gamma, D[b]);                            // discount * d_t, learning.py:202
  const float Rb = R[b];
  if (on0) { p[i0] = e0 / se; zc[i0] = fminf(fmaxf(__fadd_rn(Rb, __fmul_rn(dg, z0)), vmin), vmax); }   // distributional.py:27
  if (on1) { p[i1] = e1 / se; zc[i1] = fminf(fmaxf(__fadd_rn(Rb, __fmul_rn(dg, z1)), vmin), vmax); }
  __syncwarp();
  // neighbours of my atoms in the support (distributional.py:66-76: the edge spacings wrap to vmin / vmax)
  const float zp0 = __shfl_up_sync(full, z0, 1), zn0 = __shfl_down_sync(full, z0, 1);
  const float zp1 = __shfl_up_sync(full, z1, 1), zn1 = __shfl_down_sync(full, z1, 1);
  const float z1_first = __shfl_sync(full, z1, 0), z0_last = __shfl_sync(full, z0, 31);
  auto project = [&](int i, float zi, float below, float above) -> float {
    // below / above = z_{i-1} / z_{i+1} where they exist
    const float d_pos = (i + 1 < K ? above : vmin) - zi;
    const float d_neg = zi - (i > 0 ? below : vmax);
    int lo = 0, hi = K;
    if (dg >= 0.f) {
      if (i > 0) {              // first j with z'_j > z_{i-1}
        int a = 0, c = K;
        while (a < c) { const int mid = (a + c) >> 1; if (zc[mid] > below) c = mid; else a = mid + 1; }
        lo = a;
      }
      if (i + 1 < K) {          // first j with z'_j >= z_{i+1}
        int a = lo, c = K;
        while (a < c) { const int mid = (a + c) >> 1; if (zc[mid] >= above) c = mid; else a = mid + 1; }
        hi = a;
      }
    }
    float tgt = 0.f;
    for (int j = lo; j < hi; ++j) {
      const float delta = zc[j] - zi;
      const float dh = (delta >= 0.f) ? (delta / d_pos) : -(delta / d_neg);
      const float wgt = fminf(fmaxf(1.f - dh, 0.f), 1.f);
      tgt = __fadd_rn(tgt, __fmul_rn(wgt, p[j]));
    }
    return tgt;
  };
  const float t0 = on0 ? project(i0, z0, zp0, lane == 31 ? z1_first : zn0) : 0.f;
  const float t1 = on1 ? project(i1, z1, lane == 0 ? z0_last : zp1, zn1) : 0.f;
  if (target_out) {
    if (on0) target_out[row + i0] = t0;
    if (on1) target_out[row + i1] = t1;
  }
  // softmax cross-entropy of logits_tm1 against the (stop-gradient) target
  const float l0 = on0 ? logits_tm1[row + i0] : -INFINITY, l1 = on1 ? logits_tm1[row + i1] : -INFINITY;
  const float m1 = wmax(fmaxf(l0, l1));
  const float f0 = on0 ? expf(l0 - m1) : 0.f, f1 = on1 ? expf(l1 - m1) : 0.f;
  const float s1 = wsum(f0 + f1);
  const float lse = m1 + logf(s1);
  const float loss = wsum((on0 ? -t0 * (l0 - lse) : 0.f) + (on1 ? -t1 * (l1 - lse) : 0.f));
  const float tsum = wsum(t0 + t1);
  if constexpr (W) {
    const float w = is_weight_of(iw, b);
    const float gs = __fmul_rn(w, grad_scale);
    if (dlogits) {
      if (on0) dlogits[row + i0] = ((f0 / s1) * tsum - t0) * gs;
      if (on1) dlogits[row + i1] = ((f1 / s1) * tsum - t1) * gs;
    }
    if (lane == 0) {
      loss_ps[b] = __fmul_rn(loss, w);
      iw.weight[b] = w;
      iw.priority[b] = loss;                                          // the unweighted cross-entropy
    }
    weighted_mean_tail(iw, loss_ps, 1);
  } else {
    if (dlogits) {
      if (on0) dlogits[row + i0] = ((f0 / s1) * tsum - t0) * grad_scale;
      if (on1) dlogits[row + i1] = ((f1 / s1) * tsum - t1) * grad_scale;
    }
    if (lane == 0 && loss_ps) loss_ps[b] = loss;
  }
}

// trfl.td_learning as called at acme/agents/tf/ddpg/learning.py:193 (public trfl formula; trfl is not in the tree):
// target = r + pcont * v_t (stop-gradient), td = target - v_tm1, loss = 0.5 td^2; d(mean loss)/d v_tm1 = -td / B.
template <bool W>
__global__ void td_learning_kernel(int B, const float* __restrict__ v_tm1, const float* __restrict__ v_t,
                                   const float* __restrict__ R, const float* __restrict__ D, float gamma, float grad_scale,
                                   float* __restrict__ td_out, float* __restrict__ loss_ps, float* __restrict__ dv,
                                   IsWeighted iw) {
  pdl_launch_dependents();
  pdl_wait();
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if constexpr (W) {
    // every lane stays for the warp's mean tail
    if (b < B) {
      const float pcont = __fmul_rn(gamma, D[b]);
      const float target = __fadd_rn(R[b], __fmul_rn(pcont, v_t[b]));
      const float td = __fsub_rn(target, v_tm1[b]);
      const float w = is_weight_of(iw, b);
      if (td_out) td_out[b] = td;
      loss_ps[b] = __fmul_rn(__fmul_rn(0.5f, __fmul_rn(td, td)), w);
      iw.weight[b] = w;
      iw.priority[b] = fabsf(td);                                     // dqn/learning.py:152 (no epsilon)
      if (dv) dv[b] = -td * __fmul_rn(w, grad_scale);
    }
    weighted_mean_tail(iw, loss_ps, __popc(__ballot_sync(0xffffffffu, b < B)));
    return;
  }
  if (b >= B) return;
  const float pcont = __fmul_rn(gamma, D[b]);                        // discount * d_t, learning.py:169,193
  const float target = __fadd_rn(R[b], __fmul_rn(pcont, v_t[b]));
  const float td = __fsub_rn(target, v_tm1[b]);
  if (td_out) td_out[b] = td;
  loss_ps[b] = __fmul_rn(0.5f, __fmul_rn(td, td));
  if (dv) dv[b] = -td * grad_scale;
}

__global__ void __launch_bounds__(1024) mean_kernel(const float* __restrict__ x, int n, float* __restrict__ out) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ float scratch[32];
  float s = 0.f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) s += x[i];
  s = block_reduce(s, SumF(), 0.f, scratch);
  if (threadIdx.x == 0) *out = s / (float)n;
}

// distributions.py:64-66: q = sum_i softmax(l)_i z_i ; warp per row
__global__ void c51_mean_kernel(int B, int K, float vmin, float vmax, const float* __restrict__ logits,
                                const float* __restrict__ dq, float* __restrict__ q, float* __restrict__ dlogits) {
  pdl_launch_dependents();
  pdl_wait();
  const int lane = threadIdx.x & 31;
  const int b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (b >= B) return;
  const float* l = logits + (size_t)b * K;
  float mx = -INFINITY;
  for (int i = lane; i < K; i += 32) mx = fmaxf(mx, l[i]);
  for (int d = 16; d > 0; d >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, d));
  float se = 0.f, sz = 0.f;
  for (int i = lane; i < K; i += 32) {
    float e = expf(l[i] - mx);
    se += e;
    sz += e * atom_value(i, K, vmin, vmax);
  }
  for (int d = 16; d > 0; d >>= 1) {
    se += __shfl_xor_sync(0xffffffffu, se, d);
    sz += __shfl_xor_sync(0xffffffffu, sz, d);
  }
  const float mean = sz / se;
  if (q && lane == 0) q[b] = mean;
  if (dlogits) {
    const float g = dq ? dq[b] : 1.f;
    for (int i = lane; i < K; i += 32)
      dlogits[(size_t)b * K + i] = (expf(l[i] - mx) / se) * (atom_value(i, K, vmin, vmax) - mean) * g;
  }
}

// acme/tf/losses/dpg.py:41-57 (tf.clip_by_norm: t * clip / max(||t||, clip)); warp per row
__global__ void dpg_kernel(int B, int A, const float* __restrict__ dqda, float clip, int clip_norm,
                           float grad_scale, float* __restrict__ da, float* __restrict__ loss_ps) {
  pdl_launch_dependents();
  pdl_wait();
  const int lane = threadIdx.x & 31;
  const int b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (b >= B) return;
  const float* g = dqda + (size_t)b * A;
  float ss = 0.f;
  for (int i = lane; i < A; i += 32) ss += g[i] * g[i];
  for (int d = 16; d > 0; d >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, d);
  const float nrm = sqrtf(ss);
  float l = 0.f;
  for (int i = lane; i < A; i += 32) {
    float v = g[i];
    if (clip > 0.f) v = clip_norm ? (v * clip) / fmaxf(nrm, clip) : fminf(fmaxf(v, -clip), clip);
    da[(size_t)b * A + i] = -v * grad_scale;
    l += v * v;
  }
  for (int d = 16; d > 0; d >>= 1) l += __shfl_xor_sync(0xffffffffu, l, d);
  if (lane == 0 && loss_ps) loss_ps[b] = 0.5f * l;
}

// ------------------------------------------------------------------------------------------ K7
// snt.optimizers.Adam.apply as recalled in SURVEY App. A.5 (source not in the reference tree).
struct AdamConsts { float bc1, bc2, b1f, b2f, omb1, omb2, gs, k1, lr, eps; int eps_mode; };
__device__ __forceinline__ float adam_one(float& p, float g, float& m, float& v, const AdamConsts& c) {
  const float gj = c.gs == 1.f ? g : __fmul_rn(g, c.gs);
  m = __fadd_rn(__fmul_rn(c.b1f, m), __fmul_rn(c.omb1, gj));
  v = __fadd_rn(__fmul_rn(c.b2f, v), __fmul_rn(c.omb2, __fmul_rn(gj, gj)));
  // Moments of (nearly) dead units decay through the subnormal range and stay there for hundreds of steps; the IEEE
  // division / square-root sequences below take a slow path on subnormal operands (measured: the kernel went from
  // 55 to 88 us after 3000 updates).  Flushing |m|, v < FLT_MIN to zero changes the update by < 1e-30.
  m = fabsf(m) < 1.17549435e-38f ? 0.f : m;
  v = v < 1.17549435e-38f ? 0.f : v;
  // Exact zeros (weights of dead units keep g = m = v = 0 for good) would send the IEEE square root and division down
  // their slow paths -- a warp takes the slow path if ANY lane needs it; measured: 62.7 us for the 8M-parameter pass with
  // 70% zero moments against 41.9 us without (tools/adam_micro.py).  Substitute harmless operands and select the exact
  // results afterwards (sqrt(0) = 0, 0 / x = 0): bit-identical values, no slow path.
  const bool vz = v == 0.f, mz = m == 0.f;
  const float v_in = vz ? 1.f : v, m_in = mz ? 1.f : m;
  float upd;
  if (c.eps_mode == 0) {
    const float root = vz ? 0.f : __fsqrt_rn(__fdiv_rn(v_in, c.bc2));
    upd = __fdiv_rn(__fdiv_rn(m_in, c.bc1), __fadd_rn(root, c.eps));
  } else {
    const float root = vz ? 0.f : __fsqrt_rn(v_in);
    upd = __fdiv_rn(__fmul_rn(c.k1, m_in), __fadd_rn(root, c.eps));
  }
  upd = mz ? 0.f : upd;
  p = __fsub_rn(p, __fmul_rn(c.lr, upd));
  return p;
}
// 8 elements (two float4 per array = 8 independent 16-byte loads) per thread per iteration: enough bytes in
// flight to run at HBM speed; p/m/v are read-modify-write, g is read once (streamed through the read-only path).
// Measured on B200: four float4 per array per thread is SLOWER (0.347 vs 0.318 ms per step at full occupancy, no gain
// beside other kernels): the extra registers per thread cost more than the extra loads in flight bring.
__global__ void __launch_bounds__(256)
adam_kernel(long long n, float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
            float* __restrict__ v, const long long* __restrict__ step_dev, float lr, double b1,
            double b2, float eps, int eps_mode, const float* __restrict__ gscale_dev,
            __nv_bfloat16* __restrict__ shadow) {
  // the double-precision powers cost a few hundred FP64 instructions: one thread per CTA evaluates them
  __shared__ float bc_sh[2];
  pdl_launch_dependents();
  pdl_wait();
  if (threadIdx.x == 0) {
    const double t = (double)(*step_dev + 1);
    bc_sh[0] = (float)(1.0 - pow(b1, t));
    bc_sh[1] = (float)(1.0 - pow(b2, t));
  }
  __syncthreads();
  AdamConsts c;
  c.bc1 = bc_sh[0]; c.bc2 = bc_sh[1];
  c.b1f = (float)b1; c.b2f = (float)b2; c.omb1 = (float)(1.0 - b1); c.omb2 = (float)(1.0 - b2);
  c.gs = gscale_dev ? *gscale_dev : 1.f;
  c.k1 = sqrtf(c.bc2) / c.bc1; c.lr = lr; c.eps = eps; c.eps_mode = eps_mode;
  constexpr int VPT = 2, EPT = 4 * VPT;              // float4 vectors / elements per array per thread per iteration
  const long long n8 = n - n % EPT;
  long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * EPT;
  const long long stride = (long long)gridDim.x * blockDim.x * EPT;
  for (; i < n8; i += stride) {
    float4 pq[VPT], gq[VPT], mq[VPT], vq[VPT];
#pragma unroll
    for (int h = 0; h < VPT; ++h) {
      pq[h] = *reinterpret_cast<const float4*>(p + i + 4 * h);
      gq[h] = __ldg(reinterpret_cast<const float4*>(g + i + 4 * h));
      mq[h] = *reinterpret_cast<const float4*>(m + i + 4 * h);
      vq[h] = *reinterpret_cast<const float4*>(v + i + 4 * h);
    }
#pragma unroll
    for (int h = 0; h < VPT; ++h) {
      adam_one(pq[h].x, gq[h].x, mq[h].x, vq[h].x, c);
      adam_one(pq[h].y, gq[h].y, mq[h].y, vq[h].y, c);
      adam_one(pq[h].z, gq[h].z, mq[h].z, vq[h].z, c);
      adam_one(pq[h].w, gq[h].w, mq[h].w, vq[h].w, c);
      *reinterpret_cast<float4*>(p + i + 4 * h) = pq[h];
      *reinterpret_cast<float4*>(m + i + 4 * h) = mq[h];
      *reinterpret_cast<float4*>(v + i + 4 * h) = vq[h];
    }
    if (shadow) {
      uint4 pk;
      __nv_bfloat162 t0 = __floats2bfloat162_rn(pq[0].x, pq[0].y), t1 = __floats2bfloat162_rn(pq[0].z, pq[0].w);
      __nv_bfloat162 t2 = __floats2bfloat162_rn(pq[1].x, pq[1].y), t3 = __floats2bfloat162_rn(pq[1].z, pq[1].w);
      pk.x = *reinterpret_cast<uint32_t*>(&t0); pk.y = *reinterpret_cast<uint32_t*>(&t1);
      pk.z = *reinterpret_cast<uint32_t*>(&t2); pk.w = *reinterpret_cast<uint32_t*>(&t3);
      *reinterpret_cast<uint4*>(shadow + i) = pk;
    }
  }
  if (blockIdx.x == 0 && threadIdx.x < (int)(n - n8)) {   // ragged tail (< EPT elements)
    const long long j = n8 + threadIdx.x;
    float pv = p[j], mv = m[j], vv = v[j];
    adam_one(pv, g[j], mv, vv, c);
    p[j] = pv; m[j] = mv; v[j] = vv;
    if (shadow) shadow[j] = __float2bfloat16_rn(pv);
  }
}

// tf.clip_by_global_norm (acme/agents/tf/d4pg/learning.py:235-237), two fixed-order stages
__global__ void __launch_bounds__(256) sumsq_partial_kernel(long long n, const float* __restrict__ g, float* __restrict__ partial) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ double scratch[32];
  double s = 0.0;
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (; i < n; i += stride) { double x = g[i]; s += x * x; }
  s = block_reduce(s, SumD(), 0.0, scratch);
  if (threadIdx.x == 0) partial[blockIdx.x] = (float)s;
}
__global__ void __launch_bounds__(256) norm_finish_kernel(int nparts, const float* __restrict__ partial, float clip,
                                                         float* __restrict__ scale_out, float* __restrict__ norm_out) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ double scratch[32];
  double s = 0.0;
  for (int i = threadIdx.x; i < nparts; i += blockDim.x) s += (double)partial[i];
  s = block_reduce(s, SumD(), 0.0, scratch);
  if (threadIdx.x == 0) {
    float nrm = (float)sqrt(s);
    if (norm_out) *norm_out = nrm;
    *scale_out = clip / fmaxf(nrm, clip);
  }
}

__global__ void copy_if_period_kernel(long long n16, int4* __restrict__ dst, const int4* __restrict__ src,
                                      const long long* __restrict__ step_dev, long long period, long long phase) {
  pdl_launch_dependents();
  pdl_wait();
  if (((*step_dev) + phase) % period != 0) return;
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (; i < n16; i += stride) dst[i] = __ldg(src + i);
}
__global__ void step_increment_kernel(long long* step) {
  pdl_launch_dependents();
  pdl_wait(); *step += 1; }

// The end of a learner step in one launch: target <- online (parameters and, if given, their bf16 shadow) when
// (*step + phase) % period == 0, then *step += 1 and (if given) *counter2 += 1.  Every CTA reads *step when it starts;
// the increments are done by the CTA that finishes LAST (ticket), i.e. after every CTA has taken its decision.
__device__ unsigned int g_tail_ticket[8];
__global__ void __launch_bounds__(256)
learner_tail_kernel(long long n16_a, int4* __restrict__ dst_a, const int4* __restrict__ src_a, long long n16_b,
                    int4* __restrict__ dst_b, const int4* __restrict__ src_b, long long* __restrict__ step_dev, long long period,
                    long long phase, long long* __restrict__ counter2, int ticket) {
  pdl_wait();
  const bool due = period > 0 && ((*step_dev) + phase) % period == 0;
  if (due) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n16_a; i += stride) dst_a[i] = __ldg(src_a + i);
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n16_b; i += stride) dst_b[i] = __ldg(src_b + i);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    if (atomicAdd(&g_tail_ticket[ticket], 1u) == gridDim.x - 1) {
      g_tail_ticket[ticket] = 0;
      *step_dev += 1;
      if (counter2) *counter2 += 1;
    }
  }
}

// ------------------------------------------------------------------------------ element-wise
__device__ __forceinline__ float act_grad_from_output(float y, int act) {
  switch (act) {
    case B200RL_ACT_RELU: return y > 0.f ? 1.f : 0.f;
    case B200RL_ACT_ELU: return y > 0.f ? 1.f : y + 1.f;
    case B200RL_ACT_TANH: return 1.f - y * y;
    default: return 1.f;
  }
}
__global__ void act_bwd_kernel(long long n, float* __restrict__ dy, const float* __restrict__ y, int act) {
  pdl_launch_dependents();
  pdl_wait();
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (; i < n; i += stride) dy[i] *= act_grad_from_output(y[i], act);
}

// acme/tf/networks/duelling.py:51-59
__global__ void duelling_fwd_kernel(int B, int A, const float* __restrict__ value, const float* __restrict__ adv, float* __restrict__ q) {
  pdl_launch_dependents();
  pdl_wait();
  int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  float s = 0.f;
  for (int a = 0; a < A; ++a) s += adv[(size_t)b * A + a];
  const float mean = s / (float)A, v = value[b];
  for (int a = 0; a < A; ++a) q[(size_t)b * A + a] = v + (adv[(size_t)b * A + a] - mean);
}
__global__ void duelling_bwd_kernel(int B, int A, const float* __restrict__ dq, float* __restrict__ dvalue, float* __restrict__ dadv) {
  pdl_launch_dependents();
  pdl_wait();
  int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  float s = 0.f;
  for (int a = 0; a < A; ++a) s += dq[(size_t)b * A + a];
  dvalue[b] = s;
  const float mean = s / (float)A;
  for (int a = 0; a < A; ++a) dadv[(size_t)b * A + a] = dq[(size_t)b * A + a] - mean;
}


// Fused duelling head (acme/tf/networks/duelling.py:37-59): value = h[:, :H] . wv + bv, adv = h[:, H:] . wa^T + ba,
// q = value + (adv - mean(adv)).  One warp per sample: the 2H-wide hidden row sits in registers (H = 32 * HPL),
// the weight rows stream through with HPL independent loads in flight per dot product.
// The (A+1) x H weight rows are staged in shared memory once per CTA (one coalesced sweep, all loads
// independent) so that the per-sample dot products never wait on L2.
__device__ __forceinline__ void stage_head_weights(float* sw, const float* __restrict__ wv, const float* __restrict__ wa,
                                                   int A, int H) {
  const int nv = H / 4, na = A * H / 4;
  for (int i = threadIdx.x; i < nv; i += blockDim.x) reinterpret_cast<float4*>(sw)[i] = __ldg(reinterpret_cast<const float4*>(wv) + i);
  for (int i = threadIdx.x; i < na; i += blockDim.x) reinterpret_cast<float4*>(sw + H)[i] = __ldg(reinterpret_cast<const float4*>(wa) + i);
  __syncthreads();
}

template <int HPL>
__global__ void __launch_bounds__(256)
duelling_head_fwd_kernel(int B, int A, const float* __restrict__ h, int ldh, const float* __restrict__ wv,
                         const float* __restrict__ bv, const float* __restrict__ wa, const float* __restrict__ ba,
                         float* __restrict__ val, float* __restrict__ adv, float* __restrict__ q) {
  pdl_launch_dependents();
  pdl_wait();
  constexpr int H = 32 * HPL;
  extern __shared__ __align__(16) float sw[];   // [A + 1][H]: value row, then advantage rows
  stage_head_weights(sw, wv, wa, A, H);
  const int lane = threadIdx.x & 31;
  const int b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (b >= B) return;
  float hv[HPL], ha[HPL];
#pragma unroll
  for (int j = 0; j < HPL; ++j) {
    hv[j] = h[(size_t)b * ldh + lane + 32 * j];
    ha[j] = h[(size_t)b * ldh + H + lane + 32 * j];
  }
  float sv = 0.f;
#pragma unroll
  for (int j = 0; j < HPL; ++j) sv = fmaf(hv[j], sw[lane + 32 * j], sv);
  for (int d = 16; d > 0; d >>= 1) sv += __shfl_xor_sync(0xffffffffu, sv, d);
  sv += bv[0];
  float total = 0.f, mine = 0.f;
  for (int a = 0; a < A; ++a) {
    const float* w = sw + (size_t)(a + 1) * H;
    float s = 0.f;
#pragma unroll
    for (int j = 0; j < HPL; ++j) s = fmaf(ha[j], w[lane + 32 * j], s);
    for (int d = 16; d > 0; d >>= 1) s += __shfl_xor_sync(0xffffffffu, s, d);
    s += ba[a];
    total += s;
    if (lane == (a & 31)) mine = s;
    if (A > 32 && lane == 0) adv[(size_t)b * A + a] = s;
  }
  const float mean = total / (float)A;
  if (lane == 0) val[b] = sv;
  if (A <= 32) {
    if (lane < A) { adv[(size_t)b * A + lane] = mine; q[(size_t)b * A + lane] = sv + (mine - mean); }
  } else {
    __syncwarp();
    for (int a = lane; a < A; a += 32) q[(size_t)b * A + a] = sv + (adv[(size_t)b * A + a] - mean);
  }
}

// ------------------------------------------------------------------------------ K4 fused into the duelling head
// The three duelling heads (online(o_tm1), target(o_t), online(o_t); duelling.py:37-59), the double-Q TD error / Huber /
// importance weight / priority (learning.py:127-154) and the head's data gradient dh = [dval * wv, dadv @ wa] * relu'(h)
// in ONE launch -- three head kernels, the single-CTA TD kernel and the head-backward kernel of the unfused path sat
// back to back on the step's critical path.  Three warps per sample (one per head) so the 3 x (A + 1) dot products of a
// sample are not one serial chain; the warp that owns the o_tm1 head keeps its hidden row in registers and finishes the
// sample (TD, dq, dh) once the other two have published their q rows in shared memory.  The arithmetic of every piece
// is the unfused kernels', operation for operation (same dot-product order, same __f*_rn sequence), so the two paths
// agree bit for bit.  Needs A <= 32 and the batch-max importance weight precomputed (b200rl_is_weight_max).
constexpr int kHeadSamples = 4;                       // samples per CTA
constexpr int kHeadThreads = 96 * kHeadSamples;       // 3 warps per sample

// q row of one head from a hidden row held in registers; lane a < A returns q[a].  Dot products run four at a time
// (their shuffle reductions interleave), each one in the order of duelling_head_fwd_kernel.
template <int HPL>
__device__ __forceinline__ float head_q(const float* __restrict__ sw, const float* __restrict__ bv, const float* __restrict__ ba,
                                        int A, int lane, const float (&hv)[HPL], const float (&ha)[HPL]) {
  constexpr int H = 32 * HPL;
  float sv = 0.f;
#pragma unroll
  for (int j = 0; j < HPL; ++j) sv = fmaf(hv[j], sw[lane + 32 * j], sv);
  for (int d = 16; d > 0; d >>= 1) sv += __shfl_xor_sync(0xffffffffu, sv, d);
  sv += bv[0];
  float total = 0.f, mine = 0.f;
  for (int a0 = 0; a0 < A; a0 += 4) {
    float s[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      s[q] = 0.f;
      if (a0 + q < A) {
        const float* w = sw + (size_t)(a0 + q + 1) * H;
#pragma unroll
        for (int j = 0; j < HPL; ++j) s[q] = fmaf(ha[j], w[lane + 32 * j], s[q]);
      }
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
#pragma unroll
      for (int q = 0; q < 4; ++q) s[q] += __shfl_xor_sync(0xffffffffu, s[q], d);
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      if (a0 + q < A) {
        const float t = s[q] + ba[a0 + q];
        total += t;
        if (lane == a0 + q) mine = t;
      }
    }
  }
  const float mean = total / (float)A;
  return sv + (mine - mean);
}

struct HeadTdArgs {
  int B, A, ldh, lddh, flags, dh_bf16;
  const float *h_tm1, *h_sel, *h_tgt;
  const float *wv, *bv, *wa, *ba, *twv, *tbv, *twa, *tba;
  const int* a_tm1;
  const float *R, *D, *prob;
  float gamma, delta, max_abs_r, grad_scale;
  double beta;
  const double* wmax_dev;
  float *q_tm1, *q_tv, *q_ts, *td, *loss_ps, *weight, *priority, *dq, *dval, *dadv;
  void* dh;
};

template <int HPL>
__global__ void __launch_bounds__(kHeadThreads)
dqn_head_td_kernel(HeadTdArgs p) {
  constexpr int H = 32 * HPL;
  extern __shared__ __align__(16) float sw[];   // online [A + 1][H], then target [A + 1][H]
  __shared__ __align__(8) unsigned long long bar;
  __shared__ float q_other[kHeadSamples][2][32];  // [sample][0 = target(o_t), 1 = online(o_t)][action]
  float* swt = sw + (size_t)(p.A + 1) * H;
  pdl_launch_dependents();
  pdl_wait();
  // the four weight blocks arrive by bulk async copies (one instruction each, completion on an mbarrier) while the
  // warps already fetch their hidden rows
  if (threadIdx.x == 0) {
    const uint32_t b32 = (uint32_t)__cvta_generic_to_shared(&bar);
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(b32) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    const uint32_t nv = H * 4, na = p.A * H * 4;
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(b32), "r"(2 * (nv + na)) : "memory");
    const float* src[4] = {p.wv, p.wa, p.twv, p.twa};
    float* dst[4] = {sw, sw + H, swt, swt + H};
    const uint32_t nb[4] = {nv, na, nv, na};
#pragma unroll
    for (int i = 0; i < 4; ++i)
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                       (uint32_t)__cvta_generic_to_shared(dst[i])),
                   "l"(src[i]), "r"(nb[i]), "r"(b32)
                   : "memory");
  }
  __syncthreads();   // the barrier is initialised before anyone waits on it
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int sl = warp / 3, head = warp - 3 * sl;           // head: 0 = online(o_tm1), 1 = target(o_t), 2 = online(o_t)
  const int b = blockIdx.x * kHeadSamples + sl;
  const bool valid = b < p.B;
  const int A = p.A;
  float hv[HPL], ha[HPL];
  if (valid) {
    const float* row = (head == 0 ? p.h_tm1 : (head == 1 ? p.h_tgt : p.h_sel)) + (size_t)b * p.ldh;
#pragma unroll
    for (int j = 0; j < HPL; ++j) {
      hv[j] = row[lane + 32 * j];
      ha[j] = row[H + lane + 32 * j];
    }
  }
  {
    const uint32_t b32 = (uint32_t)__cvta_generic_to_shared(&bar);
    uint32_t ok;
    do {
      asm volatile(
          "{\n.reg .pred q;\nmbarrier.try_wait.parity.shared::cta.b64 q, [%1], 0;\nselp.u32 %0, 1, 0, q;\n}\n"
          : "=r"(ok)
          : "r"(b32)
          : "memory");
    } while (!ok);
  }
  float q = 0.f;
  if (valid) {
    q = head == 1 ? head_q<HPL>(swt, p.tbv, p.tba, A, lane, hv, ha) : head_q<HPL>(sw, p.bv, p.ba, A, lane, hv, ha);
    float* qout = head == 0 ? p.q_tm1 : (head == 1 ? p.q_tv : p.q_ts);
    if (qout && lane < A) qout[(size_t)b * A + lane] = q;
    if (head != 0) q_other[sl][head - 1][lane] = q;
  }
  __syncthreads();
  if (!valid || head != 0) return;
  const float q_tm1 = q, q_tv = q_other[sl][0][lane], q_ts = q_other[sl][1][lane];
  // trfl.double_qlearning: first maximum of the selector wins
  int best = 0;
  float bvv = __shfl_sync(0xffffffffu, q_ts, 0);
  for (int a = 1; a < A; ++a) {
    const float v = __shfl_sync(0xffffffffu, q_ts, a);
    if (v > bvv) { bvv = v; best = a; }
  }
  const int act = p.a_tm1[b];
  const float q_next = __shfl_sync(0xffffffffu, q_tv, best);
  const float q_act = __shfl_sync(0xffffffffu, q_tm1, act);
  const float r = fminf(fmaxf(p.R[b], -p.max_abs_r), p.max_abs_r);          // learning.py:129
  const float d = __fmul_rn(p.D[b], p.gamma);                               // learning.py:130
  const float target = __fadd_rn(r, __fmul_rn(d, q_next));
  const float td = __fsub_rn(target, q_act);
  const float absx = fabsf(td);
  const float quad = fminf(absx, p.delta);
  const float lin = __fsub_rn(absx, quad);
  const float hub = __fadd_rn(__fmul_rn(__fmul_rn(0.5f, quad), quad), __fmul_rn(p.delta, lin));   // huber.py:48-57
  float w = 0.f;
  if (lane == 0) w = is_weight_norm(is_weight_raw(p.prob[b], p.beta, p.flags), *p.wmax_dev, p.flags);   // learning.py:138-143
  w = __shfl_sync(0xffffffffu, w, 0);
  const float g = -(w * p.grad_scale) * fminf(fmaxf(td, -p.delta), p.delta);
  if (lane == 0) {
    p.td[b] = td;
    p.loss_ps[b] = __fmul_rn(hub, w);
    p.weight[b] = w;
    p.priority[b] = absx;                                                    // learning.py:152 (no epsilon)
  }
  // duelling backward: dval = sum_a dq, dadv = dq - mean(dq) (dq has one non-zero, g at the action taken)
  float s = 0.f;
  for (int a = 0; a < A; ++a) s += (a == act) ? g : 0.f;
  const float mean = s / (float)A;
  const float my_dq = (lane == act) ? g : 0.f;
  if (lane < A) {
    if (p.dq) p.dq[(size_t)b * A + lane] = my_dq;
    p.dadv[(size_t)b * A + lane] = my_dq - mean;
  }
  if (lane == 0) p.dval[b] = s;
  float acc[HPL];
#pragma unroll
  for (int j = 0; j < HPL; ++j) acc[j] = 0.f;
  for (int a = 0; a < A; ++a) {
    const float ga = ((a == act) ? g : 0.f) - mean;
    const float* wr = sw + (size_t)(a + 1) * H;
#pragma unroll
    for (int j = 0; j < HPL; ++j) acc[j] = fmaf(ga, wr[lane + 32 * j], acc[j]);
  }
#pragma unroll
  for (int j = 0; j < HPL; ++j) {
    const int k = lane + 32 * j;
    const float dv = hv[j] > 0.f ? s * sw[k] : 0.f;
    const float da = ha[j] > 0.f ? acc[j] : 0.f;
    if (p.dh_bf16) {
      __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(p.dh) + (size_t)b * p.lddh;
      o[k] = __float2bfloat16_rn(dv);
      o[H + k] = __float2bfloat16_rn(da);
    } else {
      float* o = reinterpret_cast<float*>(p.dh) + (size_t)b * p.lddh;
      o[k] = dv;
      o[H + k] = da;
    }
  }
}

// backward, part 1 (thread per sample x 4 hidden units): dval = sum_a dq, dadv = dq - mean(dq), and
// dh = [dval * wv, dadv @ wa] * relu'(h).  The (A+1) x H weights are 40 KB: they stay in L1/L2, the dq row is a
// warp-wide broadcast load.
__global__ void __launch_bounds__(256)
duelling_head_bwd_dh_kernel(int B, int A, int H, const float* __restrict__ dq, const float* __restrict__ h, int ldh,
                            const float* __restrict__ wv, const float* __restrict__ wa, float* __restrict__ dval,
                            float* __restrict__ dadv, float* __restrict__ dh, int lddh) {
  pdl_launch_dependents();
  pdl_wait();
  const int per = H >> 2;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)B * per) return;
  const int b = (int)(i / per), k = (int)(i % per) * 4;
  const float* q = dq + (size_t)b * A;
  float s = 0.f;
  for (int a = 0; a < A; ++a) s += __ldg(q + a);
  const float mean = s / (float)A;
  if (k == 0) {
    dval[b] = s;
    for (int a = 0; a < A; ++a) dadv[(size_t)b * A + a] = __ldg(q + a) - mean;
  }
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int a = 0; a < A; ++a) {
    const float g = __ldg(q + a) - mean;
    const float4 w = __ldg(reinterpret_cast<const float4*>(wa + (size_t)a * H + k));
    acc.x = fmaf(g, w.x, acc.x); acc.y = fmaf(g, w.y, acc.y); acc.z = fmaf(g, w.z, acc.z); acc.w = fmaf(g, w.w, acc.w);
  }
  const float4 v = __ldg(reinterpret_cast<const float4*>(wv + k));
  const float4 hv = __ldg(reinterpret_cast<const float4*>(h + (size_t)b * ldh + k));
  const float4 ha = __ldg(reinterpret_cast<const float4*>(h + (size_t)b * ldh + H + k));
  *reinterpret_cast<float4*>(dh + (size_t)b * lddh + k) =
      make_float4(hv.x > 0.f ? s * v.x : 0.f, hv.y > 0.f ? s * v.y : 0.f, hv.z > 0.f ? s * v.z : 0.f, hv.w > 0.f ? s * v.w : 0.f);
  *reinterpret_cast<float4*>(dh + (size_t)b * lddh + H + k) =
      make_float4(ha.x > 0.f ? acc.x : 0.f, ha.y > 0.f ? acc.y : 0.f, ha.z > 0.f ? acc.z : 0.f, ha.w > 0.f ? acc.w : 0.f);
}
// backward, part 2: dwv[k] = sum_b dval[b] h[b,k], dwa[a,k] = sum_b dadv[b,a] h[b,H+k] and the bias sums.
// The batch is cut into gridDim.z segments (partial sums, then a fixed-order add) so that enough
// threads are in flight; 8 independent accumulators keep 8 loads per thread outstanding.
__global__ void __launch_bounds__(128)
duelling_head_bwd_dw_kernel(int B, int A, int H, const float* __restrict__ dval, const float* __restrict__ dadv,
                            const float* __restrict__ h, int ldh, float* __restrict__ partial) {
  pdl_launch_dependents();
  pdl_wait();
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  const int a = (int)blockIdx.y - 1;   // -1 = value stream
  if (k >= H) return;
  const int seg = (B + gridDim.z - 1) / gridDim.z;
  const int b0 = blockIdx.z * seg, b1 = min(B, b0 + seg);
  const float* g = a < 0 ? dval : dadv + a;
  const int gs = a < 0 ? 1 : A;
  const float* hc = h + (a < 0 ? 0 : H) + k;
  float acc[8], bs = 0.f;
#pragma unroll
  for (int j = 0; j < 8; ++j) acc[j] = 0.f;
  int b = b0;
  for (; b + 8 <= b1; b += 8) {
    float gv[8], hv[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) { gv[j] = g[(size_t)(b + j) * gs]; hv[j] = hc[(size_t)(b + j) * ldh]; }
#pragma unroll
    for (int j = 0; j < 8; ++j) { acc[j] = fmaf(gv[j], hv[j], acc[j]); bs += gv[j]; }
  }
  for (; b < b1; ++b) { const float gv = g[(size_t)b * gs]; acc[0] = fmaf(gv, hc[(size_t)b * ldh], acc[0]); bs += gv; }
  const float t = ((acc[0] + acc[1]) + (acc[2] + acc[3])) + ((acc[4] + acc[5]) + (acc[6] + acc[7]));
  // partial layout: [seg][A+1][H + 1] (last column = bias partial, written by k == 0)
  float* row = partial + ((size_t)blockIdx.z * (A + 1) + (a + 1)) * (H + 1);
  row[k] = t;
  if (k == 0) row[H] = bs;
}
__global__ void duelling_head_bwd_finish_kernel(int A, int H, int segs, const float* __restrict__ partial,
                                                float* __restrict__ dwv, float* __restrict__ dbv,
                                                float* __restrict__ dwa, float* __restrict__ dba) {
  pdl_launch_dependents();
  pdl_wait();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;   // over (A+1) * (H+1)
  if (i >= (A + 1) * (H + 1)) return;
  float t = 0.f;
  for (int s = 0; s < segs; ++s) t += partial[(size_t)s * (A + 1) * (H + 1) + i];
  const int r = i / (H + 1), k = i % (H + 1);
  if (r == 0) { if (k < H) dwv[k] = t; else dbv[0] = t; }
  else { if (k < H) dwa[(size_t)(r - 1) * H + k] = t; else dba[r - 1] = t; }
}

// Backward of a dense head with N <= 64 outputs in the bf16 dataflow (the C51, scalar-critic and policy heads of
// LayerNormMLP): the bf16 GEMMs need N >= 64 (data gradient) and N % 64 == 0 (weight gradient).  One launch computes
//   dx[M,K] = (dy[M,N] @ w[N,K]) * act'(mask)  as bf16,   dw[N,K] = dy^T @ x,   db[N] = colsum(dy)  in fp32.
// CTA (kb, mb) owns columns [64 kb, 64 kb + 64) and rows [mb * rows_per_cta, ...), walked in chunks of 32 rows staged in
// shared memory as fp32 (bf16 -> fp32 is exact); every sum is a chain of fmaf in ascending n or m.  With one row slice
// the CTA writes dw / db directly.  With several, each writes a partial slab and the CTA of column block kb that finishes
// last (a per-stream, per-column-block ticket reset on the way out, so the kernel is CUDA-graph safe) adds the slabs in
// slice order: the order of every addition is fixed by indices, never by arrival.
constexpr int kHbRows = 32, kHbCols = 64, kHbMaxColBlocks = 32;
__device__ unsigned int g_head_tickets[64 * kHbMaxColBlocks];

__device__ __forceinline__ void bf16x8_to_f32(uint4 u, float* v) {
  const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w[j]));
    v[2 * j] = f.x;
    v[2 * j + 1] = f.y;
  }
}

__global__ void __launch_bounds__(256)
dense_head_bwd_bf16_kernel(int M, int N, int K, const float* __restrict__ dy, int lddy, const __nv_bfloat16* __restrict__ x,
                           int ldx, const __nv_bfloat16* __restrict__ w, __nv_bfloat16* __restrict__ dx, int lddx,
                           const __nv_bfloat16* __restrict__ mask, int mask_act, float* __restrict__ dw,
                           float* __restrict__ db, int rows_per_cta, float* __restrict__ partial, int ticket) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ float w_s[64][kHbCols];
  __shared__ float dy_s[kHbRows][64];
  __shared__ float x_s[kHbRows][kHbCols];
  __shared__ bool last;
  const int kb = blockIdx.x, mb = blockIdx.y;
  const int k0 = kb * kHbCols, kc = min(kHbCols, K - k0);          // kc % 8 == 0
  const int m0 = mb * rows_per_cta, m1 = min(M, m0 + rows_per_cta);
  const int t = threadIdx.x, col = t & (kHbCols - 1), rg = t >> 6;  // rg: row group 0..3
  const bool grads = dw || db;
  for (int i = t; i < 64 * (kHbCols / 8); i += 256) {
    const int n = i / (kHbCols / 8), c8 = (i % (kHbCols / 8)) * 8;
    float v[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (n < N && c8 < kc) bf16x8_to_f32(__ldg(reinterpret_cast<const uint4*>(w + (size_t)n * K + k0 + c8)), v);
#pragma unroll
    for (int j = 0; j < 8; ++j) w_s[n][c8 + j] = v[j];
  }
  float acc_w[16], acc_b = 0.f;
#pragma unroll
  for (int j = 0; j < 16; ++j) acc_w[j] = 0.f;
  for (int r0 = m0; r0 < m1; r0 += kHbRows) {
    const int rows = min(kHbRows, m1 - r0);
    __syncthreads();   // the previous chunk has been consumed
    for (int i = t; i < kHbRows * 64; i += 256) {
      const int r = i >> 6, n = i & 63;
      dy_s[r][n] = (r < rows && n < N) ? dy[(size_t)(r0 + r) * lddy + n] : 0.f;
    }
    if (dw) {
      const int r = t / (kHbCols / 8), c8 = (t % (kHbCols / 8)) * 8;   // 256 threads = 32 rows x 8 vectors
      float v[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      if (r < rows && c8 < kc) bf16x8_to_f32(__ldg(reinterpret_cast<const uint4*>(x + (size_t)(r0 + r) * ldx + k0 + c8)), v);
#pragma unroll
      for (int j = 0; j < 8; ++j) x_s[r][c8 + j] = v[j];
    }
    __syncthreads();
    if (col < kc) {
      float a[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      for (int n = 0; n < N; ++n) {
        const float wv = w_s[n][col];
#pragma unroll
        for (int j = 0; j < 8; ++j) a[j] = fmaf(dy_s[rg + 4 * j][n], wv, a[j]);
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int r = rg + 4 * j;
        if (r < rows) {
          const size_t o = (size_t)(r0 + r) * lddx + k0 + col;
          float v = a[j];
          if (mask) v = v * act_grad_from_output(__bfloat162float(mask[o]), mask_act);
          dx[o] = __float2bfloat16_rn(v);
        }
      }
      if (dw)
        for (int r = 0; r < rows; ++r) {
          const float xv = x_s[r][col];
#pragma unroll
          for (int j = 0; j < 16; ++j) acc_w[j] = fmaf(dy_s[r][rg + 4 * j], xv, acc_w[j]);
        }
    }
    if (db && kb == 0 && t < N)
      for (int r = 0; r < rows; ++r) acc_b = acc_b + dy_s[r][t];
  }
  if (!grads) return;
  if (gridDim.y == 1) {
    if (dw && col < kc)
#pragma unroll
      for (int j = 0; j < 16; ++j)
        if (rg + 4 * j < N) dw[(size_t)(rg + 4 * j) * K + k0 + col] = acc_w[j];
    if (db && kb == 0 && t < N) db[t] = acc_b;
    return;
  }
  // partial layout: [kb][mb][64][64] dw slabs, then [mb][64] bias sums
  float* slab = partial + ((size_t)kb * gridDim.y + mb) * (64 * kHbCols);
  float* bpart = partial + (size_t)gridDim.x * gridDim.y * (64 * kHbCols);
  if (dw)
#pragma unroll
    for (int j = 0; j < 16; ++j) slab[(rg + 4 * j) * kHbCols + col] = acc_w[j];
  if (db && kb == 0 && t < 64) bpart[mb * 64 + t] = acc_b;
  __threadfence();
  __syncthreads();
  unsigned int* tk = &g_head_tickets[ticket * kHbMaxColBlocks + kb];
  if (t == 0) last = atomicAdd(tk, 1u) == gridDim.y - 1;
  __syncthreads();
  if (!last) return;
  __threadfence();
  if (dw && col < kc)
    for (int j = 0; j < 16; ++j) {
      const int n = rg + 4 * j;
      if (n >= N) break;
      float s = 0.f;
      for (int q = 0; q < (int)gridDim.y; ++q) s = s + __ldcg(partial + ((size_t)kb * gridDim.y + q) * (64 * kHbCols) + n * kHbCols + col);
      dw[(size_t)n * K + k0 + col] = s;
    }
  if (db && kb == 0 && t < N) {
    float s = 0.f;
    for (int q = 0; q < (int)gridDim.y; ++q) s = s + __ldcg(bpart + q * 64 + t);
    db[t] = s;
  }
  if (t == 0) *tk = 0;
}

// snt.LayerNorm(axis=slice(1,None), scale, offset) + tanh (acme/tf/networks/continuous.py:55-58); CTA per row.
// y_bf16 (nullable): also store RN-bf16(y), the operand of the next layer in the bf16 dataflow.
__global__ void __launch_bounds__(256)
layernorm_tanh_fwd_kernel(int N, const float* __restrict__ x, const float* __restrict__ scale,
                          const float* __restrict__ offset, float eps, float* __restrict__ y,
                          float* __restrict__ xhat, float* __restrict__ rstd, __nv_bfloat16* __restrict__ y_bf16) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ float scratch[32];
  const int b = blockIdx.x;
  const float* xr = x + (size_t)b * N;
  float s = 0.f;
  for (int i = threadIdx.x; i < N; i += blockDim.x) s += xr[i];
  const float mean = block_reduce(s, SumF(), 0.f, scratch) / (float)N;
  float vs = 0.f;
  for (int i = threadIdx.x; i < N; i += blockDim.x) { float d = xr[i] - mean; vs += d * d; }
  const float var = block_reduce(vs, SumF(), 0.f, scratch) / (float)N;
  const float rs = rsqrtf(var + eps);
  for (int i = threadIdx.x; i < N; i += blockDim.x) {
    float xh = (xr[i] - mean) * rs;
    xhat[(size_t)b * N + i] = xh;
    const float yv = tanhf(xh * scale[i] + offset[i]);
    y[(size_t)b * N + i] = yv;
    if (y_bf16) y_bf16[(size_t)b * N + i] = __float2bfloat16_rn(yv);
  }
  if (threadIdx.x == 0) rstd[b] = rs;
}
__global__ void __launch_bounds__(256)
layernorm_tanh_bwd_kernel(int N, const float* __restrict__ dy, const float* __restrict__ y,
                          const float* __restrict__ xhat, const float* __restrict__ rstd,
                          const float* __restrict__ scale, float* __restrict__ dx) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ float scratch[32];
  const int b = blockIdx.x;
  const size_t o = (size_t)b * N;
  float s1 = 0.f, s2 = 0.f;
  for (int i = threadIdx.x; i < N; i += blockDim.x) {
    float dz = dy[o + i] * (1.f - y[o + i] * y[o + i]);
    float dxh = dz * scale[i];
    s1 += dxh;
    s2 += dxh * xhat[o + i];
  }
  const float m1 = block_reduce(s1, SumF(), 0.f, scratch) / (float)N;
  const float m2 = block_reduce(s2, SumF(), 0.f, scratch) / (float)N;
  const float rs = rstd[b];
  for (int i = threadIdx.x; i < N; i += blockDim.x) {
    float dz = dy[o + i] * (1.f - y[o + i] * y[o + i]);
    float dxh = dz * scale[i];
    dx[o + i] = rs * (dxh - m1 - xhat[o + i] * m2);
  }
}
__global__ void layernorm_param_grad_kernel(int B, int N, const float* __restrict__ dy, const float* __restrict__ y,
                                            const float* __restrict__ xhat, float* __restrict__ dscale, float* __restrict__ doffset) {
  pdl_launch_dependents();
  pdl_wait();
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  float ds = 0.f, dof = 0.f;
  for (int b = 0; b < B; ++b) {
    size_t o = (size_t)b * N + i;
    float dz = dy[o] * (1.f - y[o] * y[o]);
    ds += dz * xhat[o];
    dof += dz;
  }
  dscale[i] = ds;
  doffset[i] = dof;
}

// The first LayerNormMLP layer over observation-network features: z0 = z_f + a @ w_a^T + b (z_f = features @ w_f^T, a
// GEMM with an fp32 output), then LayerNorm + tanh with the arithmetic of layernorm_tanh_fwd_kernel.  CTA per row.
constexpr int kFeatMaxN = 1024, kFeatMaxA = 64, kFeatRows = 8;
__device__ unsigned int g_feature_tickets[64];

__global__ void __launch_bounds__(256)
feature_layer_fwd_kernel(int N, int A, const float* __restrict__ zf, const float* __restrict__ act,
                         const float* __restrict__ w_a, const float* __restrict__ bias, const float* __restrict__ scale,
                         const float* __restrict__ offset, float eps, float* __restrict__ y,
                         __nv_bfloat16* __restrict__ y_bf16, float* __restrict__ xhat, float* __restrict__ rstd) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ float scratch[32];
  __shared__ float z[kFeatMaxN];
  __shared__ float a_s[kFeatMaxA];
  const int b = blockIdx.x;
  if (threadIdx.x < A) a_s[threadIdx.x] = act[(size_t)b * A + threadIdx.x];
  __syncthreads();
  float s = 0.f;
  for (int i = threadIdx.x; i < N; i += blockDim.x) {
    float v = zf[(size_t)b * N + i];
    for (int k = 0; k < A; ++k) v = fmaf(a_s[k], w_a[(size_t)i * A + k], v);
    v = v + bias[i];
    z[i] = v;
    s += v;
  }
  const float mean = block_reduce(s, SumF(), 0.f, scratch) / (float)N;
  float vs = 0.f;
  for (int i = threadIdx.x; i < N; i += blockDim.x) { float d = z[i] - mean; vs += d * d; }
  const float var = block_reduce(vs, SumF(), 0.f, scratch) / (float)N;
  const float rs = rsqrtf(var + eps);
  for (int i = threadIdx.x; i < N; i += blockDim.x) {
    float xh = (z[i] - mean) * rs;
    xhat[(size_t)b * N + i] = xh;
    const float yv = tanhf(xh * scale[i] + offset[i]);
    y[(size_t)b * N + i] = yv;
    if (y_bf16) y_bf16[(size_t)b * N + i] = __float2bfloat16_rn(yv);
  }
  if (threadIdx.x == 0) rstd[b] = rs;
}

// Its backward.  CTA s owns rows [s * rows_per_cta, ...) (at most kFeatRows): per row the LayerNorm + tanh backward of
// layernorm_tanh_bwd_kernel gives dz (fp32, and RN-bf16(dz) when asked) and, when asked, da = dz @ w_a (one warp per
// action column, lanes in a fixed stride, then a fixed butterfly).  The parameter gradients are sums over the batch in
// ascending row order: d scale = sum dt * xhat, d offset = sum dt (dt = dy * (1 - y^2)), db = sum dz, dw_a = dz^T a.
// With one slice the CTA writes them; with several each writes a partial slab to `partial` and the CTA that finishes last
// (per-stream ticket, reset on exit: CUDA-graph safe) adds the slabs in slice order.
__global__ void __launch_bounds__(256)
feature_layer_bwd_kernel(int B, int N, int A, const float* __restrict__ dy, const float* __restrict__ y,
                         const float* __restrict__ xhat, const float* __restrict__ rstd, const float* __restrict__ scale,
                         const float* __restrict__ act, const float* __restrict__ w_a, float* __restrict__ dz,
                         __nv_bfloat16* __restrict__ dz_bf16, float* __restrict__ dscale, float* __restrict__ doffset,
                         float* __restrict__ db, float* __restrict__ dw_a, float* __restrict__ da, int rows_per_cta,
                         float* __restrict__ partial, int ticket) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ float scratch[32];
  __shared__ float dz_s[kFeatRows][kFeatMaxN];
  __shared__ float a_s[kFeatRows][kFeatMaxA];
  __shared__ bool last;
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const int m0 = blockIdx.x * rows_per_cta, rows = min(rows_per_cta, B - m0);
  const bool grads = dscale != nullptr;
  float acc_s[kFeatMaxN / 256], acc_o[kFeatMaxN / 256];
#pragma unroll
  for (int q = 0; q < kFeatMaxN / 256; ++q) acc_s[q] = acc_o[q] = 0.f;
  for (int r = 0; r < rows; ++r) {
    const size_t o = (size_t)(m0 + r) * N;
    float s1 = 0.f, s2 = 0.f;
    for (int i = t; i < N; i += blockDim.x) {
      float dt = dy[o + i] * (1.f - y[o + i] * y[o + i]);
      float dxh = dt * scale[i];
      s1 += dxh;
      s2 += dxh * xhat[o + i];
    }
    const float m1 = block_reduce(s1, SumF(), 0.f, scratch) / (float)N;
    const float m2 = block_reduce(s2, SumF(), 0.f, scratch) / (float)N;
    const float rs = rstd[m0 + r];
#pragma unroll
    for (int q = 0; q < kFeatMaxN / 256; ++q) {
      const int i = t + 256 * q;
      if (i < N) {
        float dt = dy[o + i] * (1.f - y[o + i] * y[o + i]);
        float dxh = dt * scale[i];
        const float v = rs * (dxh - m1 - xhat[o + i] * m2);
        dz[o + i] = v;
        if (dz_bf16) dz_bf16[o + i] = __float2bfloat16_rn(v);
        dz_s[r][i] = v;
        acc_s[q] = acc_s[q] + dt * xhat[o + i];
        acc_o[q] = acc_o[q] + dt;
      }
    }
    if (act && t < A) a_s[r][t] = act[(size_t)(m0 + r) * A + t];
  }
  __syncthreads();
  if (da)
    for (int p = warp; p < rows * A; p += 8) {
      const int r = p / A, k = p % A;
      float s = 0.f;
      for (int i = lane; i < N; i += 32) s = fmaf(dz_s[r][i], w_a[(size_t)i * A + k], s);
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) s = s + __shfl_xor_sync(0xffffffffu, s, off);
      if (lane == 0) da[(size_t)(m0 + r) * A + k] = s;
    }
  if (!grads) return;
  // this slice's sums: [d scale | d offset | db] (3N) then dw_a (N x A)
  const int per = N * (3 + A);
  float* out = gridDim.x == 1 ? nullptr : partial + (size_t)blockIdx.x * per;
#pragma unroll
  for (int q = 0; q < kFeatMaxN / 256; ++q) {
    const int i = t + 256 * q;
    if (i < N) {
      float sb = 0.f;
      for (int r = 0; r < rows; ++r) sb = sb + dz_s[r][i];
      if (out) { out[i] = acc_s[q]; out[N + i] = acc_o[q]; out[2 * N + i] = sb; }
      else { dscale[i] = acc_s[q]; doffset[i] = acc_o[q]; db[i] = sb; }
    }
  }
  for (int e = t; e < N * A; e += blockDim.x) {
    const int i = e / A, k = e % A;
    float s = 0.f;
    for (int r = 0; r < rows; ++r) s = fmaf(dz_s[r][i], a_s[r][k], s);
    if (out) out[3 * N + e] = s;
    else dw_a[e] = s;
  }
  if (!out) return;
  __threadfence();
  __syncthreads();
  if (t == 0) last = atomicAdd(&g_feature_tickets[ticket], 1u) == gridDim.x - 1;
  __syncthreads();
  if (!last) return;
  __threadfence();
  for (int e = t; e < per; e += blockDim.x) {
    float s = 0.f;
    for (int q = 0; q < (int)gridDim.x; ++q) s = s + __ldcg(partial + (size_t)q * per + e);
    if (e < N) dscale[e] = s;
    else if (e < 2 * N) doffset[e - N] = s;
    else if (e < 3 * N) db[e - 2 * N] = s;
    else dw_a[e - 3 * N] = s;
  }
  if (t == 0) g_feature_tickets[ticket] = 0u;
}

// acme/tf/networks/rescaling.py:63-74
__global__ void tanh_to_spec_fwd_kernel(long long n, int A, const float* __restrict__ x, const float* __restrict__ scale,
                                        const float* __restrict__ offset, float* __restrict__ a) {
  pdl_launch_dependents();
  pdl_wait();
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int c = (int)(i % A);
  float t = tanhf(x[i]);
  t = 0.5f * (t + 1.0f);
  a[i] = t * scale[c] + offset[c];
}
__global__ void tanh_to_spec_bwd_kernel(long long n, int A, const float* __restrict__ da, const float* __restrict__ x,
                                        const float* __restrict__ scale, float* __restrict__ dx) {
  pdl_launch_dependents();
  pdl_wait();
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int c = (int)(i % A);
  float t = tanhf(x[i]);
  dx[i] = da[i] * 0.5f * scale[c] * (1.f - t * t);
}

// acme/tf/utils.py:39-54 batch_concat of two flat tensors, and the slice of its gradient
__global__ void concat2_kernel(int B, int n0, int n1, const float* __restrict__ x0, const float* __restrict__ x1, float* __restrict__ y) {
  pdl_launch_dependents();
  pdl_wait();
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int n = n0 + n1;
  if (i >= (long long)B * n) return;
  int b = (int)(i / n), c = (int)(i % n);
  y[i] = c < n0 ? x0[(size_t)b * n0 + c] : x1[(size_t)b * n1 + (c - n0)];
}
__global__ void split_second_kernel(int B, int n0, int n1, const float* __restrict__ dy, float* __restrict__ dx1) {
  pdl_launch_dependents();
  pdl_wait();
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)B * n1) return;
  int b = (int)(i / n1), c = (int)(i % n1);
  dx1[i] = dy[(size_t)b * (n0 + n1) + n0 + c];
}

// ---- recurrent replay (SURVEY §8f-3): acme/agents/tf/r2d2/learning.py:230-236 and :170-176
__global__ void seq_priority_kernel(int T, int B, const float* __restrict__ err, float eta, float* __restrict__ out) {
  pdl_launch_dependents();
  pdl_wait();
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  float mx = 0.f, sum = 0.f;
  for (int t = 0; t < T; ++t) {                 // coalesced over b; tf.reduce_mean = sum / T
    const float a = fabsf(err[(size_t)t * B + b]);
    mx = fmaxf(mx, a);
    sum = __fadd_rn(sum, a);
  }
  const float mean = __fdiv_rn(sum, (float)T);
  out[b] = __fadd_rn(__fmul_rn(eta, mx), __fmul_rn(__fsub_rn(1.f, eta), mean));
}

__global__ void __launch_bounds__(1024)
seq_is_weights_kernel(int B, const float* __restrict__ prob, double N, double beta, float* __restrict__ w) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ double red[32];
  double m = 0.0;
  for (int b = threadIdx.x; b < B; b += blockDim.x) m = fmax(m, pow(1.0 / (N * (double)prob[b]), beta));
  for (int o = 16; o; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x < 32) {
    m = threadIdx.x < (blockDim.x + 31) / 32 ? red[threadIdx.x] : 0.0;
    for (int o = 16; o; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (threadIdx.x == 0) red[0] = m;
  }
  __syncthreads();
  const double wmax = red[0];
  for (int b = threadIdx.x; b < B; b += blockDim.x) w[b] = (float)(pow(1.0 / (N * (double)prob[b]), beta) / wmax);
}

}  // namespace b200rl

using namespace b200rl;

static inline int grid1d(long long n, int threads, int cap = kNumSMs * 16) {
  long long b = (n + threads - 1) / threads;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (int)b;
}

extern "C" int b200rl_uniform(float* out, int32_t n, uint64_t seed, const int64_t* step_dev,
                              int64_t step_offset, void* stream) {
  B200RL_REQUIRE(out && n >= 0, "bad argument");
  if (n == 0) return B200RL_OK;
  B200RL_CUDA_OK(launch_pdl_small(uniform_kernel, dim3(ceil_div(n, 256)), dim3(256), 0, as_stream(stream), out, n, seed, (const long long*)step_dev, step_offset));
  B200RL_LAUNCH_OK();
  return B200RL_OK;
}

extern "C" int b200rl_seq_priority(int32_t T, int32_t B, const float* err_tb, float eta, float* priority_out, void* stream) {
  B200RL_REQUIRE(err_tb && priority_out && T >= 1 && B >= 1, "bad argument");
  B200RL_CUDA_OK(launch_pdl_small(seq_priority_kernel, dim3((B + 127) / 128), dim3(128), 0, as_stream(stream), T, B, err_tb, eta, priority_out));
  B200RL_LAUNCH_OK();
  return B200RL_OK;
}

extern "C" int b200rl_seq_is_weights(int32_t B, const float* prob, double table_size, double is_exponent, float* w_out,
                                     void* stream) {
  B200RL_REQUIRE(prob && w_out && B >= 1 && table_size > 0, "bad argument");
  B200RL_CUDA_OK(launch_pdl_small(seq_is_weights_kernel, dim3(1), dim3(B >= 1024 ? 1024 : ((B + 31) / 32) * 32), 0, as_stream(stream), B, prob, table_size, is_exponent, w_out));
  B200RL_LAUNCH_OK();
  return B200RL_OK;
}

extern "C" int b200rl_is_weight_max(int32_t B, const float* prob, double beta, double* out, int32_t flags, void* stream) {
  B200RL_REQUIRE(prob && out && B >= 1, "bad argument");
  B200RL_CUDA_OK(launch_pdl_small(is_weight_max_kernel, dim3(1), dim3(B >= 1024 ? 1024 : ((B + 31) / 32) * 32), 0, as_stream(stream), B, prob, beta, out, flags));
  B200RL_LAUNCH_OK();
  return B200RL_OK;
}

extern "C" int b200rl_dqn_td(int32_t B, int32_t A, const float* q_tm1, const float* q_tv, const float* q_ts,
                             const int32_t* a_tm1, const float* R, const float* D, const float* prob,
                             float gamma, float delta, double beta, float max_abs_reward,
                             const double* wmax_dev, float grad_scale, float* td, float* loss_ps,
                             float* weight, float* priority, float* dq, float* loss_mean, int32_t flags, void* stream) {
  B200RL_REQUIRE(q_tm1 && q_tv && q_ts && a_tm1 && R && D && prob && td && loss_ps && weight && priority && dq,
                 "null argument");
  B200RL_REQUIRE(B >= 1 && A >= 1, "bad shape");
  B200RL_REQUIRE(delta >= 0.f, "quadratic_linear_boundary must be >= 0");  // huber.py:45-46
  int threads = B >= 1024 ? 1024 : ((B + 31) / 32) * 32;
  B200RL_CUDA_OK(launch_pdl_small(dqn_td_kernel, dim3(1), dim3(threads), 0, as_stream(stream), B, A, q_tm1, q_tv, q_ts, a_tm1, R, D, prob, gamma, delta, beta,
                                                     max_abs_reward, wmax_dev, grad_scale, td, loss_ps, weight,
                                                     priority, dq, loss_mean, flags));
  B200RL_LAUNCH_OK();
  return B200RL_OK;
}

extern "C" int b200rl_c51_loss(int32_t B, int32_t K, float vmin, float vmax, const float* logits_tm1,
                               const float* logits_t, const float* R, const float* D, float gamma,
                               float grad_scale, float* target, float* loss_ps, float* dlogits,
                               float* loss_mean, void* stream) {
  B200RL_REQUIRE(logits_tm1 && logits_t && R && D && loss_ps, "null argument");
  B200RL_REQUIRE(B >= 1 && K >= 2 && K <= 1024, "bad shape");
  static const int dense_env = getenv("B200RL_C51_DENSE") ? atoi(getenv("B200RL_C51_DENSE")) : 0;
  if (K <= 64 && !dense_env) {
    B200RL_CUDA_OK(launch_pdl_small(c51_loss_warp_kernel<false>, dim3((B + kC51WarpsPerCta - 1) / kC51WarpsPerCta), dim3(32 * kC51WarpsPerCta), 0, as_stream(stream), B, K, vmin, vmax, logits_tm1, logits_t, R, D, gamma, grad_scale, target, loss_ps, dlogits, IsWeighted{}));
  } else {
    int threads = ((K + 31) / 32) * 32;
    B200RL_CUDA_OK(launch_pdl_small(c51_loss_kernel<false>, dim3(B), dim3(threads), 3 * K * sizeof(float), as_stream(stream), K, vmin, vmax, logits_tm1, logits_t, R, D, gamma,
                                                                             grad_scale, target, loss_ps, dlogits, IsWeighted{}));
  }
  B200RL_LAUNCH_OK();
  if (loss_mean) {
    B200RL_CUDA_OK(launch_pdl_small(mean_kernel, dim3(1), dim3(256), 0, as_stream(stream), loss_ps, B, loss_mean));
    B200RL_LAUNCH_OK();
  }
  return B200RL_OK;
}

extern "C" int b200rl_td_learning(int32_t B, const float* v_tm1, const float* v_t, const float* R, const float* D, float gamma,
                                  float grad_scale, float* td, float* loss_ps, float* dv_tm1, float* loss_mean, void* stream) {
  B200RL_REQUIRE(v_tm1 && v_t && R && D && loss_ps && B >= 1, "bad argument");
  B200RL_CUDA_OK(launch_pdl_small(td_learning_kernel<false>, dim3(ceil_div(B, 128)), dim3(128), 0, as_stream(stream), B, v_tm1, v_t, R, D, gamma, grad_scale, td, loss_ps, dv_tm1, IsWeighted{}));
  B200RL_LAUNCH_OK();
  if (loss_mean) {
    B200RL_CUDA_OK(launch_pdl_small(mean_kernel, dim3(1), dim3(256), 0, as_stream(stream), loss_ps, B, loss_mean));
    B200RL_LAUNCH_OK();
  }
  return B200RL_OK;
}

// the importance-weight arguments shared by the two weighted critic losses; fills `iw` (ticket: the stream's slot)
static int weighted_args(int32_t B, const float* prob, double beta, const double* wmax_dev, float* loss_ps, float* weight,
                         float* priority, float* loss_mean, cudaStream_t st, IsWeighted* iw) {
  B200RL_REQUIRE(prob && wmax_dev && loss_ps && weight && priority, "null argument");
  B200RL_REQUIRE(B >= 1, "bad shape");
  B200RL_REQUIRE(beta >= 0.0, "importance_sampling_exponent must be >= 0");
  int ticket = 0;
  if (loss_mean) {
    ticket = ticket_for(st);
    B200RL_REQUIRE(ticket >= 0, "weighted critic loss: more than 64 streams");
  }
  *iw = IsWeighted{prob, beta, wmax_dev, weight, priority, loss_mean, ticket, B};
  return B200RL_OK;
}

extern "C" int b200rl_c51_loss_weighted(int32_t B, int32_t K, float vmin, float vmax, const float* logits_tm1,
                                        const float* logits_t, const float* R, const float* D, float gamma,
                                        const float* prob, double is_exponent, const double* wmax_dev, float grad_scale,
                                        float* target, float* loss_ps, float* weight, float* priority,
                                        float* dlogits, float* loss_mean, void* stream) {
  B200RL_REQUIRE(logits_tm1 && logits_t && R && D, "null argument");
  B200RL_REQUIRE(K >= 2 && K <= 1024, "bad shape");
  cudaStream_t st = as_stream(stream);
  IsWeighted iw;
  const int rc = weighted_args(B, prob, is_exponent, wmax_dev, loss_ps, weight, priority, loss_mean, st, &iw);
  if (rc != B200RL_OK) return rc;
  static const int dense_env = getenv("B200RL_C51_DENSE") ? atoi(getenv("B200RL_C51_DENSE")) : 0;
  if (K <= 64 && !dense_env) {
    B200RL_CUDA_OK(launch_pdl_small(c51_loss_warp_kernel<true>, dim3((B + kC51WarpsPerCta - 1) / kC51WarpsPerCta), dim3(32 * kC51WarpsPerCta), 0, st,
                                    B, K, vmin, vmax, logits_tm1, logits_t, R, D, gamma, grad_scale, target, loss_ps, dlogits, iw));
  } else {
    int threads = ((K + 31) / 32) * 32;
    B200RL_CUDA_OK(launch_pdl_small(c51_loss_kernel<true>, dim3(B), dim3(threads), 3 * K * sizeof(float), st, K, vmin, vmax, logits_tm1, logits_t,
                                    R, D, gamma, grad_scale, target, loss_ps, dlogits, iw));
  }
  B200RL_LAUNCH_OK();
  return B200RL_OK;
}

extern "C" int b200rl_td_learning_weighted(int32_t B, const float* v_tm1, const float* v_t, const float* R, const float* D,
                                           float gamma, const float* prob, double is_exponent, const double* wmax_dev,
                                           float grad_scale, float* td, float* loss_ps, float* weight, float* priority,
                                           float* dv_tm1, float* loss_mean, void* stream) {
  B200RL_REQUIRE(v_tm1 && v_t && R && D, "null argument");
  cudaStream_t st = as_stream(stream);
  IsWeighted iw;
  const int rc = weighted_args(B, prob, is_exponent, wmax_dev, loss_ps, weight, priority, loss_mean, st, &iw);
  if (rc != B200RL_OK) return rc;
  B200RL_CUDA_OK(launch_pdl_small(td_learning_kernel<true>, dim3(ceil_div(B, 128)), dim3(128), 0, st, B, v_tm1, v_t, R, D, gamma, grad_scale,
                                  td, loss_ps, dv_tm1, iw));
  B200RL_LAUNCH_OK();
  return B200RL_OK;
}

extern "C" int b200rl_c51_mean_fwd(int32_t B, int32_t K, float vmin, float vmax, const float* logits, float* q, void* stream) {
  B200RL_REQUIRE(logits && q && B >= 1 && K >= 2, "bad argument");
  B200RL_CUDA_OK(launch_pdl_small(c51_mean_kernel, dim3(ceil_div(B * 32, 128)), dim3(128), 0, as_stream(stream), B, K, vmin, vmax, logits, nullptr, q, nullptr));
  B200RL_LAUNCH_OK();
  return B200RL_OK;
}
extern "C" int b200rl_c51_mean_bwd(int32_t B, int32_t K, float vmin, float vmax, const float* logits, const float* dq,
                                   float* dlogits, void* stream) {
  B200RL_REQUIRE(logits && dlogits && B >= 1 && K >= 2, "bad argument");
  B200RL_CUDA_OK(launch_pdl_small(c51_mean_kernel, dim3(ceil_div(B * 32, 128)), dim3(128), 0, as_stream(stream), B, K, vmin, vmax, logits, dq, nullptr, dlogits));
  B200RL_LAUNCH_OK();
  return B200RL_OK;
}

extern "C" int b200rl_dpg_action_grad(int32_t B, int32_t A, const float* dqda, float clip, int clip_norm,
                                      float grad_scale, float* da, float* loss_ps, float* loss_mean, void* stream) {
  B200RL_REQUIRE(dqda && da && B >= 1 && A >= 1, "bad argument");
  B200RL_REQUIRE(!loss_mean || loss_ps, "loss_mean needs a loss_per_sample buffer");
  B200RL_CUDA_OK(launch_pdl_small(dpg_kernel, dim3(ceil_div(B * 32, 128)), dim3(128), 0, as_stream(stream), B, A, dqda, clip, clip_norm, grad_scale, da, loss_ps));
  B200RL_LAUNCH_OK();
  if (loss_mean) {
    B200RL_CUDA_OK(launch_pdl_small(mean_kernel, dim3(1), dim3(256), 0, as_stream(stream), loss_ps, B, loss_mean));
    B200RL_LAUNCH_OK();
  }
  return B200RL_OK;
}

// tools/step_phases.py: a one-thread kernel that writes the global timer, placed between the phases of a captured step
__global__ void stamp_kernel(unsigned long long* buf, int slot) {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  buf[slot] = t;
}
extern "C" int b200rl_debug_stamp(unsigned long long* buf, int slot, void* stream) {
  stamp_kernel<<<1, 1, 0, as_stream(stream)>>>(buf, slot);
  return cudaGetLastError() == cudaSuccess ? 0 : -2;
}

extern "C" int b200rl_adam(int64_t n, float* param, const float* grad, float* m, float* v, const int64_t* step_dev,
                           float lr, double b1, double b2, float eps, int eps_mode, const float* grad_scale_dev,
                           void* bf16_shadow, void* stream) {
  B200RL_REQUIRE(param && grad && m && v && step_dev, "null argument");
  B200RL_REQUIRE(n >= 0 && (eps_mode == 0 || eps_mode == 1), "bad argument");
  B200RL_REQUIRE((((uintptr_t)param | (uintptr_t)grad | (uintptr_t)m | (uintptr_t)v) & 15) == 0, "buffers must be 16-byte aligned");
  if (n == 0) return B200RL_OK;
  const int blocks = grid1d((n + 7) / 8, 256, kNumSMs * 8);   // 8 CTAs per SM, grid-stride loop beyond that
  B200RL_CUDA_OK(launch_pdl(adam_kernel, dim3(blocks), dim3(256), 0, as_stream(stream), n, param, grad, m, v,
                            (const long long*)step_dev, lr, b1, b2, eps, eps_mode, grad_scale_dev,
                            (__nv_bfloat16*)bf16_shadow));
  B200RL_LAUNCH_OK();
  return B200RL_OK;
}

extern "C" int b200rl_global_norm_scale(int64_t n, const float* grad, float clip, float* partial_ws, float* scale_out,
                                        float* norm_out, void* stream) {
  B200RL_REQUIRE(grad && partial_ws && scale_out && n >= 1, "bad argument");
  int blocks = grid1d(n, 256, 1024);
  B200RL_CUDA_OK(launch_pdl_small(sumsq_partial_kernel, dim3(blocks), dim3(256), 0, as_stream(stream), n, grad, partial_ws));
  B200RL_LAUNCH_OK();
  B200RL_CUDA_OK(launch_pdl_small(norm_finish_kernel, dim3(1), dim3(256), 0, as_stream(stream), blocks, partial_ws, clip, scale_out, norm_out));
  B200RL_LAUNCH_OK();
  return B200RL_OK;
}

extern "C" int b200rl_copy_if_period(int64_t n_bytes, void* dst, const void* src, const int64_t* step_dev, int64_t period,
                                     int64_t phase, void* stream) {
  B200RL_REQUIRE(dst && src && step_dev && period >= 1, "bad argument");
  B200RL_REQUIRE(n_bytes % 16 == 0 && (((uintptr_t)dst | (uintptr_t)src) & 15) == 0, "copy must be 16-byte aligned/sized");
  B200RL_CUDA_OK(launch_pdl_small(copy_if_period_kernel, dim3(grid1d(n_bytes / 16, 256, kNumSMs * 8)), dim3(256), 0, as_stream(stream), n_bytes / 16, (int4*)dst, (const int4*)src, (const long long*)step_dev, period, phase));
  B200RL_LAUNCH_OK();
  return B200RL_OK;
}

extern "C" int b200rl_learner_tail(int64_t n_bytes_a, void* dst_a, const void* src_a, int64_t n_bytes_b, void* dst_b,
                                   const void* src_b, int64_t* step_dev, int64_t period, int64_t phase, int64_t* counter2,
                                   void* stream) {
  B200RL_REQUIRE(step_dev && period >= 0, "bad argument");
  B200RL_REQUIRE(n_bytes_a >= 0 && n_bytes_b >= 0 && n_bytes_a % 16 == 0 && n_bytes_b % 16 == 0, "copies must be multiples of 16 bytes");
  B200RL_REQUIRE((n_bytes_a == 0 || (dst_a && src_a)) && (n_bytes_b == 0 || (dst_b && src_b)), "null buffer");
  B200RL_REQUIRE(((((uintptr_t)dst_a | (uintptr_t)src_a | (uintptr_t)dst_b | (uintptr_t)src_b)) & 15) == 0, "buffers must be 16-byte aligned");
  // one ticket per call site is enough: calls on one stream never overlap, and a learner has one tail per step
  B200RL_CUDA_OK(launch_pdl(learner_tail_kernel, dim3(kNumSMs * 4), dim3(256), 0, as_stream(stream), (long long)(n_bytes_a / 16), (int4*)dst_a,
                            (const int4*)src_a, (long long)(n_bytes_b / 16), (int4*)dst_b, (const int4*)src_b, (long long*)step_dev,
                            (long long)period, (long long)phase, (long long*)counter2, 0));
  B200RL_LAUNCH_OK();
  return B200RL_OK;
}

extern "C" int b200rl_step_increment(int64_t* step_dev, void* stream) {
  B200RL_REQUIRE(step_dev, "null argument");
  B200RL_CUDA_OK(launch_pdl_small(step_increment_kernel, dim3(1), dim3(1), 0, as_stream(stream), (long long*)step_dev));
  B200RL_LAUNCH_OK();
  return B200RL_OK;
}

extern "C" int b200rl_act_bwd(int64_t n, float* dy, const float* y, int act, void* stream) {
  B200RL_REQUIRE(dy && y && n >= 0, "bad argument");
  if (n == 0 || act == B200RL_ACT_NONE) return B200RL_OK;
  B200RL_CUDA_OK(launch_pdl_small(act_bwd_kernel, dim3(grid1d(n, 256)), dim3(256), 0, as_stream(stream), n, dy, y, act));
  B200RL_LAUNCH_OK();
  return B200RL_OK;
}

extern "C" int b200rl_duelling_fwd(int32_t B, int32_t A, const float* value, const float* adv, float* q, void* stream) {
  B200RL_REQUIRE(value && adv && q && B >= 1 && A >= 1, "bad argument");
  B200RL_CUDA_OK(launch_pdl_small(duelling_fwd_kernel, dim3(ceil_div(B, 128)), dim3(128), 0, as_stream(stream), B, A, value, adv, q));
  B200RL_LAUNCH_OK();
  return B200RL_OK;
}
extern "C" int b200rl_duelling_bwd(int32_t B, int32_t A, const float* dq, float* dvalue, float* dadv, void* stream) {
  B200RL_REQUIRE(dq && dvalue && dadv && B >= 1 && A >= 1, "bad argument");
  B200RL_CUDA_OK(launch_pdl_small(duelling_bwd_kernel, dim3(ceil_div(B, 128)), dim3(128), 0, as_stream(stream), B, A, dq, dvalue, dadv));
  B200RL_LAUNCH_OK();
  return B200RL_OK;
}


static int ensure_head_attrs() {
  static bool attr = false;
  if (!attr) {
    B200RL_CUDA_OK(cudaFuncSetAttribute(duelling_head_fwd_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    B200RL_CUDA_OK(cudaFuncSetAttribute(duelling_head_fwd_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    B200RL_CUDA_OK(cudaFuncSetAttribute(duelling_head_fwd_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    B200RL_CUDA_OK(cudaFuncSetAttribute(duelling_head_fwd_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    attr = true;
  }
  return B200RL_OK;
}

extern "C" int b200rl_duelling_head_fwd(int32_t B, int32_t A, int32_t H, const float* h, int32_t ldh, const float* wv,
                                        const float* bv, const float* wa, const float* ba, float* value, float* adv,
                                        float* q, void* stream) {
  B200RL_REQUIRE(h && wv && bv && wa && ba && value && adv && q && B >= 1 && A >= 1 && ldh >= 2 * H, "bad argument");
  const int blocks = ceil_div(B * 32, 256);
  cudaStream_t st = as_stream(stream);
  const size_t smem = (size_t)(A + 1) * H * 4;
  B200RL_REQUIRE(smem <= 200 * 1024 && H % 4 == 0, "duelling head weights do not fit in shared memory");
  if (int rc = ensure_head_attrs()) return rc;
  switch (H) {
    case 512: B200RL_CUDA_OK(launch_pdl_small(duelling_head_fwd_kernel<16>, dim3(blocks), dim3(256), smem, st, B, A, h, ldh, wv, bv, wa, ba, value, adv, q)); break;
    case 256: B200RL_CUDA_OK(launch_pdl_small(duelling_head_fwd_kernel<8>, dim3(blocks), dim3(256), smem, st, B, A, h, ldh, wv, bv, wa, ba, value, adv, q)); break;
    case 128: B200RL_CUDA_OK(launch_pdl_small(duelling_head_fwd_kernel<4>, dim3(blocks), dim3(256), smem, st, B, A, h, ldh, wv, bv, wa, ba, value, adv, q)); break;
    case 64: B200RL_CUDA_OK(launch_pdl_small(duelling_head_fwd_kernel<2>, dim3(blocks), dim3(256), smem, st, B, A, h, ldh, wv, bv, wa, ba, value, adv, q)); break;
    default: set_error("duelling head: hidden size %d not in {64,128,256,512}", H); return B200RL_EINVAL;
  }
  B200RL_LAUNCH_OK();
  return B200RL_OK;
}
extern "C" int b200rl_duelling_head_bwd(int32_t B, int32_t A, int32_t H, const float* dq, const float* h, int32_t ldh,
                                        const float* wv, const float* wa, float* dvalue, float* dadv, float* dh,
                                        int32_t lddh, float* dwv, float* dbv, float* dwa, float* dba, void* ws,
                                        int64_t ws_bytes, void* stream) {
  B200RL_REQUIRE(dq && h && wv && wa && dvalue && dadv && dh && dwv && dbv && dwa && dba && ws, "null argument");
  B200RL_REQUIRE(B >= 1 && A >= 1 && H >= 1 && ldh >= 2 * H && lddh >= 2 * H, "bad shape");
  cudaStream_t st = as_stream(stream);
  const size_t smem = (size_t)(A + 1) * H * 4;
  B200RL_REQUIRE(smem <= 200 * 1024 && H % 4 == 0, "duelling head weights do not fit in shared memory");
  if (int rc = ensure_head_attrs()) return rc;
  B200RL_REQUIRE(ldh % 4 == 0 && lddh % 4 == 0 &&
                     (((uintptr_t)h | (uintptr_t)dh | (uintptr_t)wv | (uintptr_t)wa) & 15) == 0,
                 "duelling head: rows must be 16-byte aligned");
  B200RL_CUDA_OK(launch_pdl_small(duelling_head_bwd_dh_kernel, dim3((int)ceil_div<long long>((long long)B * (H / 4), 256)), dim3(256), 0, st, B, A, H, dq, h, ldh, wv, wa,
                                                                                                     dvalue, dadv, dh, lddh));
  B200RL_LAUNCH_OK();
  int segs = std::max(1, std::min(B / 32, 8));
  const int64_t per = (int64_t)(A + 1) * (H + 1) * 4;
  segs = (int)std::max<int64_t>(1, std::min<int64_t>(segs, ws_bytes / per));
  B200RL_CUDA_OK(launch_pdl_small(duelling_head_bwd_dw_kernel, dim3(dim3(ceil_div(H, 128), A + 1, segs)), dim3(128), 0, st, B, A, H, dvalue, dadv, h, ldh, (float*)ws));
  B200RL_LAUNCH_OK();
  B200RL_CUDA_OK(launch_pdl_small(duelling_head_bwd_finish_kernel, dim3(ceil_div((A + 1) * (H + 1), 256)), dim3(256), 0, st, A, H, segs, (const float*)ws, dwv, dbv, dwa, dba));
  B200RL_LAUNCH_OK();
  return B200RL_OK;
}

extern "C" int b200rl_dqn_head_td(int32_t B, int32_t A, int32_t H, const float* h_tm1, const float* h_sel, const float* h_tgt,
                                  int32_t ldh, const float* wv, const float* bv, const float* wa, const float* ba,
                                  const float* twv, const float* tbv, const float* twa, const float* tba,
                                  const int32_t* a_tm1, const float* R, const float* D, const float* prob, float gamma,
                                  float huber_delta, double is_exponent, float max_abs_reward, const double* wmax_dev,
                                  float grad_scale, int32_t flags, float* q_tm1, float* q_tv, float* q_ts, float* td,
                                  float* loss_ps, float* weight, float* priority, float* dq, float* dval, float* dadv,
                                  void* dh, int32_t lddh, int32_t dh_bf16, void* stream) {
  B200RL_REQUIRE(h_tm1 && h_sel && h_tgt && wv && bv && wa && ba && twv && tbv && twa && tba && a_tm1 && R && D && prob &&
                     wmax_dev && td && loss_ps && weight && priority && dval && dadv && dh,
                 "null argument");
  B200RL_REQUIRE(B >= 1 && A >= 1 && A <= 32 && ldh >= 2 * H && lddh >= 2 * H, "bad shape (the fused head needs A <= 32)");
  B200RL_REQUIRE(huber_delta >= 0.f, "quadratic_linear_boundary must be >= 0");
  B200RL_REQUIRE((((uintptr_t)wv | (uintptr_t)wa | (uintptr_t)twv | (uintptr_t)twa) & 15) == 0 && H % 4 == 0,
                 "head weights must be 16-byte aligned");
  const size_t smem = 2 * (size_t)(A + 1) * H * 4;
  B200RL_REQUIRE(smem <= 200 * 1024, "duelling head weights do not fit in shared memory");
  HeadTdArgs p;
  p.B = B; p.A = A; p.ldh = ldh; p.lddh = lddh; p.flags = flags; p.dh_bf16 = dh_bf16;
  p.h_tm1 = h_tm1; p.h_sel = h_sel; p.h_tgt = h_tgt;
  p.wv = wv; p.bv = bv; p.wa = wa; p.ba = ba; p.twv = twv; p.tbv = tbv; p.twa = twa; p.tba = tba;
  p.a_tm1 = a_tm1; p.R = R; p.D = D; p.prob = prob;
  p.gamma = gamma; p.delta = huber_delta; p.max_abs_r = max_abs_reward; p.grad_scale = grad_scale; p.beta = is_exponent;
  p.wmax_dev = wmax_dev;
  p.q_tm1 = q_tm1; p.q_tv = q_tv; p.q_ts = q_ts; p.td = td; p.loss_ps = loss_ps; p.weight = weight; p.priority = priority;
  p.dq = dq; p.dval = dval; p.dadv = dadv; p.dh = dh;
  static bool attr = false;
  if (!attr) {
    B200RL_CUDA_OK(cudaFuncSetAttribute(dqn_head_td_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    B200RL_CUDA_OK(cudaFuncSetAttribute(dqn_head_td_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    B200RL_CUDA_OK(cudaFuncSetAttribute(dqn_head_td_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    B200RL_CUDA_OK(cudaFuncSetAttribute(dqn_head_td_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    attr = true;
  }
  const int blocks = ceil_div(B, kHeadSamples);
  cudaStream_t st = as_stream(stream);
  cudaError_t e = cudaSuccess;
  switch (H) {
    case 512: e = launch_pdl(dqn_head_td_kernel<16>, dim3(blocks), dim3(kHeadThreads), smem, st, p); break;
    case 256: e = launch_pdl(dqn_head_td_kernel<8>, dim3(blocks), dim3(kHeadThreads), smem, st, p); break;
    case 128: e = launch_pdl(dqn_head_td_kernel<4>, dim3(blocks), dim3(kHeadThreads), smem, st, p); break;
    case 64: e = launch_pdl(dqn_head_td_kernel<2>, dim3(blocks), dim3(kHeadThreads), smem, st, p); break;
    default: set_error("fused duelling head: hidden size %d not in {64,128,256,512}", H); return B200RL_EINVAL;
  }
  B200RL_CUDA_OK(e);
  B200RL_LAUNCH_OK();
  return B200RL_OK;
}

extern "C" int b200rl_mean(int32_t n, const float* x, float* out, void* stream) {
  B200RL_REQUIRE(x && out && n >= 1, "bad argument");
  B200RL_CUDA_OK(launch_pdl_small(mean_kernel, dim3(1), dim3(256), 0, as_stream(stream), x, n, out));
  B200RL_LAUNCH_OK();
  return B200RL_OK;
}

// parameter gradients of the duelling head alone (dwv, dbv, dwa, dba) from dval / dadv and the hidden rows: the part of
// b200rl_duelling_head_bwd that is NOT on the critical path once the fused kernel above has produced dh
extern "C" int b200rl_duelling_head_wgrad(int32_t B, int32_t A, int32_t H, const float* dvalue, const float* dadv, const float* h,
                                          int32_t ldh, float* dwv, float* dbv, float* dwa, float* dba, void* ws, int64_t ws_bytes,
                                          void* stream) {
  B200RL_REQUIRE(dvalue && dadv && h && dwv && dbv && dwa && dba && ws, "null argument");
  B200RL_REQUIRE(B >= 1 && A >= 1 && H >= 1 && ldh >= 2 * H, "bad shape");
  cudaStream_t st = as_stream(stream);
  int segs = std::max(1, std::min(B / 32, 8));
  const int64_t per = (int64_t)(A + 1) * (H + 1) * 4;
  segs = (int)std::max<int64_t>(1, std::min<int64_t>(segs, ws_bytes / per));
  B200RL_CUDA_OK(launch_pdl_small(duelling_head_bwd_dw_kernel, dim3(dim3(ceil_div(H, 128), A + 1, segs)), dim3(128), 0, st, B, A, H, dvalue, dadv, h, ldh, (float*)ws));
  B200RL_LAUNCH_OK();
  B200RL_CUDA_OK(launch_pdl_small(duelling_head_bwd_finish_kernel, dim3(ceil_div((A + 1) * (H + 1), 256)), dim3(256), 0, st, A, H, segs, (const float*)ws, dwv, dbv, dwa, dba));
  B200RL_LAUNCH_OK();
  return B200RL_OK;
}

extern "C" int b200rl_layernorm_tanh_fwd(int32_t B, int32_t N, const float* x, const float* scale, const float* offset,
                                         float eps, float* y, float* xhat, float* rstd, void* stream) {
  B200RL_REQUIRE(x && scale && offset && y && xhat && rstd && B >= 1 && N >= 1, "bad argument");
  B200RL_CUDA_OK(launch_pdl_small(layernorm_tanh_fwd_kernel, dim3(B), dim3(256), 0, as_stream(stream), N, x, scale, offset, eps, y, xhat, rstd,
                                  (__nv_bfloat16*)nullptr));
  B200RL_LAUNCH_OK();
  return B200RL_OK;
}
extern "C" int b200rl_layernorm_tanh_fwd_bf16(int32_t B, int32_t N, const float* x, const float* scale, const float* offset,
                                              float eps, float* y, void* y_bf16, float* xhat, float* rstd, void* stream) {
  B200RL_REQUIRE(x && scale && offset && y && y_bf16 && xhat && rstd && B >= 1 && N >= 1, "bad argument");
  B200RL_CUDA_OK(launch_pdl_small(layernorm_tanh_fwd_kernel, dim3(B), dim3(256), 0, as_stream(stream), N, x, scale, offset, eps, y, xhat, rstd,
                                  (__nv_bfloat16*)y_bf16));
  B200RL_LAUNCH_OK();
  return B200RL_OK;
}

extern "C" int b200rl_dense_head_bwd_bf16(int32_t M, int32_t N, int32_t K, const float* dy, int32_t lddy, const void* x_bf16,
                                          int32_t ldx, const void* w_bf16, void* dx_bf16, int32_t lddx, const void* mask_bf16,
                                          int mask_act, float* dw, float* db, void* ws, int64_t ws_bytes, void* stream) {
  B200RL_REQUIRE(dy && w_bf16 && dx_bf16 && (x_bf16 || !dw), "null argument");
  B200RL_REQUIRE(M >= 1 && N >= 1 && N <= 64 && K >= 8 && K % 8 == 0 && lddy >= N && lddx >= K,
                 "dense head backward: N = %d must be in [1, 64] and K = %d a multiple of 8", N, K);
  B200RL_REQUIRE(lddx % 8 == 0 && (!dw || (ldx >= K && ldx % 8 == 0)) &&
                     (((uintptr_t)w_bf16 | (uintptr_t)dx_bf16 | (uintptr_t)mask_bf16 | (uintptr_t)(dw ? x_bf16 : nullptr)) & 15) == 0,
                 "dense head backward: bf16 rows must be 16-byte aligned");
  cudaStream_t st = as_stream(stream);
  const int kblocks = ceil_div(K, kHbCols);
  // row slices: enough CTAs for the latency-bound batch sizes, at most 32 partial slabs per column block
  int slices = std::min(ceil_div(M, kHbRows), (dw || db) ? 32 : 4096);
  int ticket = -1;
  if ((dw || db) && slices > 1) {
    const int64_t per = ((int64_t)kblocks * 64 * kHbCols + 64) * 4;
    if (kblocks <= kHbMaxColBlocks && ws) slices = (int)std::min<int64_t>(slices, ws_bytes / per);
    else slices = 1;
    if (slices > 1) ticket = ticket_for(st);
    if (ticket < 0) slices = 1;
  }
  slices = std::max(slices, 1);
  const int rpc = ceil_div(M, slices);
  slices = ceil_div(M, rpc);
  B200RL_CUDA_OK(launch_pdl_small(dense_head_bwd_bf16_kernel, dim3(kblocks, slices), dim3(256), 0, st, M, N, K, dy, lddy,
                                  (const __nv_bfloat16*)x_bf16, ldx, (const __nv_bfloat16*)w_bf16, (__nv_bfloat16*)dx_bf16, lddx,
                                  (const __nv_bfloat16*)mask_bf16, mask_act, dw, db, rpc, (float*)ws, ticket < 0 ? 0 : ticket));
  B200RL_LAUNCH_OK();
  return B200RL_OK;
}
extern "C" int b200rl_layernorm_tanh_bwd(int32_t B, int32_t N, const float* dy, const float* y, const float* xhat,
                                         const float* rstd, const float* scale, float* dx, float* dscale,
                                         float* doffset, void* stream) {
  B200RL_REQUIRE(dy && y && xhat && rstd && scale && dx && B >= 1 && N >= 1, "bad argument");
  B200RL_CUDA_OK(launch_pdl_small(layernorm_tanh_bwd_kernel, dim3(B), dim3(256), 0, as_stream(stream), N, dy, y, xhat, rstd, scale, dx));
  B200RL_LAUNCH_OK();
  if (dscale && doffset) {
    B200RL_CUDA_OK(launch_pdl_small(layernorm_param_grad_kernel, dim3(ceil_div(N, 128)), dim3(128), 0, as_stream(stream), B, N, dy, y, xhat, dscale, doffset));
    B200RL_LAUNCH_OK();
  }
  return B200RL_OK;
}

extern "C" int b200rl_feature_layer_fwd(int32_t B, int32_t N, int32_t A, const float* zf, const float* a, const float* w_a,
                                        const float* bias, const float* scale, const float* offset, float eps, float* y,
                                        void* y_bf16, float* xhat, float* rstd, void* stream) {
  B200RL_REQUIRE(zf && bias && scale && offset && y && xhat && rstd && (A == 0 || (a && w_a)), "feature layer: null argument");
  B200RL_REQUIRE(B >= 1 && N >= 1 && N <= kFeatMaxN && A >= 0 && A <= kFeatMaxA,
                 "feature layer: N = %d must be in [1, %d] and A = %d in [0, %d]", N, kFeatMaxN, A, kFeatMaxA);
  B200RL_CUDA_OK(launch_pdl_small(feature_layer_fwd_kernel, dim3(B), dim3(256), 0, as_stream(stream), N, A, zf, a, w_a, bias,
                                  scale, offset, eps, y, (__nv_bfloat16*)y_bf16, xhat, rstd));
  B200RL_LAUNCH_OK();
  return B200RL_OK;
}

extern "C" int b200rl_feature_layer_bwd(int32_t B, int32_t N, int32_t A, const float* dy, const float* y, const float* xhat,
                                        const float* rstd, const float* scale, const float* a, const float* w_a, float* dz,
                                        void* dz_bf16, float* dscale, float* doffset, float* db, float* dw_a, float* da,
                                        void* ws, int64_t ws_bytes, void* stream) {
  const bool grads = dscale || doffset || db || dw_a;
  B200RL_REQUIRE(dy && y && xhat && rstd && scale && dz, "feature layer backward: null argument");
  B200RL_REQUIRE(B >= 1 && N >= 1 && N <= kFeatMaxN && A >= 0 && A <= kFeatMaxA,
                 "feature layer backward: N = %d must be in [1, %d] and A = %d in [0, %d]", N, kFeatMaxN, A, kFeatMaxA);
  B200RL_REQUIRE(!grads || (dscale && doffset && db && (A == 0 || dw_a)),
                 "feature layer backward: d scale, d offset, db and dw_a are requested together");
  B200RL_REQUIRE(!(grads && A > 0) || a, "feature layer backward: dw_a needs the actions");
  B200RL_REQUIRE(!da || (A > 0 && w_a), "feature layer backward: da needs A >= 1 and w_a");
  cudaStream_t st = as_stream(stream);
  int slices = ceil_div(B, kFeatRows);
  int ticket = -1;
  if (grads && slices > 1) {
    const int64_t per = (int64_t)N * (3 + A) * 4;
    slices = ws ? (int)std::min<int64_t>(slices, ws_bytes / per) : 1;
    if (slices > 1) ticket = ticket_for(st);
    if (ticket < 0) slices = 1;
  }
  slices = std::max(slices, 1);
  const int rpc = ceil_div(B, slices);
  // a slice holds at most kFeatRows rows in shared memory: with too little workspace for the slabs, refuse
  B200RL_REQUIRE(rpc <= kFeatRows, "feature layer backward: workspace of %lld bytes is too small for B = %d",
                 (long long)ws_bytes, B);
  slices = ceil_div(B, rpc);
  B200RL_CUDA_OK(launch_pdl_small(feature_layer_bwd_kernel, dim3(slices), dim3(256), 0, st, B, N, A, dy, y, xhat, rstd, scale,
                                  a, w_a, dz, (__nv_bfloat16*)dz_bf16, dscale, doffset, db, A > 0 ? dw_a : nullptr, da, rpc,
                                  (float*)ws, ticket < 0 ? 0 : ticket));
  B200RL_LAUNCH_OK();
  return B200RL_OK;
}

extern "C" int b200rl_tanh_to_spec_fwd(int32_t B, int32_t A, const float* x, const float* scale, const float* offset,
                                       float* a, void* stream) {
  B200RL_REQUIRE(x && scale && offset && a && B >= 1 && A >= 1, "bad argument");
  long long n = (long long)B * A;
  B200RL_CUDA_OK(launch_pdl_small(tanh_to_spec_fwd_kernel, dim3((int)ceil_div<long long>(n, 256)), dim3(256), 0, as_stream(stream), n, A, x, scale, offset, a));
  B200RL_LAUNCH_OK();
  return B200RL_OK;
}
extern "C" int b200rl_tanh_to_spec_bwd(int32_t B, int32_t A, const float* da, const float* x, const float* scale,
                                       float* dx, void* stream) {
  B200RL_REQUIRE(da && x && scale && dx && B >= 1 && A >= 1, "bad argument");
  long long n = (long long)B * A;
  B200RL_CUDA_OK(launch_pdl_small(tanh_to_spec_bwd_kernel, dim3((int)ceil_div<long long>(n, 256)), dim3(256), 0, as_stream(stream), n, A, da, x, scale, dx));
  B200RL_LAUNCH_OK();
  return B200RL_OK;
}

extern "C" int b200rl_concat2(int32_t B, int32_t n0, int32_t n1, const float* x0, const float* x1, float* y, void* stream) {
  B200RL_REQUIRE(x0 && x1 && y && B >= 1 && n0 >= 1 && n1 >= 1, "bad argument");
  long long n = (long long)B * (n0 + n1);
  B200RL_CUDA_OK(launch_pdl_small(concat2_kernel, dim3((int)ceil_div<long long>(n, 256)), dim3(256), 0, as_stream(stream), B, n0, n1, x0, x1, y));
  B200RL_LAUNCH_OK();
  return B200RL_OK;
}
extern "C" int b200rl_split_second(int32_t B, int32_t n0, int32_t n1, const float* dy, float* dx1, void* stream) {
  B200RL_REQUIRE(dy && dx1 && B >= 1 && n0 >= 1 && n1 >= 1, "bad argument");
  long long n = (long long)B * n1;
  B200RL_CUDA_OK(launch_pdl_small(split_second_kernel, dim3((int)ceil_div<long long>(n, 256)), dim3(256), 0, as_stream(stream), B, n0, n1, dy, dx1));
  B200RL_LAUNCH_OK();
  return B200RL_OK;
}
