// K6, fp32 parity mode: one tiled SIMT GEMM (FFMA, fp32 accumulate) with pluggable operand
// loaders, used for every dense contraction of the Q-network / critic / policy:
//   linear fwd / dgrad / wgrad           (acme/tf/networks/duelling.py:37-59, continuous.py:37-68)
//   conv2d fwd / wgrad / dgrad (NHWC, TF-SAME asymmetric padding, implicit im2col -- no col buffer)
//                                        (acme/tf/networks/atari.py:36-52)
// This mode exists to meet the 1e-5 parity bar against the fp32 oracle; the speed mode is the
// tcgen05 path in gemm_tc.cu.  C[row, col] = sum_red A(row, red) * B(red, col).
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <mutex>
#include <vector>

#include "common.cuh"
#include "gemm_common.cuh"

namespace b200rl {

constexpr int BM = 64, BN = 64, BK = 16, GEMM_THREADS = 256;

// ---- loaders.  load(outer, red) returns 4 values:
//   kRedContig  : (outer, red .. red+3)          -- 4 consecutive reduction indices
//   !kRedContig : (outer .. outer+3, red)        -- 4 consecutive outer indices
// Out-of-range elements read as zero.  `outer` is the row index for A and the column index for B.
struct DenseRed {   // element (outer, red) at p[outer * ld + red]
  static constexpr bool kRedContig = true;
  const float* p; int ld; int n_outer; int n_red;
  __device__ __forceinline__ float4 load(int outer, int red) const {
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (outer >= n_outer || red >= n_red) return v;
    const float* q = p + (size_t)outer * ld + red;
    if (red + 3 < n_red && ((((uintptr_t)q) & 15) == 0)) return __ldg(reinterpret_cast<const float4*>(q));
    v.x = __ldg(q);
    if (red + 1 < n_red) v.y = __ldg(q + 1);
    if (red + 2 < n_red) v.z = __ldg(q + 2);
    if (red + 3 < n_red) v.w = __ldg(q + 3);
    return v;
  }
};
struct DenseOuter { // element (outer, red) at p[red * ld + outer]
  static constexpr bool kRedContig = false;
  const float* p; int ld; int n_outer; int n_red;
  __device__ __forceinline__ float4 load(int outer, int red) const {
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (outer >= n_outer || red >= n_red) return v;
    const float* q = p + (size_t)red * ld + outer;
    if (outer + 3 < n_outer && ((((uintptr_t)q) & 15) == 0)) return __ldg(reinterpret_cast<const float4*>(q));
    v.x = __ldg(q);
    if (outer + 1 < n_outer) v.y = __ldg(q + 1);
    if (outer + 2 < n_outer) v.z = __ldg(q + 2);
    if (outer + 3 < n_outer) v.w = __ldg(q + 3);
    return v;
  }
};

// implicit im2col of an NHWC tensor: pixel m = (b, oy, ox), patch index k = (ky, kx, ci); C % 4 == 0
struct Im2colBase {
  const void* x; int u8; b200rl_conv_geom g; int Mtot; int Ktot;
  __device__ __forceinline__ float4 fetch(int m, int k) const {
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (m >= Mtot || k >= Ktot) return v;
    const int ox = m % g.OW; int t = m / g.OW; const int oy = t % g.OH; const int b = t / g.OH;
    const int ci = k % g.C; int t2 = k / g.C; const int kx = t2 % g.kw; const int ky = t2 / g.kw;
    const int iy = oy * g.stride - g.pad_top + ky, ix = ox * g.stride - g.pad_left + kx;
    if (iy < 0 || iy >= g.H || ix < 0 || ix >= g.W) return v;
    const size_t off = (((size_t)b * g.H + iy) * g.W + ix) * g.C + ci;
    if (u8) {
      uchar4 q = __ldg(reinterpret_cast<const uchar4*>((const uint8_t*)x + off));
      // float32(u8)/255 with a true division: equals np.float32(u/255.0) for all 256 values
      v.x = __fdiv_rn((float)q.x, 255.f); v.y = __fdiv_rn((float)q.y, 255.f);
      v.z = __fdiv_rn((float)q.z, 255.f); v.w = __fdiv_rn((float)q.w, 255.f);
    } else {
      v = __ldg(reinterpret_cast<const float4*>((const float*)x + off));
    }
    return v;
  }
};
struct Im2colRows : Im2colBase {   // A of conv fwd: (outer = pixel m, red = k)
  static constexpr bool kRedContig = true;
  __device__ __forceinline__ float4 load(int outer, int red) const { return fetch(outer, red); }
};
struct Im2colCols : Im2colBase {   // B of conv wgrad: (outer = k, red = pixel m): 4 consecutive k
  static constexpr bool kRedContig = false;
  __device__ __forceinline__ float4 load(int outer, int red) const { return fetch(red, outer); }
};

// conv dgrad in gather form: row m' = input pixel (b, iy, ix); red = (ky, kx, co); Cout % 4 == 0
struct DgradRows {
  static constexpr bool kRedContig = true;
  const float* dy; b200rl_conv_geom g; int Mtot; int Rtot;
  __device__ __forceinline__ float4 load(int m, int r) const {
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (m >= Mtot || r >= Rtot) return v;
    const int ix = m % g.W; int t = m / g.W; const int iy = t % g.H; const int b = t / g.H;
    const int co = r % g.Cout; int t2 = r / g.Cout; const int kx = t2 % g.kw; const int ky = t2 / g.kw;
    const int ny = iy + g.pad_top - ky, nx = ix + g.pad_left - kx;
    if (ny < 0 || nx < 0 || ny % g.stride || nx % g.stride) return v;
    const int oy = ny / g.stride, ox = nx / g.stride;
    if (oy >= g.OH || ox >= g.OW) return v;
    return __ldg(reinterpret_cast<const float4*>(dy + (((size_t)b * g.OH + oy) * g.OW + ox) * g.Cout + co));
  }
};
struct DgradWeights {  // B(red = (ky,kx,co), outer = ci) = w[co][ky][kx][ci]; 4 consecutive ci
  static constexpr bool kRedContig = false;
  const float* w; b200rl_conv_geom g; int Rtot;
  __device__ __forceinline__ float4 load(int ci, int r) const {
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (ci >= g.C || r >= Rtot) return v;
    const int co = r % g.Cout; int t2 = r / g.Cout; const int kx = t2 % g.kw; const int ky = t2 / g.kw;
    return __ldg(reinterpret_cast<const float4*>(w + (((size_t)co * g.kh + ky) * g.kw + kx) * g.C + ci));
  }
};

// CTA tile (16 TM) x (16 TN) with TM, TN in {4, 8}: thread (ty, tx) of the 16 x 16 grid owns rows ty*4 .. ty*4+3 (and, for
// TM = 8, the same rows + 64) and likewise columns -- the two float4 fragments of an 8-wide micro-tile sit 64 apart so
// that the shared-memory reads of a quarter-warp stay conflict-free.  128 x 128 tiles do 64 FFMA per 4 LDS.128 (the
// 64 x 64 tile of round 1: 16 per 2, LDS-bound at 16 TFLOP/s); the k order inside a thread is the same for every
// tile shape, so results only depend on the split-K count.
// conv dgrad of a strided convolution, one STRIDE PHASE at a time: with n = i + pad = s q + p an input pixel only meets
// the taps k = p + s t, so in the gather form above (all taps for every pixel) (s^2 - 1) / s^2 of the products are zeros
// (conv2, stride 2: 606 us for 1.85 useful GFLOP).  Rows of phase (py, px) are its pixels in (b, iy, ix) order (row_map,
// built per call into the workspace), the reduction runs over (ty, tx, co) with ky = py + s ty, kx = px + s tx.
struct DgradPhaseRows {
  static constexpr bool kRedContig = true;
  const float* dy; b200rl_conv_geom g; const int* row_map; int Mp; int Rp; int py, px, ntx;
  __device__ __forceinline__ float4 load(int m, int r) const {
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (m >= Mp || r >= Rp) return v;
    const int pix = row_map[m];
    const int ix = pix % g.W; int t = pix / g.W; const int iy = t % g.H; const int b = t / g.H;
    const int co = r % g.Cout; int t2 = r / g.Cout; const int kx = px + g.stride * (t2 % ntx), ky = py + g.stride * (t2 / ntx);
    const int ny = iy + g.pad_top - ky, nx = ix + g.pad_left - kx;
    if (ny < 0 || nx < 0) return v;
    const int oy = ny / g.stride, ox = nx / g.stride;      // exact: the pixel is of this phase
    if (oy >= g.OH || ox >= g.OW) return v;
    return __ldg(reinterpret_cast<const float4*>(dy + (((size_t)b * g.OH + oy) * g.OW + ox) * g.Cout + co));
  }
};
struct DgradPhaseWeights {
  static constexpr bool kRedContig = false;
  const float* w; b200rl_conv_geom g; int Rp; int py, px, ntx;
  __device__ __forceinline__ float4 load(int ci, int r) const {
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (ci >= g.C || r >= Rp) return v;
    const int co = r % g.Cout; int t2 = r / g.Cout; const int kx = px + g.stride * (t2 % ntx), ky = py + g.stride * (t2 / ntx);
    return __ldg(reinterpret_cast<const float4*>(w + (((size_t)co * g.kh + ky) * g.kw + kx) * g.C + ci));
  }
};
// row_map[base(phase) + rank of the pixel inside its phase] = pixel, for all s^2 phases at once
__global__ void dgrad_row_map_kernel(b200rl_conv_geom g, int* __restrict__ map) {
  pdl_launch_dependents();
  pdl_wait();
  const int pix = blockIdx.x * blockDim.x + threadIdx.x;
  if (pix >= g.B * g.H * g.W) return;
  const int s = g.stride;
  const int ix = pix % g.W; int t = pix / g.W; const int iy = t % g.H; const int b = t / g.H;
  const int py = (iy + g.pad_top) % s, px = (ix + g.pad_left) % s;
  auto first = [&](int p, int pad) { return ((p - pad) % s + s) % s; };          // first index of the phase
  auto count = [&](int p, int pad, int n) { const int f = first(p, pad); return f < n ? (n - f + s - 1) / s : 0; };
  int base = 0;
  for (int q = 0; q < py * s + px; ++q) base += g.B * count(q / s, g.pad_top, g.H) * count(q % s, g.pad_left, g.W);
  const int hy = count(py, g.pad_top, g.H), wx = count(px, g.pad_left, g.W);
  const int qy = (iy - first(py, g.pad_top)) / s, qx = (ix - first(px, g.pad_left)) / s;
  map[base + (b * hy + qy) * wx + qx] = pix;
}

template <class AL, class BL, int TM, int TN>
__global__ void __launch_bounds__(GEMM_THREADS)
gemm_kernel(AL a, BL b, Epilogue epi, int M, int N, int K, int k_per_split) {
  // no early pdl_launch_dependents(): this kernel runs for tens of microseconds beside other streams' GEMMs, and a
  // dependent grid parked on the SMs (a 2,000-CTA split-K finish fills every thread slot) starves them -- measured 2.40
  // -> 2.60 ms per fp32 step with the trigger here
  pdl_wait();
  constexpr int TBM = 16 * TM, TBN = 16 * TN, LA = TM / 4, LB = TN / 4;
  __shared__ __align__(16) float As[2][BK][TBM + 4];
  __shared__ __align__(16) float Bs[2][BK][TBN + 4];
  const int tid = threadIdx.x;
  const int row0 = blockIdx.y * TBM, col0 = blockIdx.x * TBN;
  const int k_begin = blockIdx.z * k_per_split;
  const int k_end = min(K, k_begin + k_per_split);
  const int tx = tid & 15, ty = tid >> 4;

  // per-thread load coordinates inside a tile: L float4 per operand; load l of a red-contiguous operand takes rows
  // + 64 l, of an outer-contiguous one (two loads) reduction rows + 8 l
  auto coord = [&](bool red_contig, int loads, int l, int& outer, int& red) {
    if (red_contig) { outer = (tid >> 2) + 64 * l; red = (tid & 3) << 2; }
    else if (loads == 1) { outer = (tid & 15) << 2; red = tid >> 4; }
    else { outer = (tid & 31) << 2; red = (tid >> 5) + 8 * l; }
  };

  float acc[TM][TN];
#pragma unroll
  for (int i = 0; i < TM; ++i)
#pragma unroll
    for (int j = 0; j < TN; ++j) acc[i][j] = 0.f;

  auto fetch = [&](int k0, float4 (&av)[LA], float4 (&bv)[LB]) {
#pragma unroll
    for (int l = 0; l < LA; ++l) { int o, r; coord(AL::kRedContig, LA, l, o, r); av[l] = a.load(row0 + o, k0 + r); }
#pragma unroll
    for (int l = 0; l < LB; ++l) { int o, r; coord(BL::kRedContig, LB, l, o, r); bv[l] = b.load(col0 + o, k0 + r); }
  };
  auto stash = [&](int buf, const float4 (&av)[LA], const float4 (&bv)[LB]) {
#pragma unroll
    for (int l = 0; l < LA; ++l) {
      int o, r; coord(AL::kRedContig, LA, l, o, r);
      if (AL::kRedContig) { As[buf][r + 0][o] = av[l].x; As[buf][r + 1][o] = av[l].y; As[buf][r + 2][o] = av[l].z; As[buf][r + 3][o] = av[l].w; }
      else *reinterpret_cast<float4*>(&As[buf][r][o]) = av[l];
    }
#pragma unroll
    for (int l = 0; l < LB; ++l) {
      int o, r; coord(BL::kRedContig, LB, l, o, r);
      if (BL::kRedContig) { Bs[buf][r + 0][o] = bv[l].x; Bs[buf][r + 1][o] = bv[l].y; Bs[buf][r + 2][o] = bv[l].z; Bs[buf][r + 3][o] = bv[l].w; }
      else *reinterpret_cast<float4*>(&Bs[buf][r][o]) = bv[l];
    }
  };

  int buf = 0;
  {
    float4 av[LA], bv[LB];
    fetch(k_begin, av, bv);
    stash(0, av, bv);
  }
  __syncthreads();
  for (int k0 = k_begin; k0 < k_end; k0 += BK) {
    const bool more = k0 + BK < k_end;
    float4 av[LA], bv[LB];
    if (more) fetch(k0 + BK, av, bv);
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      float af[TM], bf[TN];
#pragma unroll
      for (int l = 0; l < LA; ++l) {
        const float4 t = *reinterpret_cast<const float4*>(&As[buf][kk][(ty << 2) + 64 * l]);
        af[4 * l] = t.x; af[4 * l + 1] = t.y; af[4 * l + 2] = t.z; af[4 * l + 3] = t.w;
      }
#pragma unroll
      for (int l = 0; l < LB; ++l) {
        const float4 t = *reinterpret_cast<const float4*>(&Bs[buf][kk][(tx << 2) + 64 * l]);
        bf[4 * l] = t.x; bf[4 * l + 1] = t.y; bf[4 * l + 2] = t.z; bf[4 * l + 3] = t.w;
      }
#pragma unroll
      for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(af[i], bf[j], acc[i][j]);
    }
    if (more) stash(buf ^ 1, av, bv);
    __syncthreads();
    buf ^= 1;
  }
#pragma unroll
  for (int i = 0; i < TM; ++i) {
    const int row = row0 + (ty << 2) + (i & 3) + 64 * (i >> 2);
    if (row >= M) continue;
#pragma unroll
    for (int j = 0; j < TN; ++j) {
      const int col = col0 + (tx << 2) + (j & 3) + 64 * (j >> 2);
      if (col >= N) continue;
      if (epi.partial) epi.partial[((size_t)blockIdx.z * M + row) * N + col] = acc[i][j];
      else finish(epi, row, col, acc[i][j]);
    }
  }
}

__global__ void splitk_finish_kernel(Epilogue epi, int M, int N, int splits) {
  pdl_launch_dependents();
  pdl_wait();
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)M * N) return;
  const int row = (int)(i / N), col = (int)(i % N);
  // fixed order: four interleaved accumulators (s % 4), combined pairwise; the loads of a group of 8
  // splits are independent and issue together
  float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
  const float* p = epi.partial + (size_t)row * N + col;
  const size_t stride = (size_t)M * N;
  int s = 0;
  for (; s + 8 <= splits; s += 8) {
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = p[(size_t)(s + j) * stride];
    a0 += v[0]; a1 += v[1]; a2 += v[2]; a3 += v[3];
    a0 += v[4]; a1 += v[5]; a2 += v[6]; a3 += v[7];
  }
  for (; s < splits; ++s) {
    const float v = p[(size_t)s * stride];
    switch (s & 3) { case 0: a0 += v; break; case 1: a1 += v; break; case 2: a2 += v; break; default: a3 += v; }
  }
  finish(epi, row, col, (a0 + a1) + (a2 + a3));
}

// out[n] = sum_m x[m, n].  Rows are split over gridDim.y CTAs (each a 32-column x 8-row-lane tile with a
// fixed-order tree), partial sums go to `partial` [gridDim.y][N] and a second pass adds them in
// order: deterministic and parallel over the (long) row dimension.
__global__ void colsum_partial_kernel(int M, int N, const float* __restrict__ x, int ld, int rows_per_block,
                                      float* __restrict__ partial) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ float part[8][33];
  const int col = blockIdx.x * 32 + threadIdx.x;
  const int m0 = blockIdx.y * rows_per_block, m1 = min(M, m0 + rows_per_block);
  float s = 0.f;
  if (col < N)
    for (int m = m0 + threadIdx.y; m < m1; m += 8) s += x[(size_t)m * ld + col];
  part[threadIdx.y][threadIdx.x] = s;
  __syncthreads();
  if (threadIdx.y == 0 && col < N) {
    float t = 0.f;
    for (int r = 0; r < 8; ++r) t += part[r][threadIdx.x];
    partial[(size_t)blockIdx.y * N + col] = t;
  }
}
__global__ void colsum_finish_kernel(int N, int splits, const float* __restrict__ partial, float* __restrict__ out) {
  pdl_launch_dependents();
  pdl_wait();
  const int col = blockIdx.x * blockDim.x + threadIdx.x;
  if (col >= N) return;
  float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
  int s = 0;
  for (; s + 8 <= splits; s += 8) {
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = partial[(size_t)(s + j) * N + col];
    a0 += v[0]; a1 += v[1]; a2 += v[2]; a3 += v[3];
    a0 += v[4]; a1 += v[5]; a2 += v[6]; a3 += v[7];
  }
  for (; s < splits; ++s) {
    const float v = partial[(size_t)s * N + col];
    switch (s & 3) { case 0: a0 += v; break; case 1: a1 += v; break; case 2: a2 += v; break; default: a3 += v; }
  }
  out[col] = (a0 + a1) + (a2 + a3);
}

int launch_splitk_finish(const Epilogue& epi, int M, int N, int splits, cudaStream_t stream) {
  B200RL_CUDA_OK(launch_pdl(splitk_finish_kernel, dim3((int)ceil_div<long long>((long long)M * N, 256)), dim3(256), 0, stream, epi, M, N, splits));
  B200RL_LAUNCH_OK();
  return B200RL_OK;
}

template <class AL, class BL>
static int launch_gemm(const AL& a, const BL& b, Epilogue epi, int M, int N, int K, void* ws, int64_t ws_bytes,
                       cudaStream_t stream) {
  // tile shape: 128 x 128 where that still fills the GPU, 128 x 64 for the narrow (conv) outputs, else 64 x 64
  static const int big_env = getenv("B200RL_SIMT_BIG") ? atoi(getenv("B200RL_SIMT_BIG")) : 1;
  int tm = 4, tn = 4;
  if (big_env && M >= 128 && N >= 128 && ceil_div(M, 128) * ceil_div(N, 128) >= kNumSMs) { tm = 8; tn = 8; }
  else if (big_env && M >= 128 && ceil_div(M, 128) * ceil_div(N, 64) >= kNumSMs) { tm = 8; tn = 4; }
  const int bm = 16 * tm, bn = 16 * tn;
  const int tiles = ceil_div(M, bm) * ceil_div(N, bn);
  int splits = 1;
  if (tiles < 2 * kNumSMs && K >= 4 * BK) {
    splits = ceil_div(2 * kNumSMs, tiles);
    splits = std::min(splits, K / (2 * BK));
    splits = std::min(splits, 64);
    const int64_t cap = ws ? ws_bytes / ((int64_t)M * N * 4) : 0;
    splits = (int)std::min<int64_t>(splits, cap);
    if (splits < 1) splits = 1;
  }
  int k_per_split = ceil_div(ceil_div(K, splits), BK) * BK;
  splits = ceil_div(K, k_per_split);
  dim3 grid(ceil_div(N, bn), ceil_div(M, bm), splits);
  if (splits > 1) epi.partial = (float*)ws; else epi.partial = nullptr;
  if (tm == 8 && tn == 8) B200RL_CUDA_OK(launch_pdl_small(gemm_kernel<AL, BL, 8, 8>, dim3(grid), dim3(GEMM_THREADS), 0, stream, a, b, epi, M, N, K, k_per_split));
  else if (tm == 8) B200RL_CUDA_OK(launch_pdl_small(gemm_kernel<AL, BL, 8, 4>, dim3(grid), dim3(GEMM_THREADS), 0, stream, a, b, epi, M, N, K, k_per_split));
  else B200RL_CUDA_OK(launch_pdl_small(gemm_kernel<AL, BL, 4, 4>, dim3(grid), dim3(GEMM_THREADS), 0, stream, a, b, epi, M, N, K, k_per_split));
  B200RL_LAUNCH_OK();
  if (splits > 1) {
    B200RL_CUDA_OK(launch_pdl(splitk_finish_kernel, dim3((int)ceil_div<long long>((long long)M * N, 256)), dim3(256), 0, stream, epi, M, N, splits));
    B200RL_LAUNCH_OK();
  }
  return B200RL_OK;
}

// Vectorised column sum in ONE launch: a CTA of 256 threads is a (256 / (N/4)) x (N/4) grid of float4 lanes that
// walks its slice of rows with fully coalesced 16-byte loads, reduces its row-lanes in a fixed order through shared
// memory and writes one partial row; the CTA that finishes last (a per-stream ticket in g_tail_tickets, reset on
// the way out, so the kernel is CUDA-graph safe) reduces the partial rows with the same routine.  The order of
// every addition is fixed by indices, never by arrival, so the result is deterministic.
__device__ unsigned int g_tail_tickets[64];

// one 4-column chunk of row m: fp32 (16 bytes) or bf16 (8 bytes, widened)
template <bool BF>
__device__ __forceinline__ float4 load_chunk4(const void* __restrict__ x, size_t m, int ld, int c, bool through_l2) {
  if (BF) {
    const uint2 t = __ldg(reinterpret_cast<const uint2*>(reinterpret_cast<const __nv_bfloat16*>(x) + m * ld) + c);
    const float2 lo = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&t.x));
    const float2 hi = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&t.y));
    return make_float4(lo.x, lo.y, hi.x, hi.y);
  }
  const float4* p = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(x) + m * ld) + c;
  return through_l2 ? __ldcg(p) : __ldg(p);
}

template <bool BF>
__device__ __forceinline__ float4 block_colsum(const void* __restrict__ x, int ld, int m0, int m1, int cpr, float4* red,
                                               bool through_l2) {
  const int rl = threadIdx.x / cpr, c = threadIdx.x % cpr, rpi = 256 / cpr;
  float4 a0 = make_float4(0.f, 0.f, 0.f, 0.f), a1 = a0;
  int m = m0 + rl;
  for (; m + 7 * rpi < m1; m += 8 * rpi) {   // 8 independent 16-byte loads in flight per thread
    float4 v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = load_chunk4<BF>(x, (size_t)(m + j * rpi), ld, c, through_l2);
#pragma unroll
    for (int j = 0; j < 8; j += 2) {
      a0.x += v[j].x; a0.y += v[j].y; a0.z += v[j].z; a0.w += v[j].w;
      a1.x += v[j + 1].x; a1.y += v[j + 1].y; a1.z += v[j + 1].z; a1.w += v[j + 1].w;
    }
  }
  for (; m < m1; m += rpi) {
    const float4 v0 = load_chunk4<BF>(x, (size_t)m, ld, c, through_l2);
    a0.x += v0.x; a0.y += v0.y; a0.z += v0.z; a0.w += v0.w;
  }
  red[threadIdx.x] = make_float4(a0.x + a1.x, a0.y + a1.y, a0.z + a1.z, a0.w + a1.w);
  __syncthreads();
  float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
  if (threadIdx.x < cpr)
    for (int j = 0; j < rpi; ++j) {
      const float4 v = red[j * cpr + threadIdx.x];
      t.x += v.x; t.y += v.y; t.z += v.z; t.w += v.w;
    }
  __syncthreads();
  return t;   // valid in threads < cpr
}

template <bool BF>
__global__ void __launch_bounds__(256)
colsum_vec_kernel(int M, int N, const void* __restrict__ x, int ld, int rows_per_block, float* __restrict__ partial,
                  float* __restrict__ out, int ticket) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ float4 red[256];
  __shared__ bool last;
  const int cpr = N >> 2;
  const int m0 = blockIdx.x * rows_per_block, m1 = min(M, m0 + rows_per_block);
  float4 t = block_colsum<BF>(x, ld, m0, m1, cpr, red, false);
  if (gridDim.x == 1) {
    if (threadIdx.x < cpr) reinterpret_cast<float4*>(out)[threadIdx.x] = t;
    return;
  }
  if (threadIdx.x < cpr) reinterpret_cast<float4*>(partial + (size_t)blockIdx.x * N)[threadIdx.x] = t;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) last = atomicAdd(&g_tail_tickets[ticket], 1u) == gridDim.x - 1;
  __syncthreads();
  if (!last) return;
  __threadfence();
  t = block_colsum<false>(partial, N, 0, (int)gridDim.x, cpr, red, true);
  if (threadIdx.x < cpr) reinterpret_cast<float4*>(out)[threadIdx.x] = t;
  if (threadIdx.x == 0) g_tail_tickets[ticket] = 0;
}

// kernels on one stream never overlap, so a ticket per stream is race-free (also inside a captured graph, whose
// nodes keep the capture-time stream order)
int ticket_for(cudaStream_t s) {
  static std::mutex mu;
  static std::vector<cudaStream_t> seen;
  std::lock_guard<std::mutex> lk(mu);
  for (size_t i = 0; i < seen.size(); ++i) if (seen[i] == s) return (int)i;
  if (seen.size() >= 64) return -1;
  seen.push_back(s);
  return (int)seen.size() - 1;
}

int launch_colsum(int M, int N, const float* x, int ld, float* out, void* ws, int64_t ws_bytes, cudaStream_t stream) {
  const bool vec = N >= 4 && N <= 1024 && (N & (N - 1)) == 0 && ld % 4 == 0 && ((((uintptr_t)x) | ((uintptr_t)out) | ((uintptr_t)ws)) & 15) == 0;
  const int ticket = vec ? ticket_for(stream) : -1;
  if (vec && ticket >= 0) {
    const int rpi = 256 / (N / 4);
    // ~sqrt(M) slices balance the first pass against the last CTA's pass over the partial rows
    int blocks = std::max(1, std::min((int)std::lround(std::sqrt((double)M)), 2 * kNumSMs));
    blocks = (int)std::max<int64_t>(1, std::min<int64_t>(blocks, ws ? ws_bytes / ((int64_t)N * 4) : 1));
    const int rpb = ceil_div(M, blocks);
    blocks = ceil_div(M, rpb);
    B200RL_CUDA_OK(launch_pdl_small(colsum_vec_kernel<false>, dim3(blocks), dim3(256), 0, stream, M, N, x, ld, rpb, (float*)ws, out, ticket));
    B200RL_LAUNCH_OK();
    return B200RL_OK;
  }
  const int col_blocks = ceil_div(N, 32);
  int splits = std::max(1, std::min(std::min(ceil_div(M, 64), (2 * kNumSMs) / col_blocks), 96));
  splits = (int)std::min<int64_t>(splits, ws ? ws_bytes / ((int64_t)N * 4) : 1);
  if (splits <= 1) {
    B200RL_CUDA_OK(launch_pdl_small(colsum_partial_kernel, dim3(dim3(col_blocks, 1)), dim3(dim3(32, 8)), 0, stream, M, N, x, ld, M, out));
    B200RL_LAUNCH_OK();
    return B200RL_OK;
  }
  const int rpb = ceil_div(M, splits);
  splits = ceil_div(M, rpb);
  B200RL_CUDA_OK(launch_pdl_small(colsum_partial_kernel, dim3(dim3(col_blocks, splits)), dim3(dim3(32, 8)), 0, stream, M, N, x, ld, rpb, (float*)ws));
  B200RL_LAUNCH_OK();
  B200RL_CUDA_OK(launch_pdl_small(colsum_finish_kernel, dim3(ceil_div(N, 128)), dim3(128), 0, stream, N, splits, (const float*)ws, out));
  B200RL_LAUNCH_OK();
  return B200RL_OK;
}

// bias gradients of the bf16 dataflow: out[n] = sum_m x[m, n] over bf16 rows, fp32 sums in the fixed order of
// colsum_vec_kernel (one launch; N a power of two in [4, 1024], 8-byte aligned rows)
int launch_colsum_bf16(int M, int N, const __nv_bfloat16* x, int ld, float* out, void* ws, int64_t ws_bytes, cudaStream_t stream) {
  const bool vec = N >= 4 && N <= 1024 && (N & (N - 1)) == 0 && ld % 4 == 0 && (((uintptr_t)x) & 7) == 0 &&
                   ((((uintptr_t)out) | ((uintptr_t)ws)) & 15) == 0;
  const int ticket = vec ? ticket_for(stream) : -1;
  if (!vec || ticket < 0) {
    set_error("bf16 column sum: N = %d must be a power of two in [4, 1024] with aligned rows", N);
    return B200RL_EINVAL;
  }
  int blocks = std::max(1, std::min((int)std::lround(std::sqrt((double)M)), 2 * kNumSMs));
  blocks = (int)std::max<int64_t>(1, std::min<int64_t>(blocks, ws ? ws_bytes / ((int64_t)N * 4) : 1));
  const int rpb = ceil_div(M, blocks);
  blocks = ceil_div(M, rpb);
  B200RL_CUDA_OK(launch_pdl_small(colsum_vec_kernel<true>, dim3(blocks), dim3(256), 0, stream, M, N, x, ld, rpb, (float*)ws, out, ticket));
  B200RL_LAUNCH_OK();
  return B200RL_OK;
}

// ---------------------------------------------------------------- fp32 entry points (precision 0)
int simt_linear_fwd(int M, int N, int K, const float* x, int ldx, const float* w, const float* bias, float* y,
                    int ldy, int act, void* ws, int64_t wsb, cudaStream_t s) {
  DenseRed a{x, ldx, M, K};
  DenseRed b{w, K, N, K};
  Epilogue e{y, ldy, bias, act, nullptr, 0, 0, nullptr, 0};
  return launch_gemm(a, b, e, M, N, K, ws, wsb, s);
}
int simt_linear_dgrad(int M, int N, int K, const float* dy, int lddy, const float* w, float* dx, int lddx,
                      const float* mask, int ldmask, int mask_act, void* ws, int64_t wsb, cudaStream_t s) {
  DenseRed a{dy, lddy, M, N};        // rows m, red n
  DenseOuter b{w, K, K, N};          // (outer = k, red = n) at w[n*K + k]
  Epilogue e{dx, lddx, nullptr, 0, mask, ldmask, mask_act, nullptr, 0};
  return launch_gemm(a, b, e, M, K, N, ws, wsb, s);
}
int simt_linear_wgrad(int M, int N, int K, const float* dy, int lddy, const float* x, int ldx, float* dw, float* db,
                      void* ws, int64_t wsb, cudaStream_t s) {
  DenseOuter a{dy, lddy, N, M};      // (outer = n, red = m) at dy[m*ld + n]
  DenseOuter b{x, ldx, K, M};        // (outer = k, red = m) at x[m*ld + k]
  Epilogue e{dw, K, nullptr, 0, nullptr, 0, 0, nullptr, 0};
  int rc = launch_gemm(a, b, e, N, K, M, ws, wsb, s);
  if (rc) return rc;
  if (db) return launch_colsum(M, N, dy, lddy, db, ws, wsb, s);
  return B200RL_OK;
}
int simt_conv_fwd(const void* x, int x_u8, const float* w, const float* bias, float* y, const b200rl_conv_geom& g,
                  int act, void* ws, int64_t wsb, cudaStream_t s) {
  const int M = g.B * g.OH * g.OW, K = g.kh * g.kw * g.C;
  Im2colRows a; a.x = x; a.u8 = x_u8; a.g = g; a.Mtot = M; a.Ktot = K;
  DenseRed b{w, K, g.Cout, K};
  Epilogue e{y, g.Cout, bias, act, nullptr, 0, 0, nullptr, 0};
  return launch_gemm(a, b, e, M, g.Cout, K, ws, wsb, s);
}
int simt_conv_wgrad(const void* x, int x_u8, const float* dy, float* dw, float* db, const b200rl_conv_geom& g,
                    void* ws, int64_t wsb, cudaStream_t s) {
  const int M = g.B * g.OH * g.OW, K = g.kh * g.kw * g.C;
  DenseOuter a{dy, g.Cout, g.Cout, M};                 // (outer = co, red = m)
  Im2colCols b; b.x = x; b.u8 = x_u8; b.g = g; b.Mtot = M; b.Ktot = K;
  Epilogue e{dw, K, nullptr, 0, nullptr, 0, 0, nullptr, 0};
  int rc = launch_gemm(a, b, e, g.Cout, K, M, ws, wsb, s);
  if (rc) return rc;
  if (db) return launch_colsum(M, g.Cout, dy, g.Cout, db, ws, wsb, s);
  return B200RL_OK;
}
int simt_conv_dgrad(const float* dy, const float* w, float* dx, const b200rl_conv_geom& g, const float* mask,
                    int mask_act, void* ws, int64_t wsb, cudaStream_t s) {
  const int Min = g.B * g.H * g.W, R = g.kh * g.kw * g.Cout;
  static const int phases_env = getenv("B200RL_SIMT_DGRAD_PHASES") ? atoi(getenv("B200RL_SIMT_DGRAD_PHASES")) : 1;
  const int st = g.stride;
  const int64_t map_bytes = ((int64_t)Min * 4 + 255) & ~(int64_t)255;
  if (phases_env && st > 1 && st <= g.kh && st <= g.kw && ws && wsb > map_bytes) {
    int* map = (int*)ws;
    B200RL_CUDA_OK(launch_pdl_small(dgrad_row_map_kernel, dim3(ceil_div(Min, 256)), dim3(256), 0, s, g, map));
    B200RL_LAUNCH_OK();
    auto first = [&](int p, int pad) { return ((p - pad) % st + st) % st; };
    auto count = [&](int p, int pad, int n) { const int f = first(p, pad); return f < n ? (n - f + st - 1) / st : 0; };
    int base = 0;
    for (int py = 0; py < st; ++py)
      for (int px = 0; px < st; ++px) {
        const int Mp = g.B * count(py, g.pad_top, g.H) * count(px, g.pad_left, g.W);
        const int nty = (g.kh - py + st - 1) / st, ntx = (g.kw - px + st - 1) / st;
        const int Rp = nty * ntx * g.Cout;
        if (Mp > 0) {
          DgradPhaseRows a{dy, g, map + base, Mp, Rp, py, px, ntx};
          DgradPhaseWeights b{w, g, Rp, py, px, ntx};
          Epilogue e{dx, g.C, nullptr, 0, mask, g.C, mask_act, nullptr, 0};
          e.row_map = map + base;
          int rc = launch_gemm(a, b, e, Mp, g.C, Rp, (char*)ws + map_bytes, wsb - map_bytes, s);
          if (rc) return rc;
        }
        base += Mp;
      }
    return B200RL_OK;
  }
  DgradRows a{dy, g, Min, R};
  DgradWeights b{w, g, R};
  Epilogue e{dx, g.C, nullptr, 0, mask, g.C, mask_act, nullptr, 0};
  return launch_gemm(a, b, e, Min, g.C, R, ws, wsb, s);
}

}  // namespace b200rl
