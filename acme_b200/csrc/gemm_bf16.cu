// K6, bf16 dataflow: TMA-fed bf16 GEMM / implicit-GEMM convolution on tcgen05 (kind::f16, fp32 accumulation in TMEM).
//
// Why a second tensor-core family next to gemm_tma.cu (tf32): at batch 256 the network's GEMMs are bound by the
// L2 -> shared-memory fill (LTS throughput ~ 6300 B/clk chip-wide), not by the tensor pipe -- a 128 x BN tile of fp32
// operands moves (128 + BN) * 128 B per 32-deep k-block, i.e. 16 / 10.7 / 6.4 MAC per byte for BN = 128 / 64 / 32.
// Activations, weight shadows and back-propagated gradients kept in bf16 halve every one of those bytes (and the HBM
// bytes behind them); master weights, weight gradients, accumulation and the optimizer stay fp32.
//
// One kernel template covers the dense layers and the convolutions' forward and weight gradient:
//   KE      k-elements per pipeline stage: 64 (128-byte rows) or 32 (64-byte rows: layers with 32 input channels, where
//           one filter tap only has 32 contiguous values)
//   AM / BM operand mode: 0 = K-major (reduction index contiguous in memory; rows of KE elements, swizzle = row bytes),
//           1 = MN-major in 64-wide boxes (128-byte rows, SWIZZLE_128B), 2 = MN-major in 32-wide boxes (64-byte rows,
//           SWIZZLE_64B); MN-major boxes hold KE reduction rows each and sit back to back (LBO = box bytes)
// and a second one the convolutions' data gradient (one stride-1 sub-problem per stride phase, as in gemm_tma.cu).
// Roles per CTA (192 threads): warp 0 = TMA producer, warp 1 = MMA issuer (one thread), warps 2-5 = epilogue.
#include <algorithm>
#include <cstdlib>

#include <cuda.h>
#include <cuda_bf16.h>

#include "common.cuh"
#include "gemm_common.cuh"
#include "tc_common.cuh"
#include "tma_common.cuh"

namespace b200rl {

typedef __nv_bfloat16 bf16;
constexpr int HBM_ROWS = 128, H_THREADS = 192;

// tools/h_timeline.py: global-timer stamps of one CTA's life (set-up, first operands, last MMA, epilogue, exit)
__device__ unsigned long long* g_h_timeline = nullptr;
__device__ __forceinline__ void h_mark(int slot, int cta) {
  if (g_h_timeline && (int)(blockIdx.x + blockIdx.y * gridDim.x) == cta && blockIdx.z == 0) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    g_h_timeline[slot] = t;
  }
}

// ---- tensor maps over bf16 tensors
static CUtensorMapSwizzle sw_mode(int row_bytes) { return row_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B; }

// matrix X[lines][pos] (pos contiguous, row stride ld elements); box = box_pos x box_lines, swizzle = box_pos * 2 bytes
static bool make_map_h(CUtensorMap* m, const bf16* p, int64_t lines, int64_t pos, int64_t ld, int box_pos, int box_lines) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return false;
  cuuint64_t dims[2] = {(cuuint64_t)pos, (cuuint64_t)lines};
  cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
  cuuint32_t box[2] = {(cuuint32_t)box_pos, (cuuint32_t)box_lines};
  cuuint32_t es[2] = {1, 1};
  return enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, (void*)p, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
             sw_mode(box_pos * 2), CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
// NHWC bf16 activation tensor through TMA's im2col mode: one instruction = `pixels` consecutive output pixels x `channels`
// input channels of one filter tap (padding reads as zero); swizzle = channels * 2 bytes
static bool make_im2col_map_h(CUtensorMap* m, const bf16* x, const b200rl_conv_geom& g, int channels, int pixels) {
  EncodeIm2colFn enc = get_encode_im2col();
  if (!enc) return false;
  const int pad_bottom = (g.OH - 1) * g.stride + g.kh - g.H - g.pad_top;
  const int pad_right = (g.OW - 1) * g.stride + g.kw - g.W - g.pad_left;
  cuuint64_t dims[4] = {(cuuint64_t)g.C, (cuuint64_t)g.W, (cuuint64_t)g.H, (cuuint64_t)g.B};
  cuuint64_t strides[3] = {(cuuint64_t)g.C * 2, (cuuint64_t)g.W * g.C * 2, (cuuint64_t)g.H * g.W * g.C * 2};
  int lower[2] = {-g.pad_left, -g.pad_top};
  int upper[2] = {pad_right - (g.kw - 1), pad_bottom - (g.kh - 1)};
  cuuint32_t es[4] = {1, (cuuint32_t)g.stride, (cuuint32_t)g.stride, 1};
  return enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, (void*)x, dims, strides, lower, upper, (cuuint32_t)channels,
             (cuuint32_t)pixels, es, CU_TENSOR_MAP_INTERLEAVE_NONE, sw_mode(channels * 2), CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
static bool ok16(const void* p, int64_t ld_elems) { return (((uintptr_t)p) & 15) == 0 && (ld_elems * 2) % 16 == 0; }

// ---- descriptors.  kind::f16 with bf16 operands, fp32 accumulator (same bit layout as gemm_tc.cu)
__host__ __device__ constexpr uint32_t idesc_bf16(int M, int N, bool a_mn, bool b_mn) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((a_mn ? 1u : 0u) << 15) | ((b_mn ? 1u : 0u) << 16) |
         ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
// swizzled shared-memory operand: start address, LBO, SBO (bytes), version 1, layout 2 = SWIZZLE_128B, 4 = SWIZZLE_64B
__device__ __forceinline__ uint64_t sdesc(uint32_t saddr, uint32_t lbo, uint32_t sbo, int row_bytes) {
  const uint64_t layout = row_bytes == 128 ? 2ull : 4ull;
  return (uint64_t)((saddr >> 4) & 0x3FFFu) | ((uint64_t)((lbo >> 4) & 0x3FFFu) << 16) | ((uint64_t)((sbo >> 4) & 0x3FFFu) << 32) |
         (1ull << 46) | (layout << 61);
}
// descriptor of the kk-th 16-deep slice of an operand tile at `base`
template <int MODE, int KE>
__device__ __forceinline__ uint64_t operand_desc(uint32_t base, int kk) {
  if (MODE == 0) {   // K-major: 16 k = 32 bytes inside the swizzled row; 8-row groups 8 * row_bytes apart
    constexpr int RB = KE * 2;
    return sdesc(base + kk * 32, 16, 8 * RB, RB);
  }
  // MN-major: 16 k = 16 rows of RB bytes; the next 8-row group SBO = 8 * RB further; the next MN box LBO = KE * RB further
  constexpr int RB = MODE == 1 ? 128 : 64;
  return sdesc(base + kk * 16 * RB, KE * RB, 8 * RB, RB);
}

template <int KE, int AM, int BM, int BN, int STAGES>
__global__ void __launch_bounds__(H_THREADS)
hgemm_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b, Epilogue epi, int M, int N,
             int K, int kblocks_per_split, ConvA conv) {
  constexpr int A_BYTES = HBM_ROWS * KE * 2, B_BYTES = BN * KE * 2, STAGE = A_BYTES + B_BYTES;
  constexpr int A_WB = AM == 1 ? 64 : 32, B_WB = BM == 1 ? 64 : 32;          // MN-major box widths (elements)
  constexpr int A_BOX = A_WB * KE * 2, B_BOX = B_WB * KE * 2;                 // ... and box bytes
  constexpr int A_NBOX = HBM_ROWS / A_WB, B_NBOX = BN / B_WB;
  constexpr uint32_t TMEM_COLS = BN < 32 ? 32 : BN;
  static_assert(BM == 0 || BN % B_WB == 0, "B tile must be whole MN boxes");
  static_assert(STAGES * STAGE >= HBM_ROWS * BN * 4, "the epilogue slab reuses the drained pipeline stages");
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  __shared__ __align__(8) uint64_t bar_full[STAGES], bar_empty[STAGES], bar_done;
  __shared__ uint32_t tmem_base_smem;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (!epi.pdl_late) pdl_launch_dependents();
  const int row0 = blockIdx.y * HBM_ROWS, col0 = blockIdx.x * BN;
  const int total_kblocks = (K + KE - 1) / KE;
  const int kb_begin = blockIdx.z * kblocks_per_split;
  const int nkb = min(total_kblocks, kb_begin + kblocks_per_split) - kb_begin;

  if (tid == 0) {
    prefetch_tensormap(&map_a);
    prefetch_tensormap(&map_b);
#pragma unroll
    for (int s = 0; s < STAGES; ++s) { mbar_init(&bar_full[s], 1); mbar_init(&bar_empty[s], 1); }
    mbar_init(&bar_done, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) tmem_alloc(&tmem_base_smem, TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  pdl_wait();                  // everything above overlaps the previous kernel's tail (launch_pdl); no-op otherwise
  const uint32_t tmem_d = tmem_base_smem;

  if (warp == 0 && lane == 0) {
    // ---------------- TMA producer (every coordinate advances incrementally: no divisions in the issue loop)
    int ax = 0, ay = 0, an = 0;
    if (conv.enabled) {
      const int ox = row0 % conv.OW, t = row0 / conv.OW;
      ax = ox * conv.stride_w - conv.pad_left;
      ay = (t % conv.OH) * conv.stride_h - conv.pad_top;
      an = t / conv.OH;
    }
    int f_c0 = 0, f_tx = 0, f_ty = 0;          // conv forward: channel block / filter tap of the current k-block
    int w_ox = 0, w_oy = 0, w_n = 0;           // conv weight gradient: first pixel of the current k-block
    int w_c[A_NBOX], w_tx[A_NBOX], w_ty[A_NBOX], w_nblk = 0;
    if (conv.enabled && AM == 0) {
      const int cb = conv.C / KE, tap = kb_begin / cb;
      f_c0 = (kb_begin % cb) * KE; f_tx = tap % conv.kw; f_ty = tap / conv.kw;
    }
    if (conv.enabled && AM != 0) {
      const int p0 = kb_begin * KE, t = p0 / conv.OW;
      w_ox = p0 % conv.OW; w_oy = t % conv.OH; w_n = t / conv.OH;
#pragma unroll
      for (int j = 0; j < A_NBOX; ++j) {
        const int r = row0 + A_WB * j, tap = r / conv.C;
        w_c[j] = r % conv.C; w_tx[j] = tap % conv.kw; w_ty[j] = tap / conv.kw;
        if (tap < conv.taps) w_nblk = j + 1;   // taps ascend with j: boxes past the last tap are skipped (rows never stored)
      }
    }
    for (int i = 0; i < nkb; ++i) {
      const int s = i % STAGES;
      if (i >= STAGES) mbar_wait(&bar_empty[s], ((i / STAGES) - 1) & 1);
      const uint32_t sa = base + s * STAGE, sb = sa + A_BYTES;
      const int k0 = (kb_begin + i) * KE;
      if (AM != 0 && conv.enabled) {
        // conv weight gradient: rows = patch indices (tap, channel), reduction = pixels; box j = A_WB channels of one tap
        // for the KE pixels of this k-block
        const int px = w_ox * conv.stride_w - conv.pad_left, py = w_oy * conv.stride_h - conv.pad_top;
        mbar_expect_tx(&bar_full[s], w_nblk * A_BOX + B_BYTES);
#pragma unroll
        for (int j = 0; j < A_NBOX; ++j)
          if (j < w_nblk)
            tma_load_im2col(sa + j * A_BOX, &map_a, w_c[j], px, py, w_n, (uint16_t)w_tx[j], (uint16_t)w_ty[j], &bar_full[s]);
        w_ox += KE;
        while (w_ox >= conv.OW) {
          w_ox -= conv.OW;
          if (++w_oy == conv.OH) { w_oy = 0; ++w_n; }
        }
      } else {
        mbar_expect_tx(&bar_full[s], STAGE);
        if (AM == 0 && conv.enabled) {   // conv forward: 128 pixels x KE channels of one tap
          tma_load_im2col(sa, &map_a, f_c0, ax, ay, an, (uint16_t)f_tx, (uint16_t)f_ty, &bar_full[s]);
          f_c0 += KE;
          if (f_c0 == conv.C) {
            f_c0 = 0;
            if (++f_tx == conv.kw) { f_tx = 0; ++f_ty; }
          }
        } else if (AM != 0) {
#pragma unroll
          for (int j = 0; j < A_NBOX; ++j) tma_load_2d(sa + j * A_BOX, &map_a, row0 + A_WB * j, k0, &bar_full[s]);
        } else {
          tma_load_2d(sa, &map_a, k0, row0, &bar_full[s]);
        }
      }
      if (BM != 0) {
#pragma unroll
        for (int j = 0; j < B_NBOX; ++j) tma_load_2d(sb + j * B_BOX, &map_b, col0 + B_WB * j, k0, &bar_full[s]);
      } else {
        tma_load_2d(sb, &map_b, k0, col0, &bar_full[s]);
      }
    }
  } else if (warp == 1 && lane == 0) {
    // ---------------- MMA issuer
    constexpr uint32_t idesc = idesc_bf16(HBM_ROWS, BN, AM != 0, BM != 0);
    for (int i = 0; i < nkb; ++i) {
      const int s = i % STAGES;
      mbar_wait(&bar_full[s], (i / STAGES) & 1);
      tc_fence_after();
      const uint32_t sa = base + s * STAGE, sb = sa + A_BYTES;
#pragma unroll
      for (int kk = 0; kk < KE / 16; ++kk)
        umma_bf16(tmem_d, operand_desc<AM, KE>(sa, kk), operand_desc<BM, KE>(sb, kk), idesc, (i > 0 || kk > 0) ? 1u : 0u);
      umma_commit(&bar_empty[s]);
      if (i == nkb - 1) umma_commit(&bar_done);
    }
  } else if (warp >= 2) {
    // ---------------- epilogue: warp w reads TMEM lanes 32 * (w % 4) ..
    const int lane_base = (warp & 3) * 32;
    const int first = row0 + lane_base;
    auto row_of = [&](int r) -> long long { return first + r < M ? first + r : -1; };
    uint2 pm[32 / (32 / (BN / 4))];
    const bool have_pm = !epi.transpose_out && prefetch_relu_mask<BN>(epi, lane, col0, N, row_of, pm);
    if (nkb > 0) {
      mbar_wait(&bar_done, 0);
      tc_fence_after();
    }
    if (epi.pdl_late) pdl_launch_dependents();
    if (epi.transpose_out && !epi.partial) {
      const int row = row0 + lane_base + lane;
#pragma unroll 1
      for (int cc = 0; cc < BN; cc += 16) {
        float v[16];
        if (nkb > 0) tmem_ld16(tmem_d + ((uint32_t)lane_base << 16) + (uint32_t)cc, v);
        else {
#pragma unroll
          for (int j = 0; j < 16; ++j) v[j] = 0.f;
        }
        if (row < M) finish16(epi, row, col0 + cc, N, M, v);
      }
    } else {
      float* slab = reinterpret_cast<float*>(smem_raw + (base - smem_u32(smem_raw))) + (warp & 3) * 32 * BN;
      stage_accumulator<BN>(tmem_d + ((uint32_t)lane_base << 16), slab, lane, nkb > 0);
      store_staged_rows<BN>(epi, slab, lane, col0, N, M, row_of, have_pm ? pm : nullptr);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_d, TMEM_COLS);
}

// ------------------------------------------------------------------------------ persistent variant (A K-major)
// Same tiles, but a CTA walks a static list of them (tile t = blockIdx.x + i * gridDim.x) with TWO accumulators in TMEM:
// the epilogue of tile i (TMEM -> shared-memory slab -> global) overlaps the loads and MMAs of tile i + 1, and barrier
// set-up, TMEM allocation and tensor-map fetch are paid once per CTA instead of once per tile.  For problems of hundreds
// of small tiles (conv1: 1764 tiles of 8 k-blocks; a conv data gradient: 882 tiles of 4) those fixed costs dominate.
// RESB (convolutions: the whole weight matrix is K * BN * 2 <= 72 KB): B is loaded ONCE per CTA and stays in shared
// memory; the ring then carries A only, which cuts the L2 -> shared-memory fill -- the bound of these kernels -- by
// the B share (20-33%).
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

template <int KE, int BM, int BN, int STAGES, bool RESB>
__global__ void __launch_bounds__(H_THREADS)
hgemm_pers_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b, Epilogue epi, int M, int N,
                  int K, int kblocks_per_split, int splits, ConvA conv) {
  constexpr int A_BYTES = HBM_ROWS * KE * 2, B_BYTES = BN * KE * 2, STAGE = RESB ? A_BYTES : A_BYTES + B_BYTES;
  constexpr int B_WB = BM == 1 ? 64 : 32, B_BOX = B_WB * KE * 2, B_NBOX = BN / B_WB;
  constexpr int SLAB = HBM_ROWS * BN * 4;
  constexpr uint32_t TMEM_COLS = 2 * BN < 32 ? 32 : 2 * BN;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;       // [ring stages][epilogue slab][resident B]
  uint8_t* const smem_al = smem_raw + (base - smem_u32(smem_raw));
  __shared__ __align__(8) uint64_t bar_full[STAGES], bar_empty[STAGES], acc_full[2], acc_empty[2], bar_b;
  __shared__ uint32_t tmem_base_smem;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  pdl_launch_dependents();
  const int tiles_m = (M + HBM_ROWS - 1) / HBM_ROWS, tiles_n = (N + BN - 1) / BN, tiles_mn = tiles_m * tiles_n;
  const int total = tiles_mn * splits;
  const int total_kblocks = (K + KE - 1) / KE;
  const uint32_t res_b = base + STAGES * STAGE + SLAB;                 // resident B: total_kblocks tiles of B_BYTES

  if (tid == 0) {
    prefetch_tensormap(&map_a);
    prefetch_tensormap(&map_b);
#pragma unroll
    for (int s = 0; s < STAGES; ++s) { mbar_init(&bar_full[s], 1); mbar_init(&bar_empty[s], 1); }
#pragma unroll
    for (int a = 0; a < 2; ++a) { mbar_init(&acc_full[a], 1); mbar_init(&acc_empty[a], 4); }
    mbar_init(&bar_b, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) tmem_alloc(&tmem_base_smem, TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  pdl_wait();                  // everything above overlaps the previous kernel's tail (launch_pdl); no-op otherwise
  const uint32_t tmem_d = tmem_base_smem;

  if (warp == 0 && lane == 0) {
    // ---------------- TMA producer
    if (RESB) {   // the whole weight matrix, once (conv: splits == 1, tiles_n == 1)
      mbar_expect_tx(&bar_b, (uint32_t)(total_kblocks * B_BYTES));
      for (int kb = 0; kb < total_kblocks; ++kb) tma_load_2d(res_b + kb * B_BYTES, &map_b, kb * KE, 0, &bar_b);
    }
    int it = 0;
    for (int t = blockIdx.x; t < total; t += gridDim.x) {
      const int split = t / tiles_mn, mn = t - split * tiles_mn, m_t = mn / tiles_n, n_t = mn - m_t * tiles_n;
      const int row0 = m_t * HBM_ROWS, col0 = n_t * BN;
      const int kb_begin = split * kblocks_per_split;
      const int nkb = min(total_kblocks, kb_begin + kblocks_per_split) - kb_begin;
      int ax = 0, ay = 0, an = 0, f_c0 = 0, f_tx = 0, f_ty = 0;
      if (conv.enabled) {
        const int ox = row0 % conv.OW, q = row0 / conv.OW;
        ax = ox * conv.stride_w - conv.pad_left;
        ay = (q % conv.OH) * conv.stride_h - conv.pad_top;
        an = q / conv.OH;
        const int cb = conv.C / KE, tap = kb_begin / cb;
        f_c0 = (kb_begin % cb) * KE; f_tx = tap % conv.kw; f_ty = tap / conv.kw;
      }
      for (int i = 0; i < nkb; ++i, ++it) {
        const int s = it % STAGES;
        if (it >= STAGES) mbar_wait(&bar_empty[s], ((it / STAGES) - 1) & 1);
        const uint32_t sa = base + s * STAGE, sb = sa + A_BYTES;
        const int k0 = (kb_begin + i) * KE;
        mbar_expect_tx(&bar_full[s], STAGE);
        if (conv.enabled) {
          tma_load_im2col(sa, &map_a, f_c0, ax, ay, an, (uint16_t)f_tx, (uint16_t)f_ty, &bar_full[s]);
          f_c0 += KE;
          if (f_c0 == conv.C) {
            f_c0 = 0;
            if (++f_tx == conv.kw) { f_tx = 0; ++f_ty; }
          }
        } else {
          tma_load_2d(sa, &map_a, k0, row0, &bar_full[s]);
        }
        if (!RESB) {
          if (BM != 0) {
#pragma unroll
            for (int j = 0; j < B_NBOX; ++j) tma_load_2d(sb + j * B_BOX, &map_b, col0 + B_WB * j, k0, &bar_full[s]);
          } else {
            tma_load_2d(sb, &map_b, k0, col0, &bar_full[s]);
          }
        }
      }
    }
  } else if (warp == 1 && lane == 0) {
    // ---------------- MMA issuer
    constexpr uint32_t idesc = idesc_bf16(HBM_ROWS, BN, false, BM != 0);
    if (RESB) { mbar_wait(&bar_b, 0); tc_fence_after(); }
    int it = 0, ti = 0;
    for (int t = blockIdx.x; t < total; t += gridDim.x, ++ti) {
      const int split = t / tiles_mn;
      const int kb_begin = split * kblocks_per_split;
      const int nkb = min(total_kblocks, kb_begin + kblocks_per_split) - kb_begin;
      const int ab = ti & 1;
      mbar_wait(&acc_empty[ab], ((ti >> 1) & 1) ^ 1);     // the epilogue has drained this accumulator (first use: free)
      tc_fence_after();
      const uint32_t acc = tmem_d + (uint32_t)(ab * BN);
      for (int i = 0; i < nkb; ++i, ++it) {
        const int s = it % STAGES;
        mbar_wait(&bar_full[s], (it / STAGES) & 1);
        tc_fence_after();
        const uint32_t sa = base + s * STAGE;
        const uint32_t sb = RESB ? res_b + (kb_begin + i) * B_BYTES : sa + A_BYTES;
#pragma unroll
        for (int kk = 0; kk < KE / 16; ++kk)
          umma_bf16(acc, operand_desc<0, KE>(sa, kk), operand_desc<BM, KE>(sb, kk), idesc, (i > 0 || kk > 0) ? 1u : 0u);
        umma_commit(&bar_empty[s]);
      }
      umma_commit(&acc_full[ab]);
    }
  } else if (warp >= 2) {
    // ---------------- epilogue: warp w reads TMEM lanes 32 * (w % 4) ..; private slab per warp
    const int lane_base = (warp & 3) * 32;
    float* slab = reinterpret_cast<float*>(smem_al + STAGES * STAGE) + (warp & 3) * 32 * BN;
    int ti = 0;
    for (int t = blockIdx.x; t < total; t += gridDim.x, ++ti) {
      const int split = t / tiles_mn, mn = t - split * tiles_mn, m_t = mn / tiles_n, n_t = mn - m_t * tiles_n;
      const int row0 = m_t * HBM_ROWS, col0 = n_t * BN;
      const int ab = ti & 1;
      mbar_wait(&acc_full[ab], (ti >> 1) & 1);
      tc_fence_after();
      Epilogue e = epi;
      if (e.partial) e.partial += (size_t)split * M * N;       // the helpers add blockIdx.z (= 0 here)
      stage_accumulator<BN>(tmem_d + ((uint32_t)lane_base << 16) + (uint32_t)(ab * BN), slab, lane, true);
      tc_fence_before();
      if (lane == 0) mbar_arrive(&acc_empty[ab]);              // TMEM reads done: the MMA warp may overwrite this accumulator
      const int first = row0 + lane_base;
      store_staged_rows<BN>(e, slab, lane, col0, N, M, [&](int r) -> long long { return first + r < M ? first + r : -1; });
      __syncwarp();
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_d, TMEM_COLS);
}

int g_h_persistent = -1;   // -1 = read B200RL_PERSISTENT once (default on), else 0 / 1

static bool use_persistent() {
  if (g_h_persistent < 0) {
    const char* e = getenv("B200RL_PERSISTENT");
    // Measured on B200 (round 2): correct, but SLOWER inside the learner step (0.331-0.366 vs 0.314 ms).  The step runs the
    // target pass beside the online pass and weight gradients beside data gradients on separate streams; a persistent
    // CTA with resident weights takes 130-190 KB of shared memory, so two such kernels cannot share an SM and the
    // streams serialise, while one-tile CTAs of 40-100 KB interleave.  Off by default; B200RL_PERSISTENT=1 enables it.
    g_h_persistent = e ? atoi(e) : 0;
  }
  return g_h_persistent != 0;
}

template <int KE, int BM, int BN, bool RESB, int STAGES>
static int launch_h_pers_s(const CUtensorMap& ma, const CUtensorMap& mb, const Epilogue& epi, int M, int N, int K, int kps, int splits,
                           int smem, int grid, cudaStream_t stream, const ConvA& conv) {
  static int attr = 0;
  if (attr < smem) {
    B200RL_CUDA_OK(cudaFuncSetAttribute(hgemm_pers_kernel<KE, BM, BN, STAGES, RESB>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    attr = smem;
  }
  B200RL_CUDA_OK(launch_pdl(hgemm_pers_kernel<KE, BM, BN, STAGES, RESB>, dim3(grid), dim3(H_THREADS), smem, stream, ma, mb, epi, M, N, K, kps,
                            splits, conv));
  B200RL_LAUNCH_OK();
  return B200RL_OK;
}

template <int KE, int BM, int BN, bool RESB>
static int launch_h_pers(const CUtensorMap& ma, const CUtensorMap& mb, Epilogue epi, int M, int N, int K, int kps, int splits,
                         int res_b_bytes, cudaStream_t stream, const ConvA& conv) {
  constexpr int STAGE = RESB ? HBM_ROWS * KE * 2 : HBM_ROWS * KE * 2 + BN * KE * 2;
  constexpr int S0 = STAGE >= 24 * 1024 ? 3 : 4;
  const int fixed = HBM_ROWS * BN * 4 + (RESB ? res_b_bytes : 0) + 1024;
  const int total = ceil_div(M, HBM_ROWS) * ceil_div(N, BN) * splits;
  const int tmem_occ = 512 / (2 * BN < 32 ? 32 : 2 * BN);
  auto occ_of = [&](int stages) { return std::max(0, std::min(std::min(4, (227 * 1024) / (stages * STAGE + fixed + 1024)), tmem_occ)); };
  // What hides the L2 latency is the bytes in flight per SM = co-resident CTAs x ring depth x stage size.  Shallow rings
  // with several CTAs per SM when the fixed part (slab + resident weights) is small; one CTA per SM with a deep ring when
  // the resident weights take most of the shared memory (measured: conv2 with a 4 x 8 KB ring and one CTA per SM ran at
  // 26 us against 16 us for three co-resident one-tile CTAs).
  int stages = S0;
  if (occ_of(S0) < 2) {
    for (int cand : {12, 8, 6}) if (cand > S0 && occ_of(cand) >= 1) { stages = cand; break; }
  }
  const int occ = std::max(1, occ_of(stages));
  const int smem = stages * STAGE + fixed;
  const int grid = std::min(total, kNumSMs * occ);
  switch (stages) {
    case 12: return launch_h_pers_s<KE, BM, BN, RESB, 12>(ma, mb, epi, M, N, K, kps, splits, smem, grid, stream, conv);
    case 8: return launch_h_pers_s<KE, BM, BN, RESB, 8>(ma, mb, epi, M, N, K, kps, splits, smem, grid, stream, conv);
    case 6: return launch_h_pers_s<KE, BM, BN, RESB, 6>(ma, mb, epi, M, N, K, kps, splits, smem, grid, stream, conv);
    default: return launch_h_pers_s<KE, BM, BN, RESB, S0>(ma, mb, epi, M, N, K, kps, splits, smem, grid, stream, conv);
  }
}

constexpr int SPLITK_OCC_DEFAULT = 1, SPLITK_MIN_KB_DEFAULT = 8, SPLITK_MAX_DEFAULT = 64;   // round-1/2 values
template <int KE, int AM, int BM, int BN>
static int launch_h(const CUtensorMap& ma, const CUtensorMap& mb, Epilogue epi, int M, int N, int K, void* ws, int64_t ws_bytes,
                    cudaStream_t stream, const ConvA& conv, bool allow_split = true) {
  constexpr int STAGE = HBM_ROWS * KE * 2 + BN * KE * 2;
  constexpr int STAGES = (STAGE * 3 >= HBM_ROWS * BN * 4 && STAGE >= 24 * 1024) ? 3 : (STAGE * 4 >= HBM_ROWS * BN * 4 ? 4 : 6);
  const int tiles = ceil_div(M, HBM_ROWS) * ceil_div(N, BN);
  const int kblocks = ceil_div(K, KE);
  int splits = 1;
  // split-K fills the GPU when a layer has few output tiles (conv weight gradients: 2-5 tiles over a 30-113 K pixel
  // reduction; fc1 forward: 32 tiles over K = 7744).  A CTA's k-blocks are a serial chain of ~0.5 us ring round trips, so
  // the chain length, not the byte count, sets the kernel's duration: B200RL_SPLITK_OCC CTAs per SM (default below),
  // at least B200RL_SPLITK_MIN_KB k-blocks per split, at most B200RL_SPLITK_MAX splits.
  static const int sk_occ = getenv("B200RL_SPLITK_OCC") ? atoi(getenv("B200RL_SPLITK_OCC")) : SPLITK_OCC_DEFAULT;
  static const int sk_min = getenv("B200RL_SPLITK_MIN_KB") ? atoi(getenv("B200RL_SPLITK_MIN_KB")) : SPLITK_MIN_KB_DEFAULT;
  static const int sk_max = getenv("B200RL_SPLITK_MAX") ? atoi(getenv("B200RL_SPLITK_MAX")) : SPLITK_MAX_DEFAULT;
  if (allow_split && 2 * tiles <= kNumSMs && kblocks >= 16) {
    splits = std::min(ceil_div(sk_occ * kNumSMs, tiles), kblocks / sk_min);
    splits = std::max(1, std::min(splits, sk_max));
    const int64_t cap = ws ? ws_bytes / ((int64_t)M * N * 4) : 0;
    splits = (int)std::max<int64_t>(1, std::min<int64_t>(splits, cap));
  }
  const int kps = ceil_div(kblocks, splits);
  splits = ceil_div(kblocks, kps);
  epi.partial = splits > 1 ? (float*)ws : nullptr;
  {
    // The one case where the persistent kernel wins inside the step (measured): a convolution with SMALL resident
    // weights and thousands of tiles -- conv1: 16 KB of weights, 1764 / 882 tiles of 8 k-blocks; its persistent CTAs
    // need ~65 KB of shared memory, three fit on an SM and still leave room for the other streams' kernels
    // (target-pass conv1: 15-16 us against 26-28 us).  B200RL_PERSISTENT_SMALL=0 switches it off.
    static const int small_on = getenv("B200RL_PERSISTENT_SMALL") ? atoi(getenv("B200RL_PERSISTENT_SMALL")) : 1;
    const int res_b = ceil_div(K, KE) * BN * KE * 2;
    if (AM == 0 && BM == 0 && small_on && conv.enabled && splits == 1 && ceil_div(N, BN) == 1 && !epi.transpose_out &&
        tiles >= 4 * kNumSMs && 4 * HBM_ROWS * KE * 2 + HBM_ROWS * BN * 4 + res_b <= 72 * 1024)
      return launch_h_pers<KE, BM, BN, true>(ma, mb, epi, M, N, K, kps, splits, res_b, stream, conv);
  }
  if (AM == 0 && use_persistent() && !epi.transpose_out && tiles * splits >= 3 * kNumSMs / 2) {
    // many small tiles: walk them with persistent CTAs; convolution weights (<= 80 KB) stay resident in shared memory
    const int res_b = ceil_div(K, KE) * BN * KE * 2;
    int rc;
    if (BM == 0 && conv.enabled && splits == 1 && ceil_div(N, BN) == 1 && res_b <= 80 * 1024)
      rc = launch_h_pers<KE, BM, BN, true>(ma, mb, epi, M, N, K, kps, splits, res_b, stream, conv);
    else
      rc = launch_h_pers<KE, BM, BN, false>(ma, mb, epi, M, N, K, kps, splits, 0, stream, conv);
    if (rc) return rc;
    if (splits > 1) return launch_splitk_finish(epi, M, N, splits, stream);
    return B200RL_OK;
  }
  dim3 grid(ceil_div(N, BN), ceil_div(M, HBM_ROWS), splits);
  constexpr int smem = STAGES * STAGE + 1024;
  static bool attr = false;
  if (!attr) {
    B200RL_CUDA_OK(cudaFuncSetAttribute(hgemm_kernel<KE, AM, BM, BN, STAGES>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    attr = true;
  }
  epi.pdl_late = pdl_late_mode();
  B200RL_CUDA_OK(launch_pdl(hgemm_kernel<KE, AM, BM, BN, STAGES>, grid, dim3(H_THREADS), smem, stream, ma, mb, epi, M, N, K, kps, conv));
  B200RL_LAUNCH_OK();
  if (splits > 1) return launch_splitk_finish(epi, M, N, splits, stream);
  return B200RL_OK;
}
static const ConvA kNoConv{0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
static int bn_for(int N) { return N <= 32 ? 32 : (N <= 64 ? 64 : 128); }

static Epilogue make_epi(void* out, int ldo, const float* bias, int act, const void* mask, int ldmask, int mask_act,
                         int transpose, int out_bf16, int mask_bf16, float scale) {
  Epilogue e{(float*)out, ldo, bias, act, (const float*)mask, ldmask, mask_act, nullptr, transpose, out_bf16, mask_bf16, scale};
  return e;
}

// ---- dense layers.  Return 1 when the shapes break TMA's rules (the caller reports it: there is no bf16 fallback).
int h_linear_fwd(int M, int N, int K, const bf16* x, int ldx, const bf16* w, const float* bias, void* y, int ldy, int act,
                 int out_bf16, void* ws, int64_t wsb, cudaStream_t s) {
  if (!ok16(x, ldx) || !ok16(w, K) || K < 64) return 1;
  const int BN = bn_for(N);
  CUtensorMap ma, mb;
  if (!make_map_h(&ma, x, M, K, ldx, 64, HBM_ROWS) || !make_map_h(&mb, w, N, K, K, 64, BN)) return 1;
  Epilogue e = make_epi(y, ldy, bias, act, nullptr, 0, 0, 0, out_bf16, 0, 0.f);
  if (BN == 32) return launch_h<64, 0, 0, 32>(ma, mb, e, M, N, K, ws, wsb, s, kNoConv);
  if (BN == 64) return launch_h<64, 0, 0, 64>(ma, mb, e, M, N, K, ws, wsb, s, kNoConv);
  return launch_h<64, 0, 0, 128>(ma, mb, e, M, N, K, ws, wsb, s, kNoConv);
}
int h_linear_dgrad(int M, int N, int K, const bf16* dy, int lddy, const bf16* w, void* dx, int lddx, const void* mask,
                   int ldmask, int mask_act, int out_bf16, int mask_bf16, void* ws, int64_t wsb, cudaStream_t s) {
  // dx[m, k] = sum_n dy[m, n] w[n, k]: A = dy K-major (reduction n contiguous), B = w MN-major (line = n, pos = k)
  if (!ok16(dy, lddy) || !ok16(w, K) || N < 64 || K % 64 != 0) return 1;
  int BN = K >= 128 ? 128 : 64;
  if (BN == 128 && ceil_div(M, HBM_ROWS) * ceil_div(K, 128) < kNumSMs) BN = 64;   // more, smaller tiles: no split-K here
  CUtensorMap ma, mb;
  if (!make_map_h(&ma, dy, M, N, lddy, 64, HBM_ROWS) || !make_map_h(&mb, w, N, K, K, 64, 64)) return 1;
  Epilogue e = make_epi(dx, lddx, nullptr, 0, mask, ldmask, mask_act, 0, out_bf16, mask_bf16, 0.f);
  // no split-K for a data gradient: its finish pass would re-read the whole output
  return BN == 64 ? launch_h<64, 0, 1, 64>(ma, mb, e, M, K, N, ws, wsb, s, kNoConv, false)
                  : launch_h<64, 0, 1, 128>(ma, mb, e, M, K, N, ws, wsb, s, kNoConv, false);
}
int launch_colsum_bf16(int M, int N, const bf16* x, int ld, float* out, void* ws, int64_t ws_bytes, cudaStream_t stream);

int h_linear_wgrad(int M, int N, int K, const bf16* dy, int lddy, const bf16* x, int ldx, float* dw, float* db, void* ws,
                   int64_t wsb, cudaStream_t s) {
  // dw[n, k] = sum_m dy[m, n] x[m, k]: both operands MN-major (line = reduction m)
  if (!ok16(dy, lddy) || !ok16(x, ldx) || N % 64 != 0 || K % 64 != 0) return 1;
  const int BN = K >= 128 ? 128 : 64;
  CUtensorMap ma, mb;
  if (!make_map_h(&ma, dy, M, N, lddy, 64, 64) || !make_map_h(&mb, x, M, K, ldx, 64, 64)) return 1;
  Epilogue e = make_epi(dw, K, nullptr, 0, nullptr, 0, 0, 0, 0, 0, 0.f);
  int rc = BN == 64 ? launch_h<64, 1, 1, 64>(ma, mb, e, N, K, M, ws, wsb, s, kNoConv)
                    : launch_h<64, 1, 1, 128>(ma, mb, e, N, K, M, ws, wsb, s, kNoConv);
  if (rc) return rc;
  if (db) return launch_colsum_bf16(M, N, dy, lddy, db, ws, wsb, s);
  return B200RL_OK;
}

// ---- convolutions on bf16 NHWC activations with C in {32, 64, 128...}: forward and weight gradient
int h_conv_fwd(const bf16* x, const bf16* w, const float* bias, void* y, const b200rl_conv_geom& g, int act, int out_bf16,
               void* ws, int64_t wsb, cudaStream_t s) {
  const int M = g.B * g.OH * g.OW, K = g.kh * g.kw * g.C;
  if ((g.C != 32 && g.C % 64 != 0) || !ok16(x, g.C) || !ok16(w, K) || (g.Cout != 32 && g.Cout != 64 && g.Cout != 128)) return 1;
  const int KE = g.C == 32 ? 32 : 64;
  CUtensorMap ma, mb;
  if (!make_im2col_map_h(&ma, x, g, KE, HBM_ROWS) || !make_map_h(&mb, w, g.Cout, K, K, KE, g.Cout)) return 1;
  Epilogue e = make_epi(y, g.Cout, bias, act, nullptr, 0, 0, 0, out_bf16, 0, 0.f);
  ConvA conv{1, g.C, g.kw, g.OW, g.OH, g.stride, g.stride, g.pad_left, g.pad_top, g.kh * g.kw};
  if (KE == 32) {
    if (g.Cout == 32) return launch_h<32, 0, 0, 32>(ma, mb, e, M, g.Cout, K, ws, wsb, s, conv);
    if (g.Cout == 64) return launch_h<32, 0, 0, 64>(ma, mb, e, M, g.Cout, K, ws, wsb, s, conv);
    return launch_h<32, 0, 0, 128>(ma, mb, e, M, g.Cout, K, ws, wsb, s, conv);
  }
  if (g.Cout == 32) return launch_h<64, 0, 0, 32>(ma, mb, e, M, g.Cout, K, ws, wsb, s, conv);
  if (g.Cout == 64) return launch_h<64, 0, 0, 64>(ma, mb, e, M, g.Cout, K, ws, wsb, s, conv);
  return launch_h<64, 0, 0, 128>(ma, mb, e, M, g.Cout, K, ws, wsb, s, conv);
}
// dW^T[(tap, ci), co] = sum_pixel col[pixel, (tap, ci)] dy[pixel, co], stored transposed as dw[co][(tap, ci)] (fp32)
int h_conv_wgrad(const bf16* x, const bf16* dy, float* dw, float* db, const b200rl_conv_geom& g, void* ws, int64_t wsb,
                 cudaStream_t s) {
  const int M = g.B * g.OH * g.OW, K = g.kh * g.kw * g.C;
  if ((g.C != 32 && g.C % 64 != 0) || (g.Cout != 32 && g.Cout != 64) || !ok16(x, g.C) || !ok16(dy, g.Cout)) return 1;
  const int WB = g.C == 32 ? 32 : 64, WBb = g.Cout == 32 ? 32 : 64;
  CUtensorMap ma, mb;
  if (!make_im2col_map_h(&ma, x, g, WB, 64) || !make_map_h(&mb, dy, M, g.Cout, g.Cout, WBb, 64)) return 1;
  Epilogue e = make_epi(dw, K, nullptr, 0, nullptr, 0, 0, 1, 0, 0, 0.f);
  ConvA conv{1, g.C, g.kw, g.OW, g.OH, g.stride, g.stride, g.pad_left, g.pad_top, g.kh * g.kw};
  int rc;
  if (WB == 64 && WBb == 64) rc = launch_h<64, 1, 1, 64>(ma, mb, e, K, g.Cout, M, ws, wsb, s, conv);
  else if (WB == 32 && WBb == 64) rc = launch_h<64, 2, 1, 64>(ma, mb, e, K, g.Cout, M, ws, wsb, s, conv);
  else if (WB == 32 && WBb == 32) rc = launch_h<64, 2, 2, 32>(ma, mb, e, K, g.Cout, M, ws, wsb, s, conv);
  else rc = launch_h<64, 1, 2, 32>(ma, mb, e, K, g.Cout, M, ws, wsb, s, conv);
  if (rc) return rc;
  if (db) return launch_colsum_bf16(M, g.Cout, dy, g.Cout, db, ws, wsb, s);
  return B200RL_OK;
}

// ---- first layer on uint8 frames.  The frames are rewritten once per batch as a zero-padded bf16
// ROW IMAGE holding the INTEGER pixel values 0..255 (exact in bf16); the 1/255 of `atari_wrapper.py:303-304` is applied to
// the fp32 accumulator in the epilogue, so the pixel operand carries no rounding at all.  A filter row (kw * Cp values)
// is contiguous in the padded NHWC row: the convolution is a kh x 1 filter over overlapping kw * Cp-channel "wide
// pixels" (tensor-map stride stride * Cp elements < extent), loaded by TMA's im2col mode in 32- or 64-channel blocks.
// Frames of C channels (1 <= C <= 16) get Cp = rows_cp(C) in {4, 8, 16} channels per pixel, channels C .. Cp-1 zero,
// so that a filter row is 32, 64 or 128 values (one 32-channel block, or one / two 64-channel blocks) at kw = 8; the
// filter is [Cout][kh][kw][Cp].  Atari frames (C = 4) take the original 32-channel kernels unchanged.
struct RowsView { int Cp, Hp, row_elems, wide_stride, wide; int64_t bytes; };
int rows_cp(int C) { return C <= 4 ? 4 : (C <= 8 ? 8 : 16); }
static bool rows_eligible(const b200rl_conv_geom& g) {
  if (g.C < 1 || g.C > 16) return false;
  const int cp = rows_cp(g.C), wide = g.kw * cp;
  return (wide == 32 || wide == 64 || wide == 128) && (g.Cout == 32 || g.Cout == 64) && (g.stride * cp * 2) % 16 == 0;
}
static RowsView rows_view(const b200rl_conv_geom& g) {
  RowsView v;
  v.Cp = rows_cp(g.C);
  const int pad_bottom = std::max((g.OH - 1) * g.stride + g.kh - g.H - g.pad_top, 0);
  const int pad_right = std::max((g.OW - 1) * g.stride + g.kw - g.W - g.pad_left, 0);
  v.Hp = g.H + g.pad_top + pad_bottom;
  v.row_elems = (g.W + g.pad_left + pad_right) * v.Cp;
  v.row_elems = (v.row_elems + 7) & ~7;          // 16-byte rows
  v.wide_stride = g.stride * v.Cp;
  v.wide = g.kw * v.Cp;
  v.bytes = (int64_t)g.B * v.Hp * v.row_elems * 2;
  return v;
}
int64_t h_rows_bytes(const b200rl_conv_geom& g) { return rows_eligible(g) ? rows_view(g).bytes : 0; }
// layout of the row image for replay.cu's gather (which writes it directly): padded rows per frame, bf16 elements per row
int h_rows_layout(const b200rl_conv_geom& g, int* Hp, int* row_elems) {
  if (!rows_eligible(g)) return 1;
  const RowsView v = rows_view(g);
  *Hp = v.Hp;
  *row_elems = v.row_elems;
  return 0;
}

__global__ void __launch_bounds__(256)
u8_rows_to_bf16_kernel(const uint8_t* __restrict__ x, bf16* __restrict__ out, int H, int W, int Hp, int per_row /* pixels */,
                       int pad_left, int pad_top, int total_rows, int rows_per_cta) {
  // a CTA converts rows_per_cta consecutive padded rows (b, hp); one thread = 2 pixels = 8 channels = one 16-byte store
  const int row0 = blockIdx.x * rows_per_cta;
  const int nrows = min(rows_per_cta, total_rows - row0);
  const int pairs = per_row >> 1;
  for (int e = threadIdx.x; e < nrows * pairs; e += blockDim.x) {
    const int r = e / pairs, q = e - r * pairs;
    const int row = row0 + r, b = row / Hp, hp = row - b * Hp, ys = hp - pad_top;
    uint32_t w[4] = {0u, 0u, 0u, 0u};
    if (ys >= 0 && ys < H) {
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int xs = 2 * q + h - pad_left;
        if (xs >= 0 && xs < W) {
          const uchar4 p = __ldg(reinterpret_cast<const uchar4*>(x) + ((size_t)b * H + ys) * W + xs);
          const __nv_bfloat162 lo = __floats2bfloat162_rn((float)p.x, (float)p.y), hi = __floats2bfloat162_rn((float)p.z, (float)p.w);
          w[2 * h] = *reinterpret_cast<const uint32_t*>(&lo);
          w[2 * h + 1] = *reinterpret_cast<const uint32_t*>(&hi);
        }
      }
    }
    reinterpret_cast<uint4*>(out)[(size_t)row * (per_row >> 1) + q] = make_uint4(w[0], w[1], w[2], w[3]);
  }
}
// any C (1..16) into Cp-channel pixels: one thread = 8 consecutive elements of a padded row = one 16-byte store
__global__ void __launch_bounds__(256)
u8_rows_to_bf16_c_kernel(const uint8_t* __restrict__ x, uint4* __restrict__ out, int H, int W, int C, int Cp, int Hp,
                         int row_v16, int pad_left, int pad_top, int64_t total) {
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t row = e / row_v16;
    const int q = (int)(e - row * row_v16);
    const int b = (int)(row / Hp), ys = (int)(row - (int64_t)b * Hp) - pad_top;
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int el = 8 * q + j, px = el / Cp, c = el - px * Cp, xs = px - pad_left;
      v[j] = (ys >= 0 && ys < H && xs >= 0 && xs < W && c < C) ? (float)__ldg(x + (((size_t)b * H + ys) * W + xs) * C + c) : 0.f;
    }
    uint32_t w[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const __nv_bfloat162 t = __floats2bfloat162_rn(v[2 * j], v[2 * j + 1]);
      w[j] = *reinterpret_cast<const uint32_t*>(&t);
    }
    out[e] = make_uint4(w[0], w[1], w[2], w[3]);
  }
}
// the row image of B frames of g.C channels (no size / alignment checks: callers check them)
int h_rows_write(const uint8_t* x, const b200rl_conv_geom& g, bf16* rows, cudaStream_t s) {
  if (!rows_eligible(g)) return 1;
  const RowsView v = rows_view(g);
  if (g.C == 4) {
    const int total = g.B * v.Hp, rpc = 8;
    u8_rows_to_bf16_kernel<<<ceil_div(total, rpc), 256, 0, s>>>(x, rows, g.H, g.W, v.Hp, v.row_elems / g.C, g.pad_left, g.pad_top,
                                                                total, rpc);
  } else {
    const int64_t total = (int64_t)g.B * v.Hp * (v.row_elems / 8);
    const int blocks = (int)std::min<int64_t>(ceil_div<int64_t>(total, 256), 148 * 16);
    u8_rows_to_bf16_c_kernel<<<blocks, 256, 0, s>>>(x, (uint4*)rows, g.H, g.W, g.C, v.Cp, v.Hp, v.row_elems / 8, g.pad_left,
                                                   g.pad_top, total);
  }
  B200RL_LAUNCH_OK();
  return B200RL_OK;
}
int h_rows_from_u8(const uint8_t* x, const b200rl_conv_geom& g, bf16* rows, int64_t bytes, cudaStream_t s) {
  if (!rows_eligible(g) || !rows || (((uintptr_t)rows) & 127) != 0) return 1;
  if (rows_view(g).bytes > bytes) return 1;
  return h_rows_write(x, g, rows, s);
}
static bool make_rows_map(CUtensorMap* m, const bf16* rows, const b200rl_conv_geom& g, const RowsView& v, int channels,
                          int pixels) {
  EncodeIm2colFn enc = get_encode_im2col();
  if (!enc) return false;
  cuuint64_t dims[4] = {(cuuint64_t)v.wide, (cuuint64_t)g.OW, (cuuint64_t)v.Hp, (cuuint64_t)g.B};
  cuuint64_t strides[3] = {(cuuint64_t)v.wide_stride * 2, (cuuint64_t)v.row_elems * 2, (cuuint64_t)v.Hp * v.row_elems * 2};
  int lower[2] = {0, 0};
  int upper[2] = {0, -(g.kh - 1)};
  cuuint32_t es[4] = {1, 1, (cuuint32_t)g.stride, 1};
  return enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, (void*)rows, dims, strides, lower, upper, (cuuint32_t)channels,
             (cuuint32_t)pixels, es, CU_TENSOR_MAP_INTERLEAVE_NONE, sw_mode(channels * 2), CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
static int conv_fwd_rows(const bf16* rows, const bf16* w, const float* bias, void* y, const b200rl_conv_geom& g, int act,
                         int out_bf16, float scale, void* ws, int64_t wsb, cudaStream_t s) {
  if (!rows_eligible(g)) return 1;
  const RowsView v = rows_view(g);
  const int M = g.B * g.OH * g.OW, K = g.kh * v.wide, KE = v.wide == 32 ? 32 : 64;
  if (!ok16(w, K)) return 1;
  CUtensorMap ma, mb;
  if (!make_rows_map(&ma, rows, g, v, KE, HBM_ROWS) || !make_map_h(&mb, w, g.Cout, K, K, KE, g.Cout)) return 1;
  Epilogue e = make_epi(y, g.Cout, bias, act, nullptr, 0, 0, 0, out_bf16, 0, scale);
  ConvA conv{1, v.wide, 1, g.OW, g.OH, 1, g.stride, 0, 0, g.kh};
  if (KE == 32) {
    if (g.Cout == 32) return launch_h<32, 0, 0, 32>(ma, mb, e, M, g.Cout, K, ws, wsb, s, conv);
    return launch_h<32, 0, 0, 64>(ma, mb, e, M, g.Cout, K, ws, wsb, s, conv);
  }
  if (g.Cout == 32) return launch_h<64, 0, 0, 32>(ma, mb, e, M, g.Cout, K, ws, wsb, s, conv);
  return launch_h<64, 0, 0, 64>(ma, mb, e, M, g.Cout, K, ws, wsb, s, conv);
}
int h_conv_fwd_rows(const bf16* rows, const bf16* w, const float* bias, void* y, const b200rl_conv_geom& g, int act, int out_bf16,
                    void* ws, int64_t wsb, cudaStream_t s) {
  return conv_fwd_rows(rows, w, bias, y, g, act, out_bf16, 1.0f / 255.0f, ws, wsb, s);
}
// the raw fp32 accumulator (no bias, no activation, no 1/255): one product of a split filter, summed by fp32x3.cu's combine
int h_conv_fwd_rows_raw(const bf16* rows, const bf16* w, float* y, const b200rl_conv_geom& g, void* ws, int64_t wsb, cudaStream_t s) {
  return conv_fwd_rows(rows, w, nullptr, y, g, B200RL_ACT_NONE, 0, 1.0f, ws, wsb, s);
}
int h_conv_wgrad_rows(const bf16* rows, const bf16* dy, float* dw, float* db, const b200rl_conv_geom& g, void* ws, int64_t wsb,
                      cudaStream_t s) {
  if (!rows_eligible(g) || !ok16(dy, g.Cout)) return 1;
  const RowsView v = rows_view(g);
  const int M = g.B * g.OH * g.OW, K = g.kh * v.wide, WB = v.wide == 32 ? 32 : 64;
  CUtensorMap ma, mb;
  const int WBb = g.Cout == 32 ? 32 : 64;
  if (!make_rows_map(&ma, rows, g, v, WB, 64) || !make_map_h(&mb, dy, M, g.Cout, g.Cout, WBb, 64)) return 1;
  Epilogue e = make_epi(dw, K, nullptr, 0, nullptr, 0, 0, 1, 0, 0, 1.0f / 255.0f);
  ConvA conv{1, v.wide, 1, g.OW, g.OH, 1, g.stride, 0, 0, g.kh};
  int rc;
  if (WB == 32) rc = WBb == 32 ? launch_h<64, 2, 2, 32>(ma, mb, e, K, g.Cout, M, ws, wsb, s, conv)
                               : launch_h<64, 2, 1, 64>(ma, mb, e, K, g.Cout, M, ws, wsb, s, conv);
  else rc = WBb == 32 ? launch_h<64, 1, 2, 32>(ma, mb, e, K, g.Cout, M, ws, wsb, s, conv)
                      : launch_h<64, 1, 1, 64>(ma, mb, e, K, g.Cout, M, ws, wsb, s, conv);
  if (rc) return rc;
  if (db) return launch_colsum_bf16(M, g.Cout, dy, g.Cout, db, ws, wsb, s);
  return B200RL_OK;
}

// ---- conv data gradient: one stride-1 sub-problem per stride phase (derivation in gemm_tma.cu).  A = TMA im2col over
// dy (K-major, 64 output channels per k-block), B = boxes of the untransposed weight matrix [Cout][kh kw C] (MN-major,
// BN = C columns wide), accumulator rows scattered to the phase's pixels of dx with the producer's ReLU derivative.
struct HDgradPhase { int tile_begin, cnt_x, cnt_y, lower_x, lower_y, Tx, Ty, px, py, ix0, iy0; };
struct HDgradParams { HDgradPhase ph[4]; int nphase, stride, kw, C, Cout, W, H, B; };
struct HDgradMaps { CUtensorMap m[4]; };
constexpr int D_STAGES = 3;

template <int BN>
__global__ void __launch_bounds__(H_THREADS)
hconv_dgrad_kernel(const __grid_constant__ HDgradMaps maps, const __grid_constant__ CUtensorMap map_w, HDgradParams P, Epilogue epi) {
  constexpr int KE = 64, BM = BN == 32 ? 2 : 1;
  constexpr int A_BYTES = HBM_ROWS * KE * 2, B_BYTES = BN * KE * 2, STAGE = A_BYTES + B_BYTES;
  constexpr int B_WB = BN == 32 ? 32 : 64, B_BOX = B_WB * KE * 2, B_NBOX = BN / B_WB;
  constexpr uint32_t TMEM_COLS = BN < 32 ? 32 : BN;
  static_assert(D_STAGES * STAGE >= HBM_ROWS * BN * 4, "epilogue slab");
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  __shared__ __align__(8) uint64_t bar_full[D_STAGES], bar_empty[D_STAGES], bar_done;
  __shared__ uint32_t tmem_base_smem;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (!epi.pdl_late) pdl_launch_dependents();

  int phase = 0;
#pragma unroll
  for (int i = 1; i < 4; ++i) if (i < P.nphase && (int)blockIdx.x >= P.ph[i].tile_begin) phase = i;
  const HDgradPhase ph = P.ph[phase];
  const int row0 = ((int)blockIdx.x - ph.tile_begin) * HBM_ROWS;
  const int Mp = P.B * ph.cnt_y * ph.cnt_x;
  const int cb = P.Cout / KE;
  const int nkb = ph.Ty * ph.Tx * cb;
  const int mark_cta = gridDim.x / 2;
  if (tid == 0) h_mark(0, mark_cta);

  if (tid == 0) {
    prefetch_tensormap(&maps.m[phase]);
    prefetch_tensormap(&map_w);
#pragma unroll
    for (int s = 0; s < D_STAGES; ++s) { mbar_init(&bar_full[s], 1); mbar_init(&bar_empty[s], 1); }
    mbar_init(&bar_done, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) tmem_alloc(&tmem_base_smem, TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  pdl_wait();                  // everything above overlaps the previous kernel's tail (launch_pdl); no-op otherwise
  const uint32_t tmem_d = tmem_base_smem;
  if (tid == 0) h_mark(1, mark_cta);

  if (warp == 0 && lane == 0) {
    const int jx = row0 % ph.cnt_x, t = row0 / ph.cnt_x;
    const int ax = ph.lower_x + jx, ay = ph.lower_y + t % ph.cnt_y, an = t / ph.cnt_y;
    const int K = P.kw * P.C;
    int co0 = 0, off_x = 0, off_y = 0;
    for (int i = 0; i < nkb; ++i) {
      const int s = i % D_STAGES;
      if (i >= D_STAGES) mbar_wait(&bar_empty[s], ((i / D_STAGES) - 1) & 1);
      const uint32_t sa = base + s * STAGE, sb = sa + A_BYTES;
      const int ky = ph.py + P.stride * (ph.Ty - 1 - off_y), kx = ph.px + P.stride * (ph.Tx - 1 - off_x);
      mbar_expect_tx(&bar_full[s], STAGE);
      tma_load_im2col(sa, &maps.m[phase], co0, ax, ay, an, (uint16_t)off_x, (uint16_t)off_y, &bar_full[s]);
#pragma unroll
      for (int j = 0; j < B_NBOX; ++j) tma_load_2d(sb + j * B_BOX, &map_w, ky * K + kx * P.C + B_WB * j, co0, &bar_full[s]);
      co0 += KE;
      if (co0 == P.Cout) {
        co0 = 0;
        if (++off_x == ph.Tx) { off_x = 0; ++off_y; }
      }
    }
  } else if (warp == 1 && lane == 0) {
    constexpr uint32_t idesc = idesc_bf16(HBM_ROWS, BN, false, true);
    for (int i = 0; i < nkb; ++i) {
      const int s = i % D_STAGES;
      mbar_wait(&bar_full[s], (i / D_STAGES) & 1);
      if (i == 0) h_mark(2, mark_cta);
      if (i == nkb - 1) h_mark(3, mark_cta);
      tc_fence_after();
      const uint32_t sa = base + s * STAGE, sb = sa + A_BYTES;
#pragma unroll
      for (int kk = 0; kk < KE / 16; ++kk)
        umma_bf16(tmem_d, operand_desc<0, KE>(sa, kk), operand_desc<BM, KE>(sb, kk), idesc, (i > 0 || kk > 0) ? 1u : 0u);
      umma_commit(&bar_empty[s]);
      if (i == nkb - 1) umma_commit(&bar_done);
    }
  } else if (warp >= 2) {
    const int lane_base = (warp & 3) * 32;
    const int row = row0 + lane_base + lane;
    long long orow = -1;
    if (row < Mp) {
      const int jx = row % ph.cnt_x, t = row / ph.cnt_x;
      const int jy = t % ph.cnt_y, b = t / ph.cnt_y;
      orow = ((long long)b * P.H + (ph.iy0 + P.stride * jy)) * P.W + (ph.ix0 + P.stride * jx);
    }
    auto row_of = [&](int r) -> long long { return __shfl_sync(0xffffffffu, orow, r); };
    uint2 pm[32 / (32 / (BN / 4))];
    const bool have_pm = prefetch_relu_mask<BN>(epi, lane, 0, P.C, row_of, pm);   // in flight while the MMAs run
    mbar_wait(&bar_done, 0);
    if (tid == 64) h_mark(4, mark_cta);
    tc_fence_after();
    if (epi.pdl_late) pdl_launch_dependents();
    float* slab = reinterpret_cast<float*>(smem_raw + (base - smem_u32(smem_raw))) + (warp & 3) * 32 * BN;
    stage_accumulator<BN>(tmem_d + ((uint32_t)lane_base << 16), slab, lane, true);
    if (tid == 64) h_mark(5, mark_cta);
    store_staged_rows<BN>(epi, slab, lane, 0, P.C, 0, row_of, have_pm ? pm : nullptr);
    if (tid == 64) h_mark(6, mark_cta);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_d, TMEM_COLS);
  if (tid == 32) h_mark(7, mark_cta);
}

// persistent data-gradient kernel: static tile walk over all phases, two TMEM accumulators, the WHOLE weight matrix
// resident in shared memory (box (tap, co-block) at a fixed offset), so the ring carries the dy tiles only
template <int BN, int STAGES>
__global__ void __launch_bounds__(H_THREADS)
hconv_dgrad_pers_kernel(const __grid_constant__ HDgradMaps maps, const __grid_constant__ CUtensorMap map_w, HDgradParams P, Epilogue epi,
                        int total_tiles, int kh) {
  constexpr int KE = 64, BM = BN == 32 ? 2 : 1;
  constexpr int A_BYTES = HBM_ROWS * KE * 2, B_BYTES = BN * KE * 2;
  constexpr int B_WB = BN == 32 ? 32 : 64, B_BOX = B_WB * KE * 2, B_NBOX = BN / B_WB;
  constexpr int SLAB = HBM_ROWS * BN * 4;
  constexpr uint32_t TMEM_COLS = 2 * BN < 32 ? 32 : 2 * BN;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* const smem_al = smem_raw + (base - smem_u32(smem_raw));
  __shared__ __align__(8) uint64_t bar_full[STAGES], bar_empty[STAGES], acc_full[2], acc_empty[2], bar_b;
  __shared__ uint32_t tmem_base_smem;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  pdl_launch_dependents();
  const int cb = P.Cout / KE;
  const uint32_t res_b = base + STAGES * A_BYTES + SLAB;     // box ((ky * kw + kx) * cb + co-block)

  if (tid == 0) {
#pragma unroll
    for (int i = 0; i < 4; ++i) if (i < P.nphase) prefetch_tensormap(&maps.m[i]);
    prefetch_tensormap(&map_w);
#pragma unroll
    for (int s = 0; s < STAGES; ++s) { mbar_init(&bar_full[s], 1); mbar_init(&bar_empty[s], 1); }
#pragma unroll
    for (int a = 0; a < 2; ++a) { mbar_init(&acc_full[a], 1); mbar_init(&acc_empty[a], 4); }
    mbar_init(&bar_b, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) tmem_alloc(&tmem_base_smem, TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  pdl_wait();                  // everything above overlaps the previous kernel's tail (launch_pdl); no-op otherwise
  const uint32_t tmem_d = tmem_base_smem;

  auto phase_of = [&](int t) {
    int ph = 0;
#pragma unroll
    for (int i = 1; i < 4; ++i) if (i < P.nphase && t >= P.ph[i].tile_begin) ph = i;
    return ph;
  };

  if (warp == 0 && lane == 0) {
    const int K = P.kw * P.C, taps = kh * P.kw;
    mbar_expect_tx(&bar_b, (uint32_t)(taps * cb * B_BYTES));
    for (int tap = 0; tap < taps; ++tap)
      for (int c = 0; c < cb; ++c)
#pragma unroll
        for (int j = 0; j < B_NBOX; ++j)
          tma_load_2d(res_b + (tap * cb + c) * B_BYTES + j * B_BOX, &map_w, (tap / P.kw) * K + (tap % P.kw) * P.C + B_WB * j, c * KE, &bar_b);
    int it = 0;
    for (int t = blockIdx.x; t < total_tiles; t += gridDim.x) {
      const int phase = phase_of(t);
      const HDgradPhase& ph = P.ph[phase];
      const int row0 = (t - ph.tile_begin) * HBM_ROWS;
      const int jx = row0 % ph.cnt_x, q = row0 / ph.cnt_x;
      const int ax = ph.lower_x + jx, ay = ph.lower_y + q % ph.cnt_y, an = q / ph.cnt_y;
      const int nkb = ph.Ty * ph.Tx * cb;
      int co0 = 0, off_x = 0, off_y = 0;
      for (int i = 0; i < nkb; ++i, ++it) {
        const int s = it % STAGES;
        if (it >= STAGES) mbar_wait(&bar_empty[s], ((it / STAGES) - 1) & 1);
        mbar_expect_tx(&bar_full[s], A_BYTES);
        tma_load_im2col(base + s * A_BYTES, &maps.m[phase], co0, ax, ay, an, (uint16_t)off_x, (uint16_t)off_y, &bar_full[s]);
        co0 += KE;
        if (co0 == P.Cout) {
          co0 = 0;
          if (++off_x == ph.Tx) { off_x = 0; ++off_y; }
        }
      }
    }
  } else if (warp == 1 && lane == 0) {
    constexpr uint32_t idesc = idesc_bf16(HBM_ROWS, BN, false, true);
    mbar_wait(&bar_b, 0);
    tc_fence_after();
    int it = 0, ti = 0;
    for (int t = blockIdx.x; t < total_tiles; t += gridDim.x, ++ti) {
      const HDgradPhase& ph = P.ph[phase_of(t)];
      const int nkb = ph.Ty * ph.Tx * cb;
      const int ab = ti & 1;
      mbar_wait(&acc_empty[ab], ((ti >> 1) & 1) ^ 1);
      tc_fence_after();
      const uint32_t acc = tmem_d + (uint32_t)(ab * BN);
      int c = 0, off_x = 0, off_y = 0;
      for (int i = 0; i < nkb; ++i, ++it) {
        const int s = it % STAGES;
        mbar_wait(&bar_full[s], (it / STAGES) & 1);
        tc_fence_after();
        const int ky = ph.py + P.stride * (ph.Ty - 1 - off_y), kx = ph.px + P.stride * (ph.Tx - 1 - off_x);
        const uint32_t sa = base + s * A_BYTES, sb = res_b + ((ky * P.kw + kx) * cb + c) * B_BYTES;
#pragma unroll
        for (int kk = 0; kk < KE / 16; ++kk)
          umma_bf16(acc, operand_desc<0, KE>(sa, kk), operand_desc<BM, KE>(sb, kk), idesc, (i > 0 || kk > 0) ? 1u : 0u);
        umma_commit(&bar_empty[s]);
        if (++c == cb) {
          c = 0;
          if (++off_x == ph.Tx) { off_x = 0; ++off_y; }
        }
      }
      umma_commit(&acc_full[ab]);
    }
  } else if (warp >= 2) {
    const int lane_base = (warp & 3) * 32;
    float* slab = reinterpret_cast<float*>(smem_al + STAGES * A_BYTES) + (warp & 3) * 32 * BN;
    int ti = 0;
    for (int t = blockIdx.x; t < total_tiles; t += gridDim.x, ++ti) {
      const HDgradPhase& ph = P.ph[phase_of(t)];
      const int row = (t - ph.tile_begin) * HBM_ROWS + lane_base + lane;
      const int Mp = P.B * ph.cnt_y * ph.cnt_x;
      long long orow = -1;
      if (row < Mp) {
        const int jx = row % ph.cnt_x, q = row / ph.cnt_x;
        const int jy = q % ph.cnt_y, b = q / ph.cnt_y;
        orow = ((long long)b * P.H + (ph.iy0 + P.stride * jy)) * P.W + (ph.ix0 + P.stride * jx);
      }
      const int ab = ti & 1;
      mbar_wait(&acc_full[ab], (ti >> 1) & 1);
      tc_fence_after();
      stage_accumulator<BN>(tmem_d + ((uint32_t)lane_base << 16) + (uint32_t)(ab * BN), slab, lane, true);
      tc_fence_before();
      if (lane == 0) mbar_arrive(&acc_empty[ab]);
      store_staged_rows<BN>(epi, slab, lane, 0, P.C, 0, [&](int r) -> long long { return __shfl_sync(0xffffffffu, orow, r); });
      __syncwarp();
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_d, TMEM_COLS);
}

template <int BN, int STAGES>
static int launch_hdgrad_pers_s(const HDgradMaps& maps, const CUtensorMap& mw, const HDgradParams& P, int tiles, const Epilogue& e,
                                int kh, int smem, cudaStream_t s) {
  static int attr = 0;
  if (attr < smem) {
    B200RL_CUDA_OK(cudaFuncSetAttribute(hconv_dgrad_pers_kernel<BN, STAGES>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    attr = smem;
  }
  B200RL_CUDA_OK(launch_pdl(hconv_dgrad_pers_kernel<BN, STAGES>, dim3(std::min(tiles, kNumSMs)), dim3(H_THREADS), smem, s, maps, mw, P, e, tiles, kh));
  B200RL_LAUNCH_OK();
  return B200RL_OK;
}
template <int BN>
static int launch_hdgrad_pers(const HDgradMaps& maps, const CUtensorMap& mw, const HDgradParams& P, int tiles, const Epilogue& e,
                              int kh, cudaStream_t s) {
  const int res_b = kh * P.kw * (P.Cout / 64) * BN * 64 * 2;
  const int fixed = HBM_ROWS * BN * 4 + res_b + 1024, A = HBM_ROWS * 64 * 2;
  // one CTA per SM (the resident weights take 64-72 KB): the ring gets the rest of the shared memory
  if (8 * A + fixed <= 224 * 1024) return launch_hdgrad_pers_s<BN, 8>(maps, mw, P, tiles, e, kh, 8 * A + fixed, s);
  if (6 * A + fixed <= 224 * 1024) return launch_hdgrad_pers_s<BN, 6>(maps, mw, P, tiles, e, kh, 6 * A + fixed, s);
  if (4 * A + fixed <= 224 * 1024) return launch_hdgrad_pers_s<BN, 4>(maps, mw, P, tiles, e, kh, 4 * A + fixed, s);
  return 1;
}

template <int BN>
static int launch_hdgrad(const HDgradMaps& maps, const CUtensorMap& mw, const HDgradParams& P, int tiles, const Epilogue& e,
                         cudaStream_t s) {
  constexpr int smem = D_STAGES * (HBM_ROWS * 64 * 2 + BN * 64 * 2) + 1024;
  static bool attr = false;
  if (!attr) {
    B200RL_CUDA_OK(cudaFuncSetAttribute(hconv_dgrad_kernel<BN>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    attr = true;
  }
  Epilogue el = e;
  el.pdl_late = pdl_late_mode();
  B200RL_CUDA_OK(launch_pdl(hconv_dgrad_kernel<BN>, dim3(tiles), dim3(H_THREADS), smem, s, maps, mw, P, el));
  B200RL_LAUNCH_OK();
  return B200RL_OK;
}

int h_conv_dgrad(const bf16* dy, const bf16* w, void* dx, const b200rl_conv_geom& g, const void* mask, int mask_act, int out_bf16,
                 int mask_bf16, cudaStream_t s) {
  const int K = g.kh * g.kw * g.C, st = g.stride;
  if (st > 2 || g.kh < st || g.kw < st || g.Cout % 64 != 0 || (g.C != 32 && g.C != 64 && g.C != 128) || !ok16(dy, g.Cout) ||
      !ok16(w, K) || (int64_t)g.B * g.H * g.W >= (1ll << 31) / g.C)
    return 1;
  EncodeIm2colFn enc = get_encode_im2col();
  if (!enc) return 1;
  HDgradMaps maps;
  HDgradParams P;
  P.nphase = st * st; P.stride = st; P.kw = g.kw; P.C = g.C; P.Cout = g.Cout; P.W = g.W; P.H = g.H; P.B = g.B;
  auto fdiv = [](int a, int b) { return a >= 0 ? a / b : -((-a + b - 1) / b); };
  int tiles = 0;
  for (int py = 0; py < st; ++py)
    for (int px = 0; px < st; ++px) {
      HDgradPhase& ph = P.ph[py * st + px];
      const int Ty = (g.kh - py + st - 1) / st, Tx = (g.kw - px + st - 1) / st;
      const int qy0 = -fdiv(-(g.pad_top - py), st), qx0 = -fdiv(-(g.pad_left - px), st);
      const int qy1 = fdiv(g.H - 1 + g.pad_top - py, st), qx1 = fdiv(g.W - 1 + g.pad_left - px, st);
      ph.tile_begin = tiles;
      ph.cnt_x = qx1 - qx0 + 1; ph.cnt_y = qy1 - qy0 + 1;
      ph.Tx = Tx; ph.Ty = Ty; ph.px = px; ph.py = py;
      ph.lower_x = qx0 - (Tx - 1); ph.lower_y = qy0 - (Ty - 1);
      ph.ix0 = st * qx0 + px - g.pad_left; ph.iy0 = st * qy0 + py - g.pad_top;
      if (ph.cnt_x <= 0 || ph.cnt_y <= 0) return 1;
      tiles += ceil_div(g.B * ph.cnt_x * ph.cnt_y, HBM_ROWS);
      cuuint64_t dims[4] = {(cuuint64_t)g.Cout, (cuuint64_t)g.OW, (cuuint64_t)g.OH, (cuuint64_t)g.B};
      cuuint64_t strides[3] = {(cuuint64_t)g.Cout * 2, (cuuint64_t)g.OW * g.Cout * 2, (cuuint64_t)g.OH * g.OW * g.Cout * 2};
      int lower[2] = {ph.lower_x, ph.lower_y};
      int upper[2] = {(qx1 - (Tx - 1)) - (g.OW - 1), (qy1 - (Ty - 1)) - (g.OH - 1)};
      cuuint32_t es[4] = {1, 1, 1, 1};
      if (enc(&maps.m[py * st + px], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, (void*)dy, dims, strides, lower, upper, 64, HBM_ROWS, es,
              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
        return 1;
    }
  for (int i = P.nphase; i < 4; ++i) { P.ph[i] = P.ph[0]; maps.m[i] = maps.m[0]; }
  CUtensorMap mw;
  const int WB = g.C == 32 ? 32 : 64;
  if (!make_map_h(&mw, w, g.Cout, K, K, WB, 64)) return 1;
  Epilogue e = make_epi(dx, g.C, nullptr, 0, mask, g.C, mask_act, 0, out_bf16, mask_bf16, 0.f);
  if (use_persistent() && tiles > kNumSMs && (g.C == 32 || g.C == 64)) {
    const int rc = g.C == 32 ? launch_hdgrad_pers<32>(maps, mw, P, tiles, e, g.kh, s) : launch_hdgrad_pers<64>(maps, mw, P, tiles, e, g.kh, s);
    if (rc != 1) return rc;     // 1 = weights too large to stay resident: one tile per CTA instead
  }
  if (g.C == 32) return launch_hdgrad<32>(maps, mw, P, tiles, e, s);
  if (g.C == 64) return launch_hdgrad<64>(maps, mw, P, tiles, e, s);
  return launch_hdgrad<128>(maps, mw, P, tiles, e, s);
}

// ---- fp32 -> bf16 shadow of a parameter buffer (initialisation, restore, after a data-parallel exchange)
__global__ void __launch_bounds__(256) f32_to_bf16_kernel(long long n8, const float4* __restrict__ src, uint4* __restrict__ dst) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (; i < n8; i += stride) {
    const float4 a = __ldg(src + 2 * i), b = __ldg(src + 2 * i + 1);
    const __nv_bfloat162 t0 = __floats2bfloat162_rn(a.x, a.y), t1 = __floats2bfloat162_rn(a.z, a.w);
    const __nv_bfloat162 t2 = __floats2bfloat162_rn(b.x, b.y), t3 = __floats2bfloat162_rn(b.z, b.w);
    uint4 pk;
    pk.x = *reinterpret_cast<const uint32_t*>(&t0); pk.y = *reinterpret_cast<const uint32_t*>(&t1);
    pk.z = *reinterpret_cast<const uint32_t*>(&t2); pk.w = *reinterpret_cast<const uint32_t*>(&t3);
    dst[i] = pk;
  }
}
int h_f32_to_bf16(int64_t n, const float* src, bf16* dst, cudaStream_t s) {
  if (n % 8 != 0 || (((uintptr_t)src) & 15) != 0 || (((uintptr_t)dst) & 15) != 0) return 1;
  const long long n8 = n / 8;
  const int blocks = (int)std::min<long long>(ceil_div<long long>(n8, 256), kNumSMs * 8);
  f32_to_bf16_kernel<<<std::max(blocks, 1), 256, 0, s>>>(n8, (const float4*)src, (uint4*)dst);
  B200RL_LAUNCH_OK();
  return B200RL_OK;
}

}  // namespace b200rl

extern "C" int b200rl_debug_set_persistent(int on) { b200rl::g_h_persistent = on; return 0; }
extern "C" int b200rl_debug_h_timeline(unsigned long long* buf_dev) {
  cudaError_t e = cudaMemcpyToSymbol(b200rl::g_h_timeline, &buf_dev, sizeof(buf_dev));
  return e == cudaSuccess ? 0 : -2;
}
