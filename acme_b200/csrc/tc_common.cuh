// tcgen05 / TMEM / mbarrier PTX wrappers and the register-level epilogue shared by the tensor-core
// GEMM kernels (gemm_tc.cu: loader-fed bf16, gemm_tma.cu: TMA-fed tf32).
#pragma once
#include <cuda_bf16.h>

#include "common.cuh"
#include "gemm_common.cuh"

namespace b200rl {

// ------------------------------------------------------------------------------ PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  const uint32_t addr = smem_u32(bar);
  do {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(addr), "r"(parity)
        : "memory");
  } while (!ok);
}
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// Epilogue of 16 consecutive columns of one row held by one thread: vectorised (float4) whenever the
// destination allows it, so every 32-byte sector is written whole.  The transcendental activations are
// kept out of line: inlining them 16x per column group bloats the kernel past the instruction caches
// (a 128-column epilogue then runs at instruction-fetch speed).
static __device__ __noinline__ float act_eval_slow(float v, int act) { return apply_act(v, act); }
static __device__ __noinline__ float act_grad_slow(float y, int act) { return act_grad_out(y, act); }

__device__ __forceinline__ void finish16(const Epilogue& e, int row, int c0, int N, int M, float (&v)[16]) {
  const bool full = c0 + 15 < N;
  if (e.partial) {
    float* dst = e.partial + ((size_t)blockIdx.z * M + row) * N + c0;
    if (full && ((((uintptr_t)dst) & 15) == 0)) {
#pragma unroll
      for (int q = 0; q < 4; ++q) reinterpret_cast<float4*>(dst)[q] = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
    } else {
#pragma unroll
      for (int j = 0; j < 16; ++j) if (c0 + j < N) dst[j] = v[j];
    }
    return;
  }
  // bias, activation, activation-derivative mask -- each decided once per 16 columns
  if (e.out_bf16 || e.mask_bf16) {   // the bf16 dataflow reaches this (unaligned / transposed) path rarely: scalar form
#pragma unroll
    for (int j = 0; j < 16; ++j) if (c0 + j < N) finish(e, row, c0 + j, v[j]);
    return;
  }
  if (e.scale != 0.f) {
#pragma unroll
    for (int j = 0; j < 16; ++j) v[j] *= e.scale;
  }
  if (e.bias) {
#pragma unroll
    for (int j = 0; j < 16; ++j) if (c0 + j < N) v[j] += __ldg(e.bias + c0 + j);
  }
  if (e.act == B200RL_ACT_RELU) {
#pragma unroll
    for (int j = 0; j < 16; ++j) v[j] = fmaxf(v[j], 0.f);
  } else if (e.act != B200RL_ACT_NONE) {
#pragma unroll
    for (int j = 0; j < 16; ++j) v[j] = act_eval_slow(v[j], e.act);
  }
  if (e.mask) {
    const float* msk = e.mask + (size_t)row * e.ldmask + c0;
    if (e.mask_act == B200RL_ACT_RELU) {
#pragma unroll
      for (int j = 0; j < 16; ++j) if (c0 + j < N) v[j] = __ldg(msk + j) > 0.f ? v[j] : 0.f;
    } else {
#pragma unroll
      for (int j = 0; j < 16; ++j) if (c0 + j < N) v[j] *= act_grad_slow(__ldg(msk + j), e.mask_act);
    }
  }
  if (e.transpose_out) {   // lanes hold consecutive rows -> consecutive addresses for a fixed column
#pragma unroll
    for (int j = 0; j < 16; ++j) if (c0 + j < N) e.out[(size_t)(c0 + j) * e.ldo + row] = v[j];
    return;
  }
  float* dst = e.out + (size_t)row * e.ldo + c0;
  if (full && ((((uintptr_t)dst) & 15) == 0)) {
#pragma unroll
    for (int q = 0; q < 4; ++q) reinterpret_cast<float4*>(dst)[q] = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
  } else {
#pragma unroll
    for (int j = 0; j < 16; ++j) if (c0 + j < N) dst[j] = v[j];
  }
}


// Epilogue of 4 consecutive columns (col .. col+3) of one row: the row-wise, coalesced counterpart of finish16 used
// after the accumulator tile has been transposed through shared memory (a warp then writes whole 128-byte lines).
__device__ __forceinline__ void finish4(const Epilogue& e, size_t row, int col, int N, int M, float4 a) {
  float v[4] = {a.x, a.y, a.z, a.w};
  const bool full = col + 3 < N;
  float* dst;
  if (e.partial) {
    dst = e.partial + ((size_t)blockIdx.z * M + row) * N + col;
  } else {
    if (e.bias) {
#pragma unroll
      for (int j = 0; j < 4; ++j) if (col + j < N) v[j] += __ldg(e.bias + col + j);
    }
    if (e.act == B200RL_ACT_RELU) {
#pragma unroll
      for (int j = 0; j < 4; ++j) v[j] = fmaxf(v[j], 0.f);
    } else if (e.act != B200RL_ACT_NONE) {
#pragma unroll
      for (int j = 0; j < 4; ++j) v[j] = act_eval_slow(v[j], e.act);
    }
    if (e.mask) {
      const float* msk = e.mask + row * e.ldmask + col;
      float m[4];
      if (full && ((((uintptr_t)msk) & 15) == 0)) {
        const float4 t = __ldg(reinterpret_cast<const float4*>(msk));
        m[0] = t.x; m[1] = t.y; m[2] = t.z; m[3] = t.w;
      } else {
#pragma unroll
        for (int j = 0; j < 4; ++j) m[j] = col + j < N ? __ldg(msk + j) : 0.f;
      }
      if (e.mask_act == B200RL_ACT_RELU) {
#pragma unroll
        for (int j = 0; j < 4; ++j) v[j] = m[j] > 0.f ? v[j] : 0.f;
      } else {
#pragma unroll
        for (int j = 0; j < 4; ++j) v[j] *= act_grad_slow(m[j], e.mask_act);
      }
    }
    dst = e.out + row * e.ldo + col;
  }
  if (full && ((((uintptr_t)dst) & 15) == 0)) {
    *reinterpret_cast<float4*>(dst) = make_float4(v[0], v[1], v[2], v[3]);
  } else {
#pragma unroll
    for (int j = 0; j < 4; ++j) if (col + j < N) dst[j] = v[j];
  }
}

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]),
        "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]),
        "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// TMEM accumulator (this warp's 32 lanes x BN columns) -> the warp's private shared-memory slab, 16-byte chunks
// XOR-swizzled by row so both the lane-per-row writes and the row-wise reads are bank-conflict free.
template <int BN>
__device__ __forceinline__ void stage_accumulator(uint32_t tmem_warp, float* slab, int lane, bool have) {
  constexpr int CPR = BN / 4;
#pragma unroll
  for (int cc = 0; cc < BN; cc += 32) {
    float v[32];
    if (have) tmem_ld32(tmem_warp + (uint32_t)cc, v);
    else {
#pragma unroll
      for (int j = 0; j < 32; ++j) v[j] = 0.f;
    }
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      const int chunk = (cc >> 2) + q;
      reinterpret_cast<float4*>(slab)[lane * CPR + (chunk ^ (lane & 7))] = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
    }
  }
  __syncwarp();
}
template <int BN>
__device__ __forceinline__ float4 staged_chunk(const float* slab, int r, int c) {
  return reinterpret_cast<const float4*>(slab)[r * (BN / 4) + (c ^ (r & 7))];
}

// Row-wise epilogue over a staged slab: lane -> (row lane, 16-byte column chunk); four rows are in flight at a time
// (their shared-memory reads and mask loads are issued before any is consumed: one warp per scheduler has nothing
// else to hide latency with).  dst_row(r) -> destination row of slab row r, or < 0 to skip; it is called by all lanes.
// The ReLU-derivative mask of a data gradient is the producer layer's OUTPUT: it does not depend on the accumulator, so the
// epilogue warps fetch it into registers BEFORE they wait for the MMAs (a CTA's timeline showed the masked store phase
// taking 3-5 us of a 6-10 us tile: four rounds of dependent mask loads).  bf16 masks, ReLU only; `pm[it]` belongs to the
// same (row, column chunk) that iteration `it` of store_staged_rows handles.  Returns false (warp-uniform) if the
// fast-path conditions do not hold: store_staged_rows then loads the mask itself.
template <int BN, class RowFn>
__device__ __forceinline__ bool prefetch_relu_mask(const Epilogue& e, int lane, int col0, int N, RowFn dst_row,
                                                   uint2 (&pm)[32 / (32 / (BN / 4))]) {
  constexpr int CPR = BN / 4, RPI = 32 / CPR, ITERS = 32 / RPI;
  const int c = lane % CPR, rl = lane / CPR, col = col0 + 4 * c;
  const bool ok = e.mask && e.mask_bf16 && !e.partial && e.mask_act == B200RL_ACT_RELU && col + 3 < N && (e.ldmask & 3) == 0 &&
                  ((uintptr_t)e.mask & 7) == 0;
  if (!__all_sync(0xffffffffu, ok)) return false;
#pragma unroll
  for (int it = 0; it < ITERS; ++it) {
    const long long row = dst_row(it * RPI + rl);
    pm[it] = row >= 0 ? __ldg(reinterpret_cast<const uint2*>(reinterpret_cast<const __nv_bfloat16*>(e.mask) + (size_t)row * e.ldmask + col))
                      : make_uint2(0u, 0u);
  }
  return true;
}

template <int BN, class RowFn>
__device__ __forceinline__ void store_staged_rows(const Epilogue& e, const float* slab, int lane, int col0, int N, int M,
                                                  RowFn dst_row, const uint2* pm = nullptr) {
  constexpr int CPR = BN / 4, RPI = 32 / CPR, ITERS = 32 / RPI, G = 4;
  const int c = lane % CPR, rl = lane / CPR, col = col0 + 4 * c;
  float* const base = e.partial ? e.partial + (size_t)blockIdx.z * M * N : e.out;
  const int ldo = e.partial ? N : e.ldo;
  const bool use_mask = e.mask && !e.partial;
  const bool obf = e.out_bf16 && !e.partial, mbf = e.mask_bf16 != 0;
  const bool fast = col + 3 < N && (ldo & 3) == 0 && ((uintptr_t)base & (obf ? 7 : 15)) == 0 &&
                    (!use_mask || ((e.ldmask & 3) == 0 && ((uintptr_t)e.mask & (mbf ? 7 : 15)) == 0));
  if (!__all_sync(0xffffffffu, fast)) {
#pragma unroll 1
    for (int it = 0; it < ITERS; ++it) {
      const int r = it * RPI + rl;
      const long long row = dst_row(r);
      if (row < 0 || col >= N) continue;
      const float4 a = staged_chunk<BN>(slab, r, c);
      // a split-K partial is stored raw (finish4); finish() would apply the epilogue and write `out` instead
      if (!e.partial && (obf || mbf || e.scale != 0.f)) {
        const float v[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) if (col + j < N) finish(e, (int)row, col + j, v[j]);
      } else {
        finish4(e, (size_t)row, col, N, M, a);
      }
    }
    return;
  }
  const float sc = e.partial ? 1.f : epi_scale(e);
  float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
  if (e.bias && !e.partial) b4 = make_float4(__ldg(e.bias + col), __ldg(e.bias + col + 1), __ldg(e.bias + col + 2), __ldg(e.bias + col + 3));
  const int act = e.partial ? B200RL_ACT_NONE : e.act;
#pragma unroll 1
  for (int it = 0; it < ITERS; it += G) {
    long long rows[G];
    float4 a[G], m[G];
#pragma unroll
    for (int g = 0; g < G; ++g) {
      const int r = (it + g) * RPI + rl;
      rows[g] = dst_row(r);
      a[g] = staged_chunk<BN>(slab, r, c);
    }
    if (use_mask && pm) {   // fetched ahead of the accumulator (prefetch_relu_mask)
#pragma unroll
      for (int g = 0; g < G; ++g) {
        const uint2 t = pm[it + g];
        const float2 lo = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&t.x));
        const float2 hi = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&t.y));
        m[g] = make_float4(lo.x, lo.y, hi.x, hi.y);
      }
    } else if (use_mask) {
#pragma unroll
      for (int g = 0; g < G; ++g) {
        if (rows[g] < 0) continue;
        if (mbf) {
          const uint2 t = __ldg(reinterpret_cast<const uint2*>(reinterpret_cast<const __nv_bfloat16*>(e.mask) + (size_t)rows[g] * e.ldmask + col));
          const float2 lo = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&t.x));
          const float2 hi = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&t.y));
          m[g] = make_float4(lo.x, lo.y, hi.x, hi.y);
        } else {
          m[g] = __ldg(reinterpret_cast<const float4*>(e.mask + (size_t)rows[g] * e.ldmask + col));
        }
      }
    }
#pragma unroll
    for (int g = 0; g < G; ++g) {
      if (rows[g] < 0) continue;
      float4 v = make_float4(fmaf(a[g].x, sc, b4.x), fmaf(a[g].y, sc, b4.y), fmaf(a[g].z, sc, b4.z), fmaf(a[g].w, sc, b4.w));
      if (act == B200RL_ACT_RELU) {
        v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f);
      } else if (act != B200RL_ACT_NONE) {
        v.x = act_eval_slow(v.x, act); v.y = act_eval_slow(v.y, act); v.z = act_eval_slow(v.z, act); v.w = act_eval_slow(v.w, act);
      }
      if (use_mask) {
        if (e.mask_act == B200RL_ACT_RELU) {
          v.x = m[g].x > 0.f ? v.x : 0.f; v.y = m[g].y > 0.f ? v.y : 0.f; v.z = m[g].z > 0.f ? v.z : 0.f; v.w = m[g].w > 0.f ? v.w : 0.f;
        } else {
          v.x *= act_grad_slow(m[g].x, e.mask_act); v.y *= act_grad_slow(m[g].y, e.mask_act);
          v.z *= act_grad_slow(m[g].z, e.mask_act); v.w *= act_grad_slow(m[g].w, e.mask_act);
        }
      }
      if (obf) {
        const __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
        uint2 pk;
        pk.x = *reinterpret_cast<const uint32_t*>(&lo);
        pk.y = *reinterpret_cast<const uint32_t*>(&hi);
        *reinterpret_cast<uint2*>(reinterpret_cast<__nv_bfloat16*>(base) + (size_t)rows[g] * ldo + col) = pk;
      } else {
        *reinterpret_cast<float4*>(base + (size_t)rows[g] * ldo + col) = v;
      }
    }
  }
}

}  // namespace b200rl
