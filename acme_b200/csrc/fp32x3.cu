// K6, precision 3: fp32-accurate network layers on the bf16 tensor cores by three-way operand splitting.
//
// Every fp32 operand value x is split, in fp32, into three bf16 planes
//   hi = RN(x),  mid = RN(x - hi),  lo = RN(x - hi - mid)          (both subtractions are exact)
// and a product a * b becomes the six bf16 products
//   hi_a hi_b + hi_a mid_b + mid_a hi_b + hi_a lo_b + mid_a mid_b + lo_a hi_b
// summed in the fp32 accumulator; the dropped terms (mid lo, lo mid, lo lo) and the split residual are O(2^-25 |a||b|).
// An operand that is exact in bf16 (the integer pixel values of conv1's row image) has only its hi plane: three products.
//
// The kernels here only PREPARE the operands of the existing bf16 GEMMs (gemm_bf16.cu) and, where needed, add their
// outputs.  Each entry point picks one path from the shape alone:
//   (a) the split kernel writes the planes into the workspace concatenated along the reduction dimension, in matching
//       segment order, zero-padded to the multiples the bf16 kernels need; ONE bf16 GEMM launch then sums all products in
//       TMEM and applies bias / activation / mask in its own epilogue;
//   (b) conv1's forward on frames (the row-image kernel fixes C = 4 and Cout in {32, 64}): one raw fp32 launch per
//       filter plane into workspace slabs, then ONE combine kernel adds them (smallest terms first) and applies the
//       1/255 scale, bias and activation;
//   (c) everything else, and dense layers under 2^26 multiply-adds: the fp32 FFMA path (precision 0) unchanged.
// Bias gradients are the fp32 column sums of the unsplit dy (precision 0's kernel).
#include <algorithm>

#include <cuda_bf16.h>

#include "common.cuh"
#include "gemm_common.cuh"

namespace b200rl {
typedef __nv_bfloat16 bf16;
int check_geom(const b200rl_conv_geom* g);                        // layers_api.cu
int check_conv_ptr(const void* p, int u8, const char* what);
int check_geom_frames(const b200rl_conv_geom* g);
int rows_cp(int C);
int h_linear_fwd(int M, int N, int K, const bf16* x, int ldx, const bf16* w, const float* bias, void* y, int ldy, int act,
                 int out_bf16, void* ws, int64_t wsb, cudaStream_t s);   // gemm_bf16.cu
int h_linear_dgrad(int M, int N, int K, const bf16* dy, int lddy, const bf16* w, void* dx, int lddx, const void* mask, int ldmask,
                   int mask_act, int out_bf16, int mask_bf16, void* ws, int64_t wsb, cudaStream_t s);
int h_linear_wgrad(int M, int N, int K, const bf16* dy, int lddy, const bf16* x, int ldx, float* dw, float* db, void* ws,
                   int64_t wsb, cudaStream_t s);
int h_conv_fwd(const bf16* x, const bf16* w, const float* bias, void* y, const b200rl_conv_geom& g, int act, int out_bf16,
               void* ws, int64_t wsb, cudaStream_t s);
int h_conv_wgrad(const bf16* x, const bf16* dy, float* dw, float* db, const b200rl_conv_geom& g, void* ws, int64_t wsb,
                 cudaStream_t s);
int h_conv_dgrad(const bf16* dy, const bf16* w, void* dx, const b200rl_conv_geom& g, const void* mask, int mask_act, int out_bf16,
                 int mask_bf16, cudaStream_t s);
int64_t h_rows_bytes(const b200rl_conv_geom& g);
int h_rows_from_u8(const uint8_t* x, const b200rl_conv_geom& g, bf16* rows, int64_t bytes, cudaStream_t s);
int h_conv_fwd_rows_raw(const bf16* rows, const bf16* w, float* y, const b200rl_conv_geom& g, void* ws, int64_t wsb, cudaStream_t s);
int h_conv_wgrad_rows(const bf16* rows, const bf16* dy, float* dw, float* db, const b200rl_conv_geom& g, void* ws, int64_t wsb,
                      cudaStream_t s);

// ---------------------------------------------------------------------------------------------- split
// Segment s of an operand holds plane (pattern >> 2s) & 3 (0 hi, 1 mid, 2 lo).  The two operands of a GEMM use patterns
// whose segments pair up into the six (or, for an exact operand, three) products.
constexpr uint32_t PAT_A = 0u | 0u << 2 | 1u << 4 | 0u << 6 | 1u << 8 | 2u << 10;   // hi hi  mid hi  mid lo
constexpr uint32_t PAT_B = 0u | 1u << 2 | 0u << 4 | 2u << 6 | 1u << 8 | 0u << 10;   // hi mid hi  lo  mid hi
constexpr uint32_t PAT_HML = 0u | 1u << 2 | 2u << 4;                                // hi mid lo (against an exact operand)

// fp32 matrix src[R][Cc] (row stride ld) -> nseg bf16 segments.  by_rows = 0: segments side by side in every row,
// dst[r][s * Cp + c] (row length nseg * Cp, columns Cc..Cp-1 zero); by_rows = 1: segments stacked, dst[s * Rp + r][c]
// (rows R..Rp-1 zero).  One thread writes four consecutive columns of every segment (Cp, and Cc when by_rows, % 4 == 0).
struct SplitJob {
  const float* src; int64_t ld;
  int R, Cc, Rp, Cp, by_rows, nseg;
  uint32_t pattern;
  bf16* dst;
  int64_t groups;   // (by_rows ? Rp * Cc : R * Cp) / 4
};
struct SplitJobs { SplitJob j[2]; };

__device__ __forceinline__ void split3(float x, bf16& hi, bf16& mid, bf16& lo) {
  hi = __float2bfloat16_rn(x);
  const float r1 = __fsub_rn(x, __bfloat162float(hi));
  mid = __float2bfloat16_rn(r1);
  lo = __float2bfloat16_rn(__fsub_rn(r1, __bfloat162float(mid)));
}

__global__ void __launch_bounds__(256) x3_split_kernel(SplitJobs jobs, int njobs) {
  const int64_t total = jobs.j[0].groups + (njobs > 1 ? jobs.j[1].groups : 0);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const bool second = i >= jobs.j[0].groups;
    const SplitJob& J = second ? jobs.j[1] : jobs.j[0];
    const int64_t gi = second ? i - jobs.j[0].groups : i;
    const int width = (J.by_rows ? J.Cc : J.Cp) >> 2;
    const int r = (int)(gi / width), c = (int)(gi - (int64_t)r * width) * 4;
    uint32_t h[2], m[2], l[2];   // the three planes of the four values, packed two bf16 per word (kept in registers)
#pragma unroll
    for (int e = 0; e < 4; e += 2) {
      bf16 ph[2], pm[2], pl[2];
#pragma unroll
      for (int t = 0; t < 2; ++t) {
        const float x = (r < J.R && c + e + t < J.Cc) ? __ldg(J.src + (int64_t)r * J.ld + c + e + t) : 0.f;
        split3(x, ph[t], pm[t], pl[t]);
      }
      h[e / 2] = (uint32_t)__bfloat16_as_ushort(ph[0]) | (uint32_t)__bfloat16_as_ushort(ph[1]) << 16;
      m[e / 2] = (uint32_t)__bfloat16_as_ushort(pm[0]) | (uint32_t)__bfloat16_as_ushort(pm[1]) << 16;
      l[e / 2] = (uint32_t)__bfloat16_as_ushort(pl[0]) | (uint32_t)__bfloat16_as_ushort(pl[1]) << 16;
    }
    for (int s = 0; s < J.nseg; ++s) {
      const int pl = (J.pattern >> (2 * s)) & 3;
      const uint2 v = pl == 0 ? make_uint2(h[0], h[1]) : (pl == 1 ? make_uint2(m[0], m[1]) : make_uint2(l[0], l[1]));
      const int64_t o = J.by_rows ? ((int64_t)s * J.Rp + r) * J.Cc + c : (int64_t)r * J.nseg * J.Cp + (int64_t)s * J.Cp + c;
      *reinterpret_cast<uint2*>(J.dst + o) = v;
    }
  }
}

static SplitJob col_job(const float* src, int64_t ld, int R, int Cc, int Cp, int nseg, uint32_t pat, bf16* dst) {
  return SplitJob{src, ld, R, Cc, R, Cp, 0, nseg, pat, dst, (int64_t)R * Cp / 4};
}
static SplitJob row_job(const float* src, int64_t ld, int R, int Cc, int Rp, int nseg, uint32_t pat, bf16* dst) {
  return SplitJob{src, ld, R, Cc, Rp, Cc, 1, nseg, pat, dst, (int64_t)Rp * Cc / 4};
}
static int launch_split(const SplitJob& a, const SplitJob* b, cudaStream_t s) {
  SplitJobs jobs;
  jobs.j[0] = a;
  jobs.j[1] = b ? *b : a;
  const int64_t total = a.groups + (b ? b->groups : 0);
  const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>(ceil_div<int64_t>(total, 256), kNumSMs * 16));
  x3_split_kernel<<<blocks, 256, 0, s>>>(jobs, b ? 2 : 1);
  B200RL_LAUNCH_OK();
  return B200RL_OK;
}

// ---------------------------------------------------------------------------------------------- combine
// y[m, n] = act(scale * (slab[n_s - 1] + ... + slab[0]) + bias[n]); slab k = the product with plane k of the split operand,
// so the smallest terms are added first
__global__ void __launch_bounds__(256) x3_combine_kernel(const float* __restrict__ slabs, int nslab, int M, int N, float* __restrict__ y,
                                                         int ldy, const float* __restrict__ bias, int act, float scale) {
  const int64_t total = (int64_t)M * N, stride = total;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    float acc = __ldg(slabs + (nslab - 1) * stride + i);
    for (int k = nslab - 2; k >= 0; --k) acc = __fadd_rn(acc, __ldg(slabs + k * stride + i));
    const int m = (int)(i / N), n = (int)(i - (int64_t)m * N);
    acc = __fmul_rn(acc, scale);
    if (bias) acc = __fadd_rn(acc, __ldg(bias + n));
    y[(int64_t)m * ldy + n] = apply_act(acc, act);
  }
}

// ---------------------------------------------------------------------------------------------- the path rule
enum { PATH_FFMA = 0, PATH_CONCAT = 1, PATH_STACK = 2 };
static inline int rup(int a, int m) { return (a + m - 1) / m * m; }
static inline int64_t al256(int64_t b) { return (b + 255) & ~(int64_t)255; }
static bool rows_geom(const b200rl_conv_geom& g) { return h_rows_bytes(g) > 0; }
// first layer on frames of C channels: the filter has rows_cp(C) channels (padding columns zero, gemm_bf16.cu)
static b200rl_conv_geom filter_geom(const b200rl_conv_geom& g) {
  b200rl_conv_geom f = g;
  f.C = rows_cp(g.C);
  return f;
}

static int path_of(int op, int M, int N, int K, const b200rl_conv_geom* g, int x_u8) {
  switch (op) {
    case B200RL_X3_LINEAR_FWD:
      if ((int64_t)M * N * K < (1ll << 26)) return PATH_FFMA;
      return 6 * rup(K, 8) >= 64 ? PATH_CONCAT : PATH_FFMA;
    case B200RL_X3_LINEAR_DGRAD:
      if ((int64_t)M * N * K < (1ll << 26)) return PATH_FFMA;
      return (K % 64 == 0 && 6 * rup(N, 8) >= 64) ? PATH_CONCAT : PATH_FFMA;
    case B200RL_X3_LINEAR_WGRAD:
      if ((int64_t)M * N * K < (1ll << 26)) return PATH_FFMA;
      return (N % 64 == 0 && K % 64 == 0) ? PATH_CONCAT : PATH_FFMA;
    case B200RL_X3_CONV_FWD:
      if (x_u8) return rows_geom(*g) ? PATH_STACK : PATH_FFMA;
      return (g->Cout == 32 || g->Cout == 64 || g->Cout == 128) ? PATH_CONCAT : PATH_FFMA;
    case B200RL_X3_CONV_WGRAD:
      if (x_u8) return rows_geom(*g) && 3ll * g->B * g->OH * g->OW < (1ll << 31) ? PATH_CONCAT : PATH_FFMA;
      return ((g->C == 32 || g->C % 64 == 0) && (g->Cout == 32 || g->Cout == 64) && 6ll * g->B * g->H * g->W < (1ll << 31) &&
              6ll * g->B * g->OH * g->OW < (1ll << 31))
                 ? PATH_CONCAT
                 : PATH_FFMA;
    case B200RL_X3_CONV_DGRAD:
      return (g->stride <= 2 && g->kh >= g->stride && g->kw >= g->stride && (g->C == 32 || g->C == 64 || g->C == 128) &&
              (int64_t)g->B * g->H * g->W < (1ll << 31) / g->C)
                 ? PATH_CONCAT
                 : PATH_FFMA;
  }
  return -1;
}

// split-K partial slabs the bf16 GEMM of shape (M, N, K) takes at its default split rule (gemm_bf16.cu launch_h)
static int64_t splitk_bytes(int M, int N, int K, int KE, int BN) {
  const int64_t tiles = (int64_t)ceil_div(M, 128) * ceil_div(N, BN);
  const int kblocks = ceil_div(K, KE);
  if (!(2 * tiles <= kNumSMs && kblocks >= 16)) return 0;
  int splits = (int)std::min<int64_t>(ceil_div<int64_t>(kNumSMs, tiles), kblocks / 8);
  splits = std::max(1, std::min(splits, 64));
  const int kps = ceil_div(kblocks, splits);
  splits = ceil_div(kblocks, kps);
  return splits > 1 ? (int64_t)splits * M * N * 4 : 0;
}
static int64_t colsum_bytes(int N) { return 2ll * kNumSMs * N * 4; }

// Workspace layout of paths (a) / (b): [operand A planes][operand B planes][frames' row image ...][tail], each part
// 256-byte aligned; the tail takes the GEMM's split-K partials, the combine slabs and the bias-gradient column sums.
struct Plan { int path; int64_t a, b, img, slabs, tail; int64_t total() const { return al256(a) + al256(b) + al256(img) + al256(slabs) + tail; } };

static Plan plan_of(int op, int M, int N, int K, const b200rl_conv_geom* g, int x_u8) {
  Plan p{path_of(op, M, N, K, g, x_u8), 0, 0, 0, 0, 0};
  if (p.path == PATH_FFMA) {   // the fp32 path at its preferred split counts (b200rl_workspace_bytes)
    switch (op) {
      case B200RL_X3_LINEAR_FWD: p.tail = 256ll * M * N; break;
      case B200RL_X3_LINEAR_DGRAD: p.tail = 256ll * M * K; break;
      case B200RL_X3_LINEAR_WGRAD: p.tail = std::max<int64_t>(256ll * N * K, colsum_bytes(N)); break;
      case B200RL_X3_CONV_FWD: p.tail = 256ll * g->B * g->OH * g->OW * g->Cout; break;
      case B200RL_X3_CONV_WGRAD: p.tail = std::max<int64_t>(256ll * g->Cout * g->kh * g->kw * g->C, colsum_bytes(g->Cout)); break;
      case B200RL_X3_CONV_DGRAD: p.tail = al256(4ll * g->B * g->H * g->W) + 256ll * g->B * g->H * g->W * g->C; break;
    }
    return p;
  }
  switch (op) {
    case B200RL_X3_LINEAR_FWD: {
      const int K6 = 6 * rup(K, 8);
      p.a = 2ll * M * K6; p.b = 2ll * N * K6;
      p.tail = splitk_bytes(M, N, K6, 64, N <= 32 ? 32 : (N <= 64 ? 64 : 128));
      break;
    }
    case B200RL_X3_LINEAR_DGRAD: {
      const int N6 = 6 * rup(N, 8);
      p.a = 2ll * M * N6; p.b = 2ll * N6 * K;
      break;
    }
    case B200RL_X3_LINEAR_WGRAD:
      p.a = 12ll * M * N; p.b = 12ll * M * K;
      p.tail = std::max<int64_t>(splitk_bytes(N, K, 6 * M, 64, K >= 128 ? 128 : 64), colsum_bytes(N));
      break;
    case B200RL_X3_CONV_FWD: {
      const int64_t Mo = (int64_t)g->B * g->OH * g->OW, taps = g->kh * g->kw;
      if (p.path == PATH_STACK) {
        p.b = 6ll * g->Cout * taps * g->C;
        if (x_u8 == 1) p.img = h_rows_bytes(*g);
        p.slabs = 12ll * Mo * g->Cout;
        p.tail = splitk_bytes((int)Mo, g->Cout, (int)(taps * g->C), 32, g->Cout);
      } else {
        const int C6 = 6 * rup(g->C, 32);
        p.a = 2ll * g->B * g->H * g->W * C6; p.b = 2ll * g->Cout * taps * C6;
        p.tail = splitk_bytes((int)Mo, g->Cout, (int)(taps * C6), 64, g->Cout);
      }
      break;
    }
    case B200RL_X3_CONV_WGRAD: {
      const int64_t taps = g->kh * g->kw;
      if (x_u8) {
        const int64_t px = 3ll * g->B * g->OH * g->OW;
        p.a = 6ll * g->B * g->OH * g->OW * g->Cout;
        p.img = 3 * h_rows_bytes(*g);
        p.tail = std::max<int64_t>(splitk_bytes((int)(taps * g->C), g->Cout, (int)px, 64, g->Cout), colsum_bytes(g->Cout));
      } else {
        const int64_t px = 6ll * g->B * g->OH * g->OW;
        p.a = 12ll * g->B * g->H * g->W * g->C; p.b = 12ll * g->B * g->OH * g->OW * g->Cout;
        p.tail = std::max<int64_t>(splitk_bytes((int)(taps * g->C), g->Cout, (int)px, 64, g->Cout), colsum_bytes(g->Cout));
      }
      break;
    }
    case B200RL_X3_CONV_DGRAD: {
      const int C6 = 6 * rup(g->Cout, 32);
      p.a = 2ll * g->B * g->OH * g->OW * C6; p.b = 2ll * C6 * g->kh * g->kw * g->C;
      break;
    }
  }
  return p;
}

struct Carve {
  char* p;
  Carve(void* ws) : p((char*)ws) {}
  template <typename T> T* take(int64_t bytes) { T* r = (T*)p; p += al256(bytes); return r; }
};

static int check_ws(const Plan& p, void* ws, int64_t wsb) {
  const int64_t need = p.total();
  B200RL_REQUIRE(wsb >= need && (need == 0 || ws), "workspace of %lld bytes, this call needs %lld (b200rl_x3_ws_bytes)",
                 (long long)wsb, (long long)need);
  B200RL_REQUIRE(p.path == PATH_FFMA || (((uintptr_t)ws) & 255) == 0, "workspace must be 256-byte aligned");
  return B200RL_OK;
}
#define X3_GEMM(expr)                                                                                   \
  do {                                                                                                  \
    int _rc = (expr);                                                                                   \
    B200RL_REQUIRE(_rc != 1, "precision 3: shape / alignment outside the bf16 tensor-core kernels");   \
    if (_rc) return _rc;                                                                                \
  } while (0)

}  // namespace b200rl

using namespace b200rl;

extern "C" int64_t b200rl_x3_ws_bytes(int op, int32_t M, int32_t N, int32_t K, const b200rl_conv_geom* g, int x_u8) {
  if (op < B200RL_X3_LINEAR_FWD || op > B200RL_X3_CONV_DGRAD) return -1;
  if (op >= B200RL_X3_CONV_FWD) {
    if (!g || x_u8 < 0 || x_u8 > 2 || (x_u8 ? check_geom_frames(g) : check_geom(g)) || (x_u8 && op == B200RL_X3_CONV_DGRAD)) return -1;
    if (x_u8 && (x_u8 == 2 || rows_cp(g->C) != g->C) && !rows_geom(*g)) return -1;
    if (x_u8) {
      b200rl_conv_geom gp = filter_geom(*g);
      const Plan p = plan_of(op, M, N, K, &gp, x_u8);
      return p.path == PATH_FFMA && rows_cp(g->C) != g->C ? -1 : p.total();
    }
  } else if (M < 1 || N < 1 || K < 1) {
    return -1;
  }
  return plan_of(op, M, N, K, g, x_u8).total();
}

extern "C" int b200rl_linear_fwd_x3(int32_t M, int32_t N, int32_t K, const float* x, int32_t ldx, const float* w,
                                    const float* bias, float* y, int32_t ldy, int act, void* ws, int64_t wsb, void* stream) {
  B200RL_REQUIRE(x && w && y && M >= 1 && N >= 1 && K >= 1 && ldx >= K && ldy >= N, "bad argument");
  const Plan p = plan_of(B200RL_X3_LINEAR_FWD, M, N, K, nullptr, 0);
  if (int rc = check_ws(p, ws, wsb)) return rc;
  if (p.path == PATH_FFMA) return b200rl_linear_fwd(M, N, K, x, ldx, w, bias, y, ldy, act, 0, ws, p.tail, stream);
  cudaStream_t s = as_stream(stream);
  const int Kp = rup(K, 8);
  Carve c(ws);
  bf16* xa = c.take<bf16>(p.a);
  bf16* wb = c.take<bf16>(p.b);
  const SplitJob jb = col_job(w, K, N, K, Kp, 6, PAT_B, wb);
  if (int rc = launch_split(col_job(x, ldx, M, K, Kp, 6, PAT_A, xa), &jb, s)) return rc;
  X3_GEMM(h_linear_fwd(M, N, 6 * Kp, xa, 6 * Kp, wb, bias, y, ldy, act, 0, c.p, p.tail, s));
  return B200RL_OK;
}

extern "C" int b200rl_linear_dgrad_x3(int32_t M, int32_t N, int32_t K, const float* dy, int32_t lddy, const float* w, float* dx,
                                      int32_t lddx, const float* mask_y, int mask_act, void* ws, int64_t wsb, void* stream) {
  B200RL_REQUIRE(dy && w && dx && M >= 1 && N >= 1 && K >= 1 && lddy >= N && lddx >= K, "bad argument");
  const Plan p = plan_of(B200RL_X3_LINEAR_DGRAD, M, N, K, nullptr, 0);
  if (int rc = check_ws(p, ws, wsb)) return rc;
  if (p.path == PATH_FFMA) return b200rl_linear_dgrad(M, N, K, dy, lddy, w, dx, lddx, mask_y, mask_act, 0, ws, p.tail, stream);
  cudaStream_t s = as_stream(stream);
  const int Np = rup(N, 8);
  Carve c(ws);
  bf16* da = c.take<bf16>(p.a);
  bf16* wb = c.take<bf16>(p.b);
  const SplitJob jb = row_job(w, K, N, K, Np, 6, PAT_B, wb);
  if (int rc = launch_split(col_job(dy, lddy, M, N, Np, 6, PAT_A, da), &jb, s)) return rc;
  X3_GEMM(h_linear_dgrad(M, 6 * Np, K, da, 6 * Np, wb, dx, lddx, mask_y, lddx, mask_act, 0, 0, c.p, p.tail, s));
  return B200RL_OK;
}

extern "C" int b200rl_linear_wgrad_x3(int32_t M, int32_t N, int32_t K, const float* dy, int32_t lddy, const float* x, int32_t ldx,
                                      float* dw, float* db, void* ws, int64_t wsb, void* stream) {
  B200RL_REQUIRE(dy && x && dw && M >= 1 && N >= 1 && K >= 1 && lddy >= N && ldx >= K, "bad argument");
  const Plan p = plan_of(B200RL_X3_LINEAR_WGRAD, M, N, K, nullptr, 0);
  if (int rc = check_ws(p, ws, wsb)) return rc;
  if (p.path == PATH_FFMA) return b200rl_linear_wgrad(M, N, K, dy, lddy, x, ldx, dw, db, 0, ws, p.tail, stream);
  cudaStream_t s = as_stream(stream);
  Carve c(ws);
  bf16* da = c.take<bf16>(p.a);
  bf16* xb = c.take<bf16>(p.b);
  const SplitJob jb = row_job(x, ldx, M, K, M, 6, PAT_B, xb);
  if (int rc = launch_split(row_job(dy, lddy, M, N, M, 6, PAT_A, da), &jb, s)) return rc;
  X3_GEMM(h_linear_wgrad(6 * M, N, K, da, N, xb, K, dw, nullptr, c.p, p.tail, s));
  if (db) return launch_colsum(M, N, dy, lddy, db, c.p, p.tail, s);
  return B200RL_OK;
}

static int conv_args(const b200rl_conv_geom* g, const void* x, int x_u8) {
  B200RL_REQUIRE(x_u8 >= 0 && x_u8 <= 2, "x_u8 must be 0 (fp32 NHWC), 1 (uint8 frames) or 2 (the bf16 row image)");
  if (int rc = x_u8 ? check_geom_frames(g) : check_geom(g)) return rc;
  B200RL_REQUIRE(!x_u8 || (x_u8 == 1 && rows_cp(g->C) == g->C) || rows_geom(*g),
                 "frames of C = %d channels need the row-image geometry (kw * Cp = 32, 64 or 128 with Cp = 4, 8 or 16; Cout 32 / 64)", g->C);
  return check_conv_ptr(x, x_u8 == 1, "conv input x");
}

extern "C" int b200rl_conv2d_fwd_x3(const void* x, int x_u8, const float* w, const float* bias, float* y, const b200rl_conv_geom* g_in,
                                    int act, void* ws, int64_t wsb, void* stream) {
  B200RL_REQUIRE(x && w && y, "null argument");
  if (int rc = conv_args(g_in, x, x_u8)) return rc;
  const b200rl_conv_geom gf = x_u8 ? filter_geom(*g_in) : *g_in, *g = &gf;   // the filter's geometry
  const Plan p = plan_of(B200RL_X3_CONV_FWD, 0, 0, 0, g, x_u8);
  if (int rc = check_ws(p, ws, wsb)) return rc;
  B200RL_REQUIRE(p.path != PATH_FFMA || g->C == g_in->C, "frames of C = %d channels: batch too large for the row-image path", g_in->C);
  if (p.path == PATH_FFMA) return b200rl_conv2d_fwd(x, x_u8, w, bias, y, g, act, 0, ws, p.tail, stream);
  cudaStream_t s = as_stream(stream);
  const int taps = g->kh * g->kw, Kw = taps * g->C;
  Carve c(ws);
  bf16* xa = c.take<bf16>(p.a);
  bf16* wb = c.take<bf16>(p.b);
  bf16* img = c.take<bf16>(p.img);
  float* slabs = c.take<float>(p.slabs);
  if (p.path == PATH_STACK) {
    // conv1 on frames: the integer row image is exact in bf16; one raw launch per filter plane, then the combine
    const int64_t Mo = (int64_t)g->B * g->OH * g->OW;
    if (int rc = launch_split(row_job(w, Kw, g->Cout, Kw, g->Cout, 3, PAT_HML, wb), nullptr, s)) return rc;
    const bf16* rows = (const bf16*)x;
    if (x_u8 == 1) {
      X3_GEMM(h_rows_from_u8((const uint8_t*)x, *g_in, img, p.img, s));
      rows = img;
    }
    for (int k = 0; k < 3; ++k)
      X3_GEMM(h_conv_fwd_rows_raw(rows, wb + (int64_t)k * g->Cout * Kw, slabs + k * Mo * g->Cout, *g, c.p, p.tail, s));
    const int blocks = (int)std::min<int64_t>(ceil_div<int64_t>(Mo * g->Cout, 256), kNumSMs * 16);
    x3_combine_kernel<<<blocks, 256, 0, s>>>(slabs, 3, (int)Mo, g->Cout, y, g->Cout, bias, act, 1.0f / 255.0f);
    B200RL_LAUNCH_OK();
    return B200RL_OK;
  }
  const int Cp = rup(g->C, 32);
  const SplitJob jb = col_job(w, g->C, g->Cout * taps, g->C, Cp, 6, PAT_B, wb);
  if (int rc = launch_split(col_job((const float*)x, g->C, g->B * g->H * g->W, g->C, Cp, 6, PAT_A, xa), &jb, s)) return rc;
  b200rl_conv_geom g6 = *g;
  g6.C = 6 * Cp;
  X3_GEMM(h_conv_fwd(xa, wb, bias, y, g6, act, 0, c.p, p.tail, s));
  return B200RL_OK;
}

extern "C" int b200rl_conv2d_wgrad_x3(const void* x, int x_u8, const float* dy, float* dw, float* db, const b200rl_conv_geom* g_in,
                                      void* ws, int64_t wsb, void* stream) {
  B200RL_REQUIRE(x && dy && dw, "null argument");
  if (int rc = conv_args(g_in, x, x_u8)) return rc;
  const b200rl_conv_geom gf = x_u8 ? filter_geom(*g_in) : *g_in, *g = &gf;   // the filter's geometry
  const Plan p = plan_of(B200RL_X3_CONV_WGRAD, 0, 0, 0, g, x_u8);
  if (int rc = check_ws(p, ws, wsb)) return rc;
  B200RL_REQUIRE(p.path != PATH_FFMA || g->C == g_in->C, "frames of C = %d channels: batch too large for the row-image path", g_in->C);
  if (p.path == PATH_FFMA) return b200rl_conv2d_wgrad(x, x_u8, dy, dw, db, g, 0, ws, p.tail, stream);
  cudaStream_t s = as_stream(stream);
  const int64_t Mo = (int64_t)g->B * g->OH * g->OW;
  const int per_img = g->OH * g->OW * g->Cout;
  Carve c(ws);
  bf16* da = c.take<bf16>(p.a);
  bf16* xb = c.take<bf16>(p.b);
  bf16* img = c.take<bf16>(p.img);
  if (x_u8) {
    // the exact row image three times along the batch against dy's hi / mid / lo planes
    const int64_t ib = p.img / 3;
    if (int rc = launch_split(row_job(dy, per_img, g->B, per_img, g->B, 3, PAT_HML, da), nullptr, s)) return rc;
    const void* src = x;
    if (x_u8 == 1) {
      X3_GEMM(h_rows_from_u8((const uint8_t*)x, *g_in, img, ib, s));
      src = img;
    }
    for (int k = src == img ? 1 : 0; k < 3; ++k)
      B200RL_CUDA_OK(cudaMemcpyAsync((char*)img + k * ib, src, ib, cudaMemcpyDeviceToDevice, s));
    b200rl_conv_geom g3 = *g;
    g3.B = 3 * g->B;
    X3_GEMM(h_conv_wgrad_rows(img, da, dw, nullptr, g3, c.p, p.tail, s));
  } else {
    const int in_img = g->H * g->W * g->C;
    const SplitJob jb = row_job(dy, per_img, g->B, per_img, g->B, 6, PAT_B, xb);
    if (int rc = launch_split(row_job((const float*)x, in_img, g->B, in_img, g->B, 6, PAT_A, da), &jb, s)) return rc;
    b200rl_conv_geom g6 = *g;
    g6.B = 6 * g->B;
    X3_GEMM(h_conv_wgrad(da, xb, dw, nullptr, g6, c.p, p.tail, s));
  }
  if (db) return launch_colsum((int)Mo, g->Cout, dy, g->Cout, db, c.p, p.tail, s);
  return B200RL_OK;
}

extern "C" int b200rl_conv2d_dgrad_x3(const float* dy, const float* w, float* dx, const b200rl_conv_geom* g, const float* mask_y,
                                      int mask_act, void* ws, int64_t wsb, void* stream) {
  B200RL_REQUIRE(dy && w && dx, "null argument");
  if (int rc = check_geom(g)) return rc;
  if (int rc = check_conv_ptr(dy, 0, "conv dgrad dy")) return rc;
  if (int rc = check_conv_ptr(w, 0, "conv dgrad w")) return rc;
  const Plan p = plan_of(B200RL_X3_CONV_DGRAD, 0, 0, 0, g, 0);
  if (int rc = check_ws(p, ws, wsb)) return rc;
  if (p.path == PATH_FFMA) return b200rl_conv2d_dgrad(dy, w, dx, g, mask_y, mask_act, 0, ws, p.tail, stream);
  cudaStream_t s = as_stream(stream);
  const int Cp = rup(g->Cout, 32), Kw = g->kh * g->kw * g->C;
  Carve c(ws);
  bf16* da = c.take<bf16>(p.a);
  bf16* wb = c.take<bf16>(p.b);
  const SplitJob jb = row_job(w, Kw, g->Cout, Kw, Cp, 6, PAT_B, wb);
  if (int rc = launch_split(col_job(dy, g->Cout, g->B * g->OH * g->OW, g->Cout, Cp, 6, PAT_A, da), &jb, s)) return rc;
  b200rl_conv_geom g6 = *g;
  g6.Cout = 6 * Cp;
  X3_GEMM(h_conv_dgrad(da, wb, dx, g6, mask_y, mask_act, 0, 0, s));
  return B200RL_OK;
}
