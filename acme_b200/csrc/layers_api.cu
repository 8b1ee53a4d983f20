// C-ABI entry points of K6: dispatch on `precision`.
//   0  fp32 FFMA path (gemm_simt.cu): the 1e-5 parity mode
//   1  tensor cores: the TMA-fed tf32 tcgen05 kernels (gemm_tma.cu) when the operands satisfy TMA's rules, else the
//      loader-fed bf16 tcgen05 kernel (gemm_tc.cu); dense layers too small to amortise a tensor-core pipeline take
//      the (exact) fp32 path.  Results never come from a less precise path than the one asked for, and a
//      precision / shape no path implements is an error.
#include <cuda_bf16.h>

#include "common.cuh"

namespace b200rl {
int simt_linear_fwd(int M, int N, int K, const float* x, int ldx, const float* w, const float* bias, float* y,
                    int ldy, int act, void* ws, int64_t wsb, cudaStream_t s);
int simt_linear_dgrad(int M, int N, int K, const float* dy, int lddy, const float* w, float* dx, int lddx,
                      const float* mask, int ldmask, int mask_act, void* ws, int64_t wsb, cudaStream_t s);
int simt_linear_wgrad(int M, int N, int K, const float* dy, int lddy, const float* x, int ldx, float* dw, float* db,
                      void* ws, int64_t wsb, cudaStream_t s);
int simt_conv_fwd(const void* x, int x_u8, const float* w, const float* bias, float* y, const b200rl_conv_geom& g,
                  int act, void* ws, int64_t wsb, cudaStream_t s);
int simt_conv_wgrad(const void* x, int x_u8, const float* dy, float* dw, float* db, const b200rl_conv_geom& g,
                    void* ws, int64_t wsb, cudaStream_t s);
int simt_conv_dgrad(const float* dy, const float* w, float* dx, const b200rl_conv_geom& g, const float* mask,
                    int mask_act, void* ws, int64_t wsb, cudaStream_t s);
int tc_linear_fwd(int M, int N, int K, const float* x, int ldx, const float* w, const float* bias, float* y,
                  int ldy, int act, void* ws, int64_t wsb, cudaStream_t s);
int tc_linear_dgrad(int M, int N, int K, const float* dy, int lddy, const float* w, float* dx, int lddx,
                    const float* mask, int ldmask, int mask_act, void* ws, int64_t wsb, cudaStream_t s);
int tc_linear_wgrad(int M, int N, int K, const float* dy, int lddy, const float* x, int ldx, float* dw, float* db,
                    void* ws, int64_t wsb, cudaStream_t s);
int tc_conv_fwd(const void* x, int x_u8, const float* w, const float* bias, float* y, const b200rl_conv_geom& g,
                int act, void* ws, int64_t wsb, cudaStream_t s);
int tc_conv_wgrad(const void* x, int x_u8, const float* dy, float* dw, float* db, const b200rl_conv_geom& g,
                  void* ws, int64_t wsb, cudaStream_t s);
int tc_conv_dgrad(const float* dy, const float* w, float* dx, const b200rl_conv_geom& g, const float* mask,
                  int mask_act, void* ws, int64_t wsb, cudaStream_t s);
// gemm_tma.cu: return 1 = shapes not eligible for TMA (fall back to the accessor-fed kernel)
int tma_linear_fwd(int M, int N, int K, const float* x, int ldx, const float* w, const float* bias, float* y,
                   int ldy, int act, void* ws, int64_t wsb, cudaStream_t s);
int tma_linear_dgrad(int M, int N, int K, const float* dy, int lddy, const float* w, float* dx, int lddx,
                     const float* mask, int ldmask, int mask_act, void* ws, int64_t wsb, cudaStream_t s);
int tma_linear_wgrad(int M, int N, int K, const float* dy, int lddy, const float* x, int ldx, float* dw, float* db,
                     void* ws, int64_t wsb, cudaStream_t s);
int tma_conv_fwd(const float* x, const float* w, const float* bias, float* y, const b200rl_conv_geom& g, int act,
                 void* ws, int64_t wsb, cudaStream_t s);
int tma_conv_wgrad(const float* x, const float* dy, float* dw, float* db, const b200rl_conv_geom& g, void* ws, int64_t wsb,
                   cudaStream_t s);
int tma_conv_dgrad(const float* dy, const float* w, float* dx, const b200rl_conv_geom& g, const float* mask, int mask_act,
                   void* ws, int64_t wsb, cudaStream_t s);
int tma_conv_fwd_u8(const uint8_t* x, const float* w, const float* bias, float* y, const b200rl_conv_geom& g, int act,
                    void* ws, int64_t wsb, cudaStream_t s);
int tma_conv_wgrad_u8(const uint8_t* x, const float* dy, float* dw, float* db, const b200rl_conv_geom& g, void* ws, int64_t wsb,
                      cudaStream_t s);
int64_t tma_rows_bytes(const b200rl_conv_geom& g);
int tma_rows_from_u8(const uint8_t* x, const b200rl_conv_geom& g, float* rows, int64_t bytes, cudaStream_t s);
int tma_conv_fwd_rows(const float* rows, const float* w, const float* bias, float* y, const b200rl_conv_geom& g, int act,
                      void* ws, int64_t wsb, cudaStream_t s);
int tma_conv_wgrad_rows(const float* rows, const float* dy, float* dw, float* db, const b200rl_conv_geom& g, void* ws,
                        int64_t wsb, cudaStream_t s);
// gemm_bf16.cu (bf16 dataflow): return 1 = shapes outside what the kernels cover (reported as an error: no fallback)
int h_linear_fwd(int M, int N, int K, const __nv_bfloat16* x, int ldx, const __nv_bfloat16* w, const float* bias, void* y, int ldy,
                 int act, int out_bf16, void* ws, int64_t wsb, cudaStream_t s);
int h_linear_dgrad(int M, int N, int K, const __nv_bfloat16* dy, int lddy, const __nv_bfloat16* w, void* dx, int lddx,
                   const void* mask, int ldmask, int mask_act, int out_bf16, int mask_bf16, void* ws, int64_t wsb, cudaStream_t s);
int h_linear_wgrad(int M, int N, int K, const __nv_bfloat16* dy, int lddy, const __nv_bfloat16* x, int ldx, float* dw, float* db,
                   void* ws, int64_t wsb, cudaStream_t s);
int h_conv_fwd(const __nv_bfloat16* x, const __nv_bfloat16* w, const float* bias, void* y, const b200rl_conv_geom& g, int act,
               int out_bf16, void* ws, int64_t wsb, cudaStream_t s);
int h_conv_wgrad(const __nv_bfloat16* x, const __nv_bfloat16* dy, float* dw, float* db, const b200rl_conv_geom& g, void* ws,
                 int64_t wsb, cudaStream_t s);
int h_conv_dgrad(const __nv_bfloat16* dy, const __nv_bfloat16* w, void* dx, const b200rl_conv_geom& g, const void* mask,
                 int mask_act, int out_bf16, int mask_bf16, cudaStream_t s);
int64_t h_rows_bytes(const b200rl_conv_geom& g);
int h_rows_from_u8(const uint8_t* x, const b200rl_conv_geom& g, __nv_bfloat16* rows, int64_t bytes, cudaStream_t s);
int h_conv_fwd_rows(const __nv_bfloat16* rows, const __nv_bfloat16* w, const float* bias, void* y, const b200rl_conv_geom& g,
                    int act, int out_bf16, void* ws, int64_t wsb, cudaStream_t s);
int h_conv_wgrad_rows(const __nv_bfloat16* rows, const __nv_bfloat16* dy, float* dw, float* db, const b200rl_conv_geom& g,
                      void* ws, int64_t wsb, cudaStream_t s);
int rows_cp(int C);
int h_f32_to_bf16(int64_t n, const float* src, __nv_bfloat16* dst, cudaStream_t s);
int launch_colsum_bf16(int M, int N, const __nv_bfloat16* x, int ld, float* out, void* ws, int64_t ws_bytes, cudaStream_t stream);
}  // namespace b200rl

using namespace b200rl;

static bool g_use_tma = true;
// Dense layers below ~0.13 GFLOP (the 256-wide D4PG / bsuite MLPs at batch 256): the tensor-core pipelines' set-up
// latency exceeds the whole FFMA GEMM, which is also exact -- measured 0.45 ms vs 0.64 ms per D4PG step.
static inline int small_dense(int precision, int M, int N, int K) {
  return (precision == 1 && (long long)M * N * K < (1ll << 26)) ? 0 : precision;
}
extern "C" int b200rl_debug_set_tma(int on) { g_use_tma = on != 0; return 0; }

// shared with the fp32x3.cu entry points
namespace b200rl {
int check_geom(const b200rl_conv_geom* g) {
  B200RL_REQUIRE(g, "null geometry");
  B200RL_REQUIRE(g->B >= 1 && g->H >= 1 && g->W >= 1 && g->C >= 1 && g->Cout >= 1, "bad conv shape");
  B200RL_REQUIRE(g->kh >= 1 && g->kw >= 1 && g->stride >= 1 && g->OH >= 1 && g->OW >= 1, "bad conv filter");
  B200RL_REQUIRE(g->C % 4 == 0 && g->Cout % 4 == 0, "channel counts must be multiples of 4");
  B200RL_REQUIRE((int64_t)g->B * g->H * g->W < (1ll << 31) && (int64_t)g->B * g->OH * g->OW < (1ll << 31), "too many pixels");
  return B200RL_OK;
}
// the first layer's input on the row-image paths (uint8 frames or their bf16 row image): any C in [1, 16]
int check_geom_frames(const b200rl_conv_geom* g) {
  B200RL_REQUIRE(g, "null geometry");
  B200RL_REQUIRE(g->C >= 1 && g->C <= 16, "frames must have 1 to 16 channels (C = %d)", g->C);
  b200rl_conv_geom g4 = *g;
  g4.C = 4;
  return check_geom(&g4);
}
// The convolution loaders of every precision read an fp32 activation / gradient / filter as float4 (im2col of x; dy and
// w of the data gradient) and a uint8 frame as one 4-byte pixel (C % 4 == 0), with no alignment test on the device.
// A misaligned pointer is therefore rejected here, before anything is launched.
int check_conv_ptr(const void* p, int u8, const char* what) {
  B200RL_REQUIRE(((uintptr_t)p & (u8 ? 3 : 15)) == 0, "%s must be %d-byte aligned", what, u8 ? 4 : 16);
  return B200RL_OK;
}
}  // namespace b200rl

#define PRECISION_SWITCH(simt_call, tc_call)                                                   \
  if (precision == 0) return simt_call;                                                        \
  if (precision == 1) return tc_call;                                                          \
  set_error("unknown precision %d (0 = fp32 SIMT, 1 = bf16 tcgen05)", precision);             \
  return B200RL_EINVAL;

extern "C" int b200rl_conv2d_fwd(const void* x, int x_u8, const float* w, const float* bias, float* y,
                                 const b200rl_conv_geom* g, int act, int precision, void* ws, int64_t wsb, void* stream) {
  B200RL_REQUIRE(x && w && y, "null argument");
  if (int rc = check_geom(g)) return rc;
  if (int rc = check_conv_ptr(x, x_u8 == 1, "conv input x")) return rc;
  if (x_u8 == 2) {   // a row image from b200rl_conv2d_rows_from_u8
    B200RL_REQUIRE(precision == 1, "row images are a tensor-core-mode input");
    int rc = tma_conv_fwd_rows((const float*)x, w, bias, y, *g, act, ws, wsb, as_stream(stream));
    B200RL_REQUIRE(rc != 1, "geometry / alignment not supported for a row-image convolution");
    return rc;
  }
  if (precision == 1 && g_use_tma) {
    int rc = x_u8 ? tma_conv_fwd_u8((const uint8_t*)x, w, bias, y, *g, act, ws, wsb, as_stream(stream))
                  : tma_conv_fwd((const float*)x, w, bias, y, *g, act, ws, wsb, as_stream(stream));
    if (rc != 1) return rc;
  }
  PRECISION_SWITCH(simt_conv_fwd(x, x_u8, w, bias, y, *g, act, ws, wsb, as_stream(stream)),
                   tc_conv_fwd(x, x_u8, w, bias, y, *g, act, ws, wsb, as_stream(stream)));
}
extern "C" int b200rl_conv2d_wgrad(const void* x, int x_u8, const float* dy, float* dw, float* db,
                                   const b200rl_conv_geom* g, int precision, void* ws, int64_t wsb, void* stream) {
  B200RL_REQUIRE(x && dy && dw, "null argument");
  if (int rc = check_geom(g)) return rc;
  if (int rc = check_conv_ptr(x, x_u8 == 1, "conv input x")) return rc;
  if (x_u8 == 2) {
    B200RL_REQUIRE(precision == 1, "row images are a tensor-core-mode input");
    int rc = tma_conv_wgrad_rows((const float*)x, dy, dw, db, *g, ws, wsb, as_stream(stream));
    B200RL_REQUIRE(rc != 1, "geometry / alignment not supported for a row-image weight gradient");
    return rc;
  }
  if (precision == 1 && g_use_tma) {
    int rc = x_u8 ? tma_conv_wgrad_u8((const uint8_t*)x, dy, dw, db, *g, ws, wsb, as_stream(stream))
                  : tma_conv_wgrad((const float*)x, dy, dw, db, *g, ws, wsb, as_stream(stream));
    if (rc != 1) return rc;
  }
  PRECISION_SWITCH(simt_conv_wgrad(x, x_u8, dy, dw, db, *g, ws, wsb, as_stream(stream)),
                   tc_conv_wgrad(x, x_u8, dy, dw, db, *g, ws, wsb, as_stream(stream)));
}
extern "C" int64_t b200rl_conv2d_rows_bytes(const b200rl_conv_geom* g) {
  if (!g || check_geom(g)) return 0;
  return tma_rows_bytes(*g);
}
extern "C" int b200rl_conv2d_rows_from_u8(const void* x_u8, const b200rl_conv_geom* g, float* rows, int64_t rows_bytes,
                                          void* stream) {
  B200RL_REQUIRE(x_u8 && rows, "null argument");
  if (int rc = check_geom(g)) return rc;
  if (int rc = check_conv_ptr(x_u8, 1, "uint8 frames")) return rc;
  int rc = tma_rows_from_u8((const uint8_t*)x_u8, *g, rows, rows_bytes, as_stream(stream));
  B200RL_REQUIRE(rc != 1, "geometry not eligible for a row image, buffer too small or not 128-byte aligned");
  return rc;
}

// one thread per 4-byte word of the padded pixels: word q of pixel p holds channels 4q .. 4q+3
__global__ void __launch_bounds__(256)
frames_pad_u8_kernel(const uint8_t* __restrict__ x, uint32_t* __restrict__ out, int64_t words, int C, int Cp) {
  const int wpp = Cp >> 2;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < words; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t p = i / wpp;
    const int c0 = (int)(i - p * wpp) * 4;
    const uint8_t* src = x + p * C;
    uint32_t v = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (c0 + j < C) v |= (uint32_t)__ldg(src + c0 + j) << (8 * j);
    out[i] = v;
  }
}
extern "C" int b200rl_frames_pad_u8(const void* x_u8, int64_t npix, int32_t C, int32_t Cp, void* out, void* stream) {
  B200RL_REQUIRE(x_u8 && out && npix >= 0, "bad argument");
  B200RL_REQUIRE(C >= 1 && C <= Cp && Cp <= 16 && Cp % 4 == 0, "need 1 <= C <= Cp <= 16 and Cp %% 4 == 0 (C = %d, Cp = %d)", C, Cp);
  if (int rc = check_conv_ptr(out, 1, "padded frames")) return rc;
  const int64_t words = npix * (Cp / 4);
  if (words == 0) return B200RL_OK;
  const int blocks = (int)std::min<int64_t>(ceil_div<int64_t>(words, 256), 148 * 16);
  frames_pad_u8_kernel<<<blocks, 256, 0, as_stream(stream)>>>((const uint8_t*)x_u8, (uint32_t*)out, words, C, Cp);
  B200RL_LAUNCH_OK();
  return B200RL_OK;
}

extern "C" int b200rl_conv2d_dgrad(const float* dy, const float* w, float* dx, const b200rl_conv_geom* g,
                                   const float* mask_y, int mask_act, int precision, void* ws, int64_t wsb, void* stream) {
  B200RL_REQUIRE(dy && w && dx, "null argument");
  if (int rc = check_geom(g)) return rc;
  if (int rc = check_conv_ptr(dy, 0, "conv dgrad dy")) return rc;
  if (int rc = check_conv_ptr(w, 0, "conv dgrad w")) return rc;
  if (precision == 1 && g_use_tma) {
    int rc = tma_conv_dgrad(dy, w, dx, *g, mask_y, mask_act, ws, wsb, as_stream(stream));
    if (rc != 1) return rc;
  }
  B200RL_REQUIRE(precision != 1 || (g->Cout % 8 == 0 && g->C % 8 == 0), "bf16 conv dgrad needs C %% 8 == 0 and Cout %% 8 == 0");
  PRECISION_SWITCH(simt_conv_dgrad(dy, w, dx, *g, mask_y, mask_act, ws, wsb, as_stream(stream)),
                   tc_conv_dgrad(dy, w, dx, *g, mask_y, mask_act, ws, wsb, as_stream(stream)));
}
extern "C" int b200rl_linear_fwd(int32_t M, int32_t N, int32_t K, const float* x, int32_t ldx, const float* w,
                                 const float* bias, float* y, int32_t ldy, int act, int precision, void* ws,
                                 int64_t wsb, void* stream) {
  precision = small_dense(precision, M, N, K);
  B200RL_REQUIRE(x && w && y && M >= 1 && N >= 1 && K >= 1 && ldx >= K && ldy >= N, "bad argument");
  if (precision == 1 && g_use_tma) {
    int rc = tma_linear_fwd(M, N, K, x, ldx, w, bias, y, ldy, act, ws, wsb, as_stream(stream));
    if (rc != 1) return rc;
  }
  PRECISION_SWITCH(simt_linear_fwd(M, N, K, x, ldx, w, bias, y, ldy, act, ws, wsb, as_stream(stream)),
                   tc_linear_fwd(M, N, K, x, ldx, w, bias, y, ldy, act, ws, wsb, as_stream(stream)));
}
extern "C" int b200rl_linear_dgrad(int32_t M, int32_t N, int32_t K, const float* dy, int32_t lddy, const float* w,
                                   float* dx, int32_t lddx, const float* mask_y, int mask_act, int precision,
                                   void* ws, int64_t wsb, void* stream) {
  precision = small_dense(precision, M, N, K);
  B200RL_REQUIRE(dy && w && dx && M >= 1 && N >= 1 && K >= 1 && lddy >= N && lddx >= K, "bad argument");
  if (precision == 1 && g_use_tma && (!mask_y || (((uintptr_t)mask_y | (uintptr_t)dx) & 15) == 0)) {
    int rc = tma_linear_dgrad(M, N, K, dy, lddy, w, dx, lddx, mask_y, lddx, mask_act, ws, wsb, as_stream(stream));
    if (rc != 1) return rc;
  }
  PRECISION_SWITCH(simt_linear_dgrad(M, N, K, dy, lddy, w, dx, lddx, mask_y, lddx, mask_act, ws, wsb, as_stream(stream)),
                   tc_linear_dgrad(M, N, K, dy, lddy, w, dx, lddx, mask_y, lddx, mask_act, ws, wsb, as_stream(stream)));
}
extern "C" int b200rl_linear_wgrad(int32_t M, int32_t N, int32_t K, const float* dy, int32_t lddy, const float* x,
                                   int32_t ldx, float* dw, float* db, int precision, void* ws, int64_t wsb, void* stream) {
  precision = small_dense(precision, M, N, K);
  B200RL_REQUIRE(dy && x && dw && M >= 1 && N >= 1 && K >= 1 && lddy >= N && ldx >= K, "bad argument");
  if (precision == 1 && g_use_tma) {
    int rc = tma_linear_wgrad(M, N, K, dy, lddy, x, ldx, dw, db, ws, wsb, as_stream(stream));
    if (rc != 1) return rc;
  }
  PRECISION_SWITCH(simt_linear_wgrad(M, N, K, dy, lddy, x, ldx, dw, db, ws, wsb, as_stream(stream)),
                   tc_linear_wgrad(M, N, K, dy, lddy, x, ldx, dw, db, ws, wsb, as_stream(stream)));
}
extern "C" int64_t b200rl_workspace_bytes(int64_t max_out_elems) { return 64 * max_out_elems * 4; }


// ------------------------------------------------------------------------------ bf16 dataflow (precision 2)
#define H_CALL(expr, what)                                                                                  \
  do {                                                                                                      \
    int _rc = (expr);                                                                                       \
    if (_rc == 1) {                                                                                         \
      set_error("%s: shape / alignment outside the bf16 tensor-core kernels (there is no fallback)", what); \
      return B200RL_EINVAL;                                                                                 \
    }                                                                                                       \
    return _rc;                                                                                             \
  } while (0)
typedef __nv_bfloat16 bf16_t;

extern "C" int b200rl_bf16_from_f32(int64_t n, const float* src, void* dst_bf16, void* stream) {
  B200RL_REQUIRE(src && dst_bf16 && n >= 0, "bad argument");
  if (n == 0) return B200RL_OK;
  H_CALL(h_f32_to_bf16(n, src, (bf16_t*)dst_bf16, as_stream(stream)), "bf16_from_f32 (n % 8 == 0, 16-byte aligned)");
}
extern "C" int64_t b200rl_conv2d_rows_bf16_bytes(const b200rl_conv_geom* g) {
  if (!g || check_geom_frames(g)) return 0;
  return h_rows_bytes(*g);
}
extern "C" int b200rl_conv2d_rows_bf16_from_u8(const void* x_u8, const b200rl_conv_geom* g, void* rows, int64_t rows_bytes,
                                               void* stream) {
  B200RL_REQUIRE(x_u8 && rows, "null argument");
  if (int rc = check_geom_frames(g)) return rc;
  H_CALL(h_rows_from_u8((const uint8_t*)x_u8, *g, (bf16_t*)rows, rows_bytes, as_stream(stream)), "bf16 row image");
}
extern "C" int b200rl_conv2d_fwd_bf16(const void* x, int x_rows, const void* w, const float* bias, void* y, int y_bf16,
                                      const b200rl_conv_geom* g, int act, void* ws, int64_t wsb, void* stream) {
  B200RL_REQUIRE(x && w && y, "null argument");
  if (int rc = x_rows ? check_geom_frames(g) : check_geom(g)) return rc;
  if (x_rows)
    H_CALL(h_conv_fwd_rows((const bf16_t*)x, (const bf16_t*)w, bias, y, *g, act, y_bf16, ws, wsb, as_stream(stream)), "conv2d_fwd_bf16(rows)");
  H_CALL(h_conv_fwd((const bf16_t*)x, (const bf16_t*)w, bias, y, *g, act, y_bf16, ws, wsb, as_stream(stream)), "conv2d_fwd_bf16");
}
extern "C" int b200rl_conv2d_wgrad_bf16(const void* x, int x_rows, const void* dy, float* dw, float* db, const b200rl_conv_geom* g,
                                        void* ws, int64_t wsb, void* stream) {
  B200RL_REQUIRE(x && dy && dw && ws, "null argument");
  if (int rc = x_rows ? check_geom_frames(g) : check_geom(g)) return rc;
  if (x_rows)
    H_CALL(h_conv_wgrad_rows((const bf16_t*)x, (const bf16_t*)dy, dw, db, *g, ws, wsb, as_stream(stream)), "conv2d_wgrad_bf16(rows)");
  H_CALL(h_conv_wgrad((const bf16_t*)x, (const bf16_t*)dy, dw, db, *g, ws, wsb, as_stream(stream)), "conv2d_wgrad_bf16");
}
extern "C" int b200rl_conv2d_dgrad_bf16(const void* dy, const void* w, void* dx, int dx_bf16, const b200rl_conv_geom* g,
                                        const void* mask_y, int mask_bf16, int mask_act, void* stream) {
  B200RL_REQUIRE(dy && w && dx, "null argument");
  if (int rc = check_geom(g)) return rc;
  H_CALL(h_conv_dgrad((const bf16_t*)dy, (const bf16_t*)w, dx, *g, mask_y, mask_act, dx_bf16, mask_bf16, as_stream(stream)),
         "conv2d_dgrad_bf16");
}
extern "C" int b200rl_linear_fwd_bf16(int32_t M, int32_t N, int32_t K, const void* x, int32_t ldx, const void* w, const float* bias,
                                      void* y, int32_t ldy, int y_bf16, int act, void* ws, int64_t wsb, void* stream) {
  B200RL_REQUIRE(x && w && y && M >= 1 && N >= 1 && K >= 1 && ldx >= K && ldy >= N, "bad argument");
  H_CALL(h_linear_fwd(M, N, K, (const bf16_t*)x, ldx, (const bf16_t*)w, bias, y, ldy, act, y_bf16, ws, wsb, as_stream(stream)),
         "linear_fwd_bf16");
}
extern "C" int b200rl_linear_dgrad_bf16(int32_t M, int32_t N, int32_t K, const void* dy, int32_t lddy, const void* w, void* dx,
                                        int32_t lddx, int dx_bf16, const void* mask_y, int mask_bf16, int mask_act, void* ws,
                                        int64_t wsb, void* stream) {
  B200RL_REQUIRE(dy && w && dx && M >= 1 && N >= 1 && K >= 1 && lddy >= N && lddx >= K, "bad argument");
  H_CALL(h_linear_dgrad(M, N, K, (const bf16_t*)dy, lddy, (const bf16_t*)w, dx, lddx, mask_y, lddx, mask_act, dx_bf16, mask_bf16, ws,
                        wsb, as_stream(stream)),
         "linear_dgrad_bf16");
}
extern "C" int b200rl_linear_wgrad_bf16(int32_t M, int32_t N, int32_t K, const void* dy, int32_t lddy, const void* x, int32_t ldx,
                                        float* dw, float* db, void* ws, int64_t wsb, void* stream) {
  B200RL_REQUIRE(dy && x && dw && ws && M >= 1 && N >= 1 && K >= 1 && lddy >= N && ldx >= K, "bad argument");
  H_CALL(h_linear_wgrad(M, N, K, (const bf16_t*)dy, lddy, (const bf16_t*)x, ldx, dw, db, ws, wsb, as_stream(stream)),
         "linear_wgrad_bf16");
}

/* out[n] = sum_m x[m, n] over bf16 rows: a layer's bias gradient on its own stream (the wgrad calls above do it in-line
 * when db != NULL) */
extern "C" int b200rl_colsum_bf16(int32_t M, int32_t N, const void* x_bf16, int32_t ld, float* out, void* ws, int64_t wsb,
                                  void* stream) {
  B200RL_REQUIRE(x_bf16 && out && ws && M >= 1 && N >= 1 && ld >= N, "bad argument");
  return launch_colsum_bf16(M, N, (const bf16_t*)x_bf16, ld, out, ws, wsb, as_stream(stream));
}
