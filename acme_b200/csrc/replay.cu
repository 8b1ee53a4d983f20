// Replay shard runtime: HBM ring of observation slots + ring of items + sum tree, the pinned
// staging that feeds it, and K3 (gather + n-step build).
//
// Stands in for the Reverb table/writer/sampler the reference builds at
// acme/agents/tf/dqn/agent.py:95-116 and drives from acme/adders/reverb/{base,transition}.py.
// The host half of this file is the native counterpart of Reverb's C++ table bookkeeping (FIFO
// remover, key allocation, writer history); the arithmetic lives in the kernels.
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstring>
#include <cstdlib>
#include <deque>
#include <mutex>
#include <vector>

#include <cuda_bf16.h>

#include "common.cuh"

namespace b200rl {
int h_rows_layout(const b200rl_conv_geom& g, int* Hp, int* row_elems);   // gemm_bf16.cu
int h_rows_write(const uint8_t* x, const b200rl_conv_geom& g, __nv_bfloat16* rows, cudaStream_t s);

static thread_local std::string g_last_error;
static unsigned long long g_launches = 0;
void count_launch() { __atomic_add_fetch(&g_launches, 1, __ATOMIC_RELAXED); }
static int g_pdl_override = -1;   // b200rl_debug_set_pdl: 0 / 1 for the launches that follow, -1 = the environment's choice
bool pdl_enabled() {
  static const bool on = getenv("B200RL_PDL") ? atoi(getenv("B200RL_PDL")) != 0 : B200RL_PDL_DEFAULT;
  return g_pdl_override < 0 ? on : g_pdl_override != 0;
}
bool pdl_small_enabled() {
  static const bool on = getenv("B200RL_PDL_SMALL") ? atoi(getenv("B200RL_PDL_SMALL")) != 0 : false;
  return on;
}
int pdl_late_mode() {
  static const int late = getenv("B200RL_PDL_LATE") ? atoi(getenv("B200RL_PDL_LATE")) : B200RL_PDL_LATE_DEFAULT;
  return late;
}

void set_error(const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_last_error = buf;
}

// from sumtree.cu
int tree_staged_levels(const TreeView& t, int64_t budget_bytes);
int tree_sample(const TreeView& t, const ReplayState* st_dev, int64_t M, int B, const float* u, const int64_t* philox_counter,
                uint64_t philox_seed, float* u_out, int stratified, int shard_count, const float* denom_dev, int64_t* idx,
                uint64_t* keys, float* prob, cudaStream_t stream, int* staged_out);
int tree_rebuild(const TreeView& t, cudaStream_t stream);
int tree_scatter_positions(const TreeView& t, int64_t M, int n, const int64_t* pos_dev,
                           const float* w_dev, const ReplayState* st_dev, unsigned long long* stamp,
                           unsigned long long* epoch_dev, cudaStream_t stream);
int tree_scatter_keys(const TreeView& t, int64_t M, int n, const uint64_t* keys_dev,
                      const float* prio_dev, double alpha, const ReplayState* st_dev,
                      unsigned long long* stamp, unsigned long long* epoch_dev, cudaStream_t stream);

// ------------------------------------------------------------------------------ device side
struct SlotFill {   // scalars of one finished step, scattered into the slot arrays at flush
  int32_t slot;
  int32_t next;
  float rew;
  float disc;
};
constexpr int kMaxFrameStack = 8;
struct ItemRec {    // one new item (len > 0) or a tree-only update (len == 0, e.g. eviction)
  int64_t pos;
  int32_t start;
  int32_t end;
  int32_t len;
  float weight;
  // frame-deduplicated rings: slots of the F-1 observations before `start` / before `end` in the same episode, nearest
  // first; -1 = before the episode's first observation (the frame stacker's blank frames)
  int32_t prev[2][kMaxFrameStack - 1];
};

struct RingView {
  uint8_t* obs;
  uint8_t* act;
  float* rew;
  float* disc;
  int32_t* next;
  int32_t* item_start;
  int32_t* item_end;
  int32_t* item_len;
  int64_t obs_stride;
  int32_t obs_bytes;      // bytes of one observation as the table's signature (and a gathered batch row) has it
  int32_t act_stride;
  int32_t act_bytes;
  float gamma;
  // frame deduplication (SURVEY §8f-1): observations are stacks of F single-byte-element frames on their LAST axis
  // (acme/wrappers/frame_stacking.py:64-88); a slot stores only the newest frame (slot_bytes = obs_bytes / F) and
  // item_prev holds, per item, the slots of the older frames of its two observations
  int32_t frame_stack;    // F (1 = off)
  int32_t slot_bytes;
  int32_t* item_prev;     // [M][2][F - 1]
};

__global__ void scatter_fills_kernel(RingView r, const SlotFill* __restrict__ fills,
                                     const uint8_t* __restrict__ acts, int n) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  SlotFill f = fills[i];
  r.rew[f.slot] = f.rew;
  r.disc[f.slot] = f.disc;
  r.next[f.slot] = f.next;
  const uint8_t* src = acts + (size_t)i * r.act_stride;
  uint8_t* dst = r.act + (size_t)f.slot * r.act_stride;
  for (int b = 0; b < r.act_bytes; ++b) dst[b] = src[b];
}

// The staged item records arrive in one blob behind the new key range (item_head / item_tail): thread 0 publishes the
// range (K1 / K2 read it from `state_dst`, after this kernel in stream order), the others scatter the item records.
__global__ void scatter_items_kernel(RingView r, const ItemRec* __restrict__ recs, int n,
                                     long long* __restrict__ pos_out, float* __restrict__ w_out,
                                     const ReplayState* __restrict__ state_src, ReplayState* __restrict__ state_dst) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i == 0 && state_src) *state_dst = *state_src;
  if (i >= n) return;
  ItemRec it = recs[i];
  if (it.len > 0) {
    r.item_start[it.pos] = it.start;
    r.item_end[it.pos] = it.end;
    r.item_len[it.pos] = it.len;
    if (r.frame_stack > 1) {
      const int fm = r.frame_stack - 1;
      for (int w = 0; w < 2; ++w)
        for (int j = 0; j < fm; ++j) r.item_prev[((size_t)it.pos * 2 + w) * fm + j] = it.prev[w][j];
    }
  }
  pos_out[i] = it.pos;
  w_out[i] = it.weight;
}

// K3.  grid = (B, 2): y = 0 copies o_tm1 (+ action, n-step R/D by thread 0), y = 1 copies o_t.
// Observation rows are moved with 16-byte vectors (ring rows are 16-byte aligned; batch rows are
// when obs_bytes % 16 == 0, otherwise the 4-byte or byte path is taken).
template <int VEC>
__global__ void __launch_bounds__(256)
gather_kernel(RingView r, const long long* __restrict__ idx, uint8_t* __restrict__ o_tm1,
              uint8_t* __restrict__ a_tm1, float* __restrict__ R, float* __restrict__ D,
              uint8_t* __restrict__ o_t) {
  pdl_launch_dependents();
  pdl_wait();                  // K1's indices
  const int b = blockIdx.x;
  const long long pos = idx[b];
  const int which = blockIdx.y;
  const int slot = which == 0 ? r.item_start[pos] : r.item_end[pos];
  const uint8_t* src = r.obs + (size_t)slot * r.obs_stride;
  uint8_t* dst = (which == 0 ? o_tm1 : o_t) + (size_t)b * r.obs_bytes;
  if (VEC == 16) {
    const int4* s4 = reinterpret_cast<const int4*>(src);
    int4* d4 = reinterpret_cast<int4*>(dst);
    const int nv = r.obs_bytes >> 4;
    // 4 independent 16-byte loads in flight per thread before the stores
    int i = threadIdx.x;
    for (; i + 3 * 256 < nv; i += 4 * 256) {
      int4 v0 = __ldg(s4 + i), v1 = __ldg(s4 + i + 256), v2 = __ldg(s4 + i + 512), v3 = __ldg(s4 + i + 768);
      d4[i] = v0; d4[i + 256] = v1; d4[i + 512] = v2; d4[i + 768] = v3;
    }
    for (; i < nv; i += 256) d4[i] = __ldg(s4 + i);
  } else if (VEC == 4) {
    const int* s1 = reinterpret_cast<const int*>(src);
    int* d1 = reinterpret_cast<int*>(dst);
    for (int i = threadIdx.x; i < (r.obs_bytes >> 2); i += 256) d1[i] = __ldg(s1 + i);
  } else {
    for (int i = threadIdx.x; i < r.obs_bytes; i += 256) dst[i] = src[i];
  }
  if (which == 0) {
    const uint8_t* as = r.act + (size_t)slot * r.act_stride;
    uint8_t* ad = a_tm1 + (size_t)b * r.act_bytes;
    for (int i = threadIdx.x; i < r.act_bytes; i += 256) ad[i] = as[i];
    if (threadIdx.x == 0) {
      // acme/adders/reverb/transition.py:135-145, fp32, every op rounded separately (no FMA)
      int cur = slot;
      const int len = r.item_len[pos];
      float Rv = r.rew[cur], Dv = r.disc[cur];
      cur = r.next[cur];
      for (int j = 1; j < len; ++j) {
        Dv = __fmul_rn(Dv, r.gamma);
        Rv = __fadd_rn(Rv, __fmul_rn(r.rew[cur], Dv));
        Dv = __fmul_rn(Dv, r.disc[cur]);
        cur = r.next[cur];
      }
      R[b] = Rv;
      D[b] = Dv;
    }
  }
}

// K3 with the first layer's input fused in: besides the uint8 batch rows the kernel writes the frames straight into the
// zero-padded bf16 ROW IMAGE that conv1 reads through TMA (gemm_bf16.cu: integer pixel values, exact in bf16; padding
// stays zero from allocation), so no separate conversion pass runs between replay and the network.
// Frames are [H][W][4] uint8; one 16-byte vector = 4 pixels x 4 channels -> 16 bf16 = two 16-byte stores.
__global__ void __launch_bounds__(256)
gather_rows_kernel(RingView r, const long long* __restrict__ idx, uint8_t* __restrict__ o_tm1, uint8_t* __restrict__ a_tm1,
                   float* __restrict__ R, float* __restrict__ D, uint8_t* __restrict__ o_t, uint4* __restrict__ rows_tm1,
                   uint4* __restrict__ rows_t, int W4 /* 16-byte vectors per image row */, int pad_left, int pad_top, int Hp,
                   int row_v16 /* 16-byte units per padded row */) {
  pdl_launch_dependents();
  pdl_wait();                  // K1's indices
  const int b = blockIdx.x;
  const long long pos = idx[b];
  const int which = blockIdx.y;
  const int slot = which == 0 ? r.item_start[pos] : r.item_end[pos];
  const int4* s4 = reinterpret_cast<const int4*>(r.obs + (size_t)slot * r.obs_stride);
  int4* d4 = reinterpret_cast<int4*>((which == 0 ? o_tm1 : o_t) + (size_t)b * r.obs_bytes);
  uint4* rows = (which == 0 ? rows_tm1 : rows_t) + (size_t)b * Hp * row_v16;
  const int nv = r.obs_bytes >> 4;
  // gridDim.z CTAs share a frame (a frame is only 1764 vectors: one CTA per frame leaves the stores latency-bound)
  for (int i = blockIdx.z * 256 + threadIdx.x; i < nv; i += 256 * gridDim.z) {
    const int4 v = __ldg(s4 + i);
    d4[i] = v;
    const int y = i / W4, xv = i - y * W4;
    const uint32_t px[4] = {(uint32_t)v.x, (uint32_t)v.y, (uint32_t)v.z, (uint32_t)v.w};
    uint32_t o[8];
#pragma unroll
    for (int p = 0; p < 4; ++p) {
      const __nv_bfloat162 lo = __floats2bfloat162_rn((float)(px[p] & 0xffu), (float)((px[p] >> 8) & 0xffu));
      const __nv_bfloat162 hi = __floats2bfloat162_rn((float)((px[p] >> 16) & 0xffu), (float)(px[p] >> 24));
      o[2 * p] = *reinterpret_cast<const uint32_t*>(&lo);
      o[2 * p + 1] = *reinterpret_cast<const uint32_t*>(&hi);
    }
    // pixel x = 4 xv sits at bf16 element (x + pad_left) * 4 of the padded row = 16-byte unit (x + pad_left) / 2
    uint4* dst = rows + (size_t)(y + pad_top) * row_v16 + ((4 * xv + pad_left) >> 1);
    dst[0] = make_uint4(o[0], o[1], o[2], o[3]);
    dst[1] = make_uint4(o[4], o[5], o[6], o[7]);
  }
  if (which == 0 && blockIdx.z == 0) {
    const uint8_t* as = r.act + (size_t)slot * r.act_stride;
    uint8_t* ad = a_tm1 + (size_t)b * r.act_bytes;
    for (int i = threadIdx.x; i < r.act_bytes; i += 256) ad[i] = as[i];
    if (threadIdx.x == 0) {
      // acme/adders/reverb/transition.py:135-145, fp32, every op rounded separately (no FMA)
      int cur = slot;
      const int len = r.item_len[pos];
      float Rv = r.rew[cur], Dv = r.disc[cur];
      cur = r.next[cur];
      for (int j = 1; j < len; ++j) {
        Dv = __fmul_rn(Dv, r.gamma);
        Rv = __fadd_rn(Rv, __fmul_rn(r.rew[cur], Dv));
        Dv = __fmul_rn(Dv, r.disc[cur]);
        cur = r.next[cur];
      }
      R[b] = Rv;
      D[b] = Dv;
    }
  }
}

// K3 on a frame-deduplicated ring: a stack [H*W][F] is rebuilt from F single frames (the item's own slot = newest
// frame = channel F-1, item_prev = the older ones, missing ones read as zero: FrameStacker's blank frames).  F = 4,
// uint8: thread i loads bytes [4i, 4i+4) of each frame (coalesced), transposes 4x4 bytes and stores 16 bytes = 4 pixels
// x 4 channels of the batch row; with ROWS it also writes conv1's bf16 row image like gather_rows_kernel.
template <bool ROWS>
__global__ void __launch_bounds__(256)
gather_frames4_kernel(RingView r, const long long* __restrict__ idx, uint8_t* __restrict__ o_tm1, uint8_t* __restrict__ a_tm1,
                      float* __restrict__ R, float* __restrict__ D, uint8_t* __restrict__ o_t, uint4* __restrict__ rows_tm1,
                      uint4* __restrict__ rows_t, int W4, int pad_left, int pad_top, int Hp, int row_v16) {
  const int b = blockIdx.x;
  const long long pos = idx[b];
  const int which = blockIdx.y;
  const int slot = which == 0 ? r.item_start[pos] : r.item_end[pos];
  const int32_t* pv = r.item_prev + ((size_t)pos * 2 + which) * 3;
  const uint32_t* f[4];   // channel c = frame of observation k - (3 - c)
  f[3] = reinterpret_cast<const uint32_t*>(r.obs + (size_t)slot * r.obs_stride);
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    const int ps = pv[j];
    f[2 - j] = ps >= 0 ? reinterpret_cast<const uint32_t*>(r.obs + (size_t)ps * r.obs_stride) : nullptr;
  }
  int4* d4 = reinterpret_cast<int4*>((which == 0 ? o_tm1 : o_t) + (size_t)b * r.obs_bytes);
  uint4* rows = ROWS ? (which == 0 ? rows_tm1 : rows_t) + (size_t)b * Hp * row_v16 : nullptr;
  const int nv = r.obs_bytes >> 4;
  for (int i = blockIdx.z * 256 + threadIdx.x; i < nv; i += 256 * gridDim.z) {
    uint32_t w[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) w[c] = f[c] ? __ldg(f[c] + i) : 0u;
    uint32_t px[4];   // pixel p of the vector: bytes (w0.p, w1.p, w2.p, w3.p)
#pragma unroll
    for (int p = 0; p < 4; ++p)
      px[p] = ((w[0] >> (8 * p)) & 0xffu) | (((w[1] >> (8 * p)) & 0xffu) << 8) | (((w[2] >> (8 * p)) & 0xffu) << 16) |
              (((w[3] >> (8 * p)) & 0xffu) << 24);
    d4[i] = make_int4((int)px[0], (int)px[1], (int)px[2], (int)px[3]);
    if (ROWS) {
      const int y = i / W4, xv = i - y * W4;
      uint32_t o[8];
#pragma unroll
      for (int p = 0; p < 4; ++p) {
        const __nv_bfloat162 lo = __floats2bfloat162_rn((float)(px[p] & 0xffu), (float)((px[p] >> 8) & 0xffu));
        const __nv_bfloat162 hi = __floats2bfloat162_rn((float)((px[p] >> 16) & 0xffu), (float)(px[p] >> 24));
        o[2 * p] = *reinterpret_cast<const uint32_t*>(&lo);
        o[2 * p + 1] = *reinterpret_cast<const uint32_t*>(&hi);
      }
      uint4* dst = rows + (size_t)(y + pad_top) * row_v16 + ((4 * xv + pad_left) >> 1);
      dst[0] = make_uint4(o[0], o[1], o[2], o[3]);
      dst[1] = make_uint4(o[4], o[5], o[6], o[7]);
    }
  }
  if (which == 0 && blockIdx.z == 0) {
    const uint8_t* as = r.act + (size_t)slot * r.act_stride;
    uint8_t* ad = a_tm1 + (size_t)b * r.act_bytes;
    for (int i = threadIdx.x; i < r.act_bytes; i += 256) ad[i] = as[i];
    if (threadIdx.x == 0) {
      // acme/adders/reverb/transition.py:135-145, fp32, every op rounded separately (no FMA)
      int cur = slot;
      const int len = r.item_len[pos];
      float Rv = r.rew[cur], Dv = r.disc[cur];
      cur = r.next[cur];
      for (int j = 1; j < len; ++j) {
        Dv = __fmul_rn(Dv, r.gamma);
        Rv = __fadd_rn(Rv, __fmul_rn(r.rew[cur], Dv));
        Dv = __fmul_rn(Dv, r.disc[cur]);
        cur = r.next[cur];
      }
      R[b] = Rv;
      D[b] = Dv;
    }
  }
}

// K3 for SEQUENCE items (SURVEY §8f-3; `acme/adders/reverb/sequence.py:77-127`): an item is T consecutive steps of one
// episode, each a full (observation, action [+ extras], reward, discount) row -- the final step of an episode and the
// zero padding after it are ordinary slots whose action / reward / discount bytes are zero.  grid = (T, B): CTA (t, b)
// copies step t of sampled item b.  A writer's slots are consecutive in the ring unless other writers interleaved, so
// step t normally sits at (start + t) mod S (recognised by end - start == len); otherwise thread 0 walks t links.
// Steps beyond the item's own length (never produced by SequenceAdder, possible with hand-made items) read as zeros.
// time_major = 1 writes [T][B] rows (`tf2_utils.batch_to_sequence`, r2d2/learning.py:115), 0 writes [B][T] rows.
template <int VEC>
__global__ void __launch_bounds__(128)
gather_seq_kernel(RingView r, const long long* __restrict__ idx, int T, int B, long long S, int time_major,
                  uint8_t* __restrict__ obs_out, uint8_t* __restrict__ act_out, float* __restrict__ rew_out,
                  float* __restrict__ disc_out) {
  const int t = blockIdx.x, b = blockIdx.y;
  const long long pos = idx[b];
  const int start = r.item_start[pos], end = r.item_end[pos], len = r.item_len[pos];
  const size_t row = time_major ? (size_t)t * B + b : (size_t)b * T + t;
  uint8_t* dst = obs_out + row * r.obs_bytes;
  uint8_t* ad = act_out + row * r.act_bytes;
  if (t >= len) {   // block-uniform
    for (int i = threadIdx.x; i < r.obs_bytes; i += 128) dst[i] = 0;
    for (int i = threadIdx.x; i < r.act_bytes; i += 128) ad[i] = 0;
    if (threadIdx.x == 0) { rew_out[row] = 0.f; disc_out[row] = 0.f; }
    return;
  }
  __shared__ int s_slot;
  long long gap = (long long)end - start;
  if (gap < 0) gap += S;
  int slot;
  if (gap == len) {   // block-uniform
    const long long sl = (long long)start + t;
    slot = (int)(sl >= S ? sl - S : sl);
  } else {
    if (threadIdx.x == 0) {
      int cur = start;
      for (int j = 0; j < t; ++j) cur = r.next[cur];
      s_slot = cur;
    }
    __syncthreads();
    slot = s_slot;
  }
  const uint8_t* src = r.obs + (size_t)slot * r.obs_stride;
  if (VEC == 16) {
    const int4* s4 = reinterpret_cast<const int4*>(src);
    int4* d4 = reinterpret_cast<int4*>(dst);
    const int nv = r.obs_bytes >> 4;
    int i = threadIdx.x;
    for (; i + 3 * 128 < nv; i += 4 * 128) {
      int4 v0 = __ldg(s4 + i), v1 = __ldg(s4 + i + 128), v2 = __ldg(s4 + i + 256), v3 = __ldg(s4 + i + 384);
      d4[i] = v0; d4[i + 128] = v1; d4[i + 256] = v2; d4[i + 384] = v3;
    }
    for (; i < nv; i += 128) d4[i] = __ldg(s4 + i);
  } else if (VEC == 4) {
    const int* s1 = reinterpret_cast<const int*>(src);
    int* d1 = reinterpret_cast<int*>(dst);
    for (int i = threadIdx.x; i < (r.obs_bytes >> 2); i += 128) d1[i] = __ldg(s1 + i);
  } else {
    for (int i = threadIdx.x; i < r.obs_bytes; i += 128) dst[i] = src[i];
  }
  const uint8_t* as = r.act + (size_t)slot * r.act_stride;
  for (int i = threadIdx.x; i < r.act_bytes; i += 128) ad[i] = as[i];
  if (threadIdx.x == 0) { rew_out[row] = r.rew[slot]; disc_out[row] = r.disc[slot]; }
}

// device observations that arrive as full stacks [n][frame_bytes][F]: keep the newest frame (last axis index F-1)
__global__ void extract_newest_frame_kernel(const uint8_t* __restrict__ stacks, uint8_t* __restrict__ ring, long long first_slot,
                                            long long S, long long obs_stride, int frame_bytes, int F, long long n) {
  const long long total = n * frame_bytes;
  long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (; e < total; e += stride) {
    const long long j = e / frame_bytes;
    const int i = (int)(e - j * frame_bytes);
    ring[((first_slot + j) % S) * obs_stride + i] = stacks[(j * frame_bytes + i) * (long long)F + (F - 1)];
  }
}

__global__ void fill_float_kernel(float* p, long long n, float v) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long stride = (long long)gridDim.x * blockDim.x;
  for (; i < n; i += stride) p[i] = v;
}

}  // namespace b200rl

// ------------------------------------------------------------------------------ host side
using namespace b200rl;

struct Writer {
  std::deque<uint64_t> hist;  // slot seqs of this episode, newest (the open slot) last
  bool in_use = false;
  int64_t k = 0;              // steps appended in the current episode
  bool has_pending = false;   // stream form: act/rew/disc of the open slot wait for the next obs
  std::vector<uint8_t> pending_act;
  float pending_rew = 0.f, pending_disc = 0.f;
};

struct Stage {   // one pinned staging set + its device mirror; two sets alternate
  uint8_t* h_obs = nullptr;
  SlotFill* h_fill = nullptr;
  uint8_t* h_act = nullptr;
  uint8_t* h_blob = nullptr;     // [ReplayState, padded to one ItemRec | stage_items x ItemRec]: one H2D copy per flush
  uint8_t* d_blob = nullptr;
  ItemRec* h_item = nullptr;     // = h_blob + sizeof(ItemRec)
  ReplayState* h_state = nullptr;   // = h_blob
  SlotFill* d_fill = nullptr;
  uint8_t* d_act = nullptr;
  ItemRec* d_item = nullptr;
  long long* d_pos = nullptr;
  float* d_w = nullptr;
  cudaEvent_t done = nullptr;
  bool in_flight = false;
};

struct b200rl_replay {
  b200rl_replay_cfg cfg;
  int64_t M = 0, S = 0;
  int64_t obs_stride = 0;
  int32_t act_stride = 0;
  int32_t F = 1;              // frame_stack (1 = off)
  int32_t slot_bytes = 0;     // bytes stored per observation slot: obs_bytes, or one frame when F > 1
  RingView ring{};
  float* d_tree = nullptr;
  int64_t tree_floats = 0;
  TreeView tree{};
  unsigned long long* d_stamp = nullptr;
  unsigned long long* d_epoch = nullptr;
  ReplayState* d_state = nullptr;
  int staged_levels = 0;

  uint64_t slot_head = 0, item_head = 0, item_tail = 0;
  std::vector<uint64_t> item_start_seq;
  // Sliding-window minimum of the live items' first-slot sequence numbers, as (key, start) with increasing start.
  // With one writer the starts are monotone in key order and this holds one entry; with interleaved writers a slow
  // writer can create an item whose window begins long before the tail item's, and the slot ring must not overwrite it.
  std::deque<std::pair<uint64_t, uint64_t>> start_min;
  std::vector<Writer> writers;

  Stage stage[2];
  int cur = 0;
  int64_t stage_slots = 0, stage_items = 0;
  int64_t n_obs = 0, n_fill = 0, n_item = 0;
  uint64_t obs_first_seq = 0;
  bool state_dirty = false;
  // Split flush (b200rl_replay_flush): the bulk of an insert -- observation rows H2D, per-slot scalars -- goes on an
  // internal stream and overlaps whatever the caller's stream is still running (the previous learner step); only the
  // item records, the key range and the tree insert, which must not race with sampling / priority updates, are ordered
  // on the caller's stream.  Not used when this flush evicts live items from the slot ring (their slots may still be
  // read by work in flight) or for implicit flushes.
  cudaStream_t payload_stream = nullptr;
  cudaEvent_t payload_done = nullptr;
  bool async_payload = true;
  bool stage_has_eviction = false;
  cudaStream_t last_flush_stream = nullptr;  // flushes on different streams are chained by event
  cudaEvent_t last_flush_event = nullptr;
  // Host bookkeeping (staging sets, writer histories, key counters) is shared by actor threads that append and the
  // learner thread that flushes / samples; ctypes drops the GIL during calls, so every entry point takes this lock
  // (Reverb's table is thread-safe too: acme runs actors and learner against one server).
  std::recursive_mutex mu;
  const float* global_mass_dev = nullptr;   // sum of all shards' masses (caller-owned device float), or NULL
};
#define B200RL_LOCK(h) std::lock_guard<std::recursive_mutex> _guard((h)->mu)

static int64_t round_up(int64_t x, int64_t m) { return (x + m - 1) / m * m; }

static int ensure_device(b200rl_replay* h) {
  B200RL_CUDA_OK(cudaSetDevice(h->cfg.device));
  return B200RL_OK;
}

extern "C" int b200rl_version(void) { return B200RL_VERSION; }
extern "C" int b200rl_debug_set_pdl(int on) { b200rl::g_pdl_override = on; return 0; }
extern "C" uint64_t b200rl_launch_count(void) { return __atomic_load_n(&g_launches, __ATOMIC_RELAXED); }
extern "C" const char* b200rl_last_error(void) { return g_last_error.c_str(); }

extern "C" int b200rl_device_check(int device) {
  cudaDeviceProp prop;
  cudaError_t e = cudaGetDeviceProperties(&prop, device);
  if (e != cudaSuccess) {
    set_error("no usable CUDA device %d: %s (this library has no CPU fallback)", device,
              cudaGetErrorString(e));
    return B200RL_ECUDA;
  }
  if (prop.major != 10) {
    set_error("device %d is sm_%d%d; this library is built for sm_100a (B200) only", device,
              prop.major, prop.minor);
    return B200RL_EARCH;
  }
  return B200RL_OK;
}

static void free_stage(Stage& s) {
  cudaFreeHost(s.h_obs); cudaFreeHost(s.h_fill); cudaFreeHost(s.h_act); cudaFreeHost(s.h_blob);
  cudaFree(s.d_fill); cudaFree(s.d_act); cudaFree(s.d_blob); cudaFree(s.d_pos); cudaFree(s.d_w);
  if (s.done) cudaEventDestroy(s.done);
  s = Stage{};
}

extern "C" int b200rl_replay_destroy(b200rl_replay* h) {
  if (!h) return B200RL_OK;
  cudaSetDevice(h->cfg.device);
  cudaFree(h->ring.obs); cudaFree(h->ring.act); cudaFree(h->ring.rew); cudaFree(h->ring.disc);
  cudaFree(h->ring.next); cudaFree(h->ring.item_start); cudaFree(h->ring.item_end);
  cudaFree(h->ring.item_len); cudaFree(h->ring.item_prev); cudaFree(h->d_tree); cudaFree(h->d_stamp); cudaFree(h->d_epoch);
  cudaFree(h->d_state);
  free_stage(h->stage[0]);
  free_stage(h->stage[1]);
  if (h->payload_stream) cudaStreamDestroy(h->payload_stream);
  if (h->payload_done) cudaEventDestroy(h->payload_done);
  delete h;
  return B200RL_OK;
}

extern "C" int b200rl_replay_create(b200rl_replay** out, const b200rl_replay_cfg* cfg) {
  B200RL_REQUIRE(out && cfg, "null argument");
  B200RL_REQUIRE(cfg->max_items >= 1 && cfg->max_items < (1ll << 31), "max_items out of range");
  B200RL_REQUIRE(cfg->obs_bytes >= 0 && cfg->act_bytes >= 0, "negative payload size");
  B200RL_REQUIRE(cfg->max_window >= 1 && cfg->max_window <= 64, "max_window must be in [1,64]");
  B200RL_REQUIRE(cfg->shard_count >= 1, "shard_count must be >= 1");
  const bool payload = cfg->obs_bytes > 0;
  const int F = cfg->frame_stack > 1 ? cfg->frame_stack : 1;
  B200RL_REQUIRE(F <= kMaxFrameStack, "frame_stack must be <= %d", kMaxFrameStack);
  B200RL_REQUIRE(F == 1 || (payload && cfg->obs_bytes % F == 0), "frame_stack must divide obs_bytes (stacks of single-byte elements)");
  B200RL_REQUIRE(!payload || (cfg->slot_capacity >= cfg->max_window + 1 + F && cfg->slot_capacity < (1ll << 31)),
                 "slot_capacity must be >= max_window + 1 + frame_stack");
  int rc = b200rl_device_check(cfg->device);
  if (rc) return rc;
  B200RL_CUDA_OK(cudaSetDevice(cfg->device));

  b200rl_replay* h = new b200rl_replay();
  h->cfg = *cfg;
  h->M = cfg->max_items;
  h->S = payload ? cfg->slot_capacity : 0;
  h->F = F;
  h->slot_bytes = cfg->obs_bytes / F;
  h->obs_stride = round_up(h->slot_bytes, 16);
  h->act_stride = (int32_t)round_up(std::max(cfg->act_bytes, 1), 4);
  RingView& r = h->ring;
  r.obs_stride = h->obs_stride;
  r.obs_bytes = cfg->obs_bytes;
  r.act_stride = h->act_stride;
  r.act_bytes = cfg->act_bytes;
  r.gamma = cfg->gamma;
  r.frame_stack = F;
  r.slot_bytes = h->slot_bytes;
  r.item_prev = nullptr;

#define ALLOC(ptr, bytes)                                                        \
  do {                                                                           \
    cudaError_t _e = cudaMalloc((void**)&(ptr), (size_t)std::max<int64_t>((bytes), 16)); \
    if (_e != cudaSuccess) {                                                     \
      set_error("cudaMalloc(%lld bytes) failed: %s", (long long)(bytes), cudaGetErrorString(_e)); \
      b200rl_replay_destroy(h);                                                  \
      return B200RL_ECUDA;                                                       \
    }                                                                            \
  } while (0)

  if (payload) {
    ALLOC(r.obs, h->S * h->obs_stride);
    ALLOC(r.act, h->S * (int64_t)h->act_stride);
    ALLOC(r.rew, h->S * 4);
    ALLOC(r.disc, h->S * 4);
    ALLOC(r.next, h->S * 4);
    ALLOC(r.item_start, h->M * 4);
    ALLOC(r.item_end, h->M * 4);
    ALLOC(r.item_len, h->M * 4);
    if (F > 1) {
      ALLOC(r.item_prev, h->M * 2 * (F - 1) * 4);
      cudaMemset(r.item_prev, 0xff, h->M * 2 * (F - 1) * 4);
    }
    cudaMemset(r.next, 0xff, h->S * 4);
    cudaMemset(r.item_len, 0, h->M * 4);
  }
  // tree geometry (oracle/sumtree.py::num_levels / level_width)
  TreeView& t = h->tree;
  int L = 1;
  {
    int64_t span = kFanout;
    while (span < h->M) { span *= kFanout; ++L; }
  }
  B200RL_REQUIRE(L < kMaxLevels, "tree too deep");
  t.L = L;
  int64_t total = 32;  // root padded
  for (int l = 1; l <= L; ++l) {
    int64_t span = 1;
    for (int i = 0; i < L - l; ++i) span *= kFanout;
    t.width[l] = round_up(ceil_div<int64_t>(h->M, span), kFanout);
    total += t.width[l];
  }
  t.width[0] = 1;
  h->tree_floats = 2 * total;   // raw values + prefix lines
  ALLOC(h->d_tree, h->tree_floats * 4);
  cudaMemset(h->d_tree, 0, h->tree_floats * 4);
  {
    float* p = h->d_tree;
    t.lvl[0] = p;
    t.pre[0] = p + total;
    p += 32;
    for (int l = 1; l <= L; ++l) { t.lvl[l] = p; t.pre[l] = p + total; p += t.width[l]; }
  }
  ALLOC(h->d_stamp, t.width[L] * 8);
  cudaMemset(h->d_stamp, 0, t.width[L] * 8);
  ALLOC(h->d_epoch, 8);
  {
    unsigned long long one = 1;
    cudaMemcpy(h->d_epoch, &one, 8, cudaMemcpyHostToDevice);
  }
  ALLOC(h->d_state, sizeof(ReplayState));
  cudaMemset(h->d_state, 0, sizeof(ReplayState));
  h->staged_levels = tree_staged_levels(t, 16 * 1024);

  h->stage_slots = cfg->stage_slots > 0 ? cfg->stage_slots : 256;
  h->stage_items = h->stage_slots * 2 + 2 * cfg->max_window + 8;
  for (int i = 0; i < 2; ++i) {
    Stage& s = h->stage[i];
    bool ok = true;
    if (payload) {
      ok = ok && cudaMallocHost((void**)&s.h_fill, h->stage_slots * sizeof(SlotFill)) == cudaSuccess;
      ok = ok && cudaMallocHost((void**)&s.h_act, h->stage_slots * (size_t)h->act_stride) == cudaSuccess;
      ok = ok && cudaMalloc((void**)&s.d_fill, h->stage_slots * sizeof(SlotFill)) == cudaSuccess;
      ok = ok && cudaMalloc((void**)&s.d_act, h->stage_slots * (size_t)h->act_stride) == cudaSuccess;
    }
    static_assert(sizeof(ReplayState) <= sizeof(ItemRec), "blob header");
    ok = ok && cudaMallocHost((void**)&s.h_blob, (h->stage_items + 1) * sizeof(ItemRec)) == cudaSuccess;
    ok = ok && cudaMalloc((void**)&s.d_blob, (h->stage_items + 1) * sizeof(ItemRec)) == cudaSuccess;
    if (ok) {
      s.h_state = (ReplayState*)s.h_blob;
      s.h_item = (ItemRec*)(s.h_blob + sizeof(ItemRec));
      s.d_item = (ItemRec*)(s.d_blob + sizeof(ItemRec));
    }
    ok = ok && cudaMalloc((void**)&s.d_pos, h->stage_items * 8) == cudaSuccess;
    ok = ok && cudaMalloc((void**)&s.d_w, h->stage_items * 4) == cudaSuccess;
    ok = ok && cudaEventCreateWithFlags(&s.done, cudaEventDisableTiming) == cudaSuccess;
    if (!ok) {
      set_error("staging allocation failed: %s", cudaGetErrorString(cudaGetLastError()));
      b200rl_replay_destroy(h);
      return B200RL_ECUDA;
    }
  }
#undef ALLOC
  if (payload) {
    const char* e = getenv("B200RL_ASYNC_INSERT");
    h->async_payload = !(e && atoi(e) == 0);
    B200RL_CUDA_OK(cudaStreamCreateWithFlags(&h->payload_stream, cudaStreamNonBlocking));
    B200RL_CUDA_OK(cudaEventCreateWithFlags(&h->payload_done, cudaEventDisableTiming));
  }
  B200RL_CUDA_OK(cudaDeviceSynchronize());
  *out = h;
  return B200RL_OK;
}

// ----------------------------------------------------------------------------------- flush
static int flush_impl(b200rl_replay* h, cudaStream_t stream, bool allow_split = false) {
  // Order `stream` after the previous flush even when nothing is staged now: an implicit flush (staging full) runs on
  // g_implicit_stream, and the sample / gather kernels the caller is about to issue on `stream` must see its copies.
  if (h->last_flush_event && h->last_flush_stream != stream) {
    B200RL_CUDA_OK(cudaStreamWaitEvent(stream, h->last_flush_event, 0));
    h->last_flush_stream = stream;   // `stream` is now ordered after that flush: later calls on it need no second wait
  }
  if (h->n_obs == 0 && h->n_fill == 0 && h->n_item == 0 && !h->state_dirty) return B200RL_OK;
  Stage& s = h->stage[h->cur];
  RingView& r = h->ring;
  const bool split = allow_split && h->async_payload && h->payload_stream && !h->stage_has_eviction &&
                     (h->n_obs > 0 || h->n_fill > 0);
  cudaStream_t ps = split ? h->payload_stream : stream;
  if (split && h->last_flush_event)   // payload copies of this flush after the previous flush's (shared device staging)
    B200RL_CUDA_OK(cudaStreamWaitEvent(ps, h->last_flush_event, 0));
  if (h->n_obs > 0) {
    // staged observations occupy consecutive slot sequence numbers -> at most two runs in the ring
    int64_t first = (int64_t)(h->obs_first_seq % (uint64_t)h->S);
    int64_t run0 = std::min<int64_t>(h->n_obs, h->S - first);
    B200RL_CUDA_OK(cudaMemcpy2DAsync(r.obs + first * r.obs_stride, r.obs_stride, s.h_obs, r.slot_bytes,
                                     r.slot_bytes, run0, cudaMemcpyHostToDevice, ps));
    if (run0 < h->n_obs)
      B200RL_CUDA_OK(cudaMemcpy2DAsync(r.obs, r.obs_stride, s.h_obs + run0 * (int64_t)r.slot_bytes,
                                       r.slot_bytes, r.slot_bytes, h->n_obs - run0,
                                       cudaMemcpyHostToDevice, ps));
  }
  if (h->n_fill > 0) {
    B200RL_CUDA_OK(cudaMemcpyAsync(s.d_fill, s.h_fill, h->n_fill * sizeof(SlotFill), cudaMemcpyHostToDevice, ps));
    B200RL_CUDA_OK(cudaMemcpyAsync(s.d_act, s.h_act, h->n_fill * (size_t)r.act_stride, cudaMemcpyHostToDevice, ps));
    scatter_fills_kernel<<<(int)ceil_div<int64_t>(h->n_fill, 128), 128, 0, ps>>>(r, s.d_fill, s.d_act, (int)h->n_fill);
    B200RL_LAUNCH_OK();
  }
  if (split) {
    B200RL_CUDA_OK(cudaEventRecord(h->payload_done, ps));
    B200RL_CUDA_OK(cudaStreamWaitEvent(stream, h->payload_done, 0));
  }
  // the key range and the item records travel in one copy; the range is published BEFORE the tree update so that its
  // kernels see the new tail / head
  s.h_state->item_head = h->item_head;
  s.h_state->item_tail = h->item_tail;
  B200RL_CUDA_OK(cudaMemcpyAsync(s.d_blob, s.h_blob, (size_t)(h->n_item + 1) * sizeof(ItemRec), cudaMemcpyHostToDevice, stream));
  scatter_items_kernel<<<(int)std::max<int64_t>(1, ceil_div<int64_t>(h->n_item, 128)), 128, 0, stream>>>(
      r, s.d_item, (int)h->n_item, s.d_pos, s.d_w, (const ReplayState*)s.d_blob, h->d_state);
  B200RL_LAUNCH_OK();
  if (h->n_item > 0) {
    int rc = tree_scatter_positions(h->tree, h->M, (int)h->n_item, (const int64_t*)s.d_pos, s.d_w,
                                    h->d_state, h->d_stamp, h->d_epoch, stream);
    if (rc) return rc;
  }
  B200RL_CUDA_OK(cudaEventRecord(s.done, stream));
  s.in_flight = true;
  h->last_flush_event = s.done;
  h->last_flush_stream = stream;
  h->n_obs = h->n_fill = h->n_item = 0;
  h->state_dirty = false;
  h->stage_has_eviction = false;
  h->cur ^= 1;
  Stage& nxt = h->stage[h->cur];
  if (nxt.in_flight) {  // the set we are about to overwrite: wait for its copies (2 flushes ago)
    B200RL_CUDA_OK(cudaEventSynchronize(nxt.done));
    nxt.in_flight = false;
  }
  return B200RL_OK;
}

extern "C" int b200rl_replay_flush(b200rl_replay* h, void* stream) {
  B200RL_REQUIRE(h, "null handle");
  B200RL_LOCK(h);
  int rc = ensure_device(h);
  if (rc) return rc;
  return flush_impl(h, as_stream(stream), /*allow_split=*/true);
}

// the stream used by implicit flushes triggered from the host-only writer calls
// (thread-local: b200rl_writer_append_stream redirects it to the caller's stream for the duration of its own call only)
static thread_local cudaStream_t g_implicit_stream = nullptr;

static int stage_tree_only(b200rl_replay* h, int64_t pos, float w) {
  if (h->n_item >= h->stage_items) {
    int rc = flush_impl(h, g_implicit_stream);
    if (rc) return rc;
  }
  ItemRec& it = h->stage[h->cur].h_item[h->n_item++];
  it.pos = pos; it.start = 0; it.end = 0; it.len = 0; it.weight = w;
  return B200RL_OK;
}

// Allocate the next slot; evict items whose first slot is about to be overwritten.
static int alloc_slot(b200rl_replay* h, const void* obs_host, uint64_t* seq_out) {
  // staged observations must fit the ring once around (tiny rings: flush before they lap it)
  if (obs_host && h->n_obs >= std::min<int64_t>(h->stage_slots, h->S)) {
    int rc = flush_impl(h, g_implicit_stream);
    if (rc) return rc;
  }
  if (obs_host && !h->stage[h->cur].h_obs) {  // host-observation staging is allocated on first use
    for (int i = 0; i < 2; ++i)
      B200RL_CUDA_OK(cudaMallocHost((void**)&h->stage[i].h_obs,
                                    (size_t)(h->stage_slots * std::max<int64_t>(h->slot_bytes, 1))));
  }
  uint64_t seq = h->slot_head++;
  if (obs_host) {
    if (h->n_obs == 0) h->obs_first_seq = seq;
    uint8_t* dst = h->stage[h->cur].h_obs + h->n_obs * (int64_t)h->slot_bytes;
    if (h->F == 1) {
      memcpy(dst, obs_host, h->slot_bytes);
    } else {   // the newest frame of the stack: last-axis index F - 1
      const uint8_t* src = (const uint8_t*)obs_host + (h->F - 1);
      const int F = h->F, nb = h->slot_bytes;
      for (int i = 0; i < nb; ++i) dst[i] = src[(size_t)i * F];
    }
    h->n_obs++;
  }
  if (h->slot_head > (uint64_t)h->S) {
    uint64_t floor_seq = h->slot_head - (uint64_t)h->S;
    // FIFO eviction until NO live item starts in a slot that is about to be overwritten (oldest keys go first,
    // like Reverb's Fifo remover, even when the offending item is not the tail)
    while (h->item_tail < h->item_head) {
      while (!h->start_min.empty() && h->start_min.front().first < h->item_tail) h->start_min.pop_front();
      if (h->start_min.empty() || h->start_min.front().second >= floor_seq) break;
      int rc = stage_tree_only(h, (int64_t)(h->item_tail % h->M), 0.f);
      if (rc) return rc;
      h->item_tail++;
      h->state_dirty = true;
      h->stage_has_eviction = true;   // live slots are being recycled: this flush stays on one stream
    }
  }
  *seq_out = seq;
  return B200RL_OK;
}

static int stage_fill(b200rl_replay* h, uint64_t slot_seq, const void* act, float rew, float disc,
                      uint64_t next_seq) {
  if (h->n_fill >= h->stage_slots) {
    int rc = flush_impl(h, g_implicit_stream);
    if (rc) return rc;
  }
  Stage& s = h->stage[h->cur];
  SlotFill& f = s.h_fill[h->n_fill];
  f.slot = (int32_t)(slot_seq % (uint64_t)h->S);
  f.next = (int32_t)(next_seq % (uint64_t)h->S);
  f.rew = rew;
  f.disc = disc;
  uint8_t* a = s.h_act + h->n_fill * (int64_t)h->act_stride;
  memset(a, 0, h->act_stride);
  if (act) memcpy(a, act, h->cfg.act_bytes);
  h->n_fill++;
  return B200RL_OK;
}

static int make_item(b200rl_replay* h, Writer& w, int32_t num_timesteps, double priority, uint64_t* key_out) {
  B200RL_REQUIRE(num_timesteps >= 1 && (int64_t)w.hist.size() >= (int64_t)num_timesteps + 1,
                 "create_item(%d): only %d steps appended in this episode", num_timesteps,
                 (int)w.hist.size() - 1);
  const int64_t i_end = (int64_t)w.hist.size() - 1, i_start = i_end - num_timesteps;
  uint64_t start_seq = w.hist[i_start];
  uint64_t end_seq = w.hist.back();
  // with frame deduplication the item also needs the F-1 slots before its first observation
  const uint64_t oldest_seq = w.hist[std::max<int64_t>(0, i_start - (h->F - 1))];
  B200RL_REQUIRE(h->slot_head <= (uint64_t)h->S || oldest_seq >= h->slot_head - (uint64_t)h->S,
                 "item window was already overwritten in the slot ring (slot_capacity too small)");
  if (h->item_start_seq.empty()) h->item_start_seq.assign(h->M, 0);
  // never stage two records for one tree position (tiny tables): cap the window at M items
  if (h->n_item >= std::min<int64_t>(h->stage_items, h->M)) {
    int rc = flush_impl(h, g_implicit_stream);
    if (rc) return rc;
  }
  uint64_t key = h->item_head++;
  if (h->item_head - h->item_tail > (uint64_t)h->M) h->item_tail++;  // Fifo remover: same tree position
  while (!h->start_min.empty() && h->start_min.front().first < h->item_tail) h->start_min.pop_front();
  int64_t pos = (int64_t)(key % (uint64_t)h->M);
  h->item_start_seq[pos] = oldest_seq;
  while (!h->start_min.empty() && h->start_min.back().second >= oldest_seq) h->start_min.pop_back();
  h->start_min.emplace_back(key, oldest_seq);
  ItemRec& it = h->stage[h->cur].h_item[h->n_item++];
  it.pos = pos;
  it.start = (int32_t)(start_seq % (uint64_t)h->S);
  it.end = (int32_t)(end_seq % (uint64_t)h->S);
  it.len = num_timesteps;
  for (int j = 0; j < kMaxFrameStack - 1; ++j) {
    const int64_t a = i_start - 1 - j, b = i_end - 1 - j;
    it.prev[0][j] = (j < h->F - 1 && a >= 0) ? (int32_t)(w.hist[a] % (uint64_t)h->S) : -1;
    it.prev[1][j] = (j < h->F - 1 && b >= 0) ? (int32_t)(w.hist[b] % (uint64_t)h->S) : -1;
  }
  float wt = (float)std::pow(priority, h->cfg.alpha);
  it.weight = (wt > 0.f && wt < 3.0e38f) ? wt : 0.f;
  h->state_dirty = true;
  if (key_out) *key_out = key;  // keys are shard-local; the owning rank is implied by the handle
  return B200RL_OK;
}

static Writer* get_writer(b200rl_replay* h, int32_t id) {
  if (id < 0 || id >= (int32_t)h->writers.size() || !h->writers[id].in_use) {
    set_error("unknown writer id %d", id);
    return nullptr;
  }
  return &h->writers[id];
}

extern "C" int b200rl_writer_open(b200rl_replay* h, int32_t* writer_id) {
  B200RL_REQUIRE(h && writer_id, "null argument");
  B200RL_LOCK(h);
  B200RL_REQUIRE(h->cfg.obs_bytes > 0, "this replay was created without payload storage");
  for (size_t i = 0; i < h->writers.size(); ++i)
    if (!h->writers[i].in_use) {
      h->writers[i] = Writer();
      h->writers[i].in_use = true;
      *writer_id = (int32_t)i;
      return B200RL_OK;
    }
  h->writers.emplace_back();
  h->writers.back().in_use = true;
  *writer_id = (int32_t)h->writers.size() - 1;
  return B200RL_OK;
}

static void push_hist(b200rl_replay* h, Writer& w, uint64_t seq) {
  w.hist.push_back(seq);
  while ((int64_t)w.hist.size() > h->cfg.max_window + 1 + (h->F - 1)) w.hist.pop_front();
}

extern "C" int b200rl_writer_append(b200rl_replay* h, int32_t writer, const void* obs, const void* act,
                                    float rew, float disc, const void* next_obs) {
  B200RL_REQUIRE(h && next_obs, "null argument");
  B200RL_LOCK(h);
  Writer* w = get_writer(h, writer);
  if (!w) return B200RL_EINVAL;
  int rc = ensure_device(h);
  if (rc) return rc;
  if (w->hist.empty()) {
    B200RL_REQUIRE(obs, "first append of an episode needs the initial observation");
    uint64_t s0;
    rc = alloc_slot(h, obs, &s0);
    if (rc) return rc;
    push_hist(h, *w, s0);
    w->k = 0;
  }
  uint64_t cur = w->hist.back(), nxt;
  rc = alloc_slot(h, next_obs, &nxt);
  if (rc) return rc;
  rc = stage_fill(h, cur, act, rew, disc, nxt);
  if (rc) return rc;
  push_hist(h, *w, nxt);
  w->k++;
  return B200RL_OK;
}

extern "C" int b200rl_writer_create_item(b200rl_replay* h, int32_t writer, int32_t num_timesteps,
                                         double priority, uint64_t* key_out) {
  B200RL_REQUIRE(h, "null handle");
  B200RL_LOCK(h);
  Writer* w = get_writer(h, writer);
  if (!w) return B200RL_EINVAL;
  int rc = ensure_device(h);
  if (rc) return rc;
  return make_item(h, *w, num_timesteps, priority, key_out);
}

extern "C" int b200rl_writer_close(b200rl_replay* h, int32_t writer) {
  B200RL_REQUIRE(h, "null handle");
  B200RL_LOCK(h);
  Writer* w = get_writer(h, writer);
  if (!w) return B200RL_EINVAL;
  w->in_use = false;
  w->hist.clear();
  return B200RL_OK;
}

// Stream insert of `n` timesteps; element i belongs to writer writers[i] (or to `writer` for every element when `writers` is
// NULL).  A writer's elements are consecutive timesteps of its stream in array order.
static int append_stream_impl(b200rl_replay* h, int64_t n, const int32_t* writers, int32_t writer, const void* obs,
                              int obs_on_device, const void* act, const float* rew, const float* disc, const uint8_t* first,
                              const uint8_t* last, int32_t n_step, double priority, cudaStream_t stream) {
  B200RL_REQUIRE(obs && rew && disc && first && last, "null argument");
  B200RL_REQUIRE(n_step >= 1 && n_step <= h->cfg.max_window, "n_step must be in [1, max_window]");
  B200RL_REQUIRE(n >= 0 && n <= h->S, "a stream chunk cannot exceed slot_capacity");
  for (int64_t i = 0; i < (writers ? n : 1); ++i)   // every writer id before any state changes
    if (!get_writer(h, writers ? writers[i] : writer)) return B200RL_EINVAL;
  int rc = ensure_device(h);
  if (rc) return rc;
  // obs_on_device: 0 = host observations as the signature has them; 1 = device observations as the signature has them;
  // 2 = device SINGLE FRAMES [n][obs_bytes / frame_stack] (frame-deduplicated tables: what the ring stores)
  B200RL_REQUIRE(obs_on_device != 2 || h->F > 1, "obs_on_device = 2 (single frames) needs a frame-deduplicated table");
  cudaStream_t saved = g_implicit_stream;
  g_implicit_stream = stream;
  const int32_t ob = h->cfg.obs_bytes;
  if (obs_on_device) {
    // pending host-staged observations must land first (slot order), then one or two D2D runs: element i takes slot
    // slot_head + i, whichever writer it belongs to
    rc = flush_impl(h, stream);
    if (rc) { g_implicit_stream = saved; return rc; }
    int64_t firsti = (int64_t)(h->slot_head % (uint64_t)h->S);
    int64_t run0 = std::min<int64_t>(n, h->S - firsti);
    RingView& r = h->ring;
    if (h->F > 1 && obs_on_device == 1) {
      if (n > 0) {
        const long long total = n * (long long)h->slot_bytes;
        extract_newest_frame_kernel<<<(int)std::min<long long>(ceil_div<long long>(total, 256), kNumSMs * 16), 256, 0, stream>>>(
            (const uint8_t*)obs, r.obs, firsti, h->S, r.obs_stride, h->slot_bytes, h->F, n);
        B200RL_LAUNCH_OK();
      }
    } else {
      const int32_t sb = h->slot_bytes;
      if (run0 > 0)
        B200RL_CUDA_OK(cudaMemcpy2DAsync(r.obs + firsti * r.obs_stride, r.obs_stride, obs, sb, sb, run0,
                                         cudaMemcpyDeviceToDevice, stream));
      if (run0 < n)
        B200RL_CUDA_OK(cudaMemcpy2DAsync(r.obs, r.obs_stride, (const uint8_t*)obs + run0 * (int64_t)sb, sb, sb,
                                         n - run0, cudaMemcpyDeviceToDevice, stream));
    }
  }
  const uint8_t* acts = (const uint8_t*)act;
  for (int64_t i = 0; i < n && rc == 0; ++i) {
    Writer* w = &h->writers[writers ? writers[i] : writer];
    if (first[i]) {  // a FIRST timestep: any unfinished episode of this writer is abandoned
      w->hist.clear();
      w->k = 0;
      w->has_pending = false;
    } else {
      if (w->hist.empty()) {
        set_error("stream element %lld is not FIRST but the writer has no open episode", (long long)i);
        rc = B200RL_EINVAL;
        break;
      }
    }
    uint64_t seq;
    rc = alloc_slot(h, obs_on_device ? nullptr : (const uint8_t*)obs + i * (int64_t)ob, &seq);
    if (rc) break;
    if (!first[i]) {
      rc = stage_fill(h, w->hist.back(), w->pending_act.data(), w->pending_rew, w->pending_disc, seq);
      if (rc) break;
    }
    push_hist(h, *w, seq);
    if (!first[i]) {
      w->k++;
      // NStepTransitionAdder._write after the k-th add: window = whole deque (transition.py:120-124)
      int32_t m = (int32_t)std::min<int64_t>(w->k, n_step);
      rc = make_item(h, *w, m, priority, nullptr);
      if (rc) break;
      if (last[i]) {  // _write_last drain (transition.py:167-172)
        for (int32_t j = 1; j < m && rc == 0; ++j) rc = make_item(h, *w, m - j, priority, nullptr);
        w->hist.clear();
        w->k = 0;
        w->has_pending = false;
        continue;
      }
    }
    if (!last[i]) {
      w->pending_act.assign(h->act_stride, 0);
      if (acts) memcpy(w->pending_act.data(), acts + i * (int64_t)h->cfg.act_bytes, h->cfg.act_bytes);
      w->pending_rew = rew[i];
      w->pending_disc = disc[i];
      w->has_pending = true;
    } else {  // FIRST and LAST at once: a one-observation episode yields nothing
      w->hist.clear();
      w->k = 0;
    }
  }
  if (rc == 0) rc = flush_impl(h, stream);
  g_implicit_stream = saved;
  return rc;
}

extern "C" int b200rl_writer_append_stream(b200rl_replay* h, int32_t writer, int64_t n, const void* obs,
                                           int obs_on_device, const void* act, const float* rew,
                                           const float* disc, const uint8_t* first,
                                           const uint8_t* last, int32_t n_step, double priority,
                                           void* stream_) {
  B200RL_REQUIRE(h, "null argument");
  B200RL_LOCK(h);
  return append_stream_impl(h, n, nullptr, writer, obs, obs_on_device, act, rew, disc, first, last, n_step, priority,
                            as_stream(stream_));
}

extern "C" int b200rl_writer_append_multi(b200rl_replay* h, int64_t n, const int32_t* writers, const void* obs,
                                          int obs_on_device, const void* act, const float* rew, const float* disc,
                                          const uint8_t* first, const uint8_t* last, int32_t n_step, double priority,
                                          void* stream_) {
  B200RL_REQUIRE(h && writers, "null argument");
  B200RL_LOCK(h);
  return append_stream_impl(h, n, writers, -1, obs, obs_on_device, act, rew, disc, first, last, n_step, priority,
                            as_stream(stream_));
}

extern "C" int b200rl_replay_reset(b200rl_replay* h, void* stream_) {
  B200RL_REQUIRE(h, "null handle");
  B200RL_LOCK(h);
  int rc = ensure_device(h);
  if (rc) return rc;
  cudaStream_t stream = as_stream(stream_);
  h->n_obs = h->n_fill = h->n_item = 0;
  h->item_tail = h->item_head;  // every key issued so far is dead
  h->start_min.clear();
  for (auto& w : h->writers) { w.hist.clear(); w.k = 0; w.has_pending = false; }
  B200RL_CUDA_OK(cudaMemsetAsync(h->d_tree, 0, h->tree_floats * 4, stream));
  h->state_dirty = true;
  return flush_impl(h, stream);
}


// ------------------------------------------------------------------------------ checkpoint / resume (SURVEY §8f-4)
// The reference never checkpoints replay contents (acme/tf/savers.py:76-167 saves learner state only); a resumed
// run there starts from an empty table.  Here the whole shard can be saved: its device arrays are exposed one by one
// (the host side copies them with any D2H mechanism) and the host bookkeeping is serialised into one blob.
enum { SEG_OBS = 0, SEG_ACT, SEG_REW, SEG_DISC, SEG_NEXT, SEG_ITEM_START, SEG_ITEM_END, SEG_ITEM_LEN, SEG_TREE, SEG_STATE, SEG_ITEM_PREV, SEG_COUNT };

extern "C" int b200rl_replay_segment(b200rl_replay* h, int32_t which, void** dev_ptr, int64_t* bytes) {
  B200RL_REQUIRE(h && dev_ptr && bytes, "null argument");
  B200RL_LOCK(h);
  const RingView& r = h->ring;
  const bool payload = h->cfg.obs_bytes > 0;
  void* p = nullptr;
  int64_t n = 0;
  switch (which) {
    case SEG_OBS: p = r.obs; n = payload ? h->S * h->obs_stride : 0; break;
    case SEG_ACT: p = r.act; n = payload ? h->S * (int64_t)h->act_stride : 0; break;
    case SEG_REW: p = r.rew; n = payload ? h->S * 4 : 0; break;
    case SEG_DISC: p = r.disc; n = payload ? h->S * 4 : 0; break;
    case SEG_NEXT: p = r.next; n = payload ? h->S * 4 : 0; break;
    case SEG_ITEM_START: p = r.item_start; n = payload ? h->M * 4 : 0; break;
    case SEG_ITEM_END: p = r.item_end; n = payload ? h->M * 4 : 0; break;
    case SEG_ITEM_LEN: p = r.item_len; n = payload ? h->M * 4 : 0; break;
    case SEG_TREE: p = h->d_tree; n = h->tree_floats * 4; break;
    case SEG_STATE: p = h->d_state; n = sizeof(ReplayState); break;
    case SEG_ITEM_PREV: p = r.item_prev; n = h->F > 1 ? h->M * 2 * (h->F - 1) * 4 : 0; break;
    default: set_error("unknown replay segment %d (0..%d)", which, SEG_COUNT - 1); return B200RL_EINVAL;
  }
  *dev_ptr = p;
  *bytes = n;
  return B200RL_OK;
}

namespace {
struct BlobWriter {
  std::vector<uint8_t> b;
  void u64(uint64_t v) { const uint8_t* p = (const uint8_t*)&v; b.insert(b.end(), p, p + 8); }
  void bytes(const void* p, size_t n) { const uint8_t* q = (const uint8_t*)p; b.insert(b.end(), q, q + n); }
};
struct BlobReader {
  const uint8_t* p; size_t n, at = 0; bool ok = true;
  uint64_t u64() { uint64_t v = 0; if (at + 8 > n) { ok = false; return 0; } memcpy(&v, p + at, 8); at += 8; return v; }
  void bytes(void* dst, size_t k) { if (at + k > n) { ok = false; return; } memcpy(dst, p + at, k); at += k; }
};
constexpr uint64_t kBlobMagic = 0x62323030726c7631ull;   // "b200rlv1"
}  // namespace

static void write_host_state(b200rl_replay* h, BlobWriter& w) {
  w.u64(kBlobMagic);
  w.u64((uint64_t)h->M); w.u64((uint64_t)h->S); w.u64((uint64_t)h->cfg.obs_bytes); w.u64((uint64_t)h->cfg.act_bytes);
  w.u64(h->slot_head); w.u64(h->item_head); w.u64(h->item_tail);
  w.u64(h->item_start_seq.size());
  w.bytes(h->item_start_seq.data(), h->item_start_seq.size() * 8);
  w.u64(h->start_min.size());
  for (auto& e : h->start_min) { w.u64(e.first); w.u64(e.second); }
  w.u64(h->writers.size());
  for (auto& wr : h->writers) {
    w.u64(wr.in_use ? 1 : 0); w.u64((uint64_t)wr.k); w.u64(wr.has_pending ? 1 : 0);
    uint32_t f[2]; memcpy(&f[0], &wr.pending_rew, 4); memcpy(&f[1], &wr.pending_disc, 4);
    w.u64(((uint64_t)f[1] << 32) | f[0]);
    w.u64(wr.hist.size());
    for (uint64_t s : wr.hist) w.u64(s);
    w.u64(wr.pending_act.size());
    w.bytes(wr.pending_act.data(), wr.pending_act.size());
  }
}

// Host bookkeeping (key counters, FIFO bounds, every open writer's episode window) as one blob.  Staged steps are
// flushed first, so the device arrays read afterwards are complete.  blob == NULL: only the size is returned.
extern "C" int b200rl_replay_host_state(b200rl_replay* h, void* blob, int64_t capacity, int64_t* size, void* stream) {
  B200RL_REQUIRE(h && size, "null argument");
  B200RL_LOCK(h);
  int rc = ensure_device(h);
  if (rc) return rc;
  rc = flush_impl(h, as_stream(stream));
  if (rc) return rc;
  BlobWriter w;
  write_host_state(h, w);
  *size = (int64_t)w.b.size();
  if (blob) {
    B200RL_REQUIRE(capacity >= *size, "blob buffer too small: need %lld bytes", (long long)*size);
    memcpy(blob, w.b.data(), w.b.size());
  }
  return B200RL_OK;
}

// Inverse of b200rl_replay_host_state: the handle must have the geometry the blob was saved from; the caller restores
// the device arrays (b200rl_replay_segment) around this call, in any order, before the next sample / append.
extern "C" int b200rl_replay_set_host_state(b200rl_replay* h, const void* blob, int64_t size) {
  B200RL_REQUIRE(h && blob && size >= 64, "bad argument");
  B200RL_LOCK(h);
  BlobReader r{(const uint8_t*)blob, (size_t)size};
  B200RL_REQUIRE(r.u64() == kBlobMagic, "not a b200rl replay state blob");
  const uint64_t M = r.u64(), S = r.u64(), ob = r.u64(), ab = r.u64();
  B200RL_REQUIRE((int64_t)M == h->M && (int64_t)S == h->S && (int64_t)ob == h->cfg.obs_bytes && (int64_t)ab == h->cfg.act_bytes,
                 "replay geometry differs from the saved one (max_items %llu, slots %llu, obs %llu B, act %llu B)",
                 (unsigned long long)M, (unsigned long long)S, (unsigned long long)ob, (unsigned long long)ab);
  h->n_obs = h->n_fill = h->n_item = 0;
  h->slot_head = r.u64(); h->item_head = r.u64(); h->item_tail = r.u64();
  uint64_t n = r.u64();
  B200RL_REQUIRE(r.ok && n <= (uint64_t)h->M, "corrupt blob");
  h->item_start_seq.assign(n, 0);
  r.bytes(h->item_start_seq.data(), n * 8);
  n = r.u64();
  B200RL_REQUIRE(r.ok && n <= (uint64_t)h->M, "corrupt blob");
  h->start_min.clear();
  for (uint64_t i = 0; i < n; ++i) { uint64_t a = r.u64(), b = r.u64(); h->start_min.emplace_back(a, b); }
  n = r.u64();
  B200RL_REQUIRE(r.ok && n <= 65536, "corrupt blob");
  h->writers.assign(n, Writer());
  for (auto& wr : h->writers) {
    wr.in_use = r.u64() != 0; wr.k = (int64_t)r.u64(); wr.has_pending = r.u64() != 0;
    const uint64_t f = r.u64();
    uint32_t lo = (uint32_t)f, hi = (uint32_t)(f >> 32);
    memcpy(&wr.pending_rew, &lo, 4); memcpy(&wr.pending_disc, &hi, 4);
    uint64_t k = r.u64();
    B200RL_REQUIRE(r.ok && k <= 1024, "corrupt blob");
    for (uint64_t i = 0; i < k; ++i) wr.hist.push_back(r.u64());
    k = r.u64();
    B200RL_REQUIRE(r.ok && k <= (1u << 20), "corrupt blob");
    wr.pending_act.resize(k);
    r.bytes(wr.pending_act.data(), k);
  }
  B200RL_REQUIRE(r.ok, "truncated blob");
  h->state_dirty = false;      // d_state is one of the restored segments
  return B200RL_OK;
}

// ----------------------------------------------------------------------------- sample path
extern "C" int b200rl_replay_sample(b200rl_replay* h, int32_t B, const float* u_dev, int stratified,
                                    int64_t* idx_dev, uint64_t* keys_dev, float* prob_dev, void* stream) {
  B200RL_REQUIRE(h && u_dev && idx_dev && prob_dev, "null argument");
  B200RL_LOCK(h);
  B200RL_REQUIRE(B >= 1, "batch must be >= 1");
  if (h->item_head == h->item_tail) {
    set_error("replay is empty (MinSize(1) not met)");
    return B200RL_EAGAIN;
  }
  int rc = ensure_device(h);
  if (rc) return rc;
  return tree_sample(h->tree, h->d_state, h->M, B, u_dev, nullptr, 0, nullptr, stratified, h->cfg.shard_count, h->global_mass_dev,
                     idx_dev, keys_dev, prob_dev, as_stream(stream), nullptr);
}

// K1 with built-in uniform draws: u_b = Philox(seed, *counter_dev)[b] -- exactly what b200rl_uniform(seed, counter_dev)
// would have written -- so a captured step needs no separate draw kernel.  u_out (nullable) receives the draws.
extern "C" int b200rl_replay_sample_philox(b200rl_replay* h, int32_t B, uint64_t seed, const int64_t* counter_dev, int stratified,
                                           float* u_out_dev, int64_t* idx_dev, uint64_t* keys_dev, float* prob_dev, void* stream) {
  B200RL_REQUIRE(h && counter_dev && idx_dev && prob_dev, "null argument");
  B200RL_LOCK(h);
  B200RL_REQUIRE(B >= 1, "batch must be >= 1");
  if (h->item_head == h->item_tail) {
    set_error("replay is empty (MinSize(1) not met)");
    return B200RL_EAGAIN;
  }
  int rc = ensure_device(h);
  if (rc) return rc;
  return tree_sample(h->tree, h->d_state, h->M, B, nullptr, counter_dev, seed, u_out_dev, stratified, h->cfg.shard_count,
                     h->global_mass_dev, idx_dev, keys_dev, prob_dev, as_stream(stream), nullptr);
}

static int gather_locked(b200rl_replay* h, int32_t B, const int64_t* idx_dev, void* o_tm1, void* a_tm1, float* R, float* D,
                         void* o_t, void* stream);
extern "C" int b200rl_replay_gather(b200rl_replay* h, int32_t B, const int64_t* idx_dev, void* o_tm1,
                                    void* a_tm1, float* R, float* D, void* o_t, void* stream) {
  B200RL_REQUIRE(h && idx_dev && o_tm1 && a_tm1 && R && D && o_t, "null argument");
  B200RL_LOCK(h);
  return gather_locked(h, B, idx_dev, o_tm1, a_tm1, R, D, o_t, stream);
}
static int gather_locked(b200rl_replay* h, int32_t B, const int64_t* idx_dev, void* o_tm1, void* a_tm1, float* R, float* D,
                         void* o_t, void* stream) {
  B200RL_REQUIRE(h->cfg.obs_bytes > 0, "this replay was created without payload storage");
  B200RL_REQUIRE(B >= 1, "batch must be >= 1");
  int rc = ensure_device(h);
  if (rc) return rc;
  if (h->F > 1) {
    B200RL_REQUIRE(h->F == 4 && h->cfg.obs_bytes % 16 == 0 && (((uintptr_t)o_tm1 | (uintptr_t)o_t) % 16 == 0),
                   "frame-deduplicated gather is implemented for stacks of 4 uint8 frames with 16-byte aligned rows");
    const int zsplit = std::max(1, std::min(4, (h->cfg.obs_bytes >> 4) / 256));
    gather_frames4_kernel<false><<<dim3(B, 2, zsplit), 256, 0, as_stream(stream)>>>(
        h->ring, (const long long*)idx_dev, (uint8_t*)o_tm1, (uint8_t*)a_tm1, R, D, (uint8_t*)o_t, nullptr, nullptr, 1, 0, 0, 0, 0);
    B200RL_LAUNCH_OK();
    return B200RL_OK;
  }
  dim3 grid(B, 2);
  const bool a16 = (h->cfg.obs_bytes % 16 == 0) && (((uintptr_t)o_tm1 | (uintptr_t)o_t) % 16 == 0);
  const bool a4 = (h->cfg.obs_bytes % 4 == 0) && (((uintptr_t)o_tm1 | (uintptr_t)o_t) % 4 == 0);
  if (a16)
    B200RL_CUDA_OK(launch_pdl(gather_kernel<16>, dim3(grid), dim3(256), 0, as_stream(stream), h->ring, (const long long*)idx_dev, (uint8_t*)o_tm1, (uint8_t*)a_tm1, R, D, (uint8_t*)o_t));
  else if (a4)
    B200RL_CUDA_OK(launch_pdl(gather_kernel<4>, dim3(grid), dim3(256), 0, as_stream(stream), h->ring, (const long long*)idx_dev, (uint8_t*)o_tm1, (uint8_t*)a_tm1, R, D, (uint8_t*)o_t));
  else
    B200RL_CUDA_OK(launch_pdl(gather_kernel<1>, dim3(grid), dim3(256), 0, as_stream(stream), h->ring, (const long long*)idx_dev, (uint8_t*)o_tm1, (uint8_t*)a_tm1, R, D, (uint8_t*)o_t));
  B200RL_LAUNCH_OK();
  return B200RL_OK;
}

extern "C" int b200rl_replay_gather_rows(b200rl_replay* h, int32_t B, const int64_t* idx_dev, void* o_tm1, void* a_tm1, float* R,
                                         float* D, void* o_t, void* rows_tm1, void* rows_t, const b200rl_conv_geom* g,
                                         void* stream) {
  B200RL_REQUIRE(h && idx_dev && o_tm1 && a_tm1 && R && D && o_t && rows_tm1 && rows_t && g, "null argument");
  B200RL_LOCK(h);
  B200RL_REQUIRE(B >= 1, "batch must be >= 1");
  B200RL_REQUIRE(g->C >= 1 && g->C <= 16 && h->cfg.obs_bytes == g->H * g->W * g->C,
                 "gather_rows: the table's observations are not [H][W][C] uint8 frames of this geometry (1 <= C <= 16)");
  int Hp = 0, row_elems = 0;
  B200RL_REQUIRE(h_rows_layout(*g, &Hp, &row_elems) == 0, "gather_rows: geometry not eligible for a row image");
  B200RL_REQUIRE(((((uintptr_t)o_tm1 | (uintptr_t)o_t | (uintptr_t)rows_tm1 | (uintptr_t)rows_t)) & 15) == 0, "buffers must be 16-byte aligned");
  if (g->C != 4) {
    // other channel counts (RGB frames, stacks of RGB frames): the batch gather, then the row image of each half written
    // from the gathered frames (padding channels zero, as b200rl_conv2d_rows_bf16_from_u8 writes them)
    if (int rc = gather_locked(h, B, idx_dev, o_tm1, a_tm1, R, D, o_t, stream)) return rc;
    b200rl_conv_geom gb = *g;
    gb.B = B;
    if (int rc = h_rows_write((const uint8_t*)o_tm1, gb, (__nv_bfloat16*)rows_tm1, as_stream(stream))) return rc;
    return h_rows_write((const uint8_t*)o_t, gb, (__nv_bfloat16*)rows_t, as_stream(stream));
  }
  B200RL_REQUIRE(g->W % 4 == 0 && g->pad_left % 2 == 0, "gather_rows: W %% 4 == 0 and an even pad_left (16-byte aligned pixel pairs)");
  int rc = ensure_device(h);
  if (rc) return rc;
  const int zsplit = std::max(1, std::min(4, (h->cfg.obs_bytes >> 4) / 256));
  if (h->F > 1) {
    B200RL_REQUIRE(h->F == 4, "frame-deduplicated gather is implemented for stacks of 4 frames");
    gather_frames4_kernel<true><<<dim3(B, 2, zsplit), 256, 0, as_stream(stream)>>>(
        h->ring, (const long long*)idx_dev, (uint8_t*)o_tm1, (uint8_t*)a_tm1, R, D, (uint8_t*)o_t, (uint4*)rows_tm1, (uint4*)rows_t,
        g->W / 4, g->pad_left, g->pad_top, Hp, row_elems / 8);
    B200RL_LAUNCH_OK();
    return B200RL_OK;
  }
  B200RL_CUDA_OK(launch_pdl(gather_rows_kernel, dim3(B, 2, zsplit), dim3(256), 0, as_stream(stream), h->ring, (const long long*)idx_dev,
                            (uint8_t*)o_tm1, (uint8_t*)a_tm1, R, D, (uint8_t*)o_t, (uint4*)rows_tm1, (uint4*)rows_t, (int)(g->W / 4),
                            (int)g->pad_left, (int)g->pad_top, (int)Hp, (int)(row_elems / 8)));
  B200RL_LAUNCH_OK();
  return B200RL_OK;
}

extern "C" int b200rl_replay_gather_sequences(b200rl_replay* h, int32_t B, const int64_t* idx_dev, int32_t T,
                                              int32_t time_major, void* obs, void* act, float* rew, float* disc,
                                              void* stream) {
  B200RL_REQUIRE(h && idx_dev && obs && act && rew && disc, "null argument");
  B200RL_LOCK(h);
  B200RL_REQUIRE(h->cfg.obs_bytes > 0, "this replay was created without payload storage");
  B200RL_REQUIRE(B >= 1 && T >= 1 && T <= h->cfg.max_window, "gather_sequences: need 1 <= T <= max_window (%d), B >= 1",
                 h->cfg.max_window);
  B200RL_REQUIRE(h->F == 1, "sequence gather from a frame-deduplicated ring is not implemented");
  int rc = ensure_device(h);
  if (rc) return rc;
  dim3 grid(T, B);
  cudaStream_t st = as_stream(stream);
  const bool a16 = (h->cfg.obs_bytes % 16 == 0) && ((uintptr_t)obs % 16 == 0);
  const bool a4 = (h->cfg.obs_bytes % 4 == 0) && ((uintptr_t)obs % 4 == 0);
#define SEQ_ARGS h->ring, (const long long*)idx_dev, T, B, (long long)h->S, time_major ? 1 : 0, (uint8_t*)obs, (uint8_t*)act, rew, disc
  if (a16) gather_seq_kernel<16><<<grid, 128, 0, st>>>(SEQ_ARGS);
  else if (a4) gather_seq_kernel<4><<<grid, 128, 0, st>>>(SEQ_ARGS);
  else gather_seq_kernel<1><<<grid, 128, 0, st>>>(SEQ_ARGS);
#undef SEQ_ARGS
  B200RL_LAUNCH_OK();
  return B200RL_OK;
}

extern "C" int b200rl_replay_update_priorities(b200rl_replay* h, int32_t B, const uint64_t* keys_dev,
                                               const float* priority_dev, void* stream) {
  B200RL_REQUIRE(h && keys_dev && priority_dev, "null argument");
  B200RL_LOCK(h);
  B200RL_REQUIRE(B >= 0, "negative batch");
  int rc = ensure_device(h);
  if (rc) return rc;
  return tree_scatter_keys(h->tree, h->M, B, keys_dev, priority_dev, h->cfg.alpha, h->d_state,
                           h->d_stamp, h->d_epoch, as_stream(stream));
}

extern "C" int b200rl_replay_info(b200rl_replay* h, int64_t* size, uint64_t* head_key, uint64_t* tail_key,
                                  float* total_mass, void* stream) {
  B200RL_REQUIRE(h, "null handle");
  B200RL_LOCK(h);
  if (size) *size = (int64_t)(h->item_head - h->item_tail);
  if (head_key) *head_key = h->item_head;
  if (tail_key) *tail_key = h->item_tail;
  if (total_mass) {
    int rc = ensure_device(h);
    if (rc) return rc;
    B200RL_CUDA_OK(cudaMemcpyAsync(total_mass, h->tree.lvl[0], 4, cudaMemcpyDeviceToHost, as_stream(stream)));
    B200RL_CUDA_OK(cudaStreamSynchronize(as_stream(stream)));
  }
  return B200RL_OK;
}

extern "C" int b200rl_replay_tree_levels(b200rl_replay* h, int32_t* num_levels, int32_t* fanout, int32_t* staged) {
  B200RL_REQUIRE(h, "null handle");
  if (num_levels) *num_levels = h->tree.L;
  if (fanout) *fanout = kFanout;
  if (staged) *staged = h->staged_levels;
  return B200RL_OK;
}

extern "C" int b200rl_replay_tree_level_width(b200rl_replay* h, int32_t level, int64_t* width) {
  B200RL_REQUIRE(h && width && level >= 0 && level <= h->tree.L, "bad level");
  *width = h->tree.width[level];
  return B200RL_OK;
}

extern "C" int b200rl_replay_tree_read(b200rl_replay* h, int32_t level, float* host_out, int64_t n, void* stream) {
  B200RL_REQUIRE(h && host_out && level >= 0 && level <= h->tree.L, "bad argument");
  B200RL_REQUIRE(n >= 0 && n <= h->tree.width[level], "n exceeds level width");
  int rc = ensure_device(h);
  if (rc) return rc;
  B200RL_CUDA_OK(cudaMemcpyAsync(host_out, h->tree.lvl[level], n * 4, cudaMemcpyDeviceToHost, as_stream(stream)));
  B200RL_CUDA_OK(cudaStreamSynchronize(as_stream(stream)));
  return B200RL_OK;
}

extern "C" int b200rl_replay_tree_read_prefix(b200rl_replay* h, int32_t level, float* host_out, int64_t n, void* stream) {
  B200RL_REQUIRE(h && host_out && level >= 1 && level <= h->tree.L, "bad argument");
  B200RL_REQUIRE(n >= 0 && n <= h->tree.width[level], "n exceeds level width");
  int rc = ensure_device(h);
  if (rc) return rc;
  B200RL_CUDA_OK(cudaMemcpyAsync(host_out, h->tree.pre[level], n * 4, cudaMemcpyDeviceToHost, as_stream(stream)));
  B200RL_CUDA_OK(cudaStreamSynchronize(as_stream(stream)));
  return B200RL_OK;
}

// Global-priority-mass normalisation (SURVEY §8e): every rank all-reduces its shard mass (b200rl_replay_mass_ptr) into
// one device float and installs it here; K1 then reports weight / sum_r M_r.  NULL restores weight / (R * M_r).
extern "C" int b200rl_replay_set_global_mass(b200rl_replay* h, const float* global_mass_dev) {
  B200RL_REQUIRE(h, "null handle");
  B200RL_LOCK(h);
  h->global_mass_dev = global_mass_dev;
  return B200RL_OK;
}

extern "C" int b200rl_replay_mass_ptr(b200rl_replay* h, float** mass_dev) {
  B200RL_REQUIRE(h && mass_dev, "null argument");
  *mass_dev = h->tree.lvl[0];
  return B200RL_OK;
}

extern "C" int b200rl_replay_set_weights(b200rl_replay* h, int64_t n, const float* weights_dev, void* stream_) {
  B200RL_REQUIRE(h && weights_dev, "null argument");
  B200RL_LOCK(h);
  B200RL_REQUIRE(n >= 1 && n <= h->M, "n must be in [1, max_items]");
  int rc = ensure_device(h);
  if (rc) return rc;
  cudaStream_t stream = as_stream(stream_);
  const int L = h->tree.L;
  B200RL_CUDA_OK(cudaMemcpyAsync(h->tree.lvl[L], weights_dev, n * 4, cudaMemcpyDeviceToDevice, stream));
  if (n < h->tree.width[L])
    B200RL_CUDA_OK(cudaMemsetAsync(h->tree.lvl[L] + n, 0, (h->tree.width[L] - n) * 4, stream));
  rc = tree_rebuild(h->tree, stream);
  if (rc) return rc;
  h->item_tail = 0;
  h->item_head = (uint64_t)n;
  h->state_dirty = true;
  return flush_impl(h, stream);
}
