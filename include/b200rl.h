/*
 * b200rl.h — C ABI of the B200-native off-policy learner hot path.
 *
 * The reference (tmtlakmal/acme v0.1.8) is pure Python and has no FFI layer of its own; its
 * seams for this path are Python ABCs and the Reverb client surface (SURVEY.md §8b).  Each entry
 * point below names the reference call site it stands in for.  Host code (acme_b200/*.py) binds
 * these with ctypes; signatures carry only plain pointers and sizes.
 *
 * Conventions
 *   - return 0 on success; <0 on failure: -1 invalid argument, -2 CUDA error, -3 would block /
 *     not enough items, -4 unsupported device (compute capability != 10.0; there is NO CPU
 *     fallback).  b200rl_last_error() gives the message (thread-local).
 *   - `*_dev` pointers are device pointers on the handle's device; `stream` is a cudaStream_t
 *     passed as void* (NULL = legacy default stream).  Hot calls never allocate, never
 *     synchronise and never create streams, so they can be captured into CUDA graphs.
 *   - buffers are caller-owned; the library allocates only in *_create and frees in *_destroy.
 *   - one writer thread + one learner thread per handle; a handle is not re-entrant.
 */
#ifndef B200RL_H_
#define B200RL_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200RL_VERSION 100

#define B200RL_OK 0
#define B200RL_EINVAL (-1)
#define B200RL_ECUDA (-2)
#define B200RL_EAGAIN (-3)
#define B200RL_EARCH (-4)

int b200rl_version(void);
/* Number of CUDA kernels this library has launched (or recorded into a graph capture) so far. */
uint64_t b200rl_launch_count(void);
const char* b200rl_last_error(void);
/* 0 iff `device` is an sm_100 part this library was built for. */
int b200rl_device_check(int device);

/* ------------------------------------------------------------------------------------------
 * Replay shard: ring of observation slots + ring of items + fan-out-32 fp32 sum-tree.
 * Stands in for reverb.Table(sampler=Prioritized(alpha), remover=Fifo(), max_size,
 * rate_limiter=MinSize(1))  — acme/agents/tf/dqn/agent.py:95-102, d4pg/agent.py:96-103.
 * ------------------------------------------------------------------------------------------ */
typedef struct b200rl_replay b200rl_replay;

typedef struct b200rl_replay_cfg {
  int64_t max_items;     /* Table max_size (items)                                         */
  int64_t slot_capacity; /* observation slots in the HBM ring (>= max_window + 2)           */
  int32_t obs_bytes;     /* bytes of one observation                                        */
  int32_t act_bytes;     /* bytes of one action                                             */
  int32_t max_window;    /* largest n_step any writer will use                              */
  int32_t shard_count;   /* R replay shards (one per rank); probability = w / (R * mass_r)  */
  int32_t shard_rank;
  int32_t device;
  int32_t stage_slots;   /* pinned-host staging capacity in slots (0 = default)             */
  int32_t frame_stack;   /* F > 1: observations are stacks of F single-byte-element frames on their LAST axis
                            (acme/wrappers/frame_stacking.py:64-88, atari_wrapper.py:277-308) and the ring stores one
                            frame per slot, rebuilding stacks (zero frames before the episode start) at gather time:
                            obs_bytes / F bytes of HBM per step instead of obs_bytes.  0 / 1 = off                  */
  float gamma;           /* agent discount, np.float32(discount): transition.py:111         */
  float reserved_f;
  double alpha;          /* priority exponent: stored weight = priority^alpha               */
} b200rl_replay_cfg;

int b200rl_replay_create(b200rl_replay** out, const b200rl_replay_cfg* cfg);
int b200rl_replay_destroy(b200rl_replay* h);
/* reverb.Client.reset(table) (acme/datasets/reverb_test.py:70): drop every item. */
int b200rl_replay_reset(b200rl_replay* h, void* stream);

/* --- insert path: reverb.Client.writer(...) / Writer.append / create_item / close
 *     (acme/adders/reverb/base.py:111-132, transition.py:162-165).  Host pointers. --- */
int b200rl_writer_open(b200rl_replay* h, int32_t* writer_id);
/* One environment step: (obs, act, rew, disc) then the observation that followed.  `obs` is read
 * only when the writer has no open episode (first step after open/close). */
int b200rl_writer_append(b200rl_replay* h, int32_t writer, const void* obs, const void* act,
                         float rew, float disc, const void* next_obs);
/* Item over the last `num_timesteps` appended steps (Reverb's meaning), priority raw. */
int b200rl_writer_create_item(b200rl_replay* h, int32_t writer, int32_t num_timesteps,
                              double priority, uint64_t* key_out);
/* End of episode (ReverbAdder.reset, base.py:126-132): forget the step history. */
int b200rl_writer_close(b200rl_replay* h, int32_t writer);
/* Bulk form used by feeders and benchmarks: `n` consecutive timesteps of ONE stream.  Element i is
 * an observation slot; first[i] marks an episode start, last[i] a terminal observation (its
 * act/rew/disc are ignored).  Items are enumerated exactly as NStepTransitionAdder does
 * (transition.py:119-172, SURVEY App. A.1) with window `n_step` and raw priority `priority`.
 * `obs` may be a device pointer (obs_on_device != 0); the other arrays are host arrays. */
int b200rl_writer_append_stream(b200rl_replay* h, int32_t writer, int64_t n, const void* obs,
                                int obs_on_device, const void* act, const float* rew,
                                const float* disc, const uint8_t* first, const uint8_t* last,
                                int32_t n_step, double priority, void* stream);
/* Make everything appended so far visible to sample/gather (H2D of staged slots + tree insert). */
int b200rl_replay_flush(b200rl_replay* h, void* stream);

/* --- sample path: what reverb.ReplayDataset yields per item (acme/datasets/reverb.py:91-139):
 *     SampleInfo(key, probability, table_size, priority) + data.                       --- */
/* K1.  u_dev: B uniforms in [0,1).  stratified: target_b = (b+u_b)/B*mass, else u_b*mass.
 * idx = tree position (item slot), keys = Reverb-style opaque key, prob = w/(R*mass). */
int b200rl_replay_sample(b200rl_replay* h, int32_t B, const float* u_dev, int stratified,
                         int64_t* idx_dev, uint64_t* keys_dev, float* prob_dev, void* stream);
/* K3.  Gather (o_tm1, a_tm1, R, D, o_t) for B tree positions; R, D built from the ring with the
 * arithmetic of transition.py:135-145 (fp32, unfused). */
/* K1 with built-in draws: u_b = Philox4x32-10(seed, *counter_dev)[b], the value b200rl_uniform(seed, counter_dev) writes,
 * so a captured learner step has no separate draw kernel; u_out_dev (nullable) receives the draws. */
int b200rl_replay_sample_philox(b200rl_replay* h, int32_t B, uint64_t seed, const int64_t* counter_dev, int stratified,
                                float* u_out_dev, int64_t* idx_dev, uint64_t* keys_dev, float* prob_dev, void* stream);
int b200rl_replay_gather(b200rl_replay* h, int32_t B, const int64_t* idx_dev, void* o_tm1_dev,
                         void* a_tm1_dev, float* R_dev, float* D_dev, void* o_t_dev, void* stream);
/* K2.  TFClient.update_priorities(table, keys, priorities) (dqn/learning.py:151-154): weight =
 * priority^alpha for every still-live key, duplicates: last wins, dead keys ignored. */
int b200rl_replay_update_priorities(b200rl_replay* h, int32_t B, const uint64_t* keys_dev,
                                    const float* priority_dev, void* stream);
/* Host view of the table (synchronises `stream`): live items, key range, total mass. */
int b200rl_replay_info(b200rl_replay* h, int64_t* size, uint64_t* head_key, uint64_t* tail_key,
                       float* total_mass, void* stream);
/* Tree geometry + raw level access (tests, checkpointing).  level 0 = root .. L = leaves (child values). */
int b200rl_replay_tree_levels(b200rl_replay* h, int32_t* num_levels, int32_t* fanout,
                              int32_t* staged_levels);
int b200rl_replay_tree_level_width(b200rl_replay* h, int32_t level, int64_t* width);
int b200rl_replay_tree_read(b200rl_replay* h, int32_t level, float* host_out, int64_t n, void* stream);
/* the sequential-prefix lines of level 1..L (what the sampler reads) */
int b200rl_replay_tree_read_prefix(b200rl_replay* h, int32_t level, float* host_out, int64_t n, void* stream);
/* Device address of the root mass (one float) for cross-shard normalisation. */
int b200rl_replay_mass_ptr(b200rl_replay* h, float** mass_dev);
/* Global-priority-mass normalisation for sharded replay (SURVEY §8e; north_star "each rank sampling locally with
 * global-priority-mass normalisation"): global_mass_dev = caller-owned device float holding sum_r M_r (all-reduce of
 * every shard's *mass_dev); K1 then reports weight / sum_r M_r instead of weight / (R * M_r).  NULL switches it off. */
int b200rl_replay_set_global_mass(b200rl_replay* h, const float* global_mass_dev);

/* K3 with the first layer's input fused in (bf16 dataflow): as b200rl_replay_gather, and the frames ([H][W][4] uint8) are
 * also written into the zero-padded bf16 row images that b200rl_conv2d_fwd_bf16(x_rows = 1) reads (layout:
 * b200rl_conv2d_rows_bf16_bytes(g with B = 1) bytes per frame; the images must be zero-initialised once -- the padding is
 * never written).  Replaces gather + b200rl_conv2d_rows_bf16_from_u8. */
struct b200rl_conv_geom;   /* defined with the network layers below */
int b200rl_replay_gather_rows(b200rl_replay* h, int32_t B, const int64_t* idx_dev, void* o_tm1, void* a_tm1, float* R,
                              float* D, void* o_t, void* rows_tm1, void* rows_t, const struct b200rl_conv_geom* g,
                              void* stream);

/* K3 for SEQUENCE items (SURVEY §8f-3): the T steps of every sampled item as full rows, for recurrent learners.  Stands in
 * for reverb.ReplayDataset(sequence_length=T) + tf2_utils.batch_to_sequence (acme/datasets/reverb.py:100-121,
 * acme/agents/tf/r2d2/learning.py:112-121) over items made by SequenceAdder (acme/adders/reverb/sequence.py:77-127:
 * create_item(num_timesteps = T) over the trailing T appended steps; the episode's final step and its zero padding are
 * ordinary steps).  obs [.][.][obs_bytes], act [.][.][act_bytes] (action + extras row), rew / disc f32 [.][.]; the two
 * leading axes are [B][T], or [T][B] with time_major = 1.  Steps past an item's own length read as zeros. */
int b200rl_replay_gather_sequences(b200rl_replay* h, int32_t B, const int64_t* idx_dev, int32_t T, int32_t time_major,
                                   void* obs, void* act, float* rew, float* disc, void* stream);

/* DQfD demonstration mixing (acme/agents/tf/dqfd/agent.py:111-122: sample_from_datasets([replay, demonstrations],
 * [1 - ratio, ratio]); :160-217: _n_step_transition_from_episode).  The demonstration episodes are flat device arrays
 * (obs [steps][obs_bytes], act [steps][act_bytes], rew / disc f32 [steps], episode_offsets i64 [num_episodes + 1]; every
 * episode has >= 3 steps).  Called after sample + gather: batch row b is REPLACED by a demonstration transition when
 * uniforms3[3b] < ratio (episode = floor(uniforms3[3b+1] * num_episodes), first step = floor(uniforms3[3b+2] *
 * (max_index - 1))), with the reference's arithmetic for its n-step reward / discount, key 0 and probability 1;
 * is_demo (nullable) receives the mask. */
int b200rl_demo_mix(int32_t B, const void* obs, int32_t obs_bytes, const void* act, int32_t act_bytes, const float* rew,
                    const float* disc, const int64_t* episode_offsets, int32_t num_episodes, int32_t n_step, float gamma,
                    const float* uniforms3, float ratio, void* o_tm1, void* a_tm1, float* R, float* D, void* o_t,
                    uint64_t* keys, float* prob, int32_t* is_demo, void* stream);

/* Checkpoint / resume of a replay shard (SURVEY §8f-4; the reference's checkpointers, acme/tf/savers.py:76-167, never save
 * replay contents).  host_state serialises the host bookkeeping (key counters, FIFO bounds, every open writer's episode
 * window) after flushing staged steps; blob == NULL only reports the size.  segment(which) exposes the device arrays to
 * copy out / in: 0 obs slots, 1 actions, 2 rewards, 3 discounts, 4 next links, 5-7 item start / end / length, 8 sum
 * tree (values + prefix lines), 9 live key range, 10 older-frame slots of every item (frame-deduplicated tables).  Restore = set_host_state + writing every segment back, on a handle
 * created with the same geometry. */
int b200rl_replay_host_state(b200rl_replay* h, void* blob, int64_t capacity, int64_t* size, void* stream);
int b200rl_replay_set_host_state(b200rl_replay* h, const void* blob, int64_t size);
int b200rl_replay_segment(b200rl_replay* h, int32_t which, void** dev_ptr, int64_t* bytes);

/* Stand-alone sum-tree (priorities only) for the sampling/update sweep (BASELINE config 4). */
int b200rl_replay_set_weights(b200rl_replay* h, int64_t n, const float* weights_dev, void* stream);

/* ------------------------------------------------------------------------------------------
 * Learner math (stateless kernels; parameters live in caller-owned device buffers).
 * ------------------------------------------------------------------------------------------ */
/* Philox4x32-10 uniforms in [0,1): out[i] = f(seed, *step_dev + step_offset, i). */
int b200rl_uniform(float* out_dev, int32_t n, uint64_t seed, const int64_t* step_dev,
                   int64_t step_offset, void* stream);

/* K4.  dqn/learning.py:127-154 + trfl.double_qlearning + losses/huber.py:48-57.
 * wmax_dev (nullable): device scalar (f64) holding the GLOBAL max importance weight for data-parallel
 * learners; NULL = batch max (the reference's tf.reduce_max).  If wmax_out_dev != NULL the local
 * max is written there instead and no normalisation happens (two-pass DP form). */
int b200rl_dqn_td(int32_t B, int32_t A, const float* q_tm1, const float* q_t_value,
                  const float* q_t_selector, const int32_t* a_tm1, const float* R, const float* D,
                  const float* prob, float gamma, float huber_delta, double is_exponent,
                  float max_abs_reward, const double* wmax_dev, float grad_scale, float* td,
                  float* loss_per_sample, float* weight, float* priority, float* dq_tm1,
                  float* loss_mean, int32_t flags, void* stream);
/* flags for b200rl_dqn_td / b200rl_dqn_head_td.  IS_WEIGHTS_F32: the JAX learner's importance weights
 * (acme/agents/jax/dqn/learning.py:94-96: 1/probs cast to f32, power and max in f32) instead of the TF learner's
 * f64 power / max / divide followed by a cast (acme/agents/tf/dqn/learning.py:138-143). */
#define B200RL_TD_IS_WEIGHTS_F32 1
/* Recurrent replay (acme/agents/tf/r2d2/learning.py):
 *   seq_priority    :230-236  priority[b] = eta * max_t |err[t][b]| + (1 - eta) * mean_t |err[t][b]|, err f32 [T][B]
 *                   (time-major, as the learner holds it); the mean is a sequential fp32 sum over t divided by T
 *   seq_is_weights  :170-176  w[b] = (1 / (table_size * prob[b]))^beta / max_b(...), f64 then cast to f32 */
int b200rl_seq_priority(int32_t T, int32_t B, const float* err_tb, float eta, float* priority_out, void* stream);
int b200rl_seq_is_weights(int32_t B, const float* prob, double table_size, double is_exponent, float* w_out, void* stream);
int b200rl_is_weight_max(int32_t B, const float* prob, double is_exponent, double* wmax_out_dev,
                         int32_t flags, void* stream);

/* K5.  losses/distributional.py:22-83: target = l2_project(R + Dg*z, softmax(logits_t), z); loss =
 * CE(logits_tm1, target); dlogits = (softmax(logits_tm1)*sum(target) - target) * grad_scale. */
int b200rl_c51_loss(int32_t B, int32_t K, float vmin, float vmax, const float* logits_tm1,
                    const float* logits_t, const float* R, const float* D, float gamma,
                    float grad_scale, float* target, float* loss_per_sample, float* dlogits_tm1,
                    float* loss_mean, void* stream);
/* DDPG critic loss (acme/agents/tf/ddpg/learning.py:193, trfl.td_learning): td = (R + gamma * D * v_t) - v_tm1,
 * loss = 0.5 td^2, dv_tm1 = -td * grad_scale.  td, dv_tm1, loss_mean nullable. */
int b200rl_td_learning(int32_t B, const float* v_tm1, const float* v_t, const float* R, const float* D, float gamma,
                       float grad_scale, float* td, float* loss_per_sample, float* dv_tm1, float* loss_mean, void* stream);
/* mean of a discrete-valued distribution and its logit gradient (distributions.py:64-66):
 * q = sum softmax(l)_i z_i;  dlogits_i = p_i (z_i - q) * dq. */
int b200rl_c51_mean_fwd(int32_t B, int32_t K, float vmin, float vmax, const float* logits, float* q,
                        void* stream);
int b200rl_c51_mean_bwd(int32_t B, int32_t K, float vmin, float vmax, const float* logits,
                        const float* dq /*nullable => 1*/, float* dlogits, void* stream);
/* losses/dpg.py:41-57: da = -clip_by_norm(dqda, clip) * grad_scale; loss = mean 0.5*||clipped||^2 */
int b200rl_dpg_action_grad(int32_t B, int32_t A, const float* dqda, float clip, int clip_norm,
                           float grad_scale, float* da, float* loss_per_sample /*nullable*/,
                           float* loss_mean /*nullable, needs loss_per_sample*/, void* stream);

/* K7.  snt.optimizers.Adam.apply (dqn/learning.py:148); step/bias corrections live on device so the
 * call is graph-replayable: t = *step_dev + 1.  eps_mode 0 = m^/(sqrt(v^)+eps), 1 = Keras form.
 * grad_scale_dev (nullable): device scalar multiplied into every gradient (global-norm clip, 1/R).
 * bf16_shadow (nullable): also writes the updated parameter rounded to bf16. */
int b200rl_adam(int64_t n, float* param, const float* grad, float* m, float* v,
                const int64_t* step_dev, float lr, double b1, double b2, float eps, int eps_mode,
                const float* grad_scale_dev, void* bf16_shadow, void* stream);
/* b200rl_adam on a grid limited to ctas_per_sm CTAs per SM (0 = default): for an update issued BESIDE other kernels */
int b200rl_adam_throttled(int64_t n, float* param, const float* grad, float* m, float* v, const int64_t* step_dev,
                          float lr, double b1, double b2, float eps, int eps_mode, const float* grad_scale_dev,
                          void* bf16_shadow, int32_t ctas_per_sm, void* stream);
/* tf.clip_by_global_norm (d4pg/learning.py:235-237): *scale_out = clip / max(||g||, clip). */
int b200rl_global_norm_scale(int64_t n, const float* grad, float clip, float* partial_ws,
                             float* scale_out_dev, float* norm_out_dev, void* stream);
/* if (*step_dev % period == 0) dst <- src   (dqn/learning.py:157-160; d4pg/learning.py:171-174) */
int b200rl_copy_if_period(int64_t n_bytes, void* dst, const void* src, const int64_t* step_dev,
                          int64_t period, int64_t phase, void* stream);
int b200rl_step_increment(int64_t* step_dev, void* stream);
/* End of a learner step in ONE launch (dqn/learning.py:157-161): if ((*step_dev + phase) % period == 0) dst_a <- src_a and
 * dst_b <- src_b (online -> target parameters and their bf16 shadow; n_bytes_b may be 0), then *step_dev += 1 and, if
 * counter2 != NULL, *counter2 += 1 (the dataset's draw counter).  period = 0: increments only. */
int b200rl_learner_tail(int64_t n_bytes_a, void* dst_a, const void* src_a, int64_t n_bytes_b, void* dst_b, const void* src_b,
                        int64_t* step_dev, int64_t period, int64_t phase, int64_t* counter2, void* stream);

/* ------------------------------------------------------------------------------------------
 * K6.  Network layers (acme/tf/networks/atari.py:36-69, duelling.py:37-59, continuous.py:37-68).
 * Activations NHWC / row-major fp32; weights [out][in] (conv: [Cout][kh][kw][Cin]) fp32.
 * precision: 0 = fp32 SIMT (parity mode, 1e-5); 1 = tcgen05 tensor cores with fp32 accumulation: tf32 operands
 * fetched by TMA where the tensors satisfy its alignment rules, bf16 operands otherwise, and the exact fp32 path for
 * dense layers too small to amortise a tensor-core pipeline (speed mode; stated tolerance in DESIGN.md).
 * ws / ws_bytes: caller-owned scratch (split-K partial sums, column-sum partials, and for a first-layer convolution
 * on uint8 frames in precision 1 the zero-padded fp32 row image, B * (H + pad) * (W + pad) * C * 4 bytes); one workspace
 * per stream -- calls on different streams must not share it.
 * Alignment (every precision): the convolution entry points read fp32 x (forward, weight gradient, row image) and the
 * data gradient's dy and w as 16-byte vectors, and uint8 frames as 4-byte pixels; a pointer that is not 16-byte
 * (fp32) / 4-byte (uint8) aligned returns B200RL_EINVAL without launching.  Dense layers take any 4-byte alignment.
 * ------------------------------------------------------------------------------------------ */
typedef struct b200rl_conv_geom {
  int32_t B, H, W, C;       /* input NHWC                         */
  int32_t kh, kw, stride;   /* filter                             */
  int32_t pad_top, pad_left;/* TF SAME: before = total/2          */
  int32_t OH, OW, Cout;
} b200rl_conv_geom;

#define B200RL_ACT_NONE 0
#define B200RL_ACT_RELU 1
#define B200RL_ACT_ELU 2
#define B200RL_ACT_TANH 3

/* Row images.  In precision 1 a first-layer convolution on uint8 frames (C = 4, kw * C = 32: the Atari torso,
 * networks/atari.py:44) first rewrites the frames as zero-padded fp32 rows float(x)/255 (atari_wrapper.py:303-304).
 * A caller that convolves the same frames several times (two networks on o_t; forward and weight gradient on o_tm1:
 * dqn/learning.py:123-125,147) builds that image once and passes it as x with x_u8 = 2.
 * rows_bytes: size of the image for geometry g, 0 if g is not eligible (then pass the uint8 frames). */
int64_t b200rl_conv2d_rows_bytes(const b200rl_conv_geom* g);
int b200rl_conv2d_rows_from_u8(const void* x_u8, const b200rl_conv_geom* g, float* rows, int64_t rows_bytes,
                               void* stream);
/* y = act(conv(x, w) + b).  x_u8 = 1: x is uint8 and is read as float(x)/255 (atari_wrapper.py:303); x_u8 = 2: x is
 * the row image of the frames (precision 1 only). */
int b200rl_conv2d_fwd(const void* x, int x_u8, const float* w, const float* bias, float* y,
                      const b200rl_conv_geom* g, int act, int precision, void* ws, int64_t ws_bytes,
                      void* stream);
/* dw[Cout][kh][kw][Cin] = sum_m dy[m,co] * col(x)[m,k];  db = colsum(dy).  dy is d(pre-activation). */
int b200rl_conv2d_wgrad(const void* x, int x_u8, const float* dy, float* dw, float* db,
                        const b200rl_conv_geom* g, int precision, void* ws, int64_t ws_bytes,
                        void* stream);
/* dx = conv_transpose(dy, w) [* act'(x_out)]: if mask_y != NULL multiplies by d act / d pre evaluated
 * from the producer layer's *output* mask_y (ReLU: y>0). */
int b200rl_conv2d_dgrad(const float* dy, const float* w, float* dx, const b200rl_conv_geom* g,
                        const float* mask_y, int mask_act, int precision, void* ws,
                        int64_t ws_bytes, void* stream);
/* y[M,N] = act(x[M,K] @ w[N,K]^T + b); ldx / ldy are row strides in elements (>= K / >= N) */
int b200rl_linear_fwd(int32_t M, int32_t N, int32_t K, const float* x, int32_t ldx, const float* w,
                      const float* bias, float* y, int32_t ldy, int act, int precision, void* ws,
                      int64_t ws_bytes, void* stream);
/* dx[M,K] = dy[M,N] @ w[N,K]  [* act'(mask_y)]; mask_y shares dx's row stride */
int b200rl_linear_dgrad(int32_t M, int32_t N, int32_t K, const float* dy, int32_t lddy,
                        const float* w, float* dx, int32_t lddx, const float* mask_y, int mask_act,
                        int precision, void* ws, int64_t ws_bytes, void* stream);
/* dw[N,K] = dy[M,N]^T @ x[M,K];  db[N] = colsum(dy) (nullable) */
int b200rl_linear_wgrad(int32_t M, int32_t N, int32_t K, const float* dy, int32_t lddy,
                        const float* x, int32_t ldx, float* dw, float* db, int precision, void* ws,
                        int64_t ws_bytes, void* stream);
/* in-place dy *= act'(y) for outputs that feed a loss directly */
int b200rl_act_bwd(int64_t n, float* dy, const float* y, int act, void* stream);
/* duelling head (duelling.py:51-59): q = v + (adv - mean(adv)); bwd: dv = sum dq, dadv = dq - mean(dq) */
int b200rl_duelling_fwd(int32_t B, int32_t A, const float* value, const float* adv, float* q, void* stream);
int b200rl_duelling_bwd(int32_t B, int32_t A, const float* dq, float* dvalue, float* dadv, void* stream);
/* whole duelling head in one pass over the hidden row h[B, 2H] (value stream = first H columns):
 * value = h[:, :H].wv + bv, adv = h[:, H:] @ wa^T + ba, q as above (duelling.py:37-59); the backward
 * also applies relu'(h) to dh and produces the four parameter gradients. */
int b200rl_duelling_head_fwd(int32_t B, int32_t A, int32_t H, const float* h, int32_t ldh, const float* wv,
                             const float* bv, const float* wa, const float* ba, float* value, float* adv,
                             float* q, void* stream);
int b200rl_duelling_head_bwd(int32_t B, int32_t A, int32_t H, const float* dq, const float* h, int32_t ldh,
                             const float* wv, const float* wa, float* dvalue, float* dadv, float* dh,
                             int32_t lddh, float* dwv, float* dbv, float* dwa, float* dba, void* ws,
                             int64_t ws_bytes, void* stream);
/* snt.LayerNorm(axis=1:, scale, offset, eps=1e-5) followed by tanh (continuous.py:55-58) */
int b200rl_layernorm_tanh_fwd(int32_t B, int32_t N, const float* x, const float* scale,
                              const float* offset, float eps, float* y, float* xhat, float* rstd,
                              void* stream);
int b200rl_layernorm_tanh_bwd(int32_t B, int32_t N, const float* dy, const float* y, const float* xhat,
                              const float* rstd, const float* scale, float* dx, float* dscale,
                              float* doffset, void* stream);
/* TanhToSpec (rescaling.py:63-74): a = 0.5*(tanh(x)+1)*scale + offset; bwd: dx = da*0.5*scale*(1-tanh^2) */
int b200rl_tanh_to_spec_fwd(int32_t B, int32_t A, const float* x, const float* scale,
                            const float* offset, float* a, void* stream);
int b200rl_tanh_to_spec_bwd(int32_t B, int32_t A, const float* da, const float* x, const float* scale,
                            float* dx, void* stream);
/* batch_concat([obs, act]) (tf/utils.py:39-54) and its split for the backward */
int b200rl_concat2(int32_t B, int32_t n0, int32_t n1, const float* x0, const float* x1, float* y, void* stream);
int b200rl_split_second(int32_t B, int32_t n0, int32_t n1, const float* dy, float* dx1, void* stream);
/* K4 fused into the duelling head (dqn/learning.py:123-154 after the three fc1 layers): for every sample the three
 * heads q_tm1 = head(h_tm1), q_t_value = target_head(h_tgt), q_t_selector = head(h_sel), the double-Q TD error, Huber
 * loss, importance weight and new priority of b200rl_dqn_td, and the head's data gradient
 * dh = [dval * wv, dadv @ wa] * relu'(h_tm1) -- one launch instead of five on the step's critical path; arithmetic
 * identical to the separate kernels.  wmax_dev is REQUIRED (b200rl_is_weight_max right after sampling; the global max
 * for data-parallel learners); A <= 32.  q_*, dq nullable.  dh_bf16 = 1 writes dh as bf16 (bf16 dataflow). */
int b200rl_dqn_head_td(int32_t B, int32_t A, int32_t H, const float* h_tm1, const float* h_sel, const float* h_tgt,
                       int32_t ldh, const float* wv, const float* bv, const float* wa, const float* ba,
                       const float* target_wv, const float* target_bv, const float* target_wa, const float* target_ba,
                       const int32_t* a_tm1, const float* R, const float* D, const float* prob, float gamma,
                       float huber_delta, double is_exponent, float max_abs_reward, const double* wmax_dev,
                       float grad_scale, int32_t flags, float* q_tm1, float* q_t_value, float* q_t_selector, float* td,
                       float* loss_per_sample, float* weight, float* priority, float* dq_tm1, float* dvalue, float* dadv,
                       void* dh, int32_t lddh, int32_t dh_bf16, void* stream);
/* out[0] = mean(x[0..n)) in a fixed order (the learner's scalar loss, dqn/learning.py:143-144) */
int b200rl_mean(int32_t n, const float* x, float* out, void* stream);
/* the four parameter gradients of the duelling head from dvalue / dadv (the part of b200rl_duelling_head_bwd that is
 * off the critical path once b200rl_dqn_head_td has produced dh) */
int b200rl_duelling_head_wgrad(int32_t B, int32_t A, int32_t H, const float* dvalue, const float* dadv, const float* h,
                               int32_t ldh, float* dwv, float* dbv, float* dwa, float* dba, void* ws, int64_t ws_bytes,
                               void* stream);

/* ------------------------------------------------------------------ K6, bf16 dataflow (speed mode of the networks)
 * Same layers as above with activations, weight SHADOWS and back-propagated gradients in bf16 (tcgen05 kind::f16, fp32
 * accumulation; TMA-fed, im2col mode for the convolutions); master weights, weight gradients, biases and the optimizer
 * stay fp32.  `*_bf16` flags name the element type of an OUTPUT or mask buffer (1 = bf16, 0 = fp32); x, w, dy are
 * always bf16 here.  Shapes outside the kernels' coverage are an error (no fallback): channel counts 32 or multiples
 * of 64, Cout in {32, 64, 128}, dense K and N multiples of 64, 16-byte aligned rows.  Stated tolerance: DESIGN.md. */
int b200rl_bf16_from_f32(int64_t n, const float* src, void* dst_bf16, void* stream);   /* n % 8 == 0: weight shadows */
/* First layer on uint8 frames (C = 4, kw * C = 32, networks/atari.py:44): zero-padded bf16 row image holding the
 * INTEGER pixel values (exact in bf16); the 1/255 of atari_wrapper.py:303-304 is applied to the fp32 accumulator. */
int64_t b200rl_conv2d_rows_bf16_bytes(const b200rl_conv_geom* g);
int b200rl_conv2d_rows_bf16_from_u8(const void* x_u8, const b200rl_conv_geom* g, void* rows_bf16, int64_t rows_bytes,
                                    void* stream);
/* x_rows = 1: x is the row image above (first layer); 0: x is an NHWC bf16 activation */
int b200rl_conv2d_fwd_bf16(const void* x, int x_rows, const void* w_bf16, const float* bias, void* y, int y_bf16,
                           const b200rl_conv_geom* g, int act, void* ws, int64_t ws_bytes, void* stream);
int b200rl_conv2d_wgrad_bf16(const void* x, int x_rows, const void* dy_bf16, float* dw, float* db,
                             const b200rl_conv_geom* g, void* ws, int64_t ws_bytes, void* stream);
int b200rl_conv2d_dgrad_bf16(const void* dy_bf16, const void* w_bf16, void* dx, int dx_bf16, const b200rl_conv_geom* g,
                             const void* mask_y, int mask_bf16, int mask_act, void* stream);
int b200rl_linear_fwd_bf16(int32_t M, int32_t N, int32_t K, const void* x_bf16, int32_t ldx, const void* w_bf16,
                           const float* bias, void* y, int32_t ldy, int y_bf16, int act, void* ws, int64_t ws_bytes,
                           void* stream);
int b200rl_linear_dgrad_bf16(int32_t M, int32_t N, int32_t K, const void* dy_bf16, int32_t lddy, const void* w_bf16,
                             void* dx, int32_t lddx, int dx_bf16, const void* mask_y, int mask_bf16, int mask_act,
                             void* ws, int64_t ws_bytes, void* stream);
/* out[n] = sum_m x[m, n] over bf16 rows (a bias gradient issued on its own stream; N a power of two in [4, 1024]) */
int b200rl_colsum_bf16(int32_t M, int32_t N, const void* x_bf16, int32_t ld, float* out, void* ws, int64_t ws_bytes,
                       void* stream);
int b200rl_linear_wgrad_bf16(int32_t M, int32_t N, int32_t K, const void* dy_bf16, int32_t lddy, const void* x_bf16,
                             int32_t ldx, float* dw, float* db, void* ws, int64_t ws_bytes, void* stream);

/* ------------------------------------------------------------------ data-parallel learner (SURVEY §8e)
 * Replaces all_reduce('mean', grads) followed by optimizer.apply on every replica
 * (acme/agents/tf/crr/recurrent_learning.py:346-359, the reference's only multi-replica learner) by ONE kernel
 * per gradient bucket over NVLink peer memory: reduce-scatter by peer loads, Adam on the owned 1/R shard,
 * all-gather of the new parameters by peer stores (see acme_b200/csrc/dp_p2p.cu).  One process per GPU.
 *   create   allocates this rank's region [params | grads | mailbox]; the learner keeps its flat parameter and
 *            gradient buffers THERE (b200rl_dp_buffers)
 *   export / import   64-byte IPC handle of the region; every rank imports every peer's (exchange them with any
 *            host-side all-gather) before the first exchange call
 *   max_f64  in-place all-reduce(MAX) of one device double (the importance-weight normaliser, dqn/learning.py:140)
 *   adam     parameters[off, off+n) of all ranks <- Adam(mean over ranks of grads[off, off+n)); m, v: this rank's
 *            full-size moment buffers (only the owned shard is touched); `bucket` (0..3) names the mailbox slot, two
 *            buckets may be in flight at once; step_dev as in b200rl_adam.  final_barrier = 0 lets the kernel end
 *            without waiting for the peers' stores: only allowed when a later exchange of the same step (issued
 *            after this one on every rank) has final_barrier = 1.  All ranks must issue the same calls in the same
 *            order each step; both calls are CUDA-graph capturable.
 *   status   < 0 if an exchange gave up waiting for a peer (~2 s) */
typedef struct b200rl_dp* b200rl_dp_t;
typedef struct b200rl_dp_cfg {
  int32_t world, rank, device, reserved;
  int64_t n_params;
} b200rl_dp_cfg;
int b200rl_dp_create(b200rl_dp_t* out, const b200rl_dp_cfg* cfg);
int b200rl_dp_destroy(b200rl_dp_t h);
int b200rl_dp_buffers(b200rl_dp_t h, float** params, float** grads);
int b200rl_dp_export(b200rl_dp_t h, void* handle64);
int b200rl_dp_import(b200rl_dp_t h, int32_t peer_rank, const void* handle64);
int b200rl_dp_max_f64(b200rl_dp_t h, double* value_dev, const int64_t* step_dev, void* stream);
int b200rl_dp_adam(b200rl_dp_t h, int64_t off, int64_t n, float* m, float* v, const int64_t* step_dev, float lr,
                   double b1, double b2, float eps, int eps_mode, int32_t bucket, int32_t final_barrier, void* stream);
int b200rl_dp_status(b200rl_dp_t h);
/* The same exchange with the bulk bytes moved by the copy engines (DMA over NVLink, graph memcpy nodes) instead of SM
 * loads / stores, in two halves that a pipelined step places where they hide: the exchange keeps no SM slots, so the
 * step's latency-bound GEMM kernels run beside it undisturbed.  Bit-identical parameters to b200rl_dp_adam.
 *   reduce_adam_ce   push, for every peer, the shard that peer owns of this rank's gradients of [off, off+n) into the
 *                    peer's landing buffer (part of its region), announce "landed", wait for every peer's
 *                    announcement, then Adam on the owned shard (sum in rank order, x 1/R) into this rank's own
 *                    parameter buffer; shadow_bf16 (NULL or this rank's bf16 copy
 *                    of the flat parameters) receives the rounded shard; max_ctas > 0 caps the Adam kernel's grid
 *                    (0 = fill the GPU) so that it can run underneath other kernels.
 *   broadcast_ce     push the owned shard of the new parameters into every peer's buffer, announce "done", and with
 *                    final_barrier wait until every peer has announced: then all of [off, off+n) is in place here.
 * Same ordering rules as b200rl_dp_adam (same calls, same order on every rank; `bucket` names the mailbox slot; both
 * halves read *step_dev before the step counter is advanced). */
/* NVSwitch multicast form.  create_external adopts a SYMMETRIC allocation the caller made on every rank (for example
 * torch.distributed._symmetric_memory: the only plumbing it supplies is the allocation and the rendezvous):
 * b200rl_dp_region_bytes(n) bytes per rank, bases[r] = this process's mapping of rank r's region, multicast_base = the
 * multicast mapping of the same regions (NULL = none).  adam_mc is b200rl_dp_adam with the reduce-scatter done by the
 * switch (one multimem.ld_reduce per 16 bytes of the owned shard) and the all-gather by one multimem.st that the switch
 * replicates into every rank's parameter buffer; max_ctas > 0 caps the grid so that it runs beside other kernels.  The
 * in-switch sum replaces the rank-order sum (ulp-level difference in the mean gradient); replicas stay bit-identical. */
int64_t b200rl_dp_region_bytes(int64_t n_params);
int b200rl_dp_create_external(b200rl_dp_t* out, const b200rl_dp_cfg* cfg, void* const* bases, void* multicast_base);
int b200rl_dp_has_multicast(b200rl_dp_t h);
int b200rl_dp_adam_mc(b200rl_dp_t h, int64_t off, int64_t n, float* m, float* v, const int64_t* step_dev, float lr,
                      double b1, double b2, float eps, int eps_mode, int32_t bucket, int32_t final_barrier,
                      int32_t max_ctas, void* stream);
/* the two halves of adam_mc on their own, interchangeable with the copy-engine halves below (same flags, same shard) */
int b200rl_dp_reduce_adam_mc(b200rl_dp_t h, int64_t off, int64_t n, float* m, float* v, const int64_t* step_dev, float lr,
                             double b1, double b2, float eps, int eps_mode, int32_t bucket, void* shadow_bf16,
                             int32_t max_ctas, void* stream);
int b200rl_dp_broadcast_mc(b200rl_dp_t h, int64_t off, int64_t n, const int64_t* step_dev, int32_t bucket,
                           int32_t final_barrier, int32_t max_ctas, void* stream);
int b200rl_dp_reduce_adam_ce(b200rl_dp_t h, int64_t off, int64_t n, float* m, float* v, const int64_t* step_dev, float lr,
                             double b1, double b2, float eps, int eps_mode, int32_t bucket, void* shadow_bf16,
                             int32_t max_ctas, void* stream);
int b200rl_dp_broadcast_ce(b200rl_dp_t h, int64_t off, int64_t n, const int64_t* step_dev, int32_t bucket,
                           int32_t final_barrier, void* stream);

/* bytes of split-K workspace that lets every layer call on outputs of up to max_out_elems
 * elements use its preferred split count (smaller workspaces only reduce the split count) */
int64_t b200rl_workspace_bytes(int64_t max_out_elems);

#ifdef __cplusplus
}
#endif
#endif /* B200RL_H_ */
