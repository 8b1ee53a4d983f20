"""DQN learner + agent on the B200 hot path.

`DQNLearner` keeps the constructor and `step()/get_variables()/state` surface of
`acme/agents/tf/dqn/learning.py:35-199`; one `step()` is:
  K1 sample -> K3 gather/n-step -> K6 three forwards -> K4 TD/Huber/IS/priorities ->
  K6 backward -> [NCCL all-reduce when data-parallel] -> K7 Adam -> K2 priority write-back ->
  conditional target copy -> step counter,
all on one stream, recorded once into a CUDA graph and replayed.  `DQN` builds the table, adder,
dataset, actor and learner like `acme/agents/tf/dqn/agent.py:45-162`.
"""

from __future__ import annotations

import contextlib
import ctypes
import os
import time
from typing import List, Optional

import numpy as np

from acme_b200 import _capi, actors, adders, agent, core, counting, loggers, networks, parallel, replay, specs

# Single-GPU pipelined update (see DQNLearner.__init__): '1' once measured faster than the one-graph serial step.
PIPELINE_1GPU_DEFAULT = '0'


class DQNLearner(core.Learner, core.Saveable):

  def __init__(self, network, target_network, discount: float, importance_sampling_exponent: float,
               learning_rate: float, target_update_period: int, dataset: replay.ReplayDataset,
               huber_loss_parameter: float = 1., replay_client: Optional[replay.Client] = None,
               counter: counting.Counter = None, logger: loggers.Logger = None, checkpoint: bool = True,
               max_abs_reward: float = 1., eps_mode: int = 0, use_cuda_graph: bool = True,
               process_group=None, adam_eps: float = 1e-8, concurrent_streams: bool = True,
               peer_exchange: Optional[bool] = None, target_update_mode: str = 'pre_increment',
               is_weights_dtype: str = 'f64'):
    """Arguments up to `checkpoint` are the reference's (`dqn/learning.py:43-58`).  The two JAX-learner variants of
    SURVEY App. A.6 are switches: `target_update_mode='post_increment'` copies the target when (steps + 1) % period == 0
    (`jax/dqn/learning.py:114-119`, `jax/utils.py:148-154`) instead of the TF learner's test before the increment
    (`dqn/learning.py:157-161`); `is_weights_dtype='f32'` computes the importance weights in f32
    (`jax/dqn/learning.py:94-96`) instead of f64-then-cast (`dqn/learning.py:138-143`)."""
    import torch
    if huber_loss_parameter < 0:
      raise ValueError('quadratic_linear_boundary must be >= 0.')   # huber.py:45-46
    if target_update_mode not in ('pre_increment', 'post_increment'):
      raise ValueError(f'unknown target_update_mode {target_update_mode!r}')
    if is_weights_dtype not in ('f64', 'f32'):
      raise ValueError(f'unknown is_weights_dtype {is_weights_dtype!r}')
    self._copy_phase = 1 if target_update_mode == 'post_increment' else 0
    self._td_flags = _capi.TD_IS_WEIGHTS_F32 if is_weights_dtype == 'f32' else 0
    self._torch = torch
    self._net, self._tgt = network, target_network
    self._dataset = dataset
    self._replay_client = replay_client
    self._discount = float(np.float32(discount))
    self._beta = float(importance_sampling_exponent)
    self._delta = float(huber_loss_parameter)
    self._lr = float(np.float32(learning_rate))
    self._period = int(target_update_period)
    self._max_abs_reward = float(max_abs_reward)
    self._eps_mode, self._adam_eps = int(eps_mode), float(adam_eps)
    self._counter = counter or counting.Counter()
    self._logger = logger or loggers.TerminalLogger('learner', time_delta=1.)
    self._timestamp = None
    self._dp = parallel.DataParallel(process_group)
    self._world = self._dp.world

    dev = torch.device('cuda', network.device)
    B, A = dataset.B, network.A
    self.B = B
    f32 = lambda *s: torch.zeros(s, dtype=torch.float32, device=dev)
    # Fused path (networks with a duelling head and features(): DQNAtariNetwork): the two online forwards
    # (learning.py:123,125) run as ONE pass over the 2B frames [o_tm1; o_t] (fc1's weights are read once, half the
    # launches), and the three heads + K4 + the head's data gradient are one kernel (b200rl_dqn_head_td).
    self._fused = hasattr(network, 'features') and A <= 32
    if self._fused:
      self._bufs_on = network.make_buffers(2 * B)                 # rows [0, B) = o_tm1, rows [B, 2B) = o_t
      self._bufs_train = dict(self._bufs_on, B=B)                 # the same storage seen as the o_tm1 batch (backward)
      self._bufs_sel = None
      self._q3 = f32(3, B, A)                                     # q_tm1, q_t_value, q_t_selector
    else:
      self._bufs_train = network.make_buffers(B)
      self._bufs_sel = network.make_buffers(B)
    self._bufs_tgt = target_network.make_buffers(B)
    self._gbufs = network.make_grad_buffers(B)
    self.td, self.loss_ps, self.weight, self.priority = f32(B), f32(B), f32(B), f32(B)
    self.dq = f32(B, A)
    self.loss = f32(1)
    self._m = torch.zeros_like(network.params.flat)
    self._v = torch.zeros_like(network.params.flat)
    self._num_steps = torch.zeros(1, dtype=torch.int64, device=dev)
    self._wmax = torch.zeros(1, dtype=torch.float64, device=dev)
    self._gscale = torch.full((1,), 1.0 / self._world, dtype=torch.float32, device=dev)
    self._loss_host = torch.zeros(1, dtype=torch.float32).pin_memory()
    # fetch_loss='async': two pinned slots + events, the loss of step i is logged when step i+1 is issued
    self._loss_ring = torch.zeros(2, dtype=torch.float32).pin_memory()
    self._loss_events = [torch.cuda.Event(), torch.cuda.Event()]
    self._loss_pending = None
    self._stamps = torch.zeros(8, dtype=torch.int64, device='cuda') if os.environ.get('B200RL_STAMPS') else None
    self._graphs = None
    self._use_graph = bool(use_cuda_graph)
    # the three forward passes are independent, and so are a layer's weight- and data-gradient: run them on
    # parallel streams (fork/join with events, also inside the captured graph)
    self._concurrent = bool(concurrent_streams) and hasattr(network, 'grad_buckets')
    # one launch ends the step (target copy of parameters + shadow, both counters): single GPU only, where the whole step
    # is one graph and the counters are bumped in one place
    self._fuse_tail = self._world == 1
    self._side = [torch.cuda.Stream(device=dev) for _ in range(6)] if self._concurrent else None
    self._wmax_done = None
    self._params_ready = None      # pipelined exchange: event the online forwards wait for
    self._k2_done = False          # K2 of this step was already issued beside the backward
    # data parallel: gradients and parameters live in a peer-mapped region and the exchange is fused with Adam
    # (parallel.PeerExchange); peer_exchange=False keeps the NCCL all-reduce + replicated Adam path
    if peer_exchange is None:
      peer_exchange = self._world > 1 and os.environ.get('B200RL_PEER_EXCHANGE', '1') != '0'
    self._px = None
    if peer_exchange and self._world > 1:
      self._px = parallel.PeerExchange(self._dp, network.params.size, network.device)
      network.params.rebind(self._px.params, self._px.grads)
    # Pipelined exchange (data parallel with a peer exchange): the optimizer update of step t is issued at the START of
    # step t+1's graph, beside K1 / K3 / the target-network forward, none of which read the online parameters; only the
    # two online forwards wait for it.  Same values as the serial order, the NVLink-bound exchange just leaves the
    # critical path.  `flush()` applies the update still in flight (collective: every rank must call it).
    self._pipeline = (self._px is not None and self._concurrent and bool(use_cuda_graph) and
                      os.environ.get('B200RL_DP_PIPELINE', '1') != '0')
    # The same pipeline on ONE GPU (B200RL_PIPELINE_1GPU): Adam of step t (HBM-bound, 225 MB) is issued at the start of
    # step t+1's graph on a side stream, torso bucket first; K1 / K3 / the target forward never wait for it, the online
    # pass waits for the torso bucket before conv1 and for the fc1 + head bucket before fc1.  Same values as the serial
    # order (K1 of step t+1 still follows K2 of step t); `flush()` applies the update still in flight.
    self._pipeline1 = (self._px is None and self._world == 1 and self._concurrent and self._fused and bool(use_cuda_graph) and
                       os.environ.get('B200RL_PIPELINE_1GPU', PIPELINE_1GPU_DEFAULT) == '1')
    self._cap_stream = None
    if self._pipeline1:
      self._pipeline = True
      self._fuse_tail = False          # the pipelined update ends with its own target copy + increment
      # The update's CTAs must not queue in front of the step's: the graph is captured on a high-priority stream (its
      # forks too) and only the update's side stream keeps the default (lowest) priority, so K1 / K3 / the forwards take
      # every SM slot the streaming Adam kernel frees (all streams equal: measured 0.281 ms per step, K1 finishing 40 us
      # into the step behind Adam's 1,184 CTAs).
      self._cap_stream = torch.cuda.Stream(device=dev, priority=-1)
      self._side = [torch.cuda.Stream(device=dev, priority=(0 if i == 3 else -1)) for i in range(6)]
    # Early tail (>= 4 ranks, where the exchange is NVLink-bound rather than HBM-bound): the fc1 + head bucket of step
    # t is exchanged as soon as step t's dense backward has produced it, underneath the convolution backward, without
    # waiting for the peers' stores; the torso bucket's exchange at the start of step t+1 ends with the barrier that
    # covers both, and is the only thing the online forwards wait for.
    # Measured on 8 GPUs: 0.500 ms/step with it vs 0.486-0.505 without (same box pool, 500-2000 steps): no clear gain,
    # the exchange contends with the convolution backward for SM slots and L2 -- kept as an option, off by default.
    # Round 2: with the bulk bytes moved by the copy engines (default; B200RL_DP_CE=0 restores the SM-issued kernel:
    # `b200rl_dp_reduce_adam_ce` under the convolution backward of step t, `b200rl_dp_broadcast_ce` beside K1 / K3 / the
    # torso forwards of step t+1) the exchange of the big bucket holds no SM slots at all.  2 GPUs, bf16 dataflow:
    # 0.310 ms per step against 0.341 (one-GPU step 0.295).
    # Measured: the DMA engines move ~310 GB/s per GPU whatever the number of peers or parallel copies (2 GPUs: 53 us per
    # 16 MB phase, step 0.310 ms against 0.341 with the SM kernel; 8 GPUs: 102 + 112 us per step for 2 x 28 MB, step
    # 0.376-0.404 against 0.383), so it only pays where the bucket's shard is big and the peers few.
    # In-switch reduction (B200RL_DP_MC, default where the exchange has a multicast mapping): `b200rl_dp_adam_mc` as the
    # early tail -- the SMs issue one multimem.ld_reduce and one multimem.st per 16 bytes of the OWNED shard (1/R of the
    # bucket), so few resident warps suffice and the links carry 32 MB per direction instead of 56 MB at R = 8.
    # B200RL_DP_REDUCE = sm | ce | mc | mcfused and B200RL_DP_BCAST = ce | mc choose the two halves of the fc1 + head
    # bucket's exchange (mcfused / sm do both in one kernel).  Defaults by world size, from the measurements in DESIGN §6.
    mc_ok = self._px is not None and self._px.multicast
    # Measured (bf16 dataflow, 500 steps, one-GPU step 0.296 ms; reduce+broadcast -> ms per step):
    #   2 GPUs: ce+ce 0.295 | mc+ce 0.311 | ce+mc 0.333 | mcfused 0.330-0.384 | sm (round-1 kernel) 0.341
    #   4 GPUs: ce+ce 0.316 | mc+mc 0.339
    #   8 GPUs: mc+ce 0.328 | ce+ce 0.334 | mc+mc 0.344 | mcfused 0.355 | ce+mc 0.360 | sm 0.383
    # DMA moves ~310 GB/s per GPU however many peers or parallel copies (2 x 28 MB = 214 us per step at 8 GPUs: more than
    # the windows it has to hide in), the in-switch reduction needs few bytes through the SMs but its kernel still holds
    # slots under the convolution backward: the DMA broadcast with the multicast reduce wins at 8, DMA for both below.
    red = os.environ.get('B200RL_DP_REDUCE', '')
    if not red:
      if os.environ.get('B200RL_DP_CE') == '0' and os.environ.get('B200RL_DP_MC', '0') == '0':
        red = 'sm'
      elif os.environ.get('B200RL_DP_MC') == '1' and mc_ok:
        red = 'mcfused'
      else:
        red = 'mc' if (self._world > 4 and mc_ok) else 'ce'
    if red in ('mc', 'mcfused') and not mc_ok:
      red = 'ce'
    bc = os.environ.get('B200RL_DP_BCAST', 'ce')
    if bc == 'mc' and not mc_ok:
      bc = 'ce'
    if not self._pipeline or self._px is None:
      red = 'sm'
    self._dp_reduce, self._dp_bcast = red, (bc if red in ('ce', 'mc') else None)
    self._dp_ce = red == 'ce'          # kept: tests and tools read these
    self._dp_mc = red in ('mc', 'mcfused')
    self._ce_ctas = int(os.environ.get('B200RL_DP_CE_CTAS', '0'))
    self._mc_ctas = int(os.environ.get('B200RL_DP_MC_CTAS', '148'))
    early_default = '1' if red != 'sm' else '0'
    self._early_tail = (self._pipeline and self._px is not None and
                        os.environ.get('B200RL_DP_EARLY_TAIL', early_default) == '1')
    if not self._early_tail:
      self._dp_reduce, self._dp_bcast, self._dp_ce, self._dp_mc = 'sm', None, False, False
    self._inc_done = None            # event: the step counter has been advanced (the early tail reads it)
    self._early_tail_now = False     # true while a graph that contains the early tail exchange is being captured
    self._tail_in_flight = False     # the pending update's fc1 + head bucket has already been exchanged
    self._pending = False            # gradients computed, update not applied yet
    self._applied_host = 0           # host mirror of the device step counter (number of applied updates)
    self._pgraphs = {}
    self._steps_done = 0
    self.kernel_launches_per_step = None

    t = dataset.table
    obs_spec = t.signature[0]
    self._obs_shape = tuple(obs_spec.shape)
    self._obs_dtype = np.dtype(obs_spec.dtype)
    self._act_dtype = np.dtype(t.signature[1].dtype)
    # bf16 dataflow on uint8 frames: K3 writes the first conv layer's row image itself (no conversion pass)
    self._gather_rows = None
    if getattr(network, 'flow', False) and hasattr(network, 'rows_frame_bytes') and not network.rows_frame_bytes():
      raise ValueError(f'precision 2 (the bf16 dataflow) needs frames with a row image; got {network.in_c} channels')
    if (self._fused and getattr(network, 'flow', False) and self._obs_dtype == np.uint8 and
        getattr(dataset, 'supports_gather_rows', True)):
      buf = network.rows_buffer(2 * B, 'all')
      fb = network.rows_frame_bytes()
      if buf is not None and fb:
        self._gather_rows = (buf.data_ptr(), buf.data_ptr() + B * fb, network.geom(0, 1))

  # ------------------------------------------------------------------ one update on the device
  def _obs_view_n(self, rows, n):
    torch = self._torch
    if self._obs_dtype == np.uint8:
      return rows.view((n,) + self._obs_shape)
    return rows.view(getattr(torch, self._obs_dtype.name)).view((n,) + self._obs_shape)

  def _actions_i32(self):
    torch = self._torch
    a = self._dataset.a_tm1
    if self._act_dtype == np.int32:
      return a.view(torch.int32).view(self.B)
    return a.view(getattr(torch, self._act_dtype.name)).view(self.B).to(torch.int32)

  def _stamp(self, slot: int):
    """tools/step_phases.py: global-timer stamps between the phases of the (captured) step; off by default."""
    if self._stamps is not None:
      _capi.load().b200rl_debug_stamp(ctypes.c_void_p(self._stamps.data_ptr()), slot, ctypes.c_void_p(_capi.current_stream()))

  def _mk(self, name: str):
    """tools/step_phases.py (B200RL_FINE=1): a named global-timer mark on the current stream; off by default."""
    if getattr(self._net, 'marks', None) is not None:
      self._net.marks.mark('step.' + name)

  def _forwards(self):
    """K1 sample, K3 gather, the three forward passes (learning.py:117-125) [+ local IS-weight max]."""
    ds, net, tgt = self._dataset, self._net, self._tgt
    st = _capi.current_stream()
    self._stamp(1)
    if self._fused:
      self._forwards_fused()
      self._stamp(2)
      return
    o_tm1, o_t = self._obs_view_n(ds.o_tm1, self.B), self._obs_view_n(ds.o_t, self.B)
    if self._concurrent:
      torch = self._torch
      main = torch.cuda.current_stream()
      start = torch.cuda.Event()
      start.record(main)
      for s in self._side[:2]:
        s.wait_event(start)
      # uint8 frames in tensor-core mode: one fp32 row image per observation batch serves every pass over it
      # (o_t: target + online forward; o_tm1: online forward + conv1's weight gradient)
      shared = hasattr(net, 'prepare_frames')
      rows_t = None
      self._rows_tm1 = None
      with torch.cuda.stream(self._side[0]):
        if shared:
          rows_t = net.prepare_frames(o_t, 't')
          if rows_t is not None:
            rows_ready = torch.cuda.Event()
            rows_ready.record(self._side[0])
            self._side[1].wait_event(rows_ready)
        tkw = dict(rows=rows_t) if rows_t is not None else {}
        tgt.lane(1).forward(o_t, self._bufs_tgt, **tkw)          # learning.py:124
      tgt.lane(0)
      if shared:
        self._rows_tm1 = net.prepare_frames(o_tm1, 'tm1')
      hook = None
      if self._params_ready is not None:
        # pipelined exchange: the torso's parameters (a 0.3 MB bucket, exchanged first) must have landed before the
        # online forwards start; the fc1 + head bucket (31.7 MB) only before their first dense layer
        ev_conv, ev_tail = self._params_ready
        self._params_ready = None
        self._side[1].wait_event(ev_conv)
        main.wait_event(ev_conv)
        hook = lambda: torch.cuda.current_stream().wait_event(ev_tail)
      kw = dict(before_fc1=hook) if hook is not None else {}
      with torch.cuda.stream(self._side[1]):
        net.lane(2).forward(o_t, self._bufs_sel, **kw, **tkw)    # learning.py:125
      if self._rows_tm1 is not None:
        kw = dict(kw, rows=self._rows_tm1)
      net.lane(0).forward(o_tm1, self._bufs_train, **kw)         # learning.py:123
      for s in self._side[:2]:
        done = torch.cuda.Event()
        done.record(s)
        main.wait_event(done)
    else:
      self._rows_tm1 = None
      net.forward(o_tm1, self._bufs_train)                       # learning.py:123
      tgt.forward(o_t, self._bufs_tgt)                           # learning.py:124
      net.forward(o_t, self._bufs_sel)                           # learning.py:125
    self._stamp(2)

  def _forwards_fused(self):
    """Target features on o_t (side stream) beside ONE online pass over the 2B frames [o_tm1; o_t]."""
    torch = self._torch
    ds, net, tgt, B = self._dataset, self._net, self._tgt, self.B
    o_all = self._obs_view_n(ds.o_both, 2 * B)
    o_t = self._obs_view_n(ds.o_t, B)
    main = torch.cuda.current_stream()
    rows_all = rows_t = None
    self._rows_tm1 = None
    if self._gather_rows is not None:
      rows_all = net.rows_buffer(2 * B, 'all')               # written by K3 (b200rl_replay_gather_rows)
      self._rows_tm1 = rows_all
      rows_t = rows_all[B * net.rows_frame_bytes():]
    elif hasattr(net, 'prepare_frames'):
      rows_all = net.prepare_frames(o_all, 'all')            # one row image of the 2B frames
      if rows_all is not None:
        self._rows_tm1 = rows_all                            # its first B frames: conv1's weight gradient
        fb = net.rows_frame_bytes()
        if fb:                                               # bf16 dataflow: the target pass reads the image's second half
          rows_t = rows_all[B * fb:]
    hook = None
    if self._params_ready is not None:
      ev_conv, ev_tail = self._params_ready
      self._params_ready = None
    else:
      ev_conv = ev_tail = None
    if self._concurrent:
      side = self._side[0]
      start = torch.cuda.Event()
      start.record(main)
      side.wait_event(start)
      with torch.cuda.stream(side):
        if rows_all is not None and rows_t is None:
          rows_t = tgt.prepare_frames(o_t, 't')              # precision 1: the row image cannot be sliced
        tgt.lane(1).features(o_t, self._bufs_tgt, **(dict(rows=rows_t) if rows_t is not None else {}))   # learning.py:124
        done = torch.cuda.Event()
        done.record(side)
      tgt.lane(0)
      if ev_conv is not None:
        # pipelined exchange: the torso's parameters (a 0.3 MB bucket, exchanged first) must have landed before the
        # online pass starts; the fc1 + head bucket (31.7 MB) only before its dense layer
        main.wait_event(ev_conv)
        hook = lambda: torch.cuda.current_stream().wait_event(ev_tail)
      kw = dict(before_fc1=hook) if hook is not None else {}
      if rows_all is not None:
        kw['rows'] = rows_all
      net.lane(0).features(o_all, self._bufs_on, **kw)       # learning.py:123 and :125 in one pass
      main.wait_event(done)
    else:
      if rows_all is not None and rows_t is None:
        rows_t = tgt.prepare_frames(o_t, 't')
      tgt.features(o_t, self._bufs_tgt, **(dict(rows=rows_t) if rows_t is not None else {}))
      if ev_conv is not None:
        main.wait_event(ev_conv)
        main.wait_event(ev_tail)
      net.features(o_all, self._bufs_on, **(dict(rows=rows_all) if rows_all is not None else {}))

  def _sample(self, uniforms=None):
    """K1, and in data-parallel mode the local max importance weight: its all-reduce(MAX) (one f64) is issued right
    after this and hides behind the gather and the forward passes."""
    ds = self._dataset
    self._bump_in_tail = self._fuse_tail and uniforms is None
    ds.sample_only(uniforms, bump=not self._fuse_tail)
    if self._world > 1 or self._fused:
      torch = self._torch
      aux = self._side[2] if (self._concurrent and (self._px is not None or self._world == 1)) else None
      if aux is not None:           # the exchange waits for the slowest rank: keep it off the gather / forward path
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream())
        aux.wait_event(ev)
      with torch.cuda.stream(aux) if aux is not None else contextlib.nullcontext():
        _capi.call('b200rl_is_weight_max', self.B, _capi.ptr(ds.prob), self._beta, _capi.ptr(self._wmax), self._td_flags,
                   _capi.current_stream())
        if self._px is not None:    # all-reduce(MAX) through the peers' mailboxes, inside the captured step
          # epoch = the dataset's draw counter: unlike the step counter it is not touched by a pipelined update
          self._px.max_f64_(self._wmax, self._dataset.counter)
        if aux is not None:
          self._wmax_done = torch.cuda.Event()
          self._wmax_done.record(aux)

  def _rows_kw(self):
    rows = getattr(self, '_rows_tm1', None)
    return dict(rows=rows) if rows is not None else {}

  def _loss_backward(self, part: str = 'all'):
    """K4 (learning.py:127-154) and the backward pass through net(o_tm1).  `part` lets the data-parallel
    step cut the backward in two ('dense' = loss + head + fc1, 'conv' = the torso) so that the all-reduce
    of the fc1/head gradients (99% of the bytes) overlaps the convolution backward."""
    ds, net = self._dataset, self._net
    o_tm1 = self._obs_view_n(ds.o_tm1, self.B)
    if part == 'conv':
      net.backward_conv_part(o_tm1, self._bufs_train, self._gbufs, self._side[0], **self._rows_kw())
      return
    st = _capi.current_stream()
    if self._wmax_done is not None:
      self._torch.cuda.current_stream().wait_event(self._wmax_done)
      self._wmax_done = None
    if self._fused:
      self._head_td_fused(part)
      return
    wmax = _capi.ptr(self._wmax) if self._world > 1 else None
    _capi.call('b200rl_dqn_td', self.B, net.A, _capi.ptr(self._bufs_train['q']), _capi.ptr(self._bufs_tgt['q']),
               _capi.ptr(self._bufs_sel['q']), _capi.ptr(self._actions_i32()), _capi.ptr(ds.R), _capi.ptr(ds.D),
               _capi.ptr(ds.prob), self._discount, self._delta, self._beta, self._max_abs_reward, wmax, 1.0 / self.B,
               _capi.ptr(self.td), _capi.ptr(self.loss_ps), _capi.ptr(self.weight), _capi.ptr(self.priority),
               _capi.ptr(self.dq), _capi.ptr(self.loss), self._td_flags, st)
    self._stamp(3)
    if part == 'dense':
      net.backward_dense_part(self._bufs_train, self._gbufs, self.dq, self._side[0])
    elif self._concurrent:
      net.backward_dense_part(self._bufs_train, self._gbufs, self.dq, self._side[0])
      if self._early_tail_now:
        torch = self._torch
        main, side = torch.cuda.current_stream(), self._side[4]
        ev = torch.cuda.Event()
        ev.record(main)
        side.wait_event(ev)
        if self._inc_done is not None:
          side.wait_event(self._inc_done)
          self._inc_done = None
        with torch.cuda.stream(side):
          self._early_tail_exchange()
          self._early_done = torch.cuda.Event()
          self._early_done.record(side)
      net.backward_conv_part(o_tm1, self._bufs_train, self._gbufs, self._side[0], **self._rows_kw())
    else:
      net.backward(o_tm1, self._bufs_train, self._gbufs, self.dq)

  def _head_td_fused(self, part: str):
    """The three duelling heads + K4 + dh in one launch, then the backward through fc1 and the torso."""
    torch = self._torch
    ds, net, tgt, B = self._dataset, self._net, self._tgt, self.B
    on, tg, gb = self._bufs_on, self._bufs_tgt, self._gbufs
    h_on = on['h']
    wv, bv, wa, ba = net.head_params()
    twv, tbv, twa, tba = tgt.head_params()
    q = self._q3
    flow = bool(getattr(net, 'flow', False))
    _capi.call('b200rl_dqn_head_td', B, net.A, 512, h_on.data_ptr(), h_on.data_ptr() + 4 * B * 1024, tg['h'].data_ptr(), 1024,
               wv, bv, wa, ba, twv, tbv, twa, tba, _capi.ptr(self._actions_i32()), _capi.ptr(ds.R), _capi.ptr(ds.D),
               _capi.ptr(ds.prob), self._discount, self._delta, self._beta, self._max_abs_reward, _capi.ptr(self._wmax),
               1.0 / B, self._td_flags, q[0].data_ptr(), q[1].data_ptr(), q[2].data_ptr(), _capi.ptr(self.td),
               _capi.ptr(self.loss_ps), _capi.ptr(self.weight), _capi.ptr(self.priority), _capi.ptr(self.dq),
               gb['dval'].data_ptr(), gb['dadv'].data_ptr(), gb['dh'].data_ptr(), 1024, int(flow), _capi.current_stream())
    self._stamp(3)
    # the scalar loss (learning.py:143-144) is only logged: off the critical path
    if self._concurrent:
      main, aux = torch.cuda.current_stream(), self._side[2]
      ev = torch.cuda.Event()
      ev.record(main)
      aux.wait_event(ev)
      with torch.cuda.stream(aux):
        _capi.call('b200rl_mean', B, _capi.ptr(self.loss_ps), _capi.ptr(self.loss), _capi.current_stream())
        if self._world == 1 and self._replay_client is not None:
          # K2 (learning.py:151-154) only needs K4's priorities: on one GPU it runs beside the backward instead of beside
          # Adam, which then has the HBM to itself
          ds.table.update_priorities_device(ds.keys, self.priority)
          self._k2_done = True
        self._loss_done = torch.cuda.Event()
        self._loss_done.record(aux)
    else:
      _capi.call('b200rl_mean', B, _capi.ptr(self.loss_ps), _capi.ptr(self.loss), _capi.current_stream())
    o_tm1 = self._obs_view_n(ds.o_tm1, B)
    bt = self._bufs_train
    if part == 'dense':
      net.backward_dense_part(bt, gb, None, self._side[0])
    elif self._concurrent:
      hook = None
      if self._early_tail_now:
        # data parallel: the fc1 + head bucket is exchanged as soon as its gradients (and fc1's data gradient, the last
        # reader of its weights) are done, underneath the convolution backward
        def hook(events):
          side = self._side[4]
          for ev in events:
            side.wait_event(ev)
          if self._inc_done is not None:      # the exchange reads the step counter: after the previous update's increment
            side.wait_event(self._inc_done)
            self._inc_done = None
          with torch.cuda.stream(side):
            self._early_tail_exchange()
            self._early_done = torch.cuda.Event()
            self._early_done.record(side)
      net.backward_after_head(o_tm1, bt, gb, self._side[0], self._side[1], on_dense_done=hook, **self._rows_kw())
    else:
      net.head_wgrad(bt, gb)
      net.backward_from_dh(o_tm1, bt, gb, **self._rows_kw())
    if getattr(self, '_loss_done', None) is not None:
      torch.cuda.current_stream().wait_event(self._loss_done)
      self._loss_done = None

  def _forward_loss(self):
    self._forwards()
    if self._world > 1 and self._px is None:
      self._dp.global_max_(self._wmax)
    self._loss_backward()
    self._stamp(4)

  def _early_tail_exchange(self):
    """The fc1 + head bucket of this step, exchanged underneath the convolution backward (current stream = a side stream
    that waited for the dense backward)."""
    (o1, n1), _ = self._net.grad_buckets()
    args = (self._m, self._v, self._num_steps, self._lr, 0.9, 0.999, self._adam_eps, self._eps_mode)
    P = self._net.params
    shadow = P.shadow.data_ptr() if P.shadow is not None else None
    if self._dp_reduce == 'mcfused':
      self._mk('mc.start')
      self._px.adam_mc(o1, n1, *args, 0, final_barrier=False, max_ctas=self._mc_ctas)
      self._mk('mc.done')
    elif self._dp_reduce == 'mc':
      self._mk('mc.start')
      self._px.reduce_adam_mc(o1, n1, *args, 0, shadow, self._mc_ctas)
      self._mk('mc.done')
    elif self._dp_reduce == 'ce':
      self._mk('ce.start')
      self._px.reduce_adam_ce(o1, n1, *args, 0, shadow, self._ce_ctas)
      self._mk('ce.done')
    else:
      self._px.adam(o1, n1, *args, 0, final_barrier=False)

  def _adam(self, off: int, n: int):
    """K7 over params[off : off + n] (snt.optimizers.Adam.apply, dqn/learning.py:147-149); with a peer exchange the
    gradient mean over the ranks, Adam on the owned shard and the parameter broadcast are one kernel."""
    if self._px is not None:
      self._px.adam(off, n, self._m, self._v, self._num_steps, self._lr, 0.9, 0.999, self._adam_eps, self._eps_mode, 0)
      self._net.params.refresh_shadow(off, n)
      return
    P, b = self._net.params, 4 * off
    shadow = (P.shadow.data_ptr() + 2 * off) if P.shadow is not None else None      # bf16 dataflow: weights' bf16 copy
    _capi.call('b200rl_adam', n, _capi.ptr(P.flat) + b, _capi.ptr(P.grad) + b, _capi.ptr(self._m) + b,
               _capi.ptr(self._v) + b, _capi.ptr(self._num_steps), self._lr, 0.9, 0.999, self._adam_eps, self._eps_mode,
               _capi.ptr(self._gscale) if self._world > 1 else None, shadow, _capi.current_stream())

  def _apply(self):
    """Adam, priority update, periodic target copy, step counter."""
    net, tgt, st = self._net, self._tgt, _capi.current_stream()
    P = net.params
    prio_done = None
    k2_done, self._k2_done = self._k2_done, False
    if self._replay_client is not None and self._concurrent and not k2_done:
      # K2 only needs the priorities K4 produced: it runs beside the optimizer / exchange
      torch = self._torch
      ev = torch.cuda.Event()
      ev.record(torch.cuda.current_stream())
      self._side[2].wait_event(ev)
      with torch.cuda.stream(self._side[2]):
        self._dataset.table.update_priorities_device(self._dataset.keys, self.priority)   # learning.py:151-154
        prio_done = torch.cuda.Event()
        prio_done.record(self._side[2])
    self._adam(0, P.size)
    self._stamp(5)
    if prio_done is not None:
      self._torch.cuda.current_stream().wait_event(prio_done)
    elif self._replay_client is not None and not k2_done:       # learning.py:151-154
      self._dataset.table.update_priorities_device(self._dataset.keys, self.priority)
    # learning.py:157-161: copy when num_steps % period == 0, evaluated before the increment
    if self._fuse_tail:
      T = tgt.params
      sh = P.shadow is not None and T.shadow is not None
      _capi.call('b200rl_learner_tail', P.size * 4, _capi.ptr(T.flat), _capi.ptr(P.flat), P.size * 2 if sh else 0,
                 _capi.ptr(T.shadow) if sh else None, _capi.ptr(P.shadow) if sh else None, _capi.ptr(self._num_steps),
                 self._period, self._copy_phase, _capi.ptr(self._dataset.counter) if self._bump_in_tail else None, st)
    else:
      self._target_copy()
      _capi.call('b200rl_step_increment', _capi.ptr(self._num_steps), st)
    self._stamp(6)

  def _target_copy(self):
    """learning.py:157-161: target <- online when (num_steps + phase) % period == 0, tested before the increment
    (phase 1 = the JAX learner's post-increment test).  The bf16 weight shadow follows its parameters."""
    P, T, st = self._net.params, self._tgt.params, _capi.current_stream()
    _capi.call('b200rl_copy_if_period', P.size * 4, _capi.ptr(T.flat), _capi.ptr(P.flat), _capi.ptr(self._num_steps),
               self._period, self._copy_phase, st)
    if P.shadow is not None and T.shadow is not None:
      _capi.call('b200rl_copy_if_period', P.size * 2, _capi.ptr(T.shadow), _capi.ptr(P.shadow), _capi.ptr(self._num_steps),
                 self._period, self._copy_phase, st)

  # ---- pipelined exchange (see __init__)
  def _apply_update(self, copy: bool = True, tail_done: bool = False):
    """The optimizer half of a step: exchange + Adam, periodic target copy, step counter.  With a peer exchange: two
    exchanges, torso bucket first, each followed by an event (returned) that the forwards can wait for.  tail_done:
    the fc1 + head bucket of this update was exchanged early (its stores are covered by the torso bucket's barrier)."""
    P, st = self._net.params, _capi.current_stream()
    events = None
    # NOTE: the owner of a parameter's moments is fixed by the bucket partition, so every update of a run must use
    # the same one: with a peer exchange and a bucketed network it is always the two-bucket form
    if self._px is not None and hasattr(self._net, 'grad_buckets'):
      torch = self._torch
      (o1, n1), (o0, n0) = self._net.grad_buckets()
      px, args = self._px, (self._m, self._v, self._num_steps, self._lr, 0.9, 0.999, self._adam_eps, self._eps_mode)
      # torso bucket first (0.3 MB: one barrier round trip), then fc1 + heads (NVLink-bound).  Running the two
      # concurrently was measured slower on 2 GPUs (0.463 vs 0.436 ms): the big kernel delays the small one
      ev_tail = None
      if tail_done and self._dp_bcast is not None:
        # second half of a two-part exchange: DMA pushes (or multicast stores) + barrier on their own stream, beside the
        # torso bucket
        cur, side = torch.cuda.current_stream(), self._side[5]
        ev = torch.cuda.Event()
        ev.record(cur)
        side.wait_event(ev)
        with torch.cuda.stream(side):
          self._mk('push.start')
          if self._dp_bcast == 'mc':
            px.broadcast_mc(o1, n1, self._num_steps, 0, final_barrier=True, max_ctas=self._mc_ctas)
          else:
            px.broadcast_ce(o1, n1, self._num_steps, 0, final_barrier=True)
          self._mk('push.done')
          self._net.params.refresh_shadow(o1, n1)
          self._mk('push.shadow')
          ev_tail = torch.cuda.Event()
          ev_tail.record(side)
      self._mk('torso.start')
      px.adam(o0, n0, *args, 1, final_barrier=True)
      self._mk('torso.done')
      self._net.params.refresh_shadow(o0, n0)
      ev_conv = torch.cuda.Event()
      ev_conv.record(torch.cuda.current_stream())
      if ev_tail is not None:
        torch.cuda.current_stream().wait_event(ev_tail)     # the counter below must not move under the pushes' barrier
      elif tail_done:
        # SM-issued early exchange: the torso bucket's barrier covered its stores; the bf16 shadow follows here
        self._net.params.refresh_shadow(o1, n1)
        ev_tail = torch.cuda.Event()
        ev_tail.record(torch.cuda.current_stream())
      else:
        px.adam(o1, n1, *args, 0, final_barrier=True)
        self._net.params.refresh_shadow(o1, n1)
        ev_tail = torch.cuda.Event()
        ev_tail.record(torch.cuda.current_stream())
      events = (ev_conv, ev_tail)
    elif self._pipeline1:
      torch = self._torch
      (o1, n1), (o0, n0) = self._net.grad_buckets()
      self._adam(o0, n0)                 # torso: 0.3 MB, what conv1 of the next online pass waits for
      ev_conv = torch.cuda.Event()
      ev_conv.record(torch.cuda.current_stream())
      self._adam(o1, n1)                 # fc1 + heads: 99% of the bytes, needed only before fc1
      ev_tail = torch.cuda.Event()
      ev_tail.record(torch.cuda.current_stream())
      events = (ev_conv, ev_tail)
    else:
      self._adam(0, P.size)
    if copy:
      self._target_copy()
    _capi.call('b200rl_step_increment', _capi.ptr(self._num_steps), st)
    if tail_done and events is not None:
      # the early tail exchange of THIS graph reads the step counter: it (not the forwards) waits for the increment
      self._inc_done = self._torch.cuda.Event()
      self._inc_done.record(self._torch.cuda.current_stream())
    return events

  def _compute(self, uniforms=None):
    """The gradient half of a step: K1, K3, forwards, K4, backward, K2."""
    self._stamp(0)
    self._mk('start')
    self._sample(uniforms)
    self._mk('k1')
    self._dataset.gather_only(self._gather_rows)
    self._mk('k3')
    self._forwards()
    self._loss_backward()
    self._stamp(4)
    self._mk('bwd.done')
    if self._replay_client is not None and not self._k2_done:
      self._dataset.table.update_priorities_device(self._dataset.keys, self.priority)
    self._k2_done = False
    self._stamp(5)
    if self._early_tail_now:
      self._torch.cuda.current_stream().wait_event(self._early_done)
    self._stamp(6)

  def _pipelined_graph(self, variant: str):
    torch = self._torch

    def body():
      self._early_tail_now = self._early_tail
      self._inc_done = None
      if variant == 'copy':          # the target network changes in this update: strict order
        self._apply_update(copy=True, tail_done=self._early_tail)
      elif variant == 'norm':        # update on a side stream; only the online forwards wait for it
        main, side = torch.cuda.current_stream(), self._side[3]
        ev = torch.cuda.Event()
        ev.record(main)
        side.wait_event(ev)
        with torch.cuda.stream(side):
          self._params_ready = self._apply_update(copy=False, tail_done=self._early_tail)
          if self._params_ready is None:
            ev = torch.cuda.Event()
            ev.record(side)
            self._params_ready = (ev, ev)
          self._update_done = torch.cuda.Event()     # the side stream must rejoin the capture's origin stream
          self._update_done.record(side)
      self._compute()
      if variant == 'norm':
        torch.cuda.current_stream().wait_event(self._update_done)
      self._early_tail_now = False
    g = self._capture(body)
    if self._px is not None:
      import torch.distributed as dist
      dist.barrier(group=self._dp.group)      # every rank has the graph before anyone spins on a peer
    return g

  def _pipelined_step(self, uniforms):
    if not self._use_graph or uniforms is not None or self._steps_done < 2:
      lib = _capi.load()
      n0 = lib.b200rl_launch_count()
      had_update = self._pending
      self.flush()
      self._compute(uniforms)
      self._pending = True
      self._tail_in_flight = False
      if had_update:
        self.kernel_launches_per_step = int(lib.b200rl_launch_count() - n0)
      return
    if self._early_tail and self._pending and not self._tail_in_flight:
      self.flush()                     # graphs assume the pending update's big bucket was exchanged by the previous graph
    if not self._pending:
      variant = 'first'
    else:
      variant = 'copy' if (self._applied_host + self._copy_phase) % self._period == 0 else 'norm'
    if not self._pgraphs:              # all three at once: no capture (and no host barrier) later inside a run
      for v in ('first', 'norm', 'copy'):
        self._pgraphs[v] = self._pipelined_graph(v)
    self._pgraphs[variant].replay()
    if self._pending:
      self._applied_host += 1
    self._pending = True
    self._tail_in_flight = self._early_tail

  def flush(self):
    """Applies the optimizer update still in flight (pipelined exchange only; COLLECTIVE: all ranks call it together).
    Called by save() / state / num_steps; get_variables() does not (actors lag by that one update)."""
    if self._pending:
      self._apply_update(copy=True, tail_done=self._tail_in_flight)
      self._applied_host += 1
      self._pending = False
      self._tail_in_flight = False

  def _eager_step(self, uniforms):
    lib = _capi.load()
    n0 = lib.b200rl_launch_count()
    self._sample(uniforms)
    self._dataset.gather_only(self._gather_rows)
    self._forward_loss()
    if self._px is None:
      self._dp.sum_(self._net.params.grad)   # all-reduce(SUM); Adam multiplies by 1/R (mean), then applies
    self._apply()
    self.kernel_launches_per_step = int(lib.b200rl_launch_count() - n0)

  def _capture(self, fn):
    torch = self._torch
    g = torch.cuda.CUDAGraph()
    torch.cuda.synchronize()
    with (torch.cuda.graph(g, stream=self._cap_stream) if self._cap_stream is not None else torch.cuda.graph(g)):
      fn()
    return g

  def _device_step(self, uniforms=None):
    """One update on the device.
    * single GPU: the whole step is ONE CUDA graph (forks onto side streams inside it);
    * data parallel with a peer exchange (default): `_pipelined_step` -- one graph per step, the optimizer half of step
      t at the start of step t+1's graph; B200RL_DP_PIPELINE=0 keeps the exchange at the end of the same graph;
    * data parallel over NCCL (`peer_exchange=False`): 4-5 graphs with the all-reduces issued between them (the fc1 +
      head bucket asynchronously, overlapped with the convolution backward).
    The first two steps of a run are eager (one-time attribute set-up inside the library, launch counting)."""
    if self._pipeline:
      self._pipelined_step(uniforms)
      return
    if not self._use_graph or uniforms is not None or self._steps_done < 2:
      self._eager_step(uniforms)      # also the un-captured warm-up (one-time attribute setup inside the library)
      return
    if self._graphs is None:
      if self._world == 1 or self._px is not None:
        def whole():
          self._stamp(0)
          self._sample()
          self._dataset.gather_only(self._gather_rows)
          self._forward_loss()
          self._apply()
        self._graphs = [self._capture(whole)]
        if self._px is not None:
          import torch.distributed as dist
          dist.barrier(group=self._dp.group)    # every rank has its graph before anyone spins on a peer
      else:
        def second():
          self._dataset.gather_only(self._gather_rows)
          self._forwards()
        if self._concurrent:
          self._graphs = [self._capture(self._sample), self._capture(second),
                          self._capture(lambda: self._loss_backward('dense')),
                          self._capture(lambda: self._loss_backward('conv')), self._capture(self._apply)]
        else:
          self._graphs = [self._capture(self._sample), self._capture(second), self._capture(self._loss_backward),
                          self._capture(self._apply)]
    if self._world == 1 or self._px is not None:
      self._graphs[0].replay()
      return
    import torch.distributed as dist
    torch, grp = self._torch, self._dp.group
    g = self._net.params.grad
    self._graphs[0].replay()                      # K1 + local max importance weight
    wmax = dist.all_reduce(self._wmax, op=dist.ReduceOp.MAX, group=grp, async_op=True)   # 1 scalar, hidden behind ...
    self._graphs[1].replay()                      # ... K3 and the three forward passes
    wmax.wait()
    if len(self._graphs) == 4:
      self._graphs[2].replay()
      self._dp.sum_(g)                            # 32 MB of gradients over NVLink; Adam applies the 1/R
      self._graphs[3].replay()
      return
    (o1, n1), (o0, n0) = self._net.grad_buckets()
    self._graphs[2].replay()                      # loss, head and fc1 backward: the tail of the gradient buffer is final
    work = dist.all_reduce(g[o1:o1 + n1], op=dist.ReduceOp.SUM, group=grp, async_op=True)
    self._graphs[3].replay()                      # convolution backward runs while NCCL moves fc1's 31.7 MB
    self._dp.sum_(g[o0:o0 + n0])                  # the convolutions' 0.3 MB
    work.wait()
    self._graphs[4].replay()                      # Adam (x 1/R), priorities, target copy, step counter

  # ------------------------------------------------------------------ acme.core.Learner
  def step(self, uniforms=None, fetch_loss=True):
    """One learner update (`dqn/learning.py:143-163`).  `fetch_loss`: True = read the loss back and log it before
    returning (the reference behaviour); 'async' = copy it to pinned memory without stalling and log it when the NEXT
    step is issued (or at `drain()`), so host-side inserts overlap the device step; False = leave it on the device."""
    table = self._dataset.table
    table.flush()
    if table.size < 1:
      raise RuntimeError('replay is empty: MinSize(1) rate limiter would block')
    self._device_step(uniforms)
    self._steps_done += 1
    result = {}
    if fetch_loss == 'async':
      slot = self._steps_done & 1
      self._loss_ring[slot:slot + 1].copy_(self.loss, non_blocking=True)
      self._loss_events[slot].record()
      previous, self._loss_pending = self._loss_pending, slot
      if previous is not None:
        self._loss_events[previous].synchronize()
        result['loss'] = float(self._loss_ring[previous])
    elif fetch_loss:
      self.drain()
      self._loss_host.copy_(self.loss, non_blocking=True)
      self._torch.cuda.current_stream().synchronize()
      result['loss'] = float(self._loss_host[0])
    timestamp = time.time()
    elapsed = timestamp - self._timestamp if self._timestamp else 0
    self._timestamp = timestamp
    result.update(self._counter.increment(steps=1, walltime=elapsed))
    self._logger.write(result)
    return None

  def drain(self):
    """Logs the loss still in flight from a `fetch_loss='async'` step; returns it (or None)."""
    if self._loss_pending is None:
      return None
    slot, self._loss_pending = self._loss_pending, None
    self._loss_events[slot].synchronize()
    loss = float(self._loss_ring[slot])
    self._logger.write({'loss': loss})
    return loss

  def q_values(self):
    """(q_tm1, q_t_value, q_t_selector) of the last update, device tensors [B, A] (`dqn/learning.py:123-125`)."""
    if self._fused:
      return self._q3[0], self._q3[1], self._q3[2]
    return self._bufs_train['q'], self._bufs_tgt['q'], self._bufs_sel['q']

  def get_variables(self, names: List[str]) -> List[List[np.ndarray]]:
    return [list(self._net.variables().values())]

  @property
  def num_steps(self) -> int:
    self.flush()
    return int(self._num_steps.item())

  @property
  def state(self):
    self.flush()
    return {'network': self._net, 'target_network': self._tgt, 'optimizer': (self._m, self._v),
            'num_steps': self._num_steps}

  def save(self):
    self.flush()
    return {'network': self._net.params.flat.cpu().numpy(), 'target_network': self._tgt.params.flat.cpu().numpy(),
            'adam_m': self._m.cpu().numpy(), 'adam_v': self._v.cpu().numpy(), 'num_steps': self.num_steps}

  def restore(self, state):
    torch = self._torch
    if self._px is not None and int(state['num_steps']) < self._applied_host:
      # the exchange's mailbox flags carry step numbers: going backwards would let barriers pass on stale flags
      raise RuntimeError('restore() to an earlier step is not supported while a peer exchange is live; '
                         'build a new learner and restore into it')
    self._pending = False
    self._applied_host = int(state['num_steps'])
    self._net.params.flat.copy_(torch.as_tensor(state['network']))
    self._tgt.params.flat.copy_(torch.as_tensor(state['target_network']))
    self._m.copy_(torch.as_tensor(state['adam_m']))
    self._v.copy_(torch.as_tensor(state['adam_v']))
    self._num_steps.fill_(int(state['num_steps']))
    self._net.params.refresh_shadow()
    self._tgt.params.refresh_shadow()


class DQN(agent.Agent):
  """`acme/agents/tf/dqn/agent.py:36-167` with the replay, adder, dataset and learner of this package."""

  def __new__(cls, *args, num_envs: int = 1, **kwargs):
    return super().__new__(agent.BatchedAgent.variant_of(cls) if num_envs > 1 else cls)

  def __init__(self, environment_spec: specs.EnvironmentSpec, network, batch_size: int = 256,
               prefetch_size: int = 4, target_update_period: int = 100, samples_per_insert: float = 32.0,
               min_replay_size: int = 1000, max_replay_size: int = 1000000,
               importance_sampling_exponent: float = 0.2, priority_exponent: float = 0.6, n_step: int = 5,
               epsilon: Optional[float] = None, learning_rate: float = 1e-3, discount: float = 0.99,
               logger: loggers.Logger = None, checkpoint: bool = False, checkpoint_subpath: str = '~/acme/',
               seed: int = 0, use_cuda_graph: bool = True, slot_capacity: Optional[int] = None, frame_stack: int = 0,
               num_envs: int = 1):
    """frame_stack: see `replay.Table` -- store one frame per step when the observations are AtariWrapper frame stacks.
    num_envs > 1: the agent is an `agent.BatchedAgent` acting for that many environments at once through
    `actors.BatchedActor` (ε-greedy on the device), to be driven by `environment_loop.BatchedEnvironmentLoop`."""
    table = replay.Table(
        name=replay.DEFAULT_PRIORITY_TABLE, sampler=replay.selectors.Prioritized(priority_exponent),
        remover=replay.selectors.Fifo(), max_size=max_replay_size,
        rate_limiter=replay.rate_limiters.MinSize(1),
        signature=adders.NStepTransitionAdder.signature(environment_spec),
        max_window=max(n_step, 1), discount=discount, device=network.device, slot_capacity=slot_capacity,
        frame_stack=frame_stack)
    self._server = replay.Server([table], port=None)
    address = f'localhost:{self._server.port}'
    replay_client = replay.TFClient(address)
    dataset = replay.make_reverb_dataset(server_address=address, batch_size=batch_size,
                                         prefetch_size=prefetch_size, seed=seed)
    epsilon = 0.05 if epsilon is None else epsilon
    if num_envs > 1:
      actor = actors.BatchedActor(actors.BatchedEpsilonGreedy(network, epsilon, seed=seed), table, num_envs, n_step,
                                  use_cuda_graph=use_cuda_graph)
    else:
      adder = adders.NStepTransitionAdder(client=replay.Client(address), n_step=n_step, discount=discount)
      actor = actors.FeedForwardActor(actors.EpsilonGreedyPolicy(network, epsilon, seed=seed), adder)
    target_network = network.clone()                 # deep-copied parameters (agent.py:127)
    learner = DQNLearner(network=network, target_network=target_network, discount=discount,
                         importance_sampling_exponent=importance_sampling_exponent,
                         learning_rate=learning_rate, target_update_period=target_update_period,
                         dataset=dataset, replay_client=replay_client, logger=logger, checkpoint=checkpoint,
                         use_cuda_graph=use_cuda_graph)
    self._learner_obj = learner
    self._table = table
    super().__init__(actor=actor, learner=learner, min_observations=max(batch_size, min_replay_size),
                     observations_per_step=float(batch_size) / samples_per_insert)
