"""D4PG learner + agent on the B200 hot path.

`D4PGLearner.step()` restates `acme/agents/tf/d4pg/learning.py:156-247` as one stream of kernels:
  target copy (if due) -> K1 sample (uniform table) -> K3 gather/n-step -> critic(o_tm1, a_tm1),
  target_critic(o_t, target_policy(o_t)) -> K5 C51 projection + cross-entropy -> critic backward ->
  policy(o_t) -> critic(o_t, a) -> d mean / d a -> K(dpg) norm-clipped action gradient -> policy
  backward -> global-norm clip (40) of each gradient set -> two Adams.
The reference's D4PG has no importance weights and never writes priorities (uniform table,
`d4pg/agent.py:96-103`); by default neither does this one.

Prioritized replay is an opt-in extension (the D4PG paper evaluates the agent both ways).  With
`importance_sampling_exponent` (beta) the learner computes the batch's maximum importance weight right after K1 (on the
target chain's stream), and the critic loss becomes the importance-weighted mean, with the DQN learner's f64 weights
w = (1 / prob)^beta / max_b (1 / prob)^beta (`dqn/learning.py:138-143`): mean(w * CE) for D4PG, mean(w * 0.5 td^2) for
DDPG.  With a `replay_client` as well, K2 writes the new priorities back for the sampled keys inside the same step: the
unweighted per-sample cross-entropy (D4PG) or |td| (DDPG).  Only the critic loss is weighted; the DPG policy loss stays
unweighted.  The agents take `priority_exponent` and `importance_sampling_exponent` together to build such a learner on a
`Prioritized` table.
"""

from __future__ import annotations

import os
import time
from typing import List, Optional

import numpy as np

from acme_b200 import _capi, actors, adders, agent, core, counting, loggers, networks, parallel, replay, specs


class D4PGLearner(core.Learner, core.Saveable):

  def __init__(self, policy_network: networks.D4PGPolicy, critic_network: networks.D4PGCritic,
               target_policy_network: networks.D4PGPolicy, target_critic_network: networks.D4PGCritic,
               discount: float, target_update_period: int, dataset: replay.ReplayDataset,
               policy_lr: float = 1e-4, critic_lr: float = 1e-4, clipping: bool = True,
               counter: counting.Counter = None, logger: loggers.Logger = None, checkpoint: bool = True,
               eps_mode: int = 0, use_cuda_graph: bool = True, process_group=None,
               importance_sampling_exponent: Optional[float] = None, replay_client: Optional[replay.Client] = None,
               observation_network: Optional[networks.AtariTorso] = None,
               target_observation_network: Optional[networks.AtariTorso] = None):
    """`process_group`: data-parallel learner over per-rank replay shards -- both gradient sets are all-reduced (mean) over
    NCCL between the gradient half and the optimizer half of the step, then clipped and applied identically on every rank
    (the ordering of the reference's only multi-replica learner, `crr/recurrent_learning.py:346-359`).
    `importance_sampling_exponent`: importance-weighted critic loss for a prioritized table (module docstring);
    `replay_client`: also write the new priorities back.  Both None: the reference's uniform, unweighted step.
    `observation_network` / `target_observation_network` (given together): D4PG / DDPG from pixels, see _check_pixels
    and _gradient_half_pixels.  None: observations are the flat state vector (the reference's `batch_concat`)."""
    if replay_client is not None and importance_sampling_exponent is None:
      raise ValueError('replay_client writes priorities for prioritized replay: it needs importance_sampling_exponent')
    if importance_sampling_exponent is not None and process_group is not None:
      raise ValueError('prioritized replay (importance_sampling_exponent) is not supported by the data-parallel learner')
    if importance_sampling_exponent is not None and importance_sampling_exponent < 0:
      raise ValueError('importance_sampling_exponent must be >= 0')
    import torch
    self._torch = torch
    self._obs_net, self._tobs_net = observation_network, target_observation_network
    if (observation_network is None) != (target_observation_network is None):
      raise ValueError('observation_network and target_observation_network are given together')
    if observation_network is not None:
      self._check_pixels(policy_network, critic_network, target_policy_network, target_critic_network, dataset, process_group)
    self._beta = None if importance_sampling_exponent is None else float(importance_sampling_exponent)
    self._replay_client = replay_client
    self._dp = parallel.DataParallel(process_group)
    self._policy, self._critic = policy_network, critic_network
    self._tpolicy, self._tcritic = target_policy_network, target_critic_network
    self._dataset = dataset
    self._discount = float(np.float32(discount))
    self._period = int(target_update_period)
    self._clipping = bool(clipping)
    self._plr, self._clr = float(np.float32(policy_lr)), float(np.float32(critic_lr))
    self._eps_mode = int(eps_mode)
    self._counter = counter or counting.Counter()
    self._logger = logger or loggers.TerminalLogger('learner', time_delta=1.)
    self._timestamp = None
    self._use_graph, self._graph, self._steps_done = bool(use_cuda_graph), None, 0

    dev = torch.device('cuda', critic_network.device)
    # the three independent chains of the step on three streams (see _gradient_half); B200RL_D4PG_STREAMS=0: one stream
    self._concurrent = os.environ.get('B200RL_D4PG_STREAMS', '1') != '0'
    self._side = [torch.cuda.Stream(device=dev) for _ in range(2)] if self._concurrent else None
    B = self.B = dataset.B
    K, A = critic_network.K, policy_network.act_dim
    f32 = lambda *s: torch.zeros(s, dtype=torch.float32, device=dev)
    # the parameter sets that one target copy, clip and Adam cover: with an observation network the critic's set is the
    # torso's and the critic's parameters in one flat buffer (d4pg/learning.py:221-227)
    self._cparams, self._tcparams = critic_network.params, target_critic_network.params
    if observation_network is not None:
      critic_network.split_action_input()
      target_critic_network.split_action_input()
      self._cparams = self._joint(observation_network, critic_network)
      self._tcparams = self._joint(target_observation_network, target_critic_network)
      self._o_bufs, self._o_g = observation_network.make_buffers(B), observation_network.make_grad_buffers(B)
      self._to_bufs = target_observation_network.make_buffers(B)
      sig = dataset.table.signature[0]
      self._obs_shape, self._obs_u8 = tuple(sig.shape), np.dtype(sig.dtype) == np.uint8
      # bf16 dataflow: K3 writes conv1's row images of o_tm1 and o_t while it gathers (as DQNLearner does)
      self._gather_rows = None
      if observation_network.flow and getattr(dataset, 'supports_gather_rows', True):
        buf, fb = observation_network.rows_buffer(2 * B, 'all'), observation_network.rows_frame_bytes()
        self._rows = (buf, buf[B * fb:])
        self._gather_rows = (buf.data_ptr(), buf.data_ptr() + B * fb, observation_network.geom(0, 1))
    self._c_train, self._c_pi, self._c_tgt = (critic_network.make_buffers(B) for _ in range(3))
    self._p_online, self._p_tgt = policy_network.make_buffers(B), target_policy_network.make_buffers(B)
    self._cg_train, self._cg_pi = critic_network.make_grad_buffers(B), critic_network.make_grad_buffers(B)
    self._pg = policy_network.make_grad_buffers(B)
    self.target, self.dlogits, self.dlogits_pi = f32(B, K), f32(B, K), f32(B, K)
    self.critic_loss_ps, self.policy_loss_ps = f32(B), f32(B)
    self.critic_loss, self.policy_loss = f32(1), f32(1)
    self.dqda, self.da = f32(B, A), f32(B, A)
    if observation_network is not None:
      self.dqda = self._cg_pi['da']      # written by the critic's backward (its A action columns only)
    self._pm, self._pv = torch.zeros_like(policy_network.params.flat), torch.zeros_like(policy_network.params.flat)
    self._cm, self._cv = torch.zeros_like(self._cparams.flat), torch.zeros_like(self._cparams.flat)
    self._num_steps = torch.zeros(1, dtype=torch.int64, device=dev)
    if self._beta is not None:
      self.weight, self.priority = f32(B), f32(B)
      self._wmax = torch.zeros(1, dtype=torch.float64, device=dev)
    self._norm_ws, self._norm_ws2 = f32(1024), f32(1024)
    self._pscale, self._cscale, self.policy_norm, self.critic_norm = f32(1), f32(1), f32(1), f32(1)
    self._loss_host = torch.zeros(2, dtype=torch.float32).pin_memory()
    self._loss_ring = torch.zeros(2, 2, dtype=torch.float32).pin_memory()      # fetch_loss='async': two slots
    self._loss_events = [torch.cuda.Event(), torch.cuda.Event()]
    self._loss_pending = None
    self._obs_dim, self._act_dim = critic_network.obs_dim, critic_network.act_dim

  def _check_pixels(self, policy, critic, tpolicy, tcritic, dataset, process_group):
    """The combinations an observation network supports (ValueError otherwise)."""
    o, to = self._obs_net, self._tobs_net
    if process_group is not None:
      raise ValueError('the data-parallel learner does not support an observation network')
    if len({n.precision for n in (o, to, policy, critic, tpolicy, tcritic)}) != 1:
      raise ValueError('the observation network, policy and critic (and their targets) must share one precision')
    for name, n in (('policy', policy), ('critic', critic), ('target policy', tpolicy), ('target critic', tcritic)):
      if n.obs_dim != o.flat_dim:
        raise ValueError(f'the {name} reads {n.obs_dim} inputs but the observation network gives {o.flat_dim} features')
    if to.flat_dim != o.flat_dim or to.params.size != o.params.size:
      raise ValueError('the target observation network must have the observation network\'s architecture')
    sig = dataset.table.signature[0]
    if o.flow and np.dtype(sig.dtype) != np.uint8:
      raise ValueError('precision 2 (the bf16 dataflow) reads uint8 frames: the observation spec must be uint8')
    if int(np.prod(sig.shape)) != o.in_hw * o.in_hw * o.in_c:
      raise ValueError(f'observations of shape {tuple(sig.shape)} are not {o.in_hw} x {o.in_hw} x {o.in_c} frames, the '
                       'observation network\'s input')
    if o.in_c != o.in_cp and np.dtype(sig.dtype) != np.uint8:
      raise ValueError(f'frames of {o.in_c} channels (conv1 padded to {o.in_cp}) must be uint8')
    if o.flow and not o.rows_frame_bytes():
      raise ValueError(f'precision 2 (the bf16 dataflow) needs frames with a row image; got {o.in_c} channels')

  def _joint(self, torso, critic):
    """One flat parameter / gradient (/ bf16 shadow) buffer holding the torso's then the critic's parameters; both
    networks are rebound onto their slices."""
    torch = self._torch
    joint = networks.ParamStore(critic.device)
    nt = torso.params.size
    joint.size = nt + critic.params.size
    joint.allocate()
    if critic.params.shadow is not None:
      joint.shadow = torch.zeros(joint.size, dtype=torch.bfloat16, device=joint.flat.device)
    for net, lo, hi in ((torso, 0, nt), (critic, nt, joint.size)):
      net.params.rebind(joint.flat[lo:hi], joint.grad[lo:hi])
      if joint.shadow is not None:
        net.params.shadow = joint.shadow[lo:hi]
    joint.refresh_shadow()
    return joint

  def _views(self):
    torch, ds, B = self._torch, self._dataset, self.B
    if self._obs_net is not None:
      obs = (lambda x: x.view((B,) + self._obs_shape)) if self._obs_u8 else \
          (lambda x: x.view(torch.float32).view((B,) + self._obs_shape))
      return obs(ds.o_tm1), ds.a_tm1.view(torch.float32).view(B, self._act_dim), obs(ds.o_t)
    o0 = ds.o_tm1.view(torch.float32).view(B, self._obs_dim)
    o1 = ds.o_t.view(torch.float32).view(B, self._obs_dim)
    a0 = ds.a_tm1.view(torch.float32).view(B, self._act_dim)
    return o0, a0, o1

  def _device_step_eager(self, uniforms=None):
    self._gradient_half(uniforms)
    self._exchange()
    self._apply_half()

  def _exchange(self):
    """Data parallel: mean of both gradient sets over the ranks (NCCL all-reduce; not capturable, sits between graphs)."""
    if not self._dp.enabled:
      return
    import torch.distributed as dist
    for net in (self._policy, self._critic):
      g = net.params.grad
      if dist.get_backend(self._dp.group) == 'nccl':
        dist.all_reduce(g, op=dist.ReduceOp.AVG, group=self._dp.group)
      else:
        dist.all_reduce(g, op=dist.ReduceOp.SUM, group=self._dp.group)
        g.mul_(1.0 / self._dp.world)

  def _target_copy(self):
    """learning.py:171-174: target <- online when num_steps % period == 0, before anything else."""
    st = _capi.current_stream()
    for src, dst in ((self._policy.params, self._tpolicy.params), (self._cparams, self._tcparams)):
      _capi.call('b200rl_copy_if_period', src.size * 4, _capi.ptr(dst.flat), _capi.ptr(src.flat),
                 _capi.ptr(self._num_steps), self._period, 0, st)
      if dst.shadow is not None:   # bf16 dataflow: the target's weight operands follow its parameters
        _capi.call('b200rl_copy_if_period', src.size * 2, _capi.ptr(dst.shadow), _capi.ptr(src.shadow),
                   _capi.ptr(self._num_steps), self._period, 0, st)

  def _gradient_half(self, uniforms=None):
    if self._obs_net is not None:
      return self._gradient_half_pixels(uniforms)
    P, C, TP, TC = self._policy, self._critic, self._tpolicy, self._tcritic
    ds, B = self._dataset, self.B
    self._target_copy()
    ds.sample_raw(uniforms)
    o0, a0, o1 = self._views()
    # The step is ~100 small launch-bound kernels; its three chains are independent until the critic loss, so they run
    # on three streams (fork / join by events, also inside the captured graph; one workspace lane per stream):
    #   main  critic(o_tm1, a_tm1)                         -> [join target] critic loss -> critic backward
    #   s1    target policy(o_t) -> target critic(o_t, .)
    #   s2    policy(o_t) -> critic(o_t, .) -> dq/da -> DPG loss -> policy backward
    torch = self._torch
    main = torch.cuda.current_stream()
    fork = self._concurrent
    if fork:
      s1, s2 = self._side
      ev = torch.cuda.Event()
      ev.record(main)
      s1.wait_event(ev)
      s2.wait_event(ev)
    else:
      s1 = s2 = main
    with torch.cuda.stream(s1):
      if self._beta is not None:    # joined before the critic loss with the target chain
        _capi.call('b200rl_is_weight_max', B, _capi.ptr(ds.prob), self._beta, _capi.ptr(self._wmax), 0, _capi.current_stream())
      a_targ = TP.lane(1).action(o1, self._p_tgt)
      logits_t = TC.lane(1).logits(o1, a_targ, self._c_tgt)
      if fork:
        tgt_done = torch.cuda.Event()
        tgt_done.record(s1)
    with torch.cuda.stream(s2):
      # actor learning (learning.py:206-218): dq/da through the online critic, parameters untouched
      st2 = _capi.current_stream()
      a_t = P.lane(2).action(o1, self._p_online)
      logits_pi = C.lane(2).logits(o1, a_t, self._c_pi)
      self._dq_dlogits(logits_pi)
      C.backward_flat(self._c_pi['x'].data_ptr(), self._c_pi, self._cg_pi, self.dlogits_pi.data_ptr(),
                      param_grads=False, input_grad=True)
      _capi.call('b200rl_split_second', B, self._obs_dim, self._act_dim, _capi.ptr(self._cg_pi['dx']), _capi.ptr(self.dqda), st2)
      _capi.call('b200rl_dpg_action_grad', B, self._act_dim, _capi.ptr(self.dqda), 1.0 if self._clipping else 0.0,
                 int(self._clipping), 1.0 / B, _capi.ptr(self.da), _capi.ptr(self.policy_loss_ps), _capi.ptr(self.policy_loss), st2)
      P.backward_action(o1, self._p_online, self._pg, self.da)
      if fork:
        pi_done = torch.cuda.Event()
        pi_done.record(s2)
    # critic learning (learning.py:198-203)
    logits_tm1 = C.lane(0).logits(o0, a0, self._c_train)
    if fork:
      main.wait_event(tgt_done)
    self._critic_loss(logits_tm1, logits_t)
    k2_done = None
    if self._replay_client is not None:   # K2 (learning.py:151-154) beside the critic backward; the next K1 reads the tree
      if fork:
        ev = torch.cuda.Event()
        ev.record(main)
        s1.wait_event(ev)
      with torch.cuda.stream(s1):
        ds.table.update_priorities_device(ds.keys, self.priority)
        if fork:
          k2_done = torch.cuda.Event()
          k2_done.record(s1)
    C.backward_flat(self._c_train['x'].data_ptr(), self._c_train, self._cg_train, self.dlogits.data_ptr(),
                    param_grads=True, input_grad=False)
    if fork:
      main.wait_event(pi_done)
      if k2_done is not None:
        main.wait_event(k2_done)
    for net in (P, C, TP, TC):
      net.lane(0)

  def _gradient_half_pixels(self, uniforms=None):
    """The step with an observation network (d4pg/learning.py:189-195): feat_tm1 = torso(o_tm1) with gradient,
    feat_t = target_torso(o_t) once, without gradient, read by the target chain and by the DPG chain.  Streams:
      main  torso(o_tm1) -> critic -> [join target] critic loss -> critic backward -> torso backward
      s1    target torso(o_t) -> [feat_t ready] target policy -> target critic
      s2    [feat_t] policy -> critic -> dq/da (the critic's A action columns only) -> DPG loss -> policy backward
    The policy loss does not reach the torso; the critic's gradient set is torso + critic (one clip, one Adam)."""
    torch = self._torch
    P, C, TP, TC, O, TO = self._policy, self._critic, self._tpolicy, self._tcritic, self._obs_net, self._tobs_net
    ds, B = self._dataset, self.B
    self._target_copy()
    ds.sample_only(uniforms)
    ds.gather_only(self._gather_rows)
    o0, a0, o1 = self._views()
    rows0, rows1 = self._rows if self._gather_rows is not None else (None, None)
    if O.pads_frames and self._obs_u8:
      # frames padded to 4-channel pixels (precisions 0 and 1): one padded operand per batch, read by forward and backward
      rows0, rows1 = O.prepare_frames(o0, 'tm1'), TO.prepare_frames(o1, 't')
    main = torch.cuda.current_stream()
    fork = self._concurrent
    if fork:
      s1, s2 = self._side
      ev = torch.cuda.Event()
      ev.record(main)
      s1.wait_event(ev)
    else:
      s1 = s2 = main
    with torch.cuda.stream(s1):
      if self._beta is not None:
        _capi.call('b200rl_is_weight_max', B, _capi.ptr(ds.prob), self._beta, _capi.ptr(self._wmax), 0, _capi.current_stream())
      feat_t = TO.lane(1).forward(o1, self._to_bufs, rows=rows1).data_ptr()
      if fork:
        feat_ready = torch.cuda.Event()
        feat_ready.record(s1)
        s2.wait_event(feat_ready)
      a_targ = TP.lane(1).action_features(feat_t, self._p_tgt)
      logits_t = TC.lane(1).forward_features(feat_t, a_targ.data_ptr(), self._c_tgt)
      if fork:
        tgt_done = torch.cuda.Event()
        tgt_done.record(s1)
    with torch.cuda.stream(s2):
      st2 = _capi.current_stream()
      a_t = P.lane(2).action_features(feat_t, self._p_online)
      logits_pi = C.lane(2).forward_features(feat_t, a_t.data_ptr(), self._c_pi)
      self._dq_dlogits(logits_pi)
      C.backward_features(feat_t, a_t.data_ptr(), self._c_pi, self._cg_pi, self.dlogits_pi.data_ptr(), param_grads=False,
                          action_grad=True)
      _capi.call('b200rl_dpg_action_grad', B, self._act_dim, _capi.ptr(self.dqda), 1.0 if self._clipping else 0.0,
                 int(self._clipping), 1.0 / B, _capi.ptr(self.da), _capi.ptr(self.policy_loss_ps), _capi.ptr(self.policy_loss), st2)
      P.backward_action_features(feat_t, self._p_online, self._pg, self.da)
      if fork:
        pi_done = torch.cuda.Event()
        pi_done.record(s2)
    feat0 = O.lane(0).forward(o0, self._o_bufs, rows=rows0)
    logits_tm1 = C.lane(0).forward_features(feat0.data_ptr(), a0.data_ptr(), self._c_train)
    if fork:
      main.wait_event(tgt_done)
    self._critic_loss(logits_tm1, logits_t)
    k2_done = None
    if self._replay_client is not None:
      if fork:
        ev = torch.cuda.Event()
        ev.record(main)
        s1.wait_event(ev)
      with torch.cuda.stream(s1):
        ds.table.update_priorities_device(ds.keys, self.priority)
        if fork:
          k2_done = torch.cuda.Event()
          k2_done.record(s1)
    # the critic's feature gradient goes into conv3's dy through conv3's ReLU
    C.backward_features(feat0.data_ptr(), a0.data_ptr(), self._c_train, self._cg_train, self.dlogits.data_ptr(),
                        param_grads=True, feat_grad=(self._o_g['dy3'].data_ptr(), feat0.data_ptr()))
    O.backward(o0, self._o_bufs, self._o_g, rows=rows0)
    if fork:
      main.wait_event(pi_done)
      if k2_done is not None:
        main.wait_event(k2_done)
    for net in (P, C, TP, TC, O, TO):
      net.lane(0)

  def _critic_loss(self, logits_tm1, logits_t):
    """K5: losses.categorical (distributional.py:22-37) and its gradient w.r.t. logits_tm1 (learning.py:202-203)."""
    C, ds, B = self._critic, self._dataset, self.B
    if self._beta is not None:   # importance-weighted; priority = the unweighted per-sample cross-entropy
      _capi.call('b200rl_c51_loss_weighted', B, C.K, C.vmin, C.vmax, _capi.ptr(logits_tm1), _capi.ptr(logits_t), _capi.ptr(ds.R),
                 _capi.ptr(ds.D), self._discount, _capi.ptr(ds.prob), self._beta, _capi.ptr(self._wmax), 1.0 / B,
                 _capi.ptr(self.target), _capi.ptr(self.critic_loss_ps), _capi.ptr(self.weight), _capi.ptr(self.priority),
                 _capi.ptr(self.dlogits), _capi.ptr(self.critic_loss), _capi.current_stream())
      return
    _capi.call('b200rl_c51_loss', B, C.K, C.vmin, C.vmax, _capi.ptr(logits_tm1), _capi.ptr(logits_t), _capi.ptr(ds.R),
               _capi.ptr(ds.D), self._discount, 1.0 / B, _capi.ptr(self.target), _capi.ptr(self.critic_loss_ps),
               _capi.ptr(self.dlogits), _capi.ptr(self.critic_loss), _capi.current_stream())

  def _dq_dlogits(self, logits_pi):
    """d mean(Z) / d logits of the critic's output at (o_t, policy(o_t)) (distributions.py:64-66; learning.py:206-208)."""
    C, B = self._critic, self.B
    _capi.call('b200rl_c51_mean_bwd', B, C.K, C.vmin, C.vmax, _capi.ptr(logits_pi), None, _capi.ptr(self.dlogits_pi),
               _capi.current_stream())

  def _apply_half(self):
    """clip each gradient set by its global norm (learning.py:235-237), then the two Adams (240-241), step counter."""
    torch = self._torch
    P, C = self._policy, self._critic
    main = torch.cuda.current_stream()

    def update(params, m, v, lr, ws, scale, norm):
      st = _capi.current_stream()
      gs = None
      if self._clipping:
        _capi.call('b200rl_global_norm_scale', params.size, _capi.ptr(params.grad), 40.0, _capi.ptr(ws),
                   _capi.ptr(scale), _capi.ptr(norm), st)
        gs = _capi.ptr(scale)
      _capi.call('b200rl_adam', params.size, _capi.ptr(params.flat), _capi.ptr(params.grad), _capi.ptr(m),
                 _capi.ptr(v), _capi.ptr(self._num_steps), lr, 0.9, 0.999, 1e-8, self._eps_mode, gs, _capi.ptr(params.shadow), st)

    # the two networks' clip + Adam are independent: policy on a side stream beside the critic
    if self._concurrent:
      side = self._side[0]
      ev = torch.cuda.Event()
      ev.record(main)
      side.wait_event(ev)
      with torch.cuda.stream(side):
        update(P.params, self._pm, self._pv, self._plr, self._norm_ws2, self._pscale, self.policy_norm)
        done = torch.cuda.Event()
        done.record(side)
      update(self._cparams, self._cm, self._cv, self._clr, self._norm_ws, self._cscale, self.critic_norm)
      main.wait_event(done)
    else:
      update(P.params, self._pm, self._pv, self._plr, self._norm_ws2, self._pscale, self.policy_norm)
      update(self._cparams, self._cm, self._cv, self._clr, self._norm_ws, self._cscale, self.critic_norm)
    _capi.call('b200rl_step_increment', _capi.ptr(self._num_steps), _capi.current_stream())

  def _device_step(self, uniforms=None):
    torch = self._torch
    if not self._use_graph or uniforms is not None or self._steps_done < 2:
      self._device_step_eager(uniforms)
      return
    if self._graph is None:
      def capture(fn):
        g = torch.cuda.CUDAGraph()
        torch.cuda.synchronize()
        with torch.cuda.graph(g):
          fn()
        return g
      if self._dp.enabled:     # the all-reduces sit between two graphs
        self._graph = (capture(lambda: self._gradient_half(None)), capture(self._apply_half))
      else:
        self._graph = (capture(lambda: self._device_step_eager(None)),)
    self._graph[0].replay()
    if self._dp.enabled:
      self._exchange()
      self._graph[1].replay()

  def step(self, uniforms=None, fetch_loss: bool = True):
    table = self._dataset.table
    table.flush()
    if table.size < 1:
      raise RuntimeError('replay is empty: MinSize(1) rate limiter would block')
    self._device_step(uniforms)
    self._steps_done += 1
    result = {}
    if fetch_loss == 'async':   # copy to pinned memory now, consume when the next step has been issued (or at drain())
      slot = self._steps_done & 1
      self._loss_ring[slot, 0:1].copy_(self.critic_loss, non_blocking=True)
      self._loss_ring[slot, 1:2].copy_(self.policy_loss, non_blocking=True)
      self._loss_events[slot].record()
      previous, self._loss_pending = self._loss_pending, slot
      if previous is not None:
        self._loss_events[previous].synchronize()
        result = {'critic_loss': float(self._loss_ring[previous, 0]), 'policy_loss': float(self._loss_ring[previous, 1])}
    elif fetch_loss:
      self._loss_host[0:1].copy_(self.critic_loss, non_blocking=True)
      self._loss_host[1:2].copy_(self.policy_loss, non_blocking=True)
      self._torch.cuda.current_stream().synchronize()
      result = {'critic_loss': float(self._loss_host[0]), 'policy_loss': float(self._loss_host[1])}
    timestamp = time.time()
    elapsed = timestamp - self._timestamp if self._timestamp else 0
    self._timestamp = timestamp
    result.update(self._counter.increment(steps=1, walltime=elapsed))
    self._logger.write(result)

  def drain(self):
    """The losses still in flight from a `fetch_loss='async'` step (or None)."""
    if self._loss_pending is None:
      return None
    slot, self._loss_pending = self._loss_pending, None
    self._loss_events[slot].synchronize()
    out = {'critic_loss': float(self._loss_ring[slot, 0]), 'policy_loss': float(self._loss_ring[slot, 1])}
    self._logger.write(out)
    return out

  def get_variables(self, names: List[str]) -> List[List[np.ndarray]]:
    nets = {'critic': [self._tcritic], 'policy': [self._tpolicy]}   # learning.py:133-140: target networks
    if self._tobs_net is not None:    # snt.Sequential([target_obs_net, target_policy])
      nets['policy'] = [self._tobs_net, self._tpolicy]
    return [[v for net in nets[name] for v in net.variables().values()] for name in names]

  @property
  def num_steps(self) -> int:
    return int(self._num_steps.item())

  def save(self):
    f = lambda t: t.cpu().numpy()
    # with an observation network 'critic' / 'target_critic' hold the torso's parameters followed by the critic's
    return {'policy': f(self._policy.params.flat), 'critic': f(self._cparams.flat),
            'target_policy': f(self._tpolicy.params.flat), 'target_critic': f(self._tcparams.flat),
            'policy_opt': (f(self._pm), f(self._pv)), 'critic_opt': (f(self._cm), f(self._cv)), 'num_steps': self.num_steps}

  def restore(self, state):
    t = self._torch.as_tensor
    self._policy.params.flat.copy_(t(state['policy']))
    self._cparams.flat.copy_(t(state['critic']))
    self._tpolicy.params.flat.copy_(t(state['target_policy']))
    self._tcparams.flat.copy_(t(state['target_critic']))
    self._pm.copy_(t(state['policy_opt'][0])); self._pv.copy_(t(state['policy_opt'][1]))
    self._cm.copy_(t(state['critic_opt'][0])); self._cv.copy_(t(state['critic_opt'][1]))
    self._num_steps.fill_(int(state['num_steps']))
    for params in (self._policy.params, self._cparams, self._tpolicy.params, self._tcparams):
      params.refresh_shadow()


class DDPGLearner(D4PGLearner):
  """`acme/agents/tf/ddpg/learning.py:140-237`: the D4PG step with a scalar critic -- critic loss = trfl.td_learning
  (0.5 td^2, line 193) instead of the categorical projection, dq/da through the scalar output directly; same target-copy
  timing (before the update, 157-160), DPG loss with dq/da norm clipping, global-norm clip 40, two Adams."""

  def __init__(self, policy_network, critic_network, target_policy_network, target_critic_network, *args, **kwargs):
    super().__init__(policy_network, critic_network, target_policy_network, target_critic_network, *args, **kwargs)
    torch = self._torch
    dev = self.dlogits.device
    self.td = torch.zeros(self.B, dtype=torch.float32, device=dev)
    self._ones = torch.ones((self.B, 1), dtype=torch.float32, device=dev)

  def _critic_loss(self, q_tm1, q_t):
    ds, B = self._dataset, self.B
    if self._beta is not None:   # importance-weighted; priority = |td|
      _capi.call('b200rl_td_learning_weighted', B, _capi.ptr(q_tm1), _capi.ptr(q_t), _capi.ptr(ds.R), _capi.ptr(ds.D),
                 self._discount, _capi.ptr(ds.prob), self._beta, _capi.ptr(self._wmax), 1.0 / B, _capi.ptr(self.td),
                 _capi.ptr(self.critic_loss_ps), _capi.ptr(self.weight), _capi.ptr(self.priority), _capi.ptr(self.dlogits),
                 _capi.ptr(self.critic_loss), _capi.current_stream())
      return
    _capi.call('b200rl_td_learning', B, _capi.ptr(q_tm1), _capi.ptr(q_t), _capi.ptr(ds.R), _capi.ptr(ds.D), self._discount,
               1.0 / B, _capi.ptr(self.td), _capi.ptr(self.critic_loss_ps), _capi.ptr(self.dlogits), _capi.ptr(self.critic_loss),
               _capi.current_stream())

  def _dq_dlogits(self, q_pi):
    self.dlogits_pi.copy_(self._ones)      # d q / d q = 1: the action gradient flows through the scalar output itself


class GaussianNoisePolicy:
  """policy -> ClippedGaussian(sigma) (`acme/agents/tf/d4pg/agent.py:117-123`, networks/noise.py:27-40)."""

  def __init__(self, policy: networks.D4PGPolicy, sigma: float, act_min, act_max, seed: int = 0,
               observation_network: Optional[networks.AtariTorso] = None):
    """observation_network: the policy acts on its features (the online torso, as the single-process agent does)."""
    import torch
    self._p, self._sigma, self._torch = policy, float(sigma), torch
    self._lo, self._hi = np.asarray(act_min, np.float32), np.asarray(act_max, np.float32)
    self._rng = np.random.default_rng(seed)
    self._bufs = policy.make_buffers(1)
    self._torso = observation_network
    if observation_network is not None:
      self._tbufs = observation_network.make_buffers(1)

  def __call__(self, observation):
    if self._torso is not None:
      obs = self._torch.as_tensor(np.ascontiguousarray(observation)[None]).cuda(self._p.device)
      feat = self._torso.forward(obs, self._tbufs)
      a = self._p.action_features(feat.data_ptr(), self._bufs).cpu().numpy()[0]
    else:
      obs = self._torch.as_tensor(np.ascontiguousarray(observation, dtype=np.float32).reshape(1, -1)).cuda(self._p.device)
      a = self._p.action(obs, self._bufs).cpu().numpy()[0]
    a = a + self._rng.standard_normal(a.shape).astype(np.float32) * self._sigma
    return np.clip(a, self._lo, self._hi).astype(np.float32)


class D4PG(agent.Agent):
  """`acme/agents/tf/d4pg/agent.py:36-180`: uniform table, n-step adder, dataset, actor, learner.  With
  `priority_exponent` (alpha) and `importance_sampling_exponent` (beta), given together, the table is
  `Prioritized(alpha)` and the learner weights its critic loss and writes priorities back (`D4PGLearner`); new items
  enter with priority 1.0, as the reference adder's constant `priority_fns` gives them."""

  _learner_cls = D4PGLearner

  def __new__(cls, *args, num_envs: int = 1, **kwargs):
    return super().__new__(agent.BatchedAgent.variant_of(cls) if num_envs > 1 else cls)

  def __init__(self, environment_spec: specs.EnvironmentSpec, policy_network: networks.D4PGPolicy,
               critic_network: networks.D4PGCritic, discount: float = 0.99, batch_size: int = 256,
               prefetch_size: int = 4, target_update_period: int = 100, min_replay_size: int = 1000,
               max_replay_size: int = 1000000, samples_per_insert: float = 32.0, n_step: int = 5,
               sigma: float = 0.3, clipping: bool = True, logger: loggers.Logger = None, checkpoint: bool = False,
               seed: int = 0, use_cuda_graph: bool = True, num_envs: int = 1,
               priority_exponent: Optional[float] = None, importance_sampling_exponent: Optional[float] = None,
               observation_network: Optional[networks.AtariTorso] = None, frame_stack: int = 0):
    """observation_network: D4PG / DDPG from pixels -- the policy and the critic read the features of this torso, trained
    by the critic loss; its target is a clone.  frame_stack: see `replay.Table` (store one frame per step when the
    observations are frame stacks).
    num_envs > 1: the agent is an `agent.BatchedAgent` acting for that many environments at once through
    `actors.BatchedActor` (Gaussian exploration on the device), to be driven by `environment_loop.BatchedEnvironmentLoop`.
    priority_exponent / importance_sampling_exponent: prioritized replay (both or neither; the default is uniform)."""
    if (priority_exponent is None) != (importance_sampling_exponent is None):
      raise ValueError('prioritized replay needs both priority_exponent and importance_sampling_exponent')
    prioritized = priority_exponent is not None
    sampler = replay.selectors.Prioritized(priority_exponent) if prioritized else replay.selectors.Uniform()
    table = replay.Table(name=replay.DEFAULT_PRIORITY_TABLE, sampler=sampler,
                         remover=replay.selectors.Fifo(), max_size=max_replay_size,
                         rate_limiter=replay.rate_limiters.MinSize(1),
                         signature=adders.NStepTransitionAdder.signature(environment_spec), max_window=n_step,
                         discount=discount, device=critic_network.device, frame_stack=frame_stack)
    self._server = replay.Server([table], port=None)
    address = f'localhost:{self._server.port}'
    dataset = replay.make_reverb_dataset(server_address=address, batch_size=batch_size, prefetch_size=prefetch_size,
                                         seed=seed, stratified=False)
    aspec = environment_spec.actions
    # the observation-network arguments are passed only when there is one: the flat-state wiring is unchanged
    torso = {} if observation_network is None else dict(observation_network=observation_network)
    if num_envs > 1:
      actor = actors.BatchedActor(actors.BatchedGaussianNoise(policy_network, sigma, aspec.minimum, aspec.maximum, seed, **torso),
                                  table, num_envs, n_step, use_cuda_graph=use_cuda_graph)
    else:
      # the reference passes priority_fns={table: lambda x: 1.} (agent.py:108): the default does the same
      adder = adders.NStepTransitionAdder(client=replay.Client(address), n_step=n_step, discount=discount)
      actor = actors.FeedForwardActor(GaussianNoisePolicy(policy_network, sigma, aspec.minimum, aspec.maximum, seed, **torso),
                                      adder)
    learner = self._learner_cls(policy_network, critic_network, policy_network.clone(), critic_network.clone(), discount,
                                target_update_period, dataset, clipping=clipping, logger=logger, checkpoint=checkpoint,
                                use_cuda_graph=use_cuda_graph, importance_sampling_exponent=importance_sampling_exponent,
                                replay_client=replay.TFClient(address) if prioritized else None,
                                **({} if observation_network is None else
                                   dict(observation_network=observation_network,
                                        target_observation_network=observation_network.clone())))
    self._table = table
    super().__init__(actor=actor, learner=learner, min_observations=max(batch_size, min_replay_size),
                     observations_per_step=float(batch_size) / samples_per_insert)


class DDPG(D4PG):
  """`acme/agents/tf/ddpg/agent.py:36-173`: the same single-process wiring (uniform table, n-step adder with constant
  priorities, Gaussian-noise behaviour policy clipped to the action spec, two Adams at 1e-4) around `DDPGLearner`;
  `critic_network` is a scalar critic (`networks.DDPGCritic`)."""

  _learner_cls = DDPGLearner
