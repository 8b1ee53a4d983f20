"""FeedForwardActor (`acme/agents/tf/actors.py:35-94`): batch-1 policy forward on the learner's own
network object (actor and learner share parameters, like the single-process reference agent),
forwarding observations to the adder."""

from typing import Callable, Optional

import numpy as np

from acme_b200 import _capi, core, tree


class FeedForwardActor(core.Actor):

  def __init__(self, policy: Callable[[np.ndarray], np.ndarray], adder=None, variable_client=None):
    self._policy, self._adder, self._variable_client = policy, adder, variable_client

  def select_action(self, observation):
    return self._policy(observation)

  def observe_first(self, timestep):
    if self._adder:
      self._adder.add_first(timestep)

  def observe(self, action, next_timestep):
    if self._adder:
      self._adder.add(action, next_timestep)

  def update(self):
    if self._variable_client:
      self._variable_client.update()


class EpsilonGreedyPolicy:
  """snt.Sequential([network, lambda q: trfl.epsilon_greedy(q, eps).sample()])
  (`acme/agents/tf/dqn/agent.py:119-124`): greedy w.p. 1-eps, uniform otherwise."""

  def __init__(self, network, epsilon: float = 0.05, seed: int = 0):
    import torch
    self._net, self._eps = network, float(epsilon)
    self._rng = np.random.default_rng(seed)
    self._bufs = network.make_buffers(1)
    self._torch = torch

  def __call__(self, observation):
    torch = self._torch
    if self._rng.random() < self._eps:
      return np.int32(self._rng.integers(self._net.A))
    obs = torch.as_tensor(np.ascontiguousarray(observation)[None]).cuda(self._net.device)
    q = self._net.forward(obs, self._bufs)
    return np.int32(int(np.argmax(q.cpu().numpy()[0])))  # first max wins, like tf.argmax


# ------------------------------------------------------------------------------------------------ batched acting
class BatchedEpsilonGreedy:
  """The batched form of EpsilonGreedyPolicy: `network.forward` at batch N, then `b200rl_epsilon_greedy` (trfl's
  distribution: a uniformly drawn action among exact ties at the maximum, where the batch-1 policy takes the first)."""

  _SEED_SALT = 0x2545F491   # the actor's draws never coincide with the dataset's (seed) or DQfD's stream

  def __init__(self, network, epsilon: float = 0.05, seed: int = 0):
    self.network, self.epsilon, self.seed = network, float(epsilon), int(seed) ^ self._SEED_SALT
    self.action_dtype, self.action_shape = np.int32, ()

  def allocate(self, N: int):
    import torch
    dev = torch.device('cuda', self.network.device)
    self.bufs = self.network.make_buffers(N)
    self.counter = torch.zeros(1, dtype=torch.int64, device=dev)
    self.actions = torch.empty(N, dtype=torch.int32, device=dev)
    self.values = self.bufs['q']          # the q the actions were selected from

  def act(self, obs):
    """obs: device [N, ...] -> self.actions (one draw per row at the current counter; the caller advances it)."""
    net, N = self.network, obs.shape[0]
    rows = net.prepare_frames(obs, 'act') if hasattr(net, 'prepare_frames') else None
    q = net.forward(obs, self.bufs, rows=rows) if rows is not None else net.forward(obs, self.bufs)
    _capi.call('b200rl_epsilon_greedy', N, net.A, _capi.ptr(q), q.stride(0), self.epsilon, self.seed, _capi.ptr(self.counter),
               _capi.ptr(self.actions), None, _capi.current_stream())
    return self.actions


class BatchedGaussianNoise:
  """The batched form of d4pg.GaussianNoisePolicy: `policy.action` at batch N, then `b200rl_gaussian_explore` (the same
  float32 arithmetic, clip(a + z * sigma, lo, hi), with device Box-Muller draws instead of NumPy's)."""

  _SEED_SALT = BatchedEpsilonGreedy._SEED_SALT

  def __init__(self, policy, sigma: float, act_min, act_max, seed: int = 0, observation_network=None):
    """observation_network (networks.AtariTorso): the policy reads its features (conv1's row image in its own 'act'
    slot)."""
    self.network, self.sigma, self.seed = policy, float(np.float32(sigma)), int(seed) ^ self._SEED_SALT
    self.torso = observation_network
    A = policy.act_dim
    self._lo = np.ascontiguousarray(np.broadcast_to(np.asarray(act_min, np.float32), (A,)))
    self._hi = np.ascontiguousarray(np.broadcast_to(np.asarray(act_max, np.float32), (A,)))
    self.action_dtype, self.action_shape = np.float32, (A,)

  def allocate(self, N: int):
    import torch
    dev = torch.device('cuda', self.network.device)
    self.bufs = self.network.make_buffers(N)
    if self.torso is not None:
      self.torso_bufs = self.torso.make_buffers(N)
    self.counter = torch.zeros(1, dtype=torch.int64, device=dev)
    self.lo, self.hi = torch.as_tensor(self._lo).to(dev), torch.as_tensor(self._hi).to(dev)
    self.actions = torch.empty((N, self.network.act_dim), dtype=torch.float32, device=dev)
    self.values = self.bufs['a']          # the noiseless policy actions

  def act(self, obs):
    N, A = obs.shape[0], self.network.act_dim
    if self.torso is not None:
      feat = self.torso.forward(obs, self.torso_bufs, rows=self.torso.prepare_frames(obs, 'act'))
      a = self.network.action_features(feat.data_ptr(), self.bufs)
    else:
      a = self.network.action(obs, self.bufs)
    _capi.call('b200rl_gaussian_explore', N, A, _capi.ptr(a), self.sigma, _capi.ptr(self.lo), _capi.ptr(self.hi), self.seed,
               _capi.ptr(self.counter), _capi.ptr(self.actions), None, _capi.current_stream())
    return self.actions


class BatchedActor:
  """Acts for N environments stepped in lockstep and records their steps with one insert per step.

  `select_actions(observations[N])` stages the rows in pinned memory and replays ONE CUDA graph (captured on first use):
  host-to-device copy of the rows, the policy's forward at batch N, its exploration kernel, the draw-counter increment and
  the device-to-host copy of the actions; then one synchronise.  `observe(actions, next_timesteps)` records, through
  `Table.append_multi`, each environment's observation the actions were selected from -- read from the device rows the
  forward read, so in the common case an observation crosses PCIe once -- with its action, reward and discount; a
  step's item therefore becomes sampleable when that environment's next observation is recorded.  Terminal observations
  are not acted on; they are recorded from host memory by a second insert in the steps where an episode ends, so every
  finished episode's items are in the table when `observe` returns.  The caller resets an environment whose timestep is
  LAST before the next `select_actions`.  Items use the reference's default priority 1.0.

  Protocol (BatchedEnvironmentLoop): observe_first(timesteps) once, then select_actions -> observe -> update per step."""

  def __init__(self, policy, table, num_envs: int, n_step: int, use_cuda_graph: bool = True):
    import torch
    if num_envs < 1:
      raise ValueError('num_envs must be at least 1')
    sig = table.signature
    if sig is None or tree.is_nest(sig[0]):
      raise ValueError('the batched actor needs a single-array observation spec')
    if table.is_sequence or table.has_extras:
      raise ValueError(f'table {table.name!r}: the batched actor writes transition tables without extras')
    self.num_envs, self.policy, self._table, self._n_step = int(num_envs), policy, table, int(n_step)
    self._use_graph, self._graph, self._graph_ws = bool(use_cuda_graph), None, None
    N = self.num_envs
    self._obs_shape, self._obs_dtype = tuple(int(d) for d in sig[0].shape), np.dtype(sig[0].dtype)
    tdt = getattr(torch, self._obs_dtype.name)
    dev = torch.device('cuda', table.device)
    self._stage = torch.empty((N,) + self._obs_shape, dtype=tdt).pin_memory()
    self._stage_np = self._stage.numpy()
    self.obs_dev = torch.empty((N,) + self._obs_shape, dtype=tdt, device=dev)
    policy.allocate(N)
    self._act_host = torch.empty(tuple(policy.actions.shape), dtype=policy.actions.dtype).pin_memory()
    self._writers = np.asarray([table.open_writer() for _ in range(N)], np.int32)
    self._first = np.ones(N, np.uint8)     # the observation acted on next starts an episode

  def _step(self):
    self.obs_dev.copy_(self._stage, non_blocking=True)
    self.policy.act(self.obs_dev)
    _capi.call('b200rl_step_increment', _capi.ptr(self.policy.counter), _capi.current_stream())
    self._act_host.copy_(self.policy.actions, non_blocking=True)

  def _capture(self):
    import torch
    saved = self.policy.counter.clone()
    self._step()                            # warm-up: allocates row images, loads kernels
    self.policy.counter.copy_(saved)
    torch.cuda.current_stream().synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
      self._step()
    self._graph, self._graph_ws = g, self.policy.network.ws

  def select_actions(self, observations) -> np.ndarray:
    import torch
    np.copyto(self._stage_np, np.asarray(observations, self._obs_dtype).reshape(self._stage_np.shape))
    if not self._use_graph:
      self._step()
    else:
      if self._graph is None or self._graph_ws != self.policy.network.ws:   # precision 3 may regrow the workspace
        self._capture()
      self._graph.replay()
    torch.cuda.current_stream().synchronize()
    return self._act_host.numpy().astype(self.policy.action_dtype, copy=True)

  def observe_first(self, timesteps):
    if len(timesteps) != self.num_envs:
      raise ValueError(f'expected {self.num_envs} timesteps, got {len(timesteps)}')
    self._first[:] = 1

  def observe(self, actions, next_timesteps):
    N = self.num_envs
    if len(next_timesteps) != N:
      raise ValueError(f'expected {N} timesteps, got {len(next_timesteps)}')
    rew = np.fromiter((ts.reward for ts in next_timesteps), np.float32, N)
    disc = np.fromiter((ts.discount for ts in next_timesteps), np.float32, N)
    last = np.fromiter((ts.last() for ts in next_timesteps), np.uint8, N)
    self._table.append_multi(self._writers, self.obs_dev, actions, rew, disc, self._first, np.zeros(N, np.uint8), self._n_step)
    ends = np.flatnonzero(last)
    if ends.size:
      term = np.stack([np.asarray(next_timesteps[i].observation, self._obs_dtype) for i in ends])
      k = ends.size
      self._table.append_multi(self._writers[ends], term, np.zeros((k,) + self.policy.action_shape, self.policy.action_dtype),
                               np.zeros(k, np.float32), np.zeros(k, np.float32), np.zeros(k, np.uint8), np.ones(k, np.uint8),
                               self._n_step)
    self._first[:] = last                  # those environments are reset before the next step

  def update(self):
    pass                                   # the policy reads the learner's own parameters
