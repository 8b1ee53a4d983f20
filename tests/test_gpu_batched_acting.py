"""Batched acting on the GPU: the exploration kernels (b200rl_epsilon_greedy, b200rl_gaussian_explore) against their
stated rules and distributions, b200rl_writer_append_multi against per-writer b200rl_writer_append_stream, and the
batched actor, loop and agents against the network, the per-step adders and the learner schedule."""
import collections
import gc

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


# ------------------------------------------------------------------------------------------------ helpers
def _uniform(n, seed, counter):
  import torch
  from acme_b200 import _capi
  out = torch.empty(n, dtype=torch.float32, device='cuda')
  _capi.call('b200rl_uniform', out.data_ptr(), n, seed, counter.data_ptr(), 0, _capi.current_stream())
  return out.cpu().numpy()


def _eps_greedy(q, eps, seed, counter, with_u=True):
  import torch
  from acme_b200 import _capi
  N, A = q.shape[0], q.shape[1]
  act = torch.empty(N, dtype=torch.int32, device='cuda')
  u = torch.empty((N, 2), dtype=torch.float32, device='cuda') if with_u else None
  _capi.call('b200rl_epsilon_greedy', N, A, q.data_ptr(), q.stride(0), eps, seed, counter.data_ptr(), act.data_ptr(),
             _capi.ptr(u), _capi.current_stream())
  return act.cpu().numpy(), (u.cpu().numpy() if with_u else None)


def _host_eps_greedy(q, eps, u):
  """This package's statement of trfl.epsilon_greedy(q, eps).sample() on the draws u [N, 2] (float32 arithmetic)."""
  out = np.empty(q.shape[0], np.int64)
  A = q.shape[1]
  for r in range(q.shape[0]):
    u0, u1 = np.float32(u[r, 0]), np.float32(u[r, 1])
    if u0 < np.float32(eps):
      out[r] = min(int(np.floor(u1 * np.float32(A))), A - 1)
    else:
      ties = np.flatnonzero(q[r] == q[r].max())
      out[r] = ties[min(int(np.floor(u1 * np.float32(len(ties)))), len(ties) - 1)]
  return out


def _gaussian(a, sigma, lo, hi, seed, counter):
  import torch
  from acme_b200 import _capi
  N, A = a.shape
  out = torch.empty_like(a)
  z = torch.empty_like(a)
  _capi.call('b200rl_gaussian_explore', N, A, a.data_ptr(), sigma, lo.data_ptr(), hi.data_ptr(), seed, counter.data_ptr(),
             out.data_ptr(), z.data_ptr(), _capi.current_stream())
  return out.cpu().numpy(), z.cpu().numpy()


# ------------------------------------------------------------------------------------------------ epsilon-greedy
@pytest.mark.parametrize('N', [1, 7, 256, 4096])
@pytest.mark.parametrize('A', [1, 3, 18])
@pytest.mark.parametrize('eps', [0.0, 0.3, 1.0])
def test_epsilon_greedy_follows_the_rule(N, A, eps):
  import torch
  from acme_b200 import _capi
  rng = np.random.default_rng(N * 100 + A)
  ld = A + 3                                         # a row stride wider than the row
  q = rng.standard_normal((N, ld)).astype(np.float32)
  for r in range(N):                                 # most rows get 2-3 actions tied at the maximum
    if A > 1 and r % 4:
      k = min(A, 2 + r % 2)
      q[r, rng.choice(A, k, replace=False)] = q[r, :A].max() + 1.0
  counter = torch.tensor([5 + N], dtype=torch.int64, device='cuda')
  qd = torch.as_tensor(q).cuda()
  act = torch.empty(N, dtype=torch.int32, device='cuda')
  u = torch.empty((N, 2), dtype=torch.float32, device='cuda')
  _capi.call('b200rl_epsilon_greedy', N, A, qd.data_ptr(), ld, eps, 99, counter.data_ptr(), act.data_ptr(), u.data_ptr(),
             _capi.current_stream())
  u = u.cpu().numpy()
  np.testing.assert_array_equal(u.reshape(-1).view(np.uint32), _uniform(2 * N, 99, counter).view(np.uint32))
  np.testing.assert_array_equal(act.cpu().numpy(), _host_eps_greedy(q[:, :A], eps, u))


def test_epsilon_greedy_distribution():
  import torch
  from scipy import stats
  N, A = 1 << 20, 18
  counter = torch.zeros(1, dtype=torch.int64, device='cuda')
  rng = np.random.default_rng(0)
  q = torch.as_tensor(rng.standard_normal((N, A)).astype(np.float32)).cuda()
  # eps = 1: uniform over all actions
  act, _ = _eps_greedy(q, 1.0, 3, counter, with_u=False)
  assert stats.chisquare(np.bincount(act, minlength=A)).pvalue > 1e-4
  # eps = 0 on all-tied rows: uniform over the tied set
  act, _ = _eps_greedy(torch.zeros((N, A), device='cuda'), 0.0, 4, counter, with_u=False)
  assert stats.chisquare(np.bincount(act, minlength=A)).pvalue > 1e-4
  tied = torch.zeros((N, A), device='cuda')
  tied[:, [2, 7, 11]] = 1.0
  act, _ = _eps_greedy(tied, 0.0, 5, counter, with_u=False)
  counts = np.bincount(act, minlength=A)
  assert counts.sum() == counts[[2, 7, 11]].sum() and stats.chisquare(counts[[2, 7, 11]]).pvalue > 1e-4
  # eps = 0.3 without ties: non-greedy with probability eps (A - 1) / A
  act, _ = _eps_greedy(q, 0.3, 6, counter, with_u=False)
  p = 0.3 * (A - 1) / A
  frac = float(np.mean(act != q.argmax(1).cpu().numpy()))
  assert abs(frac - p) <= 4 * np.sqrt(p * (1 - p) / N)


# ------------------------------------------------------------------------------------------------ Gaussian
def _ulp(x):
  return np.spacing(np.abs(x).astype(np.float32))


def test_gaussian_explore_arithmetic_and_noise():
  import torch
  N, A, sigma = 4096, 21, np.float32(0.3)
  rng = np.random.default_rng(1)
  a = rng.uniform(-1.2, 1.2, (N, A)).astype(np.float32)
  lo = -rng.uniform(0.5, 1.0, A).astype(np.float32)
  hi = rng.uniform(0.5, 1.0, A).astype(np.float32)
  counter = torch.tensor([12], dtype=torch.int64, device='cuda')
  dev = lambda x: torch.as_tensor(x).cuda()
  out, z = _gaussian(dev(a), float(sigma), dev(lo), dev(hi), 17, counter)
  # out = clip(fl(a + fl(z * sigma)), lo, hi), bit for bit given z (NumPy float32: separately rounded)
  np.testing.assert_array_equal(out.view(np.uint32), np.clip(a + z * sigma, lo, hi).astype(np.float32).view(np.uint32))
  # z = sqrt(-2 log(1 - u0)) cos(fl(2 pi u1)) on the b200rl_uniform draws, within 4 ulp
  u = _uniform(2 * N * A, 17, counter).reshape(N * A, 2)
  t = (np.float32(2 * np.pi) * u[:, 1]).astype(np.float64)
  zref = np.sqrt(-2.0 * np.log1p(-u[:, 0].astype(np.float64))) * np.cos(t)
  err = np.abs(z.reshape(-1).astype(np.float64) - zref)
  assert np.all(err <= 4 * _ulp(zref)), float((err / _ulp(zref)).max())
  # sigma = 0: clip(a)
  out0, _ = _gaussian(dev(a), 0.0, dev(lo), dev(hi), 17, counter)
  np.testing.assert_array_equal(out0, np.clip(a, lo, hi))


def test_gaussian_noise_moments():
  import torch
  N, A = 50000, 21
  counter = torch.zeros(1, dtype=torch.int64, device='cuda')
  big = torch.full((A,), 1e30, device='cuda')
  _, z = _gaussian(torch.zeros((N, A), device='cuda'), 1.0, -big, big, 23, counter)
  z = z.reshape(-1).astype(np.float64)
  n = z.size
  assert abs(z.mean()) <= 5 / np.sqrt(n)
  assert abs(z.var() - 1.0) <= 5 * np.sqrt(2.0 / n)


def test_counter_drives_the_draws():
  import torch
  from acme_b200 import _capi
  q = torch.zeros((4096, 18), device='cuda')
  counter = torch.tensor([3], dtype=torch.int64, device='cuda')
  a1, u1 = _eps_greedy(q, 0.5, 8, counter)
  a2, u2 = _eps_greedy(q, 0.5, 8, counter)
  np.testing.assert_array_equal(a1, a2)
  np.testing.assert_array_equal(u1, u2)
  lo, hi = torch.full((18,), -5.0, device='cuda'), torch.full((18,), 5.0, device='cuda')
  g1, _ = _gaussian(q, 1.0, lo, hi, 8, counter)
  g2, _ = _gaussian(q, 1.0, lo, hi, 8, counter)
  np.testing.assert_array_equal(g1, g2)
  _capi.call('b200rl_step_increment', counter.data_ptr(), _capi.current_stream())
  a3, u3 = _eps_greedy(q, 0.5, 8, counter)
  g3, _ = _gaussian(q, 1.0, lo, hi, 8, counter)
  assert np.mean(u3 != u1) > 0.99 and np.mean(g3 != g1) > 0.99 and np.mean(a3 != a1) > 0.5


# ------------------------------------------------------------------------------------------------ append_multi
def _spec(obs_shape, obs_dtype=np.uint8, num_actions=5):
  from acme_b200 import specs
  return specs.EnvironmentSpec(observations=specs.Array(obs_shape, obs_dtype), actions=specs.DiscreteArray(num_actions),
                               rewards=specs.Array((), np.float32), discounts=specs.BoundedArray((), np.float32, 0., 1.))


def _table(spec, max_size, n_step=5, frame_stack=0):
  from acme_b200 import adders, replay
  return replay.Table(replay.DEFAULT_PRIORITY_TABLE, replay.selectors.Prioritized(0.6), replay.selectors.Fifo(), max_size,
                      replay.rate_limiters.MinSize(1), signature=adders.NStepTransitionAdder.signature(spec),
                      max_window=n_step, discount=0.99, frame_stack=frame_stack)


def _element_calls(rng, num_writers, num_calls, obs_shape):
  """Calls of interleaved elements: (writer index, obs, act, rew, disc, first, last) in each call's order; episodes of
  1 (FIRST + LAST) to 9 observations; a writer may appear twice in a call."""
  state = [None] * num_writers              # remaining observations of each writer's open episode
  calls = []
  for _ in range(num_calls):
    ws = list(rng.choice(num_writers, int(rng.integers(1, num_writers + 1)), replace=False))
    if rng.random() < 0.5:
      ws.insert(int(rng.integers(0, len(ws) + 1)), ws[0])    # the same writer twice, in order
    call = []
    for w in ws:
      first = state[w] is None
      if first:
        state[w] = int(rng.integers(1, 10))
      state[w] -= 1
      last = state[w] == 0
      if last:
        state[w] = None
      obs = rng.integers(0, 256, obs_shape, dtype=np.uint8)
      call.append((w, obs, np.int32(rng.integers(5)), np.float32(rng.standard_normal()), np.float32(rng.uniform()),
                   first, last))
    calls.append(call)
  return calls


def _fields(call):
  return (np.stack([c[1] for c in call]), np.array([c[2] for c in call], np.int32), np.array([c[3] for c in call]),
          np.array([c[4] for c in call]), np.array([c[5] for c in call], np.uint8), np.array([c[6] for c in call], np.uint8))


def _append_stream(table, writer, obs, act, rew, disc, first, last, n_step, on_device):
  import torch
  from acme_b200 import _capi
  o = torch.as_tensor(obs).cuda() if on_device else np.ascontiguousarray(obs)
  _capi.call('b200rl_writer_append_stream', table.handle, writer, len(act), _capi.ptr(o), int(on_device),
             np.ascontiguousarray(act).ctypes.data, np.ascontiguousarray(rew, np.float32).ctypes.data,
             np.ascontiguousarray(disc, np.float32).ctypes.data, np.ascontiguousarray(first).ctypes.data,
             np.ascontiguousarray(last).ctypes.data, n_step, 1.0, _capi.current_stream())


def _assert_same_tables(t1, t2):
  import torch
  from acme_b200 import replay
  # the host bookkeeping (key counters, FIFO bounds, every writer's window); the device rings are compared through what the
  # live items gather (their never-written slots and row padding are uninitialised memory)
  np.testing.assert_array_equal(t1.save()['host'], t2.save()['host'])
  assert t1.size == t2.size > 0
  # every live item gathered, and the same sample
  info = t1.info()
  pos = torch.as_tensor(np.arange(info['tail_key'], info['head_key'], dtype=np.int64) % t1.max_size).cuda()
  u = torch.as_tensor(np.random.default_rng(2).random(256, dtype=np.float32)).cuda()
  out = []
  for t in (t1, t2):
    ds = replay.ReplayDataset(t, len(pos), seed=1)
    ds.idx.copy_(pos)
    ds.gather_only()
    ds2 = replay.ReplayDataset(t, 256, seed=1)
    ds2.sample_only(u)
    out.append([x.cpu().numpy() for x in (ds.o_tm1, ds.a_tm1, ds.R, ds.D, ds.o_t, ds2.idx, ds2.prob)])
  for a, b in zip(out[0], out[1]):
    np.testing.assert_array_equal(a, b)


@pytest.mark.parametrize('on_device', [False, True])
@pytest.mark.parametrize('frame_stack', [0, 4])
@pytest.mark.parametrize('max_size', [40, 1000])
def test_append_multi_equals_per_writer_stream_appends(on_device, frame_stack, max_size):
  import torch
  shape = (6, 6, 4)
  spec = _spec(shape)
  n_step, W = 3, 5
  t_multi = _table(spec, max_size, n_step=n_step, frame_stack=frame_stack)
  t_ref = _table(spec, max_size, n_step=n_step, frame_stack=frame_stack)
  w_multi = [t_multi.open_writer() for _ in range(W)]
  w_ref = [t_ref.open_writer() for _ in range(W)]
  calls = _element_calls(np.random.default_rng(frame_stack + max_size + on_device), W, 60, shape)
  assert any(c[5] and c[6] for call in calls for c in call)          # a one-observation episode occurs
  for call in calls:
    obs, act, rew, disc, first, last = _fields(call)
    writers = [w_multi[c[0]] for c in call]
    t_multi.append_multi(writers, torch.as_tensor(obs).cuda() if on_device else obs, act, rew, disc, first, last, n_step)
    for i, c in enumerate(call):
      _append_stream(t_ref, w_ref[c[0]], obs[i:i + 1], act[i:i + 1], rew[i:i + 1], disc[i:i + 1], first[i:i + 1],
                     last[i:i + 1], n_step, on_device)
  torch.cuda.synchronize()
  if max_size == 40:
    assert t_multi.info()['tail_key'] > 0                             # FIFO eviction happened
  _assert_same_tables(t_multi, t_ref)


def test_append_multi_save_restore_continues_identically():
  import torch
  shape = (6, 6, 4)
  spec = _spec(shape)
  W = 4
  calls = _element_calls(np.random.default_rng(7), W, 50, shape)
  t1, t2 = _table(spec, 500, n_step=3), _table(spec, 500, n_step=3)
  w1 = [t1.open_writer() for _ in range(W)]
  for k, call in enumerate(calls):
    if k == 25:                                                       # in the middle of episodes
      t2.restore(t1.save())
    obs, act, rew, disc, first, last = _fields(call)
    ws = [w1[c[0]] for c in call]
    t1.append_multi(ws, torch.as_tensor(obs).cuda(), act, rew, disc, first, last, 3)
    if k >= 25:
      t2.append_multi(ws, torch.as_tensor(obs).cuda(), act, rew, disc, first, last, 3)
  _assert_same_tables(t1, t2)


def test_append_multi_rejects_bad_input():
  from acme_b200 import adders, replay
  spec = _spec((4,), np.float32)
  t = _table(spec, 100)
  w = t.open_writer()
  one = np.ones(1, np.uint8)
  with pytest.raises(ValueError):          # unknown writer: nothing recorded
    t.append_multi([w, w + 7], np.zeros((2, 4), np.float32), np.zeros(2, np.int32), np.zeros(2), np.zeros(2), [1, 1], [0, 0], 3)
  assert t.info()['head_key'] == 0
  with pytest.raises(ValueError):          # not FIRST on a writer without an open episode
    t.append_multi([w], np.zeros((1, 4), np.float32), np.zeros(1, np.int32), np.zeros(1), np.zeros(1), 0 * one, 0 * one, 3)
  seq = replay.Table('s', replay.selectors.Uniform(), replay.selectors.Fifo(), 100, replay.rate_limiters.MinSize(1),
                     signature=adders.SequenceAdder.signature(spec), max_window=4)
  with pytest.raises(ValueError):
    seq.append_multi([0], np.zeros((1, 4), np.float32), np.zeros(1, np.int32), np.zeros(1), np.zeros(1), one, 0 * one, 3)
  ext = replay.Table('e', replay.selectors.Uniform(), replay.selectors.Fifo(), 100, replay.rate_limiters.MinSize(1),
                     signature=adders.NStepTransitionAdder.signature(spec, extras_spec=spec.rewards), max_window=4)
  with pytest.raises(ValueError):
    ext.append_multi([0], np.zeros((1, 4), np.float32), np.zeros(1, np.int32), np.zeros(1), np.zeros(1), one, 0 * one, 3)


# ------------------------------------------------------------------------------------------------ actor and loop
class _TrajEnv:
  """Episodes of fixed lengths; observations (env id, step counter), seeded rewards and discounts; records every
  timestep it emits."""

  def __init__(self, env_id, lengths, seed):
    from acme_b200 import dm_env
    self._dm, self.id, self.lengths, self.ep, self.t, self.count = dm_env, env_id, lengths, -1, 0, 0
    self.rng = np.random.default_rng(seed)
    self.trajectory = []                     # [(action or None, timestep)]

  def _obs(self):
    self.count += 1
    return np.array([self.id, self.count], np.float32)

  def reset(self):
    self.ep, self.t = self.ep + 1, 0
    ts = self._dm.restart(self._obs())
    self.trajectory.append((None, ts))
    return ts

  def step(self, action):
    self.t += 1
    rew, disc = np.float32(self.rng.standard_normal()), np.float32(self.rng.uniform(0.5, 1.0))
    if self.t == self.lengths[self.ep % len(self.lengths)]:
      ts = self._dm.TimeStep(self._dm.StepType.LAST, rew, disc, self._obs())
    else:
      ts = self._dm.transition(rew, self._obs(), disc)
    self.trajectory.append((action, ts))
    return ts


def _items(table):
  """(o_tm1, a, R, D, o_t) of every live item, in key order."""
  import torch
  from acme_b200 import replay
  table.flush()                              # the per-step adders leave their last steps staged
  info = table.info()
  keys = np.arange(info['tail_key'], info['head_key'], dtype=np.int64)
  ds = replay.ReplayDataset(table, len(keys), seed=0)
  ds.idx.copy_(torch.as_tensor(keys % table.max_size).cuda())
  ds.gather_only()
  return list(zip(*[x.cpu().numpy() for x in (ds.o_tm1, ds.a_tm1, ds.R, ds.D, ds.o_t)]))


def _item_key(it):
  return tuple(np.asarray(x).tobytes() for x in it)


@pytest.mark.parametrize('n_step', [3, 5])
def test_batched_loop_items_equal_the_per_step_adders(n_step):
  import torch
  from acme_b200 import actors, adders, environment_loop, loggers, networks, replay
  spec = _spec((2,), np.float32, num_actions=4)
  lengths = [[1, 4, 2, 7], [7, 7], [3, 9, 2], [5, 1, 6, 2]]          # every environment ends an episode at step 14
  envs = [_TrajEnv(i, L, seed=i) for i, L in enumerate(lengths)]
  table = _table(spec, 4000, n_step=n_step)
  net = networks.MLPQNetwork(2, [16, 4], seed=0)
  actor = actors.BatchedActor(actors.BatchedEpsilonGreedy(net, 0.5, seed=3), table, len(envs), n_step)
  loop = environment_loop.BatchedEnvironmentLoop(envs, actor, logger=loggers.NoOpLogger())
  loop.run(num_steps=4 * 14)
  assert all(e.trajectory[-2][1].last() and e.trajectory[-1][1].first() for e in envs)
  torch.cuda.synchronize()
  # the reference: one NStepTransitionAdder per environment, fed the same trajectories
  ref_table = _table(spec, 4000, n_step=n_step)
  server = replay.Server([ref_table])
  for e in envs:
    adder = adders.NStepTransitionAdder(replay.Client(server), n_step, 0.99)
    for action, ts in e.trajectory:
      if ts.first():
        adder.add_first(ts)
      else:
        adder.add(np.int32(action), ts)
    adder.reset()
  got, ref = _items(table), _items(ref_table)
  assert len(got) == len(ref) > 0
  assert collections.Counter(map(_item_key, got)) == collections.Counter(map(_item_key, ref))
  for i in range(len(envs)):               # per environment, the same key order
    mine = [_item_key(it) for it in got if it[0].view(np.float32)[0] == i]
    theirs = [_item_key(it) for it in ref if it[0].view(np.float32)[0] == i]
    assert mine == theirs
  server.stop()


def test_actor_acts_on_the_network_q_and_graph_equals_eager():
  import torch
  from acme_b200 import _capi, actors, networks
  N = 16
  spec = _spec((84, 84, 4), np.uint8, num_actions=18)
  table = _table(spec, 1000, n_step=3)
  net = networks.DQNAtariNetwork(18, seed=0, precision=_capi.PRECISION_BF16FLOW)
  greedy = actors.BatchedActor(actors.BatchedEpsilonGreedy(net, 0.0, seed=1), table, N, 3)
  rng = np.random.default_rng(0)
  obs = rng.integers(0, 256, (N, 84, 84, 4), dtype=np.uint8)
  acts = greedy.select_actions(obs)
  q = greedy.policy.values.cpu().numpy()
  ref = net.forward(torch.as_tensor(obs).cuda(), net.make_buffers(N)).cpu().numpy()
  np.testing.assert_array_equal(q.view(np.uint32), ref.view(np.uint32))
  assert all(len(np.flatnonzero(r == r.max())) == 1 for r in ref)
  np.testing.assert_array_equal(acts, ref.argmax(1))
  # the captured act step and the same step run eagerly: bit for bit, over several counter values
  g = actors.BatchedActor(actors.BatchedEpsilonGreedy(net, 0.5, seed=2), table, N, 3)
  e = actors.BatchedActor(actors.BatchedEpsilonGreedy(net, 0.5, seed=2), table, N, 3, use_cuda_graph=False)
  for k in range(4):
    o = rng.integers(0, 256, (N, 84, 84, 4), dtype=np.uint8)
    np.testing.assert_array_equal(g.select_actions(o), e.select_actions(o))
  assert int(g.policy.counter) == int(e.policy.counter) == 4


def test_gaussian_actor_acts_on_the_policy():
  import torch
  from acme_b200 import _capi, actors, networks, specs
  N, O, A = 64, 67, 21
  spec = specs.EnvironmentSpec(observations=specs.Array((O,), np.float32), actions=specs.BoundedArray((A,), np.float32, -1., 1.),
                               rewards=specs.Array((), np.float32), discounts=specs.BoundedArray((), np.float32, 0., 1.))
  table = _table(spec, 1000, n_step=3)
  pol = networks.D4PGPolicy(O, A, seed=0, precision=_capi.PRECISION_BF16FLOW)
  actor = actors.BatchedActor(actors.BatchedGaussianNoise(pol, 0.3, -1., 1., seed=0), table, N, 3)
  obs = np.random.default_rng(1).standard_normal((N, O)).astype(np.float32)
  acts = actor.select_actions(obs)
  a = actor.policy.values.cpu().numpy()
  ref = pol.action(torch.as_tensor(obs).cuda(), pol.make_buffers(N)).cpu().numpy()
  np.testing.assert_array_equal(a, ref)
  assert acts.shape == (N, A) and acts.dtype == np.float32 and np.all(np.abs(acts) <= 1) and np.any(acts != np.clip(a, -1, 1))


def test_actor_rejects_nested_observations_and_extras():
  from acme_b200 import actors, adders, networks, replay, specs
  spec = _spec((4,), np.float32)
  nested = spec._replace(observations=(spec.observations, spec.observations))
  t = replay.Table('n', replay.selectors.Uniform(), replay.selectors.Fifo(), 100, replay.rate_limiters.MinSize(1),
                   signature=adders.NStepTransitionAdder.signature(nested), max_window=3)
  net = networks.MLPQNetwork(4, [8, 5])
  with pytest.raises(ValueError):
    actors.BatchedActor(actors.BatchedEpsilonGreedy(net), t, 2, 3)
  ext = replay.Table('e', replay.selectors.Uniform(), replay.selectors.Fifo(), 100, replay.rate_limiters.MinSize(1),
                     signature=adders.NStepTransitionAdder.signature(spec, extras_spec=specs.Array((), np.float32)), max_window=3)
  with pytest.raises(ValueError):
    actors.BatchedActor(actors.BatchedEpsilonGreedy(net), ext, 2, 3)


# ------------------------------------------------------------------------------------------------ agents
def _schedule_count(observations, warmup, ratio):
  from acme_b200 import agent
  s, n = agent.LearnerSchedule(warmup, ratio), 0
  for _ in range(observations):
    s.saw_observation()
    n += s.due()
  return n


@pytest.mark.parametrize('kind', ['dqn', 'd4pg', 'ddpg'])
def test_agents_with_num_envs_run_in_the_batched_loop(kind):
  import torch
  from acme_b200 import agent, d4pg, dqn, environment_loop, loggers, networks, specs, testing
  if kind == 'dqn':
    envs = [testing.DiscreteEnvironment(num_actions=5, num_observations=10, obs_dtype=np.float32, episode_length=10)
            for _ in range(4)]
    spec = specs.make_environment_spec(envs[0])
    net = networks.MLPQNetwork(1, [50, 50, spec.actions.num_values], seed=0)
    ag = dqn.DQN(spec, net, batch_size=10, samples_per_insert=2, min_replay_size=10, max_replay_size=1000, n_step=5,
                 logger=loggers.NoOpLogger(), num_envs=4)
    n_step = 5
  else:
    envs = [testing.ContinuousEnvironment(episode_length=10, bounded=True) for _ in range(4)]
    spec = specs.make_environment_spec(envs[0])
    policy = networks.D4PGPolicy(1, 1, sizes=(10, 10), seed=0)
    critic = (networks.D4PGCritic(1, 1, sizes=(10, 10), seed=1) if kind == 'd4pg' else networks.DDPGCritic(1, 1, sizes=(10, 10), seed=1))
    cls = d4pg.D4PG if kind == 'd4pg' else d4pg.DDPG
    ag = cls(spec, policy, critic, batch_size=10, samples_per_insert=2, min_replay_size=10, max_replay_size=1000,
             logger=loggers.NoOpLogger(), num_envs=4)
    n_step = 5
  assert isinstance(ag, agent.BatchedAgent)
  # tables left in reference cycles by earlier tests must not be finalised (cudaFree) inside the learner's graph capture
  gc.collect()
  loop = environment_loop.BatchedEnvironmentLoop(envs, ag, logger=loggers.NoOpLogger())
  loop.run(num_episodes=8)
  torch.cuda.synchronize()
  assert int(ag._learner._num_steps) == _schedule_count(80, 10, 5.0)
  assert ag._table.size == 8 * (10 + min(n_step, 10) - 1)
  with pytest.raises(ValueError):
    environment_loop.BatchedEnvironmentLoop(envs[:3], ag, logger=loggers.NoOpLogger())


def test_golden_nstep_cases_as_lockstep_streams():
  """The reference's n-step cases (tests/golden/nstep_cases.json), each one writer's stream; cases sharing (n_step,
  discount) step in lockstep through one append_multi call per step.  Dict observations are their single value and
  extras are left out (append_multi writes tables without extras); each case's items, in key order, are its expected
  (o_tm1, a, R, D, o_t)."""
  import json
  import os
  import torch
  from acme_b200 import adders, replay, specs
  cases = json.load(open(os.path.join(os.path.dirname(__file__), 'golden', 'nstep_cases.json')))
  val = lambda o: o['foo'] if isinstance(o, dict) else o
  groups = collections.defaultdict(list)
  for ci, c in enumerate(cases):
    groups[(c['n_step'], c['additional_discount'])].append(ci)
  spec = specs.EnvironmentSpec(specs.Array((), np.int64), specs.Array((), np.int64), specs.Array((), np.float32),
                               specs.Array((), np.float32))
  for (n_step, discount), members in groups.items():
    table = replay.Table(replay.DEFAULT_PRIORITY_TABLE, replay.selectors.Prioritized(0.6), replay.selectors.Fifo(), 64,
                         replay.rate_limiters.MinSize(1), signature=adders.NStepTransitionAdder.signature(spec),
                         max_window=n_step, discount=discount)
    writers = {ci: table.open_writer() for ci in members}
    streams = {}
    for ci in members:                       # element t: observation t with the reward / discount that followed it
      c, off = cases[ci], 100 * ci
      obs = [val(c['first'])] + [val(s['observation']) for s in c['steps']]
      rew = [s['reward'] for s in c['steps']] + [0.]
      disc = [s['discount'] for s in c['steps']] + [0.]
      streams[ci] = [(obs[t] + off, rew[t], disc[t], t == 0, t == len(obs) - 1) for t in range(len(obs))]
    for t in range(max(len(s) for s in streams.values())):
      call = [(ci, streams[ci][t]) for ci in members if t < len(streams[ci])]
      table.append_multi([writers[ci] for ci, _ in call], torch.as_tensor(np.array([e[0] for _, e in call], np.int64)).cuda(),
                         np.zeros(len(call), np.int64), [e[1] for _, e in call], [e[2] for _, e in call],
                         [e[3] for _, e in call], [e[4] for _, e in call], n_step)
    items = _items(table)
    assert len(items) == sum(len(cases[ci]['expected']) for ci in members)
    for ci in members:
      off = 100 * ci
      mine = [it for it in items if off <= int(it[0].view(np.int64)[0]) < off + 100]
      assert len(mine) == len(cases[ci]['expected']), cases[ci]['name']
      for it, e in zip(mine, cases[ci]['expected']):
        assert int(it[0].view(np.int64)[0]) - off == val(e[0]) and int(it[4].view(np.int64)[0]) - off == val(e[4])
        assert int(it[1].view(np.int64)[0]) == e[1]
        np.testing.assert_array_almost_equal([float(it[2]), float(it[3])], [e[2], e[3]])
