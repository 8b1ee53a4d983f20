"""Prioritized replay for D4PG / DDPG: the two weighted critic losses, the learners and the agents.

Kernels (`b200rl_c51_loss_weighted`, `b200rl_td_learning_weighted`) against the unweighted entry points, `b200rl_dqn_td`'s
importance weights and NumPy f64, with one launch per call and a batch mean that is bit-identical across launches, streams
and graph replay.  Learners: beta on a Prioritized(0) table equals the uniform learner bit for bit; at the C3 shape with
alpha = 0.6 the weights, losses, gradients and priorities stay inside the bounds DESIGN.md states per precision, and the
tree leaves equal f32(pow(f64(device priority), alpha)).  The errors measured on a B200 are written to
$B200RL_PARITY_DIR/parity_c3_<learner>_<mode>_prioritized.json when that variable is set.

The file sorts after every test file whose launch-signature checks read torch.profiler (the layer suites): a profiler
capture that follows a long stretch of GPU work without one can miss the first kernels it should record (seen on a B200
with nothing but a 25 s pause between two captures), and these tests are such a stretch."""
import gc
import json
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

BETA, ALPHA = 0.4, 0.6
OBS, ACT = 67, 21
MODES = {0: 'fp32', 1: 'tf32', 2: 'bf16', 3: 'fp32x3'}
# per precision: values (weights, targets, td, per-sample losses, priorities, dlogits), losses (batch means), gradients
# (relative L2): FP32_TOL at precisions 0 and 3 (tests/test_gpu_learner.py, tests/test_gpu_fp32x3.py), the C3 table's rows
# at precisions 1 and 2 (tests/test_gpu_d4pg_bf16.py)
TOL = {0: dict(value=2e-5, loss=1e-4, grad_rel_l2=1e-3), 3: dict(value=2e-5, loss=1e-4, grad_rel_l2=1e-3),
       1: dict(value=1e-2, loss=1e-2, grad_rel_l2=5e-2), 2: dict(value=2e-2, loss=2e-2, grad_rel_l2=1e-1)}


def _capi():
  from acme_b200 import _capi
  return _capi


def _dev(x):
  import torch
  return torch.as_tensor(np.ascontiguousarray(x)).cuda()


def _bits(t):
  import torch
  return t.view(torch.int32).clone()


def _launches():
  return int(_capi().load().b200rl_launch_count())


# ------------------------------------------------------------------------------ kernels
def _loss_inputs(kind, B, K, seed, equal_prob=False):
  rng = np.random.default_rng(seed)
  if kind == 'c51':
    lt1 = (rng.standard_normal((B, K)) * 2).astype(np.float32)
    lt = (rng.standard_normal((B, K)) * 2).astype(np.float32)
  else:
    lt1 = (rng.standard_normal(B) * 3).astype(np.float32)
    lt = (rng.standard_normal(B) * 3).astype(np.float32)
  R = rng.choice(np.float32([-1., 0., 0.5, 1., 2.5]), B).astype(np.float32)
  D = rng.choice(np.float32([0., 1., 0.9]), B).astype(np.float32)
  prob = (np.full(B, 1. / 600) if equal_prob else rng.uniform(1e-4, 1e-2, B)).astype(np.float32)
  return lt1, lt, R, D, prob


class _Loss:
  """Device buffers and the two calls (uniform, weighted) of one critic loss."""

  def __init__(self, kind, B, K, seed, equal_prob=False):
    import torch
    self.kind, self.B, self.K = kind, B, K
    lt1, lt, R, D, prob = _loss_inputs(kind, B, K, seed, equal_prob)
    self.host = dict(lt1=lt1, lt=lt, R=R, D=D, prob=prob)
    self.lt1, self.lt, self.R, self.D, self.prob = (_dev(x) for x in (lt1, lt, R, D, prob))
    self.wmax = torch.zeros(1, dtype=torch.float64, device='cuda')
    nan = lambda *s: torch.full(s, float('nan'), device='cuda')
    shp = (B, K) if kind == 'c51' else (B,)
    self.u = dict(first=nan(*shp), loss_ps=nan(B), grad=nan(*shp), mean=nan(1))
    self.w = dict(first=nan(*shp), loss_ps=nan(B), weight=nan(B), priority=nan(B), grad=nan(*shp), mean=nan(1))
    _capi().call('b200rl_is_weight_max', B, self.prob.data_ptr(), BETA, self.wmax.data_ptr(), 0, _capi().current_stream())

  def uniform(self):
    c, u = _capi(), self.u
    if self.kind == 'c51':
      c.call('b200rl_c51_loss', self.B, self.K, -10., 10., self.lt1.data_ptr(), self.lt.data_ptr(), self.R.data_ptr(),
             self.D.data_ptr(), 0.99, 1.0 / self.B, u['first'].data_ptr(), u['loss_ps'].data_ptr(), u['grad'].data_ptr(),
             u['mean'].data_ptr(), c.current_stream())
    else:
      c.call('b200rl_td_learning', self.B, self.lt1.data_ptr(), self.lt.data_ptr(), self.R.data_ptr(), self.D.data_ptr(), 0.99,
             1.0 / self.B, u['first'].data_ptr(), u['loss_ps'].data_ptr(), u['grad'].data_ptr(), u['mean'].data_ptr(),
             c.current_stream())

  def weighted(self, **over):
    c = _capi()
    w = {k: v.data_ptr() for k, v in self.w.items()}
    a = dict(prob=self.prob.data_ptr(), wmax=self.wmax.data_ptr(), beta=BETA, B=self.B, K=self.K, **w)
    a.update(over)
    if self.kind == 'c51':
      c.call('b200rl_c51_loss_weighted', a['B'], a['K'], -10., 10., self.lt1.data_ptr(), self.lt.data_ptr(), self.R.data_ptr(),
             self.D.data_ptr(), 0.99, a['prob'], a['beta'], a['wmax'], 1.0 / self.B, a['first'], a['loss_ps'], a['weight'],
             a['priority'], a['grad'], a['mean'], c.current_stream())
    else:
      c.call('b200rl_td_learning_weighted', a['B'], self.lt1.data_ptr(), self.lt.data_ptr(), self.R.data_ptr(), self.D.data_ptr(),
             0.99, a['prob'], a['beta'], a['wmax'], 1.0 / self.B, a['first'], a['loss_ps'], a['weight'], a['priority'], a['grad'],
             a['mean'], c.current_stream())

  def dqn_td_weights(self):
    """b200rl_dqn_td's importance weights for the same prob and beta (A = 1, flags 0, the same batch maximum)."""
    import torch
    c, B = _capi(), self.B
    z = torch.zeros(B, device='cuda')
    a = torch.zeros(B, dtype=torch.int32, device='cuda')
    outs = [torch.zeros(B, device='cuda') for _ in range(5)]
    c.call('b200rl_dqn_td', B, 1, z.data_ptr(), z.data_ptr(), z.data_ptr(), a.data_ptr(), z.data_ptr(), z.data_ptr(),
           self.prob.data_ptr(), 0.99, 1.0, BETA, 1.0, self.wmax.data_ptr(), 1.0 / B, *[o.data_ptr() for o in outs], None, 0,
           c.current_stream())
    return outs[2]


CASES = [('c51', B, K) for B in (1, 256, 4096) for K in (21, 51, 101)] + [('td', B, 1) for B in (1, 256, 4096)]


@pytest.mark.parametrize('kind,B,K', CASES)
def test_weighted_loss_kernel(kind, B, K):
  import torch
  L = _Loss(kind, B, K, seed=B * 7 + K)
  L.uniform()
  n0 = _launches()
  L.weighted()
  torch.cuda.synchronize()
  assert _launches() - n0 == 1, 'one launch per call'
  u = {k: v.cpu().numpy() for k, v in L.u.items()}
  w = {k: v.cpu().numpy() for k, v in L.w.items()}
  # target / td and the priority: bit-identical to the unweighted entry point
  np.testing.assert_array_equal(w['first'].view(np.int32), u['first'].view(np.int32))
  prio_want = u['loss_ps'] if kind == 'c51' else np.abs(u['first'])
  np.testing.assert_array_equal(w['priority'].view(np.int32), prio_want.view(np.int32))
  # weights: b200rl_dqn_td's bit for bit, and NumPy f64 to 1e-6
  np.testing.assert_array_equal(w['weight'].view(np.int32), L.dqn_td_weights().cpu().numpy().view(np.int32))
  w64 = (1.0 / L.host['prob'].astype(np.float64))**BETA
  w64 /= w64.max()
  np.testing.assert_allclose(w['weight'], w64, rtol=1e-6, atol=0)
  # the weighted per-sample loss is fl(unweighted * w)
  np.testing.assert_array_equal(w['loss_ps'], (u['loss_ps'] * w['weight']).astype(np.float32))
  # gradient: w times the unweighted one to 1e-6, bit-identical where w == 1
  want = u['grad'].astype(np.float64) * (w['weight'][:, None] if kind == 'c51' else w['weight'])
  assert np.all(np.abs(w['grad'] - want) <= 1e-6 * np.abs(want)), np.abs(w['grad'] - want).max()
  one = w['weight'] == 1.0
  assert one.any()
  np.testing.assert_array_equal(w['grad'][one].view(np.int32), u['grad'][one].view(np.int32))
  # the batch mean: within the fp32 summation bound of the f64 mean of the per-sample losses
  mean64 = w['loss_ps'].astype(np.float64).mean()
  assert abs(float(w['mean'][0]) - mean64) <= B * 2.0**-24 * np.abs(w['loss_ps']).astype(np.float64).mean() + 1e-30
  # bit-identical: again on the same stream, on a second stream, under graph replay
  first = {k: _bits(v) for k, v in L.w.items()}

  def same(what):
    torch.cuda.synchronize()
    for k, v in L.w.items():
      assert torch.equal(_bits(v), first[k]), f'{what}: {k} differs'
      v.fill_(float('nan'))

  for k in L.w:
    L.w[k].fill_(float('nan'))
  for _ in range(3):
    L.weighted()
    same('repeat')
  s = torch.cuda.Stream()
  s.wait_stream(torch.cuda.current_stream())
  with torch.cuda.stream(s):
    L.weighted()
  torch.cuda.current_stream().wait_stream(s)
  same('second stream')
  g = torch.cuda.CUDAGraph()
  torch.cuda.synchronize()
  with torch.cuda.graph(g):
    L.weighted()
  for _ in range(3):
    g.replay()
    same('graph replay')


@pytest.mark.parametrize('kind,K', [('c51', 51), ('c51', 101), ('td', 1)])
def test_weighted_loss_kernel_unit_weights_are_the_unweighted_loss(kind, K):
  """Equal probabilities: w == 1 everywhere, and every output but the mean is the unweighted entry point's, bit for bit."""
  import torch
  L = _Loss(kind, 256, K, seed=3, equal_prob=True)
  L.uniform()
  L.weighted()
  torch.cuda.synchronize()
  assert bool((L.w['weight'] == 1).all())
  for a, b in (('first', 'first'), ('loss_ps', 'loss_ps'), ('grad', 'grad')):
    assert torch.equal(_bits(L.w[a]), _bits(L.u[b])), a


@pytest.mark.parametrize('kind', ['c51', 'td'])
def test_weighted_loss_kernel_rejects(kind):
  import torch
  L = _Loss(kind, 64, 51, seed=4)
  torch.cuda.synchronize()
  bad = [dict(prob=None), dict(wmax=None), dict(loss_ps=None), dict(weight=None), dict(priority=None), dict(B=0),
         dict(beta=-0.1)]
  if kind == 'c51':
    bad += [dict(K=1), dict(K=1025)]
  for over in bad:
    n0 = _launches()
    with pytest.raises(ValueError):
      L.weighted(**over)
    assert _launches() == n0, f'{over}: a rejected call launched'
  torch.cuda.synchronize()
  for k, v in L.w.items():
    assert bool(torch.isnan(v).all()), f'a rejected call wrote {k}'


# ------------------------------------------------------------------------------ learners
def _table(sampler, seed, episodes, max_size=4000):
  """A continuous-control table filled by the n-step adder, and the oracle table holding the same items."""
  import helpers
  from acme_b200 import adders, replay, specs
  from oracle import replay as oreplay
  alpha = getattr(sampler, 'priority_exponent')
  aspec = specs.BoundedArray((ACT,), np.float32, -1., 1.)
  spec = specs.EnvironmentSpec(specs.Array((OBS,), np.float32), aspec, specs.Array((), np.float32),
                               specs.BoundedArray((), np.float32, 0., 1.))
  table = replay.Table(replay.DEFAULT_PRIORITY_TABLE, sampler, replay.selectors.Fifo(), max_size=max_size,
                       rate_limiter=replay.rate_limiters.MinSize(1), signature=adders.NStepTransitionAdder.signature(spec),
                       max_window=5, discount=0.99)
  server = replay.Server([table])
  adder = adders.NStepTransitionAdder(replay.Client(server), n_step=5, discount=0.99)
  oracle = oreplay.Table(max_size, table.slot_capacity, (OBS,), np.float32, (ACT,), np.float32, 0.99, alpha, max_window=5)
  rng = np.random.default_rng(seed)
  for _ in range(episodes):
    helpers.feed_episode(rng, adder, oracle, int(rng.integers(20, 80)), 5, (OBS,), np.float32, 0, act_dim=ACT)
  table.flush()
  helpers.sync_oracle_leaves(table, oracle)
  return table, server, oracle


def _leaf_level(table):
  return table.tree_levels()[0]   # level L of the tree holds the leaves


def _learner(kind, policy, critic, ds, use_graph, beta=None, client=None):
  from acme_b200 import d4pg, loggers
  cls = d4pg.D4PGLearner if kind == 'd4pg' else d4pg.DDPGLearner
  return cls(policy, critic, policy.clone(), critic.clone(), 0.99, target_update_period=2, dataset=ds, logger=loggers.NoOpLogger(),
             use_cuda_graph=use_graph, importance_sampling_exponent=beta, replay_client=client)


def _state(learner):
  nets = (learner._policy, learner._critic, learner._tpolicy, learner._tcritic)
  st = [n.params.flat.clone() for n in nets]
  st += [n.params.shadow.clone() for n in nets if n.params.shadow is not None]
  return st + [t.clone() for t in (learner._pm, learner._pv, learner._cm, learner._cv, learner._num_steps)]


def _assert_same_state(a, b, what):
  import torch
  assert len(a) == len(b)
  for i, (x, y) in enumerate(zip(a, b)):
    assert torch.equal(x, y), f'{what}: state tensor {i} differs'


@pytest.mark.parametrize('precision', [1, 2])
@pytest.mark.parametrize('kind', ['d4pg', 'ddpg'])
def test_alpha_zero_equals_uniform_learner(kind, precision):
  """beta = 0.4 on a Prioritized(0) table against the uniform learner on a Uniform() table with the same items, 6 updates
  in graph mode: the same draws, and bit-identical parameters, targets, shadows, Adam moments and counters; every leaf
  stays 1.0 (1 = p^0 for any priority)."""
  import torch
  from test_gpu_d4pg_bf16 import _nets
  from acme_b200 import replay
  B = 256
  runs = {}
  for name, sampler in (('uniform', replay.selectors.Uniform()), ('prioritized', replay.selectors.Prioritized(0.0))):
    table, server, _ = _table(sampler, 21, episodes=20)
    policy, critic = _nets(kind, precision)
    ds = replay.ReplayDataset(table, B, seed=11, stratified=False)
    pr = name == 'prioritized'
    learner = _learner(kind, policy, critic, ds, True, beta=BETA if pr else None, client=replay.Client(server) if pr else None)
    idx, tgt = [], []
    for _ in range(6):
      learner.step(fetch_loss=False)
      idx.append(ds.idx.clone())
      tgt.append((learner.target if kind == 'd4pg' else learner.td).clone())
    torch.cuda.synchronize()
    if pr:
      assert bool((learner.weight == 1).all())
    runs[name] = (torch.stack(idx), torch.stack(tgt), _state(learner), table.read_tree_level(_leaf_level(table))[:table.size])
    server.stop()
  (i0, t0, s0, _), (i1, t1, s1, leaves) = runs['uniform'], runs['prioritized']
  assert torch.equal(i0, i1), 'sampled indices differ'
  assert torch.equal(t0.view(torch.int32), t1.view(torch.int32)), 'targets differ'
  _assert_same_state(s1, s0, 'prioritized (alpha = 0) vs uniform')
  np.testing.assert_array_equal(leaves, np.ones_like(leaves))


@pytest.mark.parametrize('precision', [0, 1, 2, 3])
@pytest.mark.parametrize('kind', ['d4pg', 'ddpg'])
def test_learner_c3_shape_parity_prioritized(kind, precision):
  """alpha = 0.6, beta = 0.4, ~600 items (a batch of 256 repeats keys), three updates on injected uniforms; the oracle
  adopts the device networks and Adam moments before each update and the device tree's leaves after it."""
  import torch
  import prioritized_oracle as po
  from test_gpu_d4pg_bf16 import _export_flat, _nets, _scale_err
  from oracle import nets as onets
  from oracle import sumtree
  from acme_b200 import replay
  B = 256
  tol = TOL[precision]
  table, server, oracle = _table(replay.selectors.Prioritized(ALPHA), 12, episodes=12)
  policy, critic = _nets(kind, precision)
  ds = replay.ReplayDataset(table, B, seed=11, stratified=False)
  learner = _learner(kind, policy, critic, ds, False, beta=BETA, client=replay.Client(server))
  tpolicy, tcritic = learner._tpolicy, learner._tcritic
  ocls = onets.D4PGCritic if kind == 'd4pg' else onets.DDPGCritic
  opol, ocri, otp, otc = onets.D4PGPolicy(OBS, ACT), ocls(OBS, ACT), onets.D4PGPolicy(OBS, ACT), ocls(OBS, ACT)
  ol = (po.D4PGOracleLearner if kind == 'd4pg' else po.DDPGOracleLearner)(opol, ocri, otp, otc, 0.99, 2)
  rng = np.random.default_rng(5)
  L = _leaf_level(table)
  measured = []
  for step in range(3):
    for o, net in ((opol, policy), (ocri, critic), (otp, tpolicy), (otc, tcritic)):
      o.load(net.variables())
    ol.popt.m, ol.popt.v, ol.popt.t = _export_flat(policy, learner._pm), _export_flat(policy, learner._pv), step
    ol.copt.m, ol.copt.v, ol.copt.t = _export_flat(critic, learner._cm), _export_flat(critic, learner._cv), step
    ol.num_steps = step
    u = rng.random(B, dtype=np.float32)
    keys, pos, prob = oracle.sample(u, False)
    assert len(np.unique(keys)) < B, 'the batch should repeat keys'
    ref = ol.step(*oracle.gather(pos), prob=prob, beta=BETA)
    learner.step(uniforms=torch.as_tensor(u).cuda())
    torch.cuda.synchronize()
    np.testing.assert_array_equal(ds.idx.cpu().numpy(), pos)                         # sampled indices: bit-exact
    np.testing.assert_array_equal(ds.prob.cpu().numpy(), prob)
    cscale, pscale = float(learner._cscale.cpu()[0]), float(learner._pscale.cpu()[0])
    cg, pg = _export_flat(critic, critic.params.grad), _export_flat(policy, policy.params.grad)
    rel = lambda got, want: float(np.linalg.norm(got.astype(np.float64) - want) / max(np.linalg.norm(want), 1e-30))
    prio = learner.priority.cpu().numpy()
    err = dict(step=step,
               weight=_scale_err(learner.weight.cpu().numpy(), ref['weight']),
               priority=_scale_err(prio, ref['priority']),
               critic_loss_per_sample=_scale_err(learner.critic_loss_ps.cpu().numpy(), ref['per_sample']),
               critic_loss=_scale_err(learner.critic_loss.cpu().numpy()[0], ref['critic_loss']),
               dqda=_scale_err(learner.dqda.cpu().numpy(), ref['dqda']),
               policy_loss=_scale_err(learner.policy_loss.cpu().numpy()[0], ref['policy_loss']),
               critic_norm=_scale_err(learner.critic_norm.cpu().numpy()[0], ref['critic_norm']),
               policy_norm=_scale_err(learner.policy_norm.cpu().numpy()[0], ref['policy_norm']),
               critic_grad_rel_l2={k: rel(cg[k] * cscale, g) for k, g in ref['critic_grads'].items()},
               policy_grad_rel_l2={k: rel(pg[k] * pscale, g) for k, g in ref['policy_grads'].items()})
    if kind == 'd4pg':
      err['target'] = _scale_err(learner.target.cpu().numpy(), ref['target'])
      err['dlogits'] = _scale_err(learner.dlogits.cpu().numpy(), ref['dlogits_tm1'])
    else:
      err['td'] = _scale_err(learner.td.cpu().numpy(), ref['td'])
    measured.append(err)
    # the tree after K2: leaf = f32(pow(f64(device priority), alpha)), the last occurrence of a repeated key winning
    oracle.update_priorities(keys, prio)
    leaves = table.read_tree_level(L)[:oracle.tree.levels[L].shape[0]]
    np.testing.assert_array_equal(leaves, oracle.tree.levels[L])
    last = {int(p): i for i, p in enumerate(pos)}
    sel = np.fromiter(last.keys(), np.int64)
    np.testing.assert_array_equal(leaves[sel], sumtree.weight_from_priority(prio[list(last.values())], ALPHA))
    oracle.tree.levels[L][:] = leaves
    oracle.tree.rebuild()
  out = os.environ.get('B200RL_PARITY_DIR')
  if out:
    os.makedirs(out, exist_ok=True)
    mode = MODES[precision]
    with open(os.path.join(out, f'parity_c3_{kind}_{mode}_prioritized.json'), 'w') as f:
      json.dump(dict(learner=kind, mode=mode, B=B, obs=OBS, act=ACT, n=5, alpha=ALPHA, beta=BETA, items=int(table.size),
                     tolerances=tol, measured=measured), f, indent=1)
  for err in measured:
    for k, v in err.items():
      if k == 'step':
        continue
      if isinstance(v, dict):
        assert max(v.values()) <= tol['grad_rel_l2'], (k, err['step'], v)
      else:
        assert v <= tol['loss' if k.endswith('loss') else 'value'], (k, err['step'], v)
  server.stop()


@pytest.mark.parametrize('kind', ['d4pg', 'ddpg'])
def test_prioritized_learner_launch_order_is_bit_identical(kind, monkeypatch):
  """Eager, one CUDA graph and a single stream (B200RL_D4PG_STREAMS=0): 6 updates on the learner's own draws give
  bit-identical losses, state and tree leaves; an eager step launches at most one kernel more than the uniform one."""
  import torch
  from test_gpu_d4pg_bf16 import _nets
  from acme_b200 import replay
  B = 256
  runs = {}
  for name, graph, streams in (('graph', True, '1'), ('eager', False, '1'), ('one stream', True, '0')):
    monkeypatch.setenv('B200RL_D4PG_STREAMS', streams)
    table, server, _ = _table(replay.selectors.Prioritized(ALPHA), 13, episodes=20)
    policy, critic = _nets(kind, 1)
    ds = replay.ReplayDataset(table, B, seed=11, stratified=False)
    learner = _learner(kind, policy, critic, ds, graph, beta=BETA, client=replay.Client(server))
    losses = []
    for _ in range(6):
      learner.step(fetch_loss=False)
      losses.append(torch.cat([learner.critic_loss, learner.policy_loss]).clone())
    torch.cuda.synchronize()
    runs[name] = (torch.stack(losses), _state(learner), table.read_tree_level(_leaf_level(table)))
    server.stop()
  ref_losses, ref_state, ref_leaves = runs['graph']
  assert len(np.unique(ref_leaves[ref_leaves > 0])) > 1
  for name in ('eager', 'one stream'):
    losses, state, leaves = runs[name]
    assert torch.equal(losses, ref_losses), f'{name}: losses differ from the graph run'
    _assert_same_state(state, ref_state, name)
    np.testing.assert_array_equal(leaves, ref_leaves)
  # launches per eager step
  monkeypatch.setenv('B200RL_D4PG_STREAMS', '1')
  counts = {}
  for name, sampler in (('uniform', replay.selectors.Uniform()), ('prioritized', replay.selectors.Prioritized(ALPHA))):
    table, server, _ = _table(sampler, 13, episodes=20)
    policy, critic = _nets(kind, 1)
    ds = replay.ReplayDataset(table, B, seed=11, stratified=False)
    pr = name == 'prioritized'
    learner = _learner(kind, policy, critic, ds, False, beta=BETA if pr else None, client=replay.Client(server) if pr else None)
    learner.step(fetch_loss=False)
    torch.cuda.synchronize()
    n0 = _launches()
    learner.step(fetch_loss=False)
    torch.cuda.synchronize()
    counts[name] = _launches() - n0
    server.stop()
  assert counts['prioritized'] <= counts['uniform'] + 1, counts


def test_prioritized_learner_checkpoint_roundtrip():
  """Learner save() and Table.save() after 3 updates; restoring both (a fresh learner, the table rewound) and running
  the same 3 updates on injected uniforms reproduces the uninterrupted run bit for bit, tree leaves included."""
  import torch
  from test_gpu_d4pg_bf16 import _nets
  from acme_b200 import replay
  B = 256
  table, server, _ = _table(replay.selectors.Prioritized(ALPHA), 14, episodes=20)
  rng = np.random.default_rng(8)
  us = [torch.as_tensor(rng.random(B, dtype=np.float32)).cuda() for _ in range(6)]
  policy, critic = _nets('d4pg', 2)
  a = _learner('d4pg', policy, critic, replay.ReplayDataset(table, B, seed=11, stratified=False), False, beta=BETA,
               client=replay.Client(server))
  for u in us[:3]:
    a.step(uniforms=u, fetch_loss=False)
  torch.cuda.synchronize()
  lstate, tstate = a.save(), table.save()
  for u in us[3:]:
    a.step(uniforms=u, fetch_loss=False)
  torch.cuda.synchronize()
  want_state, want_leaves = _state(a), table.read_tree_level(_leaf_level(table))
  table.restore(tstate)
  policy2, critic2 = _nets('d4pg', 2, seed=10)
  b = _learner('d4pg', policy2, critic2, replay.ReplayDataset(table, B, seed=11, stratified=False), False, beta=BETA,
               client=replay.Client(server))
  b.restore(lstate)
  for u in us[3:]:
    b.step(uniforms=u, fetch_loss=False)
  torch.cuda.synchronize()
  _assert_same_state(_state(b), want_state, 'restored learner')
  np.testing.assert_array_equal(table.read_tree_level(_leaf_level(table)), want_leaves)
  server.stop()


# ------------------------------------------------------------------------------ agents
@pytest.mark.parametrize('num_envs', [1, 16])
@pytest.mark.parametrize('kind', ['d4pg', 'ddpg'])
@pytest.mark.parametrize('prioritized', [True, False])
def test_prioritized_agents_run(kind, num_envs, prioritized):
  import torch
  from acme_b200 import d4pg, environment_loop, loggers, networks, specs, testing
  envs = [testing.ContinuousEnvironment(episode_length=10, bounded=True) for _ in range(num_envs)]
  spec = specs.make_environment_spec(envs[0])
  policy = networks.D4PGPolicy(1, 1, sizes=(10, 10), seed=0)
  critic = (networks.D4PGCritic(1, 1, sizes=(10, 10), seed=1) if kind == 'd4pg' else networks.DDPGCritic(1, 1, sizes=(10, 10), seed=1))
  cls = d4pg.D4PG if kind == 'd4pg' else d4pg.DDPG
  extra = dict(priority_exponent=ALPHA, importance_sampling_exponent=BETA) if prioritized else {}
  # batched acting makes a step's items sampleable one lockstep step later: the first update waits for 4 such steps
  ag = cls(spec, policy, critic, batch_size=10, samples_per_insert=2, min_replay_size=10 if num_envs == 1 else 4 * num_envs,
           max_replay_size=1000, logger=loggers.NoOpLogger(), num_envs=num_envs, **extra)
  gc.collect()
  if num_envs > 1:
    loop = environment_loop.BatchedEnvironmentLoop(envs, ag, logger=loggers.NoOpLogger())
    loop.run(num_episodes=2 * num_envs)
  else:
    loop = environment_loop.EnvironmentLoop(envs[0], ag, logger=loggers.NoOpLogger())
    loop.run(num_episodes=4)
  torch.cuda.synchronize()
  learner = ag._learner
  assert learner.num_steps > 0
  table = ag._table
  assert table.alpha == (ALPHA if prioritized else 0.0)
  leaves = table.read_tree_level(_leaf_level(table))[:table.size]
  if prioritized:
    assert len(np.unique(leaves)) > 1, 'the learner wrote no priorities'
  else:
    np.testing.assert_array_equal(leaves, np.ones_like(leaves))
