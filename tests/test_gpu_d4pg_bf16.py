"""The D4PG / DDPG networks in the bf16 dataflow (precision 2): the two kernels it adds, and the learners end to end.

`b200rl_layernorm_tanh_fwd_bf16` must reproduce `b200rl_layernorm_tanh_fwd` bit for bit and store RN-bf16(y) beside it.
`b200rl_dense_head_bwd_bf16` (a head of N <= 64 outputs: dx in bf16, dw / db in fp32, one launch) is held against an
fp64 reference on the same operands with the bound of the bf16 layer suite,

    |got - ref| <= 2^-16 (|A|.|B|)_ij + c_out |ref_ij|      (c_out = 2^-8 for the bf16 dx, 0 for dw / db)

inside sentinel-guarded outputs, with one launch per call and bit-identical results across calls and streams.

The learners run at the C3 shape (67-d observations, 21-d actions, 51 atoms, batch 256, n = 5) against
oracle.learner.D4PGOracleLearner / DDPGOracleLearner.  Stated bounds, as fractions of each quantity's scale (max
|reference|): C3_TOL below.  The errors measured on a B200 are written to $B200RL_PARITY_DIR/parity_c3_<learner>_<mode>.json
when that variable is set and are quoted in DESIGN.md (K6, the C3 table)."""
import json
import os

import numpy as np
import pytest
from layer_check import ELU, NONE, SENT, Out, Workspace, _capi, _check, _rejects, assert_sig, mask_factor, mask_values, run

pytestmark = pytest.mark.gpu

_KEEP = []

C3_TOL = {1: dict(value=1e-2, grad_rel_l2=5e-2), 2: dict(value=2e-2, grad_rel_l2=1e-1)}
OBS, ACT = 67, 21


def dev(x, dtype=None):
  import torch
  t = torch.as_tensor(np.ascontiguousarray(x)).cuda()
  if dtype is not None:
    t = t.to(dtype)
  _KEEP.append(t)
  return t


@pytest.fixture(autouse=True)
def _release():
  yield
  import torch
  torch.cuda.synchronize()
  _KEEP.clear()


def bf(x):
  """array rounded to bf16 (returned as float64, exact)"""
  import torch
  return torch.as_tensor(np.ascontiguousarray(x, np.float32)).to(torch.bfloat16).double().numpy()


def mat_dev(a, ld=None, bf16=True):
  """[rows][cols] device matrix with row stride ld; the padding columns hold NaN (a kernel that reads them poisons its
  sums)"""
  import torch
  rows, cols = a.shape
  ld = ld or cols
  t = torch.full((rows, ld), float('nan'), dtype=torch.bfloat16 if bf16 else torch.float32, device='cuda')
  t[:, :cols] = torch.as_tensor(np.ascontiguousarray(a, np.float32)).to(t.dtype).cuda()
  _KEEP.append(t)
  return t


def stream():
  return _capi().current_stream()


# ------------------------------------------------------------------------------ LayerNorm + tanh with a bf16 copy
@pytest.mark.parametrize('N', [256, 512])
@pytest.mark.parametrize('B', [1, 256])
def test_layernorm_tanh_fwd_bf16(B, N):
  import torch
  c = _capi()
  rng = np.random.default_rng(B + N)
  x = dev((rng.standard_normal((B, N)) * 3 + 0.5).astype(np.float32))
  sc = dev((1 + 0.3 * rng.standard_normal(N)).astype(np.float32))
  of = dev((0.2 * rng.standard_normal(N)).astype(np.float32))
  f = lambda *s: torch.full(s, float('nan'), device='cuda')
  y, xh, rs, y2, xh2, rs2 = f(B, N), f(B, N), f(B), f(B, N), f(B, N), f(B)
  yb = Out(B, N, True)
  assert_sig('layernorm fp32', run(lambda: c.call('b200rl_layernorm_tanh_fwd', B, N, x.data_ptr(), sc.data_ptr(), of.data_ptr(), 1e-5,
                                                  y.data_ptr(), xh.data_ptr(), rs.data_ptr(), stream())), ['layernorm_tanh_fwd_kernel'])
  assert_sig('layernorm bf16', run(lambda: c.call('b200rl_layernorm_tanh_fwd_bf16', B, N, x.data_ptr(), sc.data_ptr(), of.data_ptr(),
                                                  1e-5, y2.data_ptr(), yb.ptr, xh2.data_ptr(), rs2.data_ptr(), stream())),
             ['layernorm_tanh_fwd_kernel'])
  for what, a, b in (('y', y, y2), ('xhat', xh, xh2), ('rstd', rs, rs2)):
    assert torch.equal(a.view(torch.int32), b.view(torch.int32)), f'{what} differs from b200rl_layernorm_tanh_fwd'
  got = yb.read('y_bf16')
  np.testing.assert_array_equal(got, y.to(torch.bfloat16).double().cpu().numpy())


def test_layernorm_tanh_fwd_bf16_rejects_null():
  c = _capi()
  o = Out(4, 64, True)
  p = dev(np.ones((4, 64), np.float32)).data_ptr()
  _rejects('null y_bf16', 'b200rl_layernorm_tanh_fwd_bf16', o, 4, 64, p, p, p, 1e-5, p, None, p, p, None)


# ------------------------------------------------------------------------------ dense head backward
# M, N, K, options.  N: 51 = the D4PG critic's atoms, 21 = the policy's actions, 1 = the DDPG critic; K = the last hidden
# width.  grads: which of dw / db are requested; mask: the producer of the layer below (ELU) or none; ws None: no
# workspace (one row slice per column block).
HEAD_BWD = [
    (256, 51, 256, {}),
    (256, 21, 256, {}),
    (256, 1, 256, {}),
    (256, 64, 512, {}),
    (256, 51, 512, {'mask': NONE}),
    (33, 21, 512, {}),
    (33, 1, 256, {'ldx': 264, 'lddx': 320, 'lddy': 9}),
    (1, 51, 256, {}),
    (1, 64, 512, {'mask': NONE, 'lddy': 72}),
    (256, 51, 512, {'grads': ''}),
    (256, 21, 256, {'grads': 'dw'}),
    (33, 64, 256, {'grads': 'db'}),
    (256, 51, 256, {'ws': None}),
    (256, 21, 512, {'ldx': 576, 'lddx': 520, 'lddy': 64}),
]


def _hb_id(v):
  return None if not isinstance(v, dict) else '-'.join(f'{k}{v[k]}' for k in v) or 'default'


def _head_call(M, N, K, dyd, lddy, xd, ldx, wd, dx, mask, mact, dw, db, wsp, wsb):
  return lambda: _capi().call('b200rl_dense_head_bwd_bf16', M, N, K, dyd.data_ptr(), lddy, xd.data_ptr(), ldx, wd.data_ptr(), dx.ptr,
                              dx.ld, mask, mact, dw.ptr if dw else None, db.ptr if db else None, wsp, wsb, stream())


@pytest.mark.parametrize('M,N,K,opt', HEAD_BWD, ids=_hb_id)
def test_dense_head_bwd_bf16(M, N, K, opt):
  import torch
  rng = np.random.default_rng(M * 5 + N * 3 + K)
  ldx, lddx, lddy = opt.get('ldx', K), opt.get('lddx', K), opt.get('lddy', N)
  grads, mact = opt.get('grads', 'dw db'), opt.get('mask', ELU)
  dy = rng.standard_normal((M, N)).astype(np.float32).astype(np.float64)
  x = bf(mask_values(rng, (M, K), ELU))
  w = bf(rng.standard_normal((N, K)) / np.sqrt(N))
  y = bf(mask_values(rng, (M, K), ELU))
  dyd, xd, wd = mat_dev(dy, lddy, bf16=False), mat_dev(x, ldx), mat_dev(w)
  maskd = mat_dev(y, lddx) if mact != NONE else None
  ws = Workspace()
  wsp, wsb = (ws.ptr, ws.bytes) if 'ws' not in opt else (None, 0)
  dx = Out(M, K, True, ld=lddx)
  dw = Out(N, K, False) if 'dw' in grads else None
  db = Out(1, N, False) if 'db' in grads else None
  call = _head_call(M, N, K, dyd, lddy, xd, ldx, wd, dx, maskd.data_ptr() if maskd is not None else None, mact, dw, db, wsp, wsb)
  what = f'dense head bwd {M}x{N}x{K} {opt}'
  assert_sig(what, run(call), ['dense_head_bwd_bf16_kernel'])
  g, gabs = mask_factor(y, mact) if mact != NONE else (1., 1.)
  _check(f'{what} dx', dx.read('dx'), (dy @ w) * g, (np.abs(dy) @ np.abs(w)) * gabs, True)
  if dw:
    _check(f'{what} dw', dw.read('dw'), dy.T @ x, np.abs(dy).T @ np.abs(x), False)
  if db:
    _check(f'{what} db', db.read('db')[0], dy.sum(0), np.abs(dy).sum(0), False)
  outs = [o for o in (dx, dw, db) if o is not None]
  first = [o.bits() for o in outs]
  # again, on the same stream, then on another stream with another workspace: bit-identical
  ws2 = Workspace()
  for i, side in enumerate((False, True)):
    for o in outs:
      o.reset()
    if side:
      s = torch.cuda.Stream()
      s.wait_stream(torch.cuda.current_stream())
      with torch.cuda.stream(s):
        _head_call(M, N, K, dyd, lddy, xd, ldx, wd, dx, maskd.data_ptr() if maskd is not None else None, mact, dw, db,
                   ws2.ptr if wsp else None, wsb)()
      torch.cuda.current_stream().wait_stream(s)
    else:
      n, _ = run(call, profile=False)
      assert n == 1
    torch.cuda.synchronize()
    for o, b in zip(outs, first):
      assert torch.equal(o.bits(), b), f'{what}: call {i + 2} ({"side stream" if side else "same stream"}) differs'


def test_dense_head_bwd_bf16_rejects():
  c = _capi()
  M, K = 8, 64
  buf = dev(np.zeros(4096, np.float32))
  p = buf.data_ptr()
  dx = Out(M, K, True)
  ws = Workspace()
  args = lambda N=21, K=K, x=p, ldx=K, dy=p: (M, N, K, dy, max(N, 1), x, ldx, p, dx.ptr, dx.ld, None, NONE, p + 8192, p + 12288,
                                              ws.ptr, ws.bytes, None)
  for what, a in (('N = 0', args(N=0)), ('N = 65', args(N=65)), ('K % 8 != 0', args(K=60)), ('x not 16-byte aligned', args(x=p + 2)),
                  ('ldx % 8 != 0', args(ldx=K + 4)), ('null dy', args(dy=None))):
    _rejects(what, 'b200rl_dense_head_bwd_bf16', dx, *a)
  assert bool((ws.buf == SENT).all())


# ------------------------------------------------------------------------------ whole learners at the C3 shape
def _export_flat(net, flat):
  """Sonnet-shaped export of any flat buffer laid out like the network's parameters (Adam moments, gradients)."""
  saved = net.params.flat
  net.params.flat = flat
  try:
    return net.variables()
  finally:
    net.params.flat = saved


def _scale_err(got, want):
  got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
  return float(np.abs(got - want).max() / max(np.abs(want).max(), 1e-30))


def _replay(B, seed, episodes=40):
  import helpers
  rng = np.random.default_rng(seed)
  spec, table, server, adder, oracle = helpers.make_pair((OBS,), np.float32, 0, 5, 0.99, 0.0, max_size=4000, act_dim=ACT)
  for _ in range(episodes):
    helpers.feed_episode(rng, adder, oracle, int(rng.integers(20, 80)), 5, (OBS,), np.float32, 0, act_dim=ACT)
  table.flush()
  helpers.sync_oracle_leaves(table, oracle)
  return table, server, oracle


def _nets(kind, precision, seed=0):
  from acme_b200 import networks
  policy = networks.D4PGPolicy(OBS, ACT, seed=1 + seed, precision=precision)
  critic = (networks.D4PGCritic if kind == 'd4pg' else networks.DDPGCritic)(OBS, ACT, seed=2 + seed, precision=precision)
  # make the near-zero-initialised policy head non-trivial so that the actor path is exercised
  pv = policy.variables()
  pv['out/w'] = (np.random.default_rng(3 + seed).standard_normal(pv['out/w'].shape) * 0.05).astype(np.float32)
  policy.load_variables(pv)
  return policy, critic


def _learner(kind, policy, critic, ds, use_graph):
  from acme_b200 import d4pg, loggers
  cls = d4pg.D4PGLearner if kind == 'd4pg' else d4pg.DDPGLearner
  return cls(policy, critic, policy.clone(), critic.clone(), 0.99, target_update_period=2, dataset=ds, logger=loggers.NoOpLogger(),
             use_cuda_graph=use_graph)


def _assert_shadows(learner, what):
  import torch
  for name, net in (('policy', learner._policy), ('critic', learner._critic), ('target policy', learner._tpolicy),
                    ('target critic', learner._tcritic)):
    assert torch.equal(net.params.shadow.view(torch.int16), net.params.flat.to(torch.bfloat16).view(torch.int16)), \
        f'{what}: {name} shadow != bf16(parameters)'


@pytest.mark.parametrize('precision', [1, 2])
@pytest.mark.parametrize('kind', ['d4pg', 'ddpg'])
def test_learner_c3_shape_parity(kind, precision):
  """Three updates on injected uniforms.  Before each, the oracle adopts the device networks (online and target) and Adam
  moments, so every update is compared from an identical state; the target copy (period 2) happens at updates 0 and 2.
  Precision 2 also checks after every update that each bf16 weight shadow equals RN-bf16 of its parameters."""
  import torch
  from oracle import learner as olearner
  from oracle import nets as onets
  from acme_b200 import replay
  B = 256
  tolv = C3_TOL[precision]
  table, server, oracle = _replay(B, 12)
  policy, critic = _nets(kind, precision)
  ds = replay.ReplayDataset(table, B, seed=11, stratified=False)
  learner = _learner(kind, policy, critic, ds, use_graph=False)
  tpolicy, tcritic = learner._tpolicy, learner._tcritic
  ocls = onets.D4PGCritic if kind == 'd4pg' else onets.DDPGCritic
  opol, ocri, otp, otc = onets.D4PGPolicy(OBS, ACT), ocls(OBS, ACT), onets.D4PGPolicy(OBS, ACT), ocls(OBS, ACT)
  ol = (olearner.D4PGOracleLearner if kind == 'd4pg' else olearner.DDPGOracleLearner)(opol, ocri, otp, otc, 0.99, 2)
  rng = np.random.default_rng(5)
  measured = []
  for step in range(3):
    for o, net in ((opol, policy), (ocri, critic), (otp, tpolicy), (otc, tcritic)):
      o.load(net.variables())
    ol.popt.m, ol.popt.v, ol.popt.t = _export_flat(policy, learner._pm), _export_flat(policy, learner._pv), step
    ol.copt.m, ol.copt.v, ol.copt.t = _export_flat(critic, learner._cm), _export_flat(critic, learner._cv), step
    ol.num_steps = step
    u = rng.random(B, dtype=np.float32)
    keys, pos, prob = oracle.sample(u, False)
    ref = ol.step(*oracle.gather(pos))
    learner.step(uniforms=torch.as_tensor(u).cuda())
    torch.cuda.synchronize()
    np.testing.assert_array_equal(ds.idx.cpu().numpy(), pos)                         # sampled indices: bit-exact
    cscale, pscale = float(learner._cscale.cpu()[0]), float(learner._pscale.cpu()[0])
    cg, pg = _export_flat(critic, critic.params.grad), _export_flat(policy, policy.params.grad)
    rel = lambda got, want: float(np.linalg.norm(got.astype(np.float64) - want) / max(np.linalg.norm(want), 1e-30))
    err = dict(step=step,
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
    else:
      err['td'] = _scale_err(learner.td.cpu().numpy(), ref['td'])
    measured.append(err)
    if precision == 2:
      _assert_shadows(learner, f'update {step}')
  out = os.environ.get('B200RL_PARITY_DIR')
  if out:
    os.makedirs(out, exist_ok=True)
    mode = {1: 'tf32', 2: 'bf16'}[precision]
    with open(os.path.join(out, f'parity_c3_{kind}_{mode}.json'), 'w') as f:
      json.dump(dict(learner=kind, mode=mode, B=B, obs=OBS, act=ACT, n=5, tolerances=tolv, measured=measured), f, indent=1)
  for err in measured:
    for k, v in err.items():
      if k == 'step':
        continue
      if isinstance(v, dict):
        assert max(v.values()) <= tolv['grad_rel_l2'], (k, err['step'], v)
      else:
        assert v <= tolv['value'], (k, err['step'], v)
  server.stop()


def _state(learner):
  import torch
  nets = (learner._policy, learner._critic, learner._tpolicy, learner._tcritic)
  return ([n.params.flat.clone() for n in nets] + [n.params.shadow.clone() for n in nets] +
          [t.clone() for t in (learner._pm, learner._pv, learner._cm, learner._cv, learner._num_steps)])


def _assert_same(a, b, what):
  import torch
  names = ['policy', 'critic', 'target policy', 'target critic'] * 2
  names = [n + (' shadow' if i >= 4 else '') for i, n in enumerate(names)] + ['policy m', 'policy v', 'critic m', 'critic v', 'steps']
  for n, x, y in zip(names, a, b):
    assert torch.equal(x, y), f'{what}: {n} differs'


@pytest.mark.parametrize('kind', ['d4pg', 'ddpg'])
def test_bf16_learner_launch_order_is_bit_identical(kind, monkeypatch):
  """Precision 2, 6 updates on the learner's own device draws: eager, one CUDA graph (captured at the third update) and
  a single stream (B200RL_D4PG_STREAMS=0) give bit-identical losses, parameters, Adam moments and shadows."""
  import torch
  from acme_b200 import replay
  B = 256
  table, server, _ = _replay(B, 13, episodes=20)
  runs = {}
  for name, graph, streams in (('graph', True, '1'), ('eager', False, '1'), ('one stream', True, '0')):
    monkeypatch.setenv('B200RL_D4PG_STREAMS', streams)
    policy, critic = _nets(kind, 2)
    ds = replay.ReplayDataset(table, B, seed=11, stratified=False)
    learner = _learner(kind, policy, critic, ds, use_graph=graph)
    losses = []
    for _ in range(6):
      learner.step(fetch_loss=False)
      losses.append(torch.cat([learner.critic_loss, learner.policy_loss]).clone())
    torch.cuda.synchronize()
    _assert_shadows(learner, name)
    runs[name] = (torch.stack(losses), _state(learner))
  ref_losses, ref_state = runs['graph']
  for name in ('eager', 'one stream'):
    losses, state = runs[name]
    assert torch.equal(losses, ref_losses), f'{name}: losses differ from the graph run'
    _assert_same(state, ref_state, name)
  server.stop()


def test_bf16_learner_checkpoint_roundtrip():
  """save() -> a fresh learner (other initial weights) -> restore(): the next update is bit-identical."""
  import torch
  from acme_b200 import replay
  B = 256
  table, server, _ = _replay(B, 14, episodes=20)
  rng = np.random.default_rng(8)
  policy, critic = _nets('d4pg', 2)
  a = _learner('d4pg', policy, critic, replay.ReplayDataset(table, B, seed=11, stratified=False), use_graph=False)
  for _ in range(3):
    a.step(uniforms=torch.as_tensor(rng.random(B, dtype=np.float32)).cuda(), fetch_loss=False)
  state = a.save()
  policy2, critic2 = _nets('d4pg', 2, seed=10)
  b = _learner('d4pg', policy2, critic2, replay.ReplayDataset(table, B, seed=11, stratified=False), use_graph=False)
  b.restore(state)
  _assert_shadows(b, 'restored')
  u = torch.as_tensor(rng.random(B, dtype=np.float32)).cuda()
  a.step(uniforms=u, fetch_loss=False)
  b.step(uniforms=u, fetch_loss=False)
  torch.cuda.synchronize()
  assert torch.equal(a.critic_loss, b.critic_loss) and torch.equal(a.policy_loss, b.policy_loss)
  _assert_same(_state(b), _state(a), 'restored learner')
  server.stop()


# ------------------------------------------------------------------------------ interface
@pytest.mark.parametrize('sizes', [(300, 200), (512,), (512, 200), (256, 2048)])
def test_bf16_layernorm_mlp_rejects_shapes(sizes):
  from acme_b200 import networks
  with pytest.raises(ValueError, match='precision 2'):
    networks.D4PGPolicy(OBS, ACT, sizes=sizes, precision=2)


def test_bf16_layernorm_mlp_rejects_wide_head():
  from acme_b200 import networks
  with pytest.raises(ValueError, match='head'):
    networks.D4PGCritic(OBS, ACT, num_atoms=101, precision=2)


def test_gaussian_noise_policy_bf16_matches_fp32():
  """sigma = 0: the behaviour policy's action (batch 1) in precision 2 is the fp32 policy's within the precision-2 bound."""
  from acme_b200 import d4pg
  p0, _ = _nets('d4pg', 0)
  p2, _ = _nets('d4pg', 2)
  rng = np.random.default_rng(9)
  pi0 = d4pg.GaussianNoisePolicy(p0, 0.0, -np.ones(ACT, np.float32), np.ones(ACT, np.float32))
  pi2 = d4pg.GaussianNoisePolicy(p2, 0.0, -np.ones(ACT, np.float32), np.ones(ACT, np.float32))
  for _ in range(4):
    o = rng.standard_normal(OBS).astype(np.float32)
    a0, a2 = pi0(o), pi2(o)
    assert a2.dtype == np.float32 and a2.shape == (ACT,)
    assert _scale_err(a2, a0) <= C3_TOL[2]['value'], (a0, a2)
