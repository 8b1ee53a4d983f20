"""GPU parity of the learner math (K4 TD/Huber/IS, K5 C51, K6 layers fwd/bwd, K7 Adam) through the
C ABI against the fp32 oracle.  Tolerance: 1e-5 relative (north_star) with an absolute floor that
scales with the magnitude of the tensor (different fp32 summation orders)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

RTOL = 1e-5
# Layer-level tolerance of the tensor-core mode (precision=1): multiplicands are rounded to tf32 (TMA path) or bf16
# (loader-fed path), products and sums are fp32; single layers are compared at 2e-2 of the tensor's scale.  The
# whole-learner tolerances at the benchmarked shapes are TC_TOL (test_dqn_learner_c2_shape_parity).
TC_LAYER_TOL = dict(rtol=2e-2, atol_scale=2e-2)


def tol(precision, **fp32_kwargs):
  return dict(TC_LAYER_TOL) if precision == 1 else fp32_kwargs


def close(got, want, rtol=RTOL, atol_scale=1e-6, name=''):
  got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
  atol = atol_scale * max(float(np.abs(want).max()), 1e-30)
  np.testing.assert_allclose(got, want, rtol=rtol, atol=atol, err_msg=name)


_KEEP = []


def dev(x):
  """Host array -> device tensor that stays alive until the end of the test (raw pointers are passed
  to the C ABI, so a temporary would be recycled by the caching allocator)."""
  import torch
  t = torch.as_tensor(np.ascontiguousarray(x)).cuda()
  _KEEP.append(t)
  return t


@pytest.fixture(autouse=True)
def _release_device_tensors():
  yield
  import torch
  if torch.cuda.is_available():
    torch.cuda.synchronize()
  _KEEP.clear()


def empty(*shape, dtype=None):
  import torch
  return torch.empty(shape, dtype=dtype or torch.float32, device='cuda')


@pytest.mark.parametrize('B,A,wmax,wdtype', [(256, 18, None, 'f64'), (10, 3, None, 'f64'), (2048, 18, None, 'f64'),
                                             (256, 18, 7.5, 'f64'), (256, 18, None, 'f32'), (64, 5, 7.5, 'f32')])
def test_dqn_td_kernel(B, A, wmax, wdtype):
  import torch
  from acme_b200 import _capi
  from oracle import losses
  rng = np.random.default_rng(B + A)
  q_tm1, q_tv, q_ts = (rng.standard_normal((B, A)).astype(np.float32) * 3 for _ in range(3))
  q_ts[0, :] = 1.0                                          # ties -> first index
  a = rng.integers(0, A, B).astype(np.int32)
  R = (rng.standard_normal(B) * 2).astype(np.float32)
  D = rng.choice([0., 0.9801, 1.0], B).astype(np.float32)
  prob = rng.uniform(1e-7, 1e-3, B).astype(np.float32)
  ref = losses.dqn_loss(q_tm1, q_tv, q_ts, a, R, D, prob, 0.99, 1.0, 0.2, 1.0, global_wmax=wmax, weights_dtype=wdtype)
  td, lps, w, pr, dq, lm = empty(B), empty(B), empty(B), empty(B), empty(B, A), empty(1)
  wm = dev(np.array([wmax], np.float64)) if wmax else None
  flags = _capi.TD_IS_WEIGHTS_F32 if wdtype == 'f32' else 0   # jax/dqn/learning.py:94-96 vs dqn/learning.py:138-143
  _capi.call('b200rl_dqn_td', B, A, dev(q_tm1).data_ptr(), dev(q_tv).data_ptr(), dev(q_ts).data_ptr(), dev(a).data_ptr(),
             dev(R).data_ptr(), dev(D).data_ptr(), dev(prob).data_ptr(), 0.99, 1.0, 0.2, 1.0, _capi.ptr(wm), 1.0 / B,
             td.data_ptr(), lps.data_ptr(), w.data_ptr(), pr.data_ptr(), dq.data_ptr(), lm.data_ptr(), flags,
             _capi.current_stream())
  torch.cuda.synchronize()
  np.testing.assert_array_equal(td.cpu().numpy(), ref['td'])          # same fp32 op order: bit-exact
  np.testing.assert_array_equal(pr.cpu().numpy(), np.abs(ref['td']))
  close(w.cpu().numpy(), ref['weight'], name='weight')
  close(lps.cpu().numpy(), ref['per_sample'], name='per-sample loss')
  close(lm.cpu().numpy()[0], ref['loss'], name='loss')
  close(dq.cpu().numpy(), ref['dq_tm1'], name='dq')
  if wmax is None:
    out = dev(np.zeros(1, np.float64))
    _capi.call('b200rl_is_weight_max', B, dev(prob).data_ptr(), 0.2, out.data_ptr(), flags, _capi.current_stream())
    close(out.cpu().numpy()[0], ref['wmax64'], rtol=1e-12 if wdtype == 'f64' else 1e-6)


@pytest.mark.parametrize('B,K,vmin,vmax', [(256, 51, -150., 150.), (7, 51, -10., 10.), (64, 11, 0., 5.)])
def test_c51_projection_and_loss(B, K, vmin, vmax):
  import torch
  from acme_b200 import _capi
  from oracle import losses
  rng = np.random.default_rng(K + B)
  lt1, lt = rng.standard_normal((B, K)).astype(np.float32) * 2, rng.standard_normal((B, K)).astype(np.float32) * 2
  R = rng.uniform(-1, 1, B).astype(np.float32) * (vmax - vmin) / 4
  D = rng.choice([0., 0.96, 1.0], B).astype(np.float32)
  R[0], D[0] = 0.0, 1.0   # gamma=1 below for this row would land on atoms; keep generic + explicit case
  values = np.linspace(vmin, vmax, K, dtype=np.float32)
  gamma = 0.99
  ref = losses.categorical(lt1, lt, values, R, (np.float32(gamma) * D).astype(np.float32))
  tgt, lps, dl, lm = empty(B, K), empty(B), empty(B, K), empty(1)
  _capi.call('b200rl_c51_loss', B, K, vmin, vmax, dev(lt1).data_ptr(), dev(lt).data_ptr(), dev(R).data_ptr(),
             dev(D).data_ptr(), gamma, 1.0 / B, tgt.data_ptr(), lps.data_ptr(), dl.data_ptr(), lm.data_ptr(),
             _capi.current_stream())
  torch.cuda.synchronize()
  close(tgt.cpu().numpy(), ref['target'], name='projected distribution')
  close(lps.cpu().numpy(), ref['loss'], name='CE loss')
  close(dl.cpu().numpy(), ref['dlogits_tm1'], atol_scale=1e-5, name='dlogits')
  close(lm.cpu().numpy()[0], ref['loss'].mean())
  np.testing.assert_allclose(tgt.cpu().numpy().sum(-1), 1.0, atol=1e-5)   # projection conserves mass


def test_c51_atoms_landing_exactly_on_support():
  import torch
  from acme_b200 import _capi
  from oracle import losses
  B, K, vmin, vmax = 4, 51, -150., 150.
  values = np.linspace(vmin, vmax, K, dtype=np.float32)
  lt = np.random.default_rng(0).standard_normal((B, K)).astype(np.float32)
  R = np.array([0., 6., -12., 400.], np.float32)     # shifts by whole atoms; last row clips to vmax
  D = np.ones(B, np.float32)
  ref = losses.categorical(lt, lt, values, R, D)
  tgt, lps = empty(B, K), empty(B)
  _capi.call('b200rl_c51_loss', B, K, vmin, vmax, dev(lt).data_ptr(), dev(lt).data_ptr(), dev(R).data_ptr(), dev(D).data_ptr(),
             1.0, 1.0, tgt.data_ptr(), lps.data_ptr(), None, None, _capi.current_stream())
  torch.cuda.synchronize()
  close(tgt.cpu().numpy(), ref['target'])
  p = losses.softmax(lt)
  close(tgt.cpu().numpy()[0], p[0])                   # identity shift reproduces the distribution
  assert abs(tgt.cpu().numpy()[3, -1] - 1.0) < 1e-5   # everything clipped onto vmax


def test_c51_mean_and_dpg():
  import torch
  from acme_b200 import _capi
  from oracle import losses
  rng = np.random.default_rng(3)
  B, K, A = 33, 51, 21
  logits = rng.standard_normal((B, K)).astype(np.float32)
  values = np.linspace(-150, 150, K, dtype=np.float32)
  p = losses.softmax(logits)
  q_ref = (p * values).sum(-1)
  q, dl = empty(B), empty(B, K)
  _capi.call('b200rl_c51_mean_fwd', B, K, -150., 150., dev(logits).data_ptr(), q.data_ptr(), _capi.current_stream())
  _capi.call('b200rl_c51_mean_bwd', B, K, -150., 150., dev(logits).data_ptr(), None, dl.data_ptr(), _capi.current_stream())
  close(q.cpu().numpy(), q_ref, atol_scale=1e-5)
  close(dl.cpu().numpy(), p * (values[None] - q_ref[:, None]), atol_scale=1e-5)
  dqda = rng.standard_normal((B, A)).astype(np.float32) * np.linspace(0.01, 3, B, dtype=np.float32)[:, None]
  da_ref, clipped = losses.dpg_action_grad(dqda, 1.0, True)
  da, lps, lm = empty(B, A), empty(B), empty(1)
  _capi.call('b200rl_dpg_action_grad', B, A, dev(dqda).data_ptr(), 1.0, 1, 1.0 / B, da.data_ptr(), lps.data_ptr(),
             lm.data_ptr(), _capi.current_stream())
  close(da.cpu().numpy(), da_ref)
  close(lm.cpu().numpy()[0], 0.5 * (clipped**2).sum(-1).mean())


@pytest.mark.parametrize('eps_mode', [0, 1])
def test_adam_and_global_norm(eps_mode):
  import torch
  from acme_b200 import _capi
  from oracle import learner as olearner
  from oracle import losses
  rng = np.random.default_rng(eps_mode)
  n = 100_003
  p0 = rng.standard_normal(n).astype(np.float32)
  opt = olearner.Adam(1e-3, eps_mode=eps_mode)
  params = {'p': p0.copy()}
  P = torch.zeros(n + 1, device='cuda')[:n]
  P.copy_(dev(p0))
  m, v = torch.zeros_like(P), torch.zeros_like(P)
  step = torch.zeros(1, dtype=torch.int64, device='cuda')
  shadow = torch.zeros(n, dtype=torch.bfloat16, device='cuda')
  for t in range(3):
    g = (rng.standard_normal(n) * 10.0**rng.integers(-6, 1, n)).astype(np.float32)
    params = opt.apply({'p': g}, params)
    _capi.call('b200rl_adam', n, P.data_ptr(), dev(g).data_ptr(), m.data_ptr(), v.data_ptr(), step.data_ptr(), 1e-3, 0.9,
               0.999, 1e-8, eps_mode, None, shadow.data_ptr(), _capi.current_stream())
    _capi.call('b200rl_step_increment', step.data_ptr(), _capi.current_stream())
    close(P.cpu().numpy(), params['p'], name=f'params after step {t}')
    close(m.cpu().numpy(), opt.m['p'])
    close(v.cpu().numpy(), opt.v['p'], atol_scale=1e-9)
  np.testing.assert_array_equal(shadow.float().cpu().numpy(), P.to(torch.bfloat16).float().cpu().numpy())
  # decayed moments: gradients vanish, m and v shrink by 0.9 / 0.999 per update until they cross FLT_MIN, where kernel
  # and oracle both flush them to zero (VERDICT r1 weak #10: one stated arithmetic on both sides)
  tiny = np.float32(np.finfo(np.float32).tiny)
  m0 = (tiny * rng.uniform(0.2, 5.0, n)).astype(np.float32) * rng.choice([-1, 1], n).astype(np.float32)
  v0 = (tiny * rng.uniform(0.2, 5.0, n)).astype(np.float32)
  opt.m['p'], opt.v['p'] = m0.copy(), v0.copy()
  m.copy_(dev(m0)); v.copy_(dev(v0))
  zero_g = np.zeros(n, np.float32)
  params = opt.apply({'p': zero_g}, params)
  _capi.call('b200rl_adam', n, P.data_ptr(), dev(zero_g).data_ptr(), m.data_ptr(), v.data_ptr(), step.data_ptr(), 1e-3, 0.9,
             0.999, 1e-8, eps_mode, None, None, _capi.current_stream())
  np.testing.assert_array_equal(m.cpu().numpy(), opt.m['p'])
  np.testing.assert_array_equal(v.cpu().numpy(), opt.v['p'])
  assert (opt.m['p'] == 0).any() and (opt.m['p'] != 0).any()          # the case straddles the flush threshold
  close(P.cpu().numpy(), params['p'], name='params after the decayed-moment update')
  # clip_by_global_norm
  g = (rng.standard_normal(n) * 3).astype(np.float32)
  ref, norm = losses.clip_by_global_norm([g], 40.)
  part, scale, nrm = empty(1024), empty(1), empty(1)
  _capi.call('b200rl_global_norm_scale', n, dev(g).data_ptr(), 40., part.data_ptr(), scale.data_ptr(), nrm.data_ptr(),
             _capi.current_stream())
  close(nrm.cpu().numpy()[0], norm)
  close(scale.cpu().numpy()[0], 40. / max(norm, 40.))


def test_copy_if_period_and_step_counter():
  import torch
  from acme_b200 import _capi
  src, dst = torch.arange(1024, dtype=torch.float32, device='cuda'), torch.zeros(1024, device='cuda')
  step = torch.zeros(1, dtype=torch.int64, device='cuda')
  for t in range(7):
    src += 1
    _capi.call('b200rl_copy_if_period', 4096, dst.data_ptr(), src.data_ptr(), step.data_ptr(), 3, 0, _capi.current_stream())
    _capi.call('b200rl_step_increment', step.data_ptr(), _capi.current_stream())
    expect = (t // 3) * 3 + 1     # copies at steps 0, 3, 6 (dqn/learning.py:157-161)
    assert float(dst[0]) == expect, (t, float(dst[0]))
  assert int(step) == 7


# ------------------------------------------------------------------------------------ K6 layers
# single layers against an fp64 reference: test_gpu_fp32_layers.py (precisions 0 and 1), test_gpu_bf16_layers.py
@pytest.mark.parametrize('act', [0, 1, 2, 3])
def test_act_bwd_matches_fp32_derivative(act):
  """b200rl_act_bwd: dy *= act'(y) from the activation's output, bit for bit the fp32 expression (learner_math.cu is built
  without multiply-add contraction): ReLU y > 0, ELU y > 0 ? 1 : y + 1, tanh 1 - y * y; ACT_NONE leaves dy untouched."""
  from acme_b200 import _capi
  rng = np.random.default_rng(act)
  n = 100_003
  z = rng.standard_normal(n).astype(np.float32)
  y = {0: z, 1: np.maximum(z, 0), 2: np.where(z > 0, z, np.expm1(np.minimum(z, 0))), 3: np.tanh(z)}[act].astype(np.float32)
  y[:4] = np.array([0., -0., 1e-30, -1.], np.float32)
  dy = rng.standard_normal(n).astype(np.float32)
  one = np.float32(1)
  g = {0: np.ones_like(y), 1: (y > 0).astype(np.float32), 2: np.where(y > 0, one, y + one), 3: one - y * y}[act]
  d, yd = dev(dy), dev(y)
  _capi.call('b200rl_act_bwd', n, d.data_ptr(), yd.data_ptr(), act, _capi.current_stream())
  np.testing.assert_array_equal(d.cpu().numpy(), (dy * g.astype(np.float32)).astype(np.float32))


def test_layernorm_tanh_and_small_ops():
  import torch
  from acme_b200 import _capi
  rng = np.random.default_rng(9)
  B, N = 17, 512
  x = (rng.standard_normal((B, N)) * 3 + 1).astype(np.float32)
  sc, of = rng.uniform(0.5, 1.5, N).astype(np.float32), rng.standard_normal(N).astype(np.float32) * 0.1
  xt, st_, ot = torch.tensor(x, requires_grad=True), torch.tensor(sc, requires_grad=True), torch.tensor(of, requires_grad=True)
  y_ref = torch.tanh(torch.nn.functional.layer_norm(xt, (N,), st_, ot, eps=1e-5))
  dy = rng.standard_normal((B, N)).astype(np.float32)
  y_ref.backward(torch.tensor(dy))
  y, xh, rs, dx, ds, do = empty(B, N), empty(B, N), empty(B), empty(B, N), empty(N), empty(N)
  s = _capi.current_stream()
  _capi.call('b200rl_layernorm_tanh_fwd', B, N, dev(x).data_ptr(), dev(sc).data_ptr(), dev(of).data_ptr(), 1e-5, y.data_ptr(),
             xh.data_ptr(), rs.data_ptr(), s)
  _capi.call('b200rl_layernorm_tanh_bwd', B, N, dev(dy).data_ptr(), y.data_ptr(), xh.data_ptr(), rs.data_ptr(),
             dev(sc).data_ptr(), dx.data_ptr(), ds.data_ptr(), do.data_ptr(), s)
  close(y.cpu().numpy(), y_ref.detach().numpy(), atol_scale=2e-6)
  close(dx.cpu().numpy(), xt.grad.numpy(), atol_scale=1e-5)
  close(ds.cpu().numpy(), st_.grad.numpy(), atol_scale=1e-5)
  close(do.cpu().numpy(), ot.grad.numpy(), atol_scale=1e-5)
  # duelling head
  A = 18
  val, adv = rng.standard_normal((B, 1)).astype(np.float32), rng.standard_normal((B, A)).astype(np.float32)
  q = empty(B, A)
  _capi.call('b200rl_duelling_fwd', B, A, dev(val).data_ptr(), dev(adv).data_ptr(), q.data_ptr(), s)
  close(q.cpu().numpy(), val + (adv - adv.mean(-1, keepdims=True)))
  dq = rng.standard_normal((B, A)).astype(np.float32)
  dv, da = empty(B), empty(B, A)
  _capi.call('b200rl_duelling_bwd', B, A, dev(dq).data_ptr(), dv.data_ptr(), da.data_ptr(), s)
  close(dv.cpu().numpy(), dq.sum(-1))
  close(da.cpu().numpy(), dq - dq.mean(-1, keepdims=True))


# ------------------------------------------------------------------------------------ whole nets
def _dqn_pair(A=18, seed=0, precision=0):
  from acme_b200 import networks
  from oracle import nets as onets
  net = networks.DQNAtariNetwork(A, seed=seed, precision=precision)
  onet = onets.DQNAtariNetwork(A)
  onet.load(net.variables())
  return net, onet


@pytest.mark.parametrize('precision', [0, 1, 2])
def test_dqn_atari_network_forward_backward(precision):
  import torch
  net, onet = _dqn_pair(precision=precision)
  rng = np.random.default_rng(0)
  B = 6
  obs = rng.integers(0, 256, (B, 84, 84, 4), dtype=np.uint8)
  bufs, gbufs = net.make_buffers(B), net.make_grad_buffers(B)
  q = net.forward(dev(obs), bufs)
  q_ref = onet(torch.tensor(obs.astype(np.float32) / np.float32(255)))
  close(q.cpu().numpy(), q_ref.detach().numpy(), name='q values', **tol(min(precision, 1), atol_scale=5e-6))
  dq = rng.standard_normal((B, 18)).astype(np.float32)
  q_ref.backward(torch.tensor(dq))
  net.backward(dev(obs), bufs, gbufs, dev(dq))
  got = net.variables(grad=True)
  for k, v in onet.vars.items():
    if precision == 0:
      close(got[k], v.grad.numpy(), name=f'grad {k}', atol_scale=1e-5)
    else:
      # bf16 rounding + a few flipped ReLU gates, amplified by the cancellation inside a weight gradient
      # (|sum| << sum|terms|, strongest for conv1): compare in the L2 sense with a loose bound
      want = v.grad.numpy().astype(np.float64)
      rel = np.linalg.norm(got[k] - want) / max(np.linalg.norm(want), 1e-30)
      assert rel < 0.2, f'grad {k}: relative L2 error {rel:.3e}'


def test_variable_export_roundtrip():
  net, onet = _dqn_pair(A=5, seed=3)
  v = net.variables()
  assert v['conv2/w'].shape == (4, 4, 32, 64) and v['value/l0/w'].shape == (7744, 512) and v['adv/l1/w'].shape == (512, 5)
  assert sum(x.size for x in v.values()) == 8_018_611 - (18 - 5) * 513
  net2 = type(net)(5, seed=99)
  net2.load_variables(v)
  for k, x in net2.variables().items():
    np.testing.assert_array_equal(x, v[k])


@pytest.mark.parametrize('mode', ['eager', 'graph', 'pipelined'])
def test_dqn_learner_steps_match_oracle(mode, monkeypatch):
  """Full update (sample -> gather -> 3 forwards -> TD -> backward -> Adam -> priorities -> target copy)
  against oracle.learner.DQNOracleLearner fed by oracle.replay on the same uniform draws.  'pipelined' = the
  single-GPU form whose optimizer half runs at the start of the next step's graph (B200RL_PIPELINE_1GPU=1): same
  values, `flush()` applies the update still in flight."""
  import torch
  use_graph = mode != 'eager'
  monkeypatch.setenv('B200RL_PIPELINE_1GPU', '1' if mode == 'pipelined' else '0')
  import helpers
  from acme_b200 import dqn, networks, replay
  from oracle import learner as olearner
  from oracle import nets as onets
  rng = np.random.default_rng(1)
  shape, A, n, B, lr = (84, 84, 4), 6, 3, 16, 1e-3
  spec, table, server, adder, oracle = helpers.make_pair(shape, np.uint8, A, n, 0.99, 0.6, max_size=300)
  for ep in range(8):
    helpers.feed_episode(rng, adder, oracle, int(rng.integers(5, 30)), n, shape, np.uint8, A)
  table.flush()
  helpers.sync_oracle_leaves(table, oracle)
  net = networks.DQNAtariNetwork(A, seed=5)
  tgt = net.clone()
  onet, otgt = onets.DQNAtariNetwork(A), onets.DQNAtariNetwork(A)
  onet.load(net.variables())
  otgt.load(net.variables())
  ds = replay.ReplayDataset(table, B, seed=7)
  client = replay.Client(server)
  learner = dqn.DQNLearner(net, tgt, 0.99, 0.2, 1e-3, target_update_period=2, dataset=ds, replay_client=client,
                           logger=__import__('acme_b200.loggers', fromlist=['x']).NoOpLogger(), use_cuda_graph=use_graph)
  ol = olearner.DQNOracleLearner(onet, otgt, 0.99, 0.2, 1e-3, 2)
  counter = torch.zeros(1, dtype=torch.int64, device='cuda')
  u_dev = torch.empty(B, device='cuda')
  from acme_b200 import _capi
  assert learner._pipeline == (mode == 'pipelined')
  steps = 5      # pipelined: two eager steps, then the 'first', 'copy' and 'norm' graphs (longer runs: the bit-identity test below)
  for step in range(steps):
    # the uniforms the learner is about to draw (device Philox keyed by (seed, call counter))
    _capi.call('b200rl_uniform', u_dev.data_ptr(), B, 7, counter.data_ptr(), step, _capi.current_stream())
    u = u_dev.cpu().numpy()
    keys, pos, prob = oracle.sample(u, True)
    o0, a, R, D, o1 = oracle.gather(pos)
    ref = ol.step(o0, a, R, D, o1, prob)
    oracle.update_priorities(keys, ref['priority'])
    learner.step()
    torch.cuda.synchronize()
    np.testing.assert_array_equal(ds.idx.cpu().numpy(), pos)
    np.testing.assert_array_equal(ds.keys.cpu().numpy().view(np.uint64), keys)
    close(learner.td.cpu().numpy(), ref['td'], atol_scale=2e-5, name=f'td step {step}')
    close(learner.priority.cpu().numpy(), ref['priority'], atol_scale=2e-5)
    close(learner.loss.cpu().numpy()[0], ref['loss'], rtol=1e-4)
    close(learner.weight.cpu().numpy(), ref['weight'])
    # Parameters: Adam's update is lr * m^/(sqrt(v^)+eps) ~ +-lr whenever |g| >> eps, so an element whose
    # gradient is ~1e-8 turns a 1e-5-relative gradient difference into a visible fraction of lr, and the two
    # trajectories then drift apart chaotically.  The Adam kernel itself is pinned to 1e-5 in
    # test_adam_and_global_norm and the gradients in test_dqn_atari_network_forward_backward; here the
    # first two updates must agree to 2% of one learning-rate step for all but <1e-3 of the parameters.
    if mode == 'pipelined' and step in (0, 1, 4):
      learner.flush()            # updates 2 and 3 stay pending across steps: applied by the next step's graph
    pending = learner._pending
    if step < 2:
      got = net.variables()
      for k, v in onet.numpy().items():
        bad = ~np.isclose(got[k], v, rtol=1e-4, atol=0.02 * lr)
        assert bad.mean() < 1e-3, f'param {k} step {step}: {bad.sum()} of {bad.size} outside 2% of lr'
        np.testing.assert_allclose(got[k], v, rtol=1e-4, atol=0.5 * lr, err_msg=f'param {k} step {step}')
    # target copy timing (learning.py:157-161): target == online right after updates 0, 2, 4 (period 2) and
    # stays frozen in between -- exact on the device.
    if not pending:
      if step % 2 == 0:
        frozen = net.params.flat.clone()
      assert torch.equal(tgt.params.flat, frozen), f'target network wrong after update {step}'
    helpers.sync_oracle_leaves_loose(table, oracle)
  assert learner.num_steps == steps
  server.stop()


@pytest.mark.parametrize('precision', [0, 2])
def test_pipelined_single_gpu_learner_is_bit_identical_to_serial(precision, monkeypatch):
  """The single-GPU pipelined update (B200RL_PIPELINE_1GPU=1: Adam of step t inside step t+1's graph, beside K1 / K3 /
  the torso forwards; K2 beside the backward) reorders launches, not arithmetic: TD errors, priorities, losses, sampled
  indices of every step and the final parameters, moments and target network equal the serial learner's bit for bit.
  Two identical tables (same inserts), period 3 so that all three graph variants ('first', 'norm', 'copy') run."""
  import torch
  import helpers
  from acme_b200 import dqn, loggers, networks, replay
  shape, A, n, B = (84, 84, 4), 6, 3, 32
  runs = []
  for pipelined in (False, True):
    monkeypatch.setenv('B200RL_PIPELINE_1GPU', '1' if pipelined else '0')
    rng = np.random.default_rng(4)
    spec, table, server, adder, oracle = helpers.make_pair(shape, np.uint8, A, n, 0.99, 0.6, max_size=300)
    for ep in range(8):
      helpers.feed_episode(rng, adder, oracle, int(rng.integers(5, 30)), n, shape, np.uint8, A)
    table.flush()
    net = networks.DQNAtariNetwork(A, seed=5, precision=precision)
    tgt = net.clone()
    ds = replay.ReplayDataset(table, B, seed=7)
    learner = dqn.DQNLearner(net, tgt, 0.99, 0.2, 1e-3, target_update_period=3, dataset=ds, replay_client=replay.Client(server),
                             logger=loggers.NoOpLogger(), use_cuda_graph=True)
    assert learner._pipeline == pipelined
    trace = []
    for step in range(13):
      learner.step(fetch_loss=False)
      torch.cuda.synchronize()
      trace.append([x.clone() for x in (ds.idx, ds.keys.view(torch.int64), learner.td, learner.priority, learner.loss, learner.weight)])
      if pipelined and step in (5, 9):
        learner.flush()             # a flush between two graph replays: the next replay is the 'first' variant again
    assert learner.num_steps == 13  # flushes the update in flight
    torch.cuda.synchronize()
    runs.append((trace, net.params.flat.clone(), tgt.params.flat.clone(), learner._m.clone(), learner._v.clone(),
                 torch.from_numpy(table.read_tree_level(table.tree_levels()[0])).clone()))
    server.stop()
  (ta, *fa), (tb, *fb) = runs
  for step, (xa, xb) in enumerate(zip(ta, tb)):
    for name, a, b in zip(('idx', 'keys', 'td', 'priority', 'loss', 'weight'), xa, xb):
      assert torch.equal(a, b), f'{name} differs at step {step}'
  for name, a, b in zip(('params', 'target params', 'adam m', 'adam v', 'tree leaves'), fa, fb):
    assert torch.equal(a, b), f'{name} differ after 13 updates'


@pytest.mark.parametrize('use_graph', [False, True])
def test_d4pg_learner_steps_match_oracle(use_graph):
  """acme/agents/tf/d4pg/learning.py:156-247 end to end (humanoid-shaped: 67-d obs, 21-d act, C51 critic)
  against oracle.learner.D4PGOracleLearner on the same uniform draws."""
  import torch
  import helpers
  from acme_b200 import _capi, d4pg, loggers, networks, replay
  from oracle import learner as olearner
  from oracle import nets as onets
  rng = np.random.default_rng(2)
  OBS, ACT, n, B = 67, 21, 5, 32
  spec, table, server, adder, oracle = helpers.make_pair((OBS,), np.float32, 0, n, 0.99, 0.0, max_size=400, act_dim=ACT)
  for ep in range(10):
    helpers.feed_episode(rng, adder, oracle, int(rng.integers(3, 40)), n, (OBS,), np.float32, 0, act_dim=ACT)
  table.flush()
  helpers.sync_oracle_leaves(table, oracle)
  policy = networks.D4PGPolicy(OBS, ACT, seed=1)
  critic = networks.D4PGCritic(OBS, ACT, seed=2)
  # make the near-zero-initialised policy head non-trivial so that the actor path is exercised
  pv = policy.variables()
  pv['out/w'] = (np.random.default_rng(3).standard_normal(pv['out/w'].shape) * 0.05).astype(np.float32)
  policy.load_variables(pv)
  tpolicy, tcritic = policy.clone(), critic.clone()
  opol, ocri = onets.D4PGPolicy(OBS, ACT), onets.D4PGCritic(OBS, ACT)
  otp, otc = onets.D4PGPolicy(OBS, ACT), onets.D4PGCritic(OBS, ACT)
  for o, n_ in ((opol, policy), (otp, policy), (ocri, critic), (otc, critic)):
    o.load(n_.variables())
  ds = replay.ReplayDataset(table, B, seed=11, stratified=False)
  learner = d4pg.D4PGLearner(policy, critic, tpolicy, tcritic, 0.99, target_update_period=2, dataset=ds,
                             logger=loggers.NoOpLogger(), use_cuda_graph=use_graph)
  ol = olearner.D4PGOracleLearner(opol, ocri, otp, otc, 0.99, 2)
  counter = torch.zeros(1, dtype=torch.int64, device='cuda')
  u_dev = torch.empty(B, device='cuda')
  lr = 1e-4
  for step in range(4):
    _capi.call('b200rl_uniform', u_dev.data_ptr(), B, 11, counter.data_ptr(), step, _capi.current_stream())
    u = u_dev.cpu().numpy()
    keys, pos, prob = oracle.sample(u, False)
    ref = ol.step(*oracle.gather(pos))
    learner.step()
    torch.cuda.synchronize()
    np.testing.assert_array_equal(ds.idx.cpu().numpy(), pos)
    close(learner.target.cpu().numpy(), ref['target'], atol_scale=2e-5, name=f'projected distribution step {step}')
    close(learner.critic_loss_ps.cpu().numpy(), ref['per_sample'], rtol=1e-4, atol_scale=2e-5, name='critic CE')
    close(learner.critic_loss.cpu().numpy()[0], ref['critic_loss'], rtol=1e-4)
    close(learner.dqda.cpu().numpy(), ref['dqda'], rtol=1e-3, atol_scale=1e-4, name='dq/da')
    close(learner.policy_loss.cpu().numpy()[0], ref['policy_loss'], rtol=1e-3)
    if ref['critic_norm'] is not None:
      close(learner.critic_norm.cpu().numpy()[0], ref['critic_norm'], rtol=1e-4)
      close(learner.policy_norm.cpu().numpy()[0], ref['policy_norm'], rtol=1e-3)
    if step < 2:
      for net, onet, what in ((critic, ocri, 'critic'), (policy, opol, 'policy')):
        got = net.variables()
        for k, v in onet.numpy().items():
          bad = ~np.isclose(got[k], v, rtol=1e-4, atol=0.02 * lr)
          assert bad.mean() < 2e-3, f'{what} {k} step {step}: {bad.sum()} of {bad.size} outside 2% of lr'
    # target copy happens BEFORE the update when num_steps % period == 0 (learning.py:171-174)
    if step % 2 == 0:
      pass   # copied at the start of this step from the pre-update online networks
    else:
      frozen_c, frozen_p = critic.params.flat.clone(), policy.params.flat.clone()
    if step in (2,):
      assert torch.equal(tcritic.params.flat, frozen_c) and torch.equal(tpolicy.params.flat, frozen_p)
  assert learner.num_steps == 4
  server.stop()


# ------------------------------------------------------------------ whole learner at the benchmarked shapes
# Stated tolerances of the tensor-core mode (precision=1), per quantity, as fractions of the tensor's scale
# (max |reference|).  They are the bounds asserted below; the errors actually measured on B200 are written to
# $B200RL_PARITY_DIR/parity_c2_<mode>.json by the test when that variable is set (kept in profiles/, quoted in
# DESIGN.md / BASELINE.md).
TC_TOL = dict(q=1e-2, td=1e-2, loss=1e-2, weight=1e-5, priority=1e-2, grad_rel_l2=5e-2)
BF16_TOL = dict(q=2e-2, td=2e-2, loss=2e-2, weight=1e-5, priority=2e-2, grad_rel_l2=1e-1)
# fp32 mode: weight gradients are sums of ~10^5 products; the two summation orders differ by a few 1e-4 of the tensor's
# norm for the most cancelling ones (conv1), 1e-6 .. 1e-5 for the rest
FP32_TOL = dict(q=2e-5, td=2e-5, loss=1e-4, weight=1e-5, priority=2e-5, grad_rel_l2=1e-3)


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


@pytest.mark.parametrize('precision,use_cuda_graph', [pytest.param(0, False, id='0'), pytest.param(1, False, id='1'),
                                                    pytest.param(2, False, id='2'), pytest.param(2, True, id='bf16-graph')])
def test_dqn_learner_c2_shape_parity(precision, use_cuda_graph):
  """BASELINE configs[1] shapes (84x84x4 uint8, A=18, B=256, n=3) through the WHOLE learner in both precisions:
  K1 indices bit-exact, then TD errors, loss, importance weights, new priorities (the quantities north_star names) and
  the parameter gradients against the oracle, for 3 updates on injected uniform draws.  Before every update the oracle
  adopts the device learner's parameters and Adam moments, so each update is compared from an identical state
  (`acme/agents/tf/dqn/learning.py:121-154`).  'bf16-graph' is the benchmarked configuration: the step captured in one
  CUDA graph (programmatic dependent launch, side streams), 4 updates of which the last two replay the graph; there the
  draws cannot be injected, so the oracle samples with the learner's own device Philox stream (dataset seed, counter)."""
  import json
  import os
  import torch
  import helpers
  from acme_b200 import _capi, dqn, loggers, networks, replay
  from oracle import learner as olearner
  from oracle import nets as onets
  tolv = {0: FP32_TOL, 1: TC_TOL, 2: BF16_TOL}[precision]
  rng = np.random.default_rng(21)
  shape, A, n, B = (84, 84, 4), 18, 3, 256
  spec, table, server, adder, oracle = helpers.make_pair(shape, np.uint8, A, n, 0.99, 0.6, max_size=1500)
  for ep in range(12):
    helpers.feed_episode(rng, adder, oracle, int(rng.integers(60, 140)), n, shape, np.uint8, A)
  table.flush()
  helpers.sync_oracle_leaves(table, oracle)
  # spread the priorities (|N(0,1)| like the bench) so that importance weights are non-trivial
  keys = np.arange(oracle.item_tail, oracle.item_head, dtype=np.uint64)
  pr = np.abs(rng.standard_normal(keys.shape[0])).astype(np.float32)
  replay.Client(server).update_priorities(table.name, keys, pr.astype(np.float64))
  oracle.update_priorities(keys, pr)
  torch.cuda.synchronize()
  helpers.sync_oracle_leaves(table, oracle)
  net = networks.DQNAtariNetwork(A, seed=5, precision=precision)
  tgt = net.clone()
  # a target network that differs from the online one (as after training), so double-Q selection matters
  tv = tgt.variables()
  tgt.load_variables({k: (v + 0.02 * np.abs(v).mean() * rng.standard_normal(v.shape)).astype(np.float32) for k, v in tv.items()})
  onet, otgt = onets.DQNAtariNetwork(A), onets.DQNAtariNetwork(A)
  ds = replay.ReplayDataset(table, B, seed=7)
  learner = dqn.DQNLearner(net, tgt, 0.99, 0.2, 1e-3, target_update_period=100, dataset=ds,
                           replay_client=replay.Client(server), logger=loggers.NoOpLogger(), use_cuda_graph=use_cuda_graph)
  ol = olearner.DQNOracleLearner(onet, otgt, 0.99, 0.2, 1e-3, 100)
  measured = []
  counter = torch.zeros(1, dtype=torch.int64, device='cuda')
  u_dev = torch.empty(B, device='cuda')
  for step in range(4 if use_cuda_graph else 3):
    onet.load(net.variables())
    otgt.load(tgt.variables())
    ol.opt.m, ol.opt.v, ol.opt.t = _export_flat(net, learner._m), _export_flat(net, learner._v), step
    ol.num_steps = step
    if use_cuda_graph:   # the uniforms the learner is about to draw (device Philox keyed by (seed, call counter))
      _capi.call('b200rl_uniform', u_dev.data_ptr(), B, 7, counter.data_ptr(), step, _capi.current_stream())
      u = u_dev.cpu().numpy()
    else:
      u = rng.random(B, dtype=np.float32)
    keys, pos, prob = oracle.sample(u, True)
    ref = ol.step(*oracle.gather(pos), prob)
    learner.step(uniforms=None if use_cuda_graph else torch.as_tensor(u).cuda())
    torch.cuda.synchronize()
    np.testing.assert_array_equal(ds.idx.cpu().numpy(), pos)                       # sampled indices: bit-exact
    np.testing.assert_array_equal(ds.keys.cpu().numpy().view(np.uint64), keys)
    np.testing.assert_array_equal(ds.prob.cpu().numpy(), prob)
    np.testing.assert_array_equal(ds.R.cpu().numpy().view(np.uint32), oracle.gather(pos)[2].view(np.uint32))   # n-step R, D
    np.testing.assert_array_equal(ds.D.cpu().numpy().view(np.uint32), oracle.gather(pos)[3].view(np.uint32))
    got_grads = _export_flat(net, net.params.grad)
    err = dict(step=step,
               q_tm1=_scale_err(learner.q_values()[0].cpu().numpy(), ref['q_tm1']),
               td=_scale_err(learner.td.cpu().numpy(), ref['td']),
               loss=abs(float(learner.loss.cpu()[0]) - float(ref['loss'])) / abs(float(ref['loss'])),
               weight=_scale_err(learner.weight.cpu().numpy(), ref['weight']),
               priority=_scale_err(learner.priority.cpu().numpy(), ref['priority']),
               grad_rel_l2={k: float(np.linalg.norm(got_grads[k].astype(np.float64) - g) / max(np.linalg.norm(g), 1e-30))
                            for k, g in ref['grads'].items()})
    measured.append(err)
    assert err['q_tm1'] <= tolv['q'], err
    assert err['td'] <= tolv['td'], err
    assert err['loss'] <= tolv['loss'], err
    assert err['weight'] <= tolv['weight'], err
    assert err['priority'] <= tolv['priority'], err
    assert max(err['grad_rel_l2'].values()) <= tolv['grad_rel_l2'], err
    oracle.update_priorities(keys, ref['priority'])
    helpers.sync_oracle_leaves_loose(table, oracle, rtol=1e-1 if precision else 5e-3, atol=0.1 if precision else 1e-4)
  out = os.environ.get('B200RL_PARITY_DIR')
  if out:
    os.makedirs(out, exist_ok=True)
    mode = {0: 'fp32', 1: 'tf32', 2: 'bf16'}[precision] + ('_graph' if use_cuda_graph else '')
    with open(os.path.join(out, f'parity_c2_{mode}.json'), 'w') as f:
      json.dump(dict(mode=mode, B=B, A=A, tolerances=tolv, measured=measured), f, indent=1)
  server.stop()


def test_dqn_learner_jax_variants():
  """SURVEY App. A.6 switches against the oracle: post-increment target copy (jax/dqn/learning.py:114-119) and f32
  importance weights (jax/dqn/learning.py:94-96)."""
  import torch
  import helpers
  from acme_b200 import dqn, loggers, networks, replay
  from oracle import learner as olearner
  from oracle import nets as onets
  rng = np.random.default_rng(4)
  shape, A, n, B = (84, 84, 4), 5, 3, 16
  spec, table, server, adder, oracle = helpers.make_pair(shape, np.uint8, A, n, 0.99, 0.6, max_size=200)
  for ep in range(6):
    helpers.feed_episode(rng, adder, oracle, int(rng.integers(5, 30)), n, shape, np.uint8, A)
  table.flush()
  helpers.sync_oracle_leaves(table, oracle)
  net = networks.DQNAtariNetwork(A, seed=9)
  tgt = net.clone()
  onet, otgt = onets.DQNAtariNetwork(A), onets.DQNAtariNetwork(A)
  onet.load(net.variables())
  otgt.load(net.variables())
  ds = replay.ReplayDataset(table, B, seed=7)
  learner = dqn.DQNLearner(net, tgt, 0.99, 0.2, 1e-3, target_update_period=3, dataset=ds, replay_client=replay.Client(server),
                           logger=loggers.NoOpLogger(), use_cuda_graph=False, target_update_mode='post_increment',
                           is_weights_dtype='f32')
  ol = olearner.DQNOracleLearner(onet, otgt, 0.99, 0.2, 1e-3, 3, target_update_mode='post_increment', is_weights_dtype='f32')
  frozen = tgt.params.flat.clone()
  for step in range(6):
    u = rng.random(B, dtype=np.float32)
    keys, pos, prob = oracle.sample(u, True)
    ref = ol.step(*oracle.gather(pos), prob)
    oracle.update_priorities(keys, ref['priority'])
    learner.step(uniforms=torch.as_tensor(u).cuda())
    torch.cuda.synchronize()
    np.testing.assert_array_equal(ds.idx.cpu().numpy(), pos)
    close(learner.weight.cpu().numpy(), ref['weight'], name='f32 importance weights')
    close(learner.td.cpu().numpy(), ref['td'], atol_scale=5e-5, name=f'td step {step}')
    # copies after updates 2 and 5 (0-based): (steps + 1) % 3 == 0, with the NEW parameters
    if (step + 1) % 3 == 0:
      frozen = net.params.flat.clone()
    assert torch.equal(tgt.params.flat, frozen), f'target network wrong after update {step}'
    helpers.sync_oracle_leaves_loose(table, oracle)
  server.stop()


@pytest.mark.parametrize('use_graph', [False, True])
def test_ddpg_learner_steps_match_oracle(use_graph):
  """SURVEY §8f-2: `acme/agents/tf/ddpg/learning.py:140-237` (scalar critic, trfl.td_learning at 193, DPG with dq/da norm
  clipping, global-norm clip, two Adams, target copy before the update) against oracle.learner.DDPGOracleLearner."""
  import torch
  import helpers
  from acme_b200 import _capi, d4pg, loggers, networks, replay
  from oracle import learner as olearner
  from oracle import nets as onets
  rng = np.random.default_rng(6)
  OBS, ACT, n, B = 17, 6, 5, 32
  spec, table, server, adder, oracle = helpers.make_pair((OBS,), np.float32, 0, n, 0.99, 0.0, max_size=400, act_dim=ACT)
  for ep in range(10):
    helpers.feed_episode(rng, adder, oracle, int(rng.integers(3, 40)), n, (OBS,), np.float32, 0, act_dim=ACT)
  table.flush()
  helpers.sync_oracle_leaves(table, oracle)
  sizes = (64, 64)
  policy = networks.D4PGPolicy(OBS, ACT, sizes=sizes, seed=1)
  critic = networks.DDPGCritic(OBS, ACT, sizes=sizes, seed=2)
  pv = policy.variables()
  pv['out/w'] = (np.random.default_rng(3).standard_normal(pv['out/w'].shape) * 0.05).astype(np.float32)
  policy.load_variables(pv)
  opol, ocri = onets.D4PGPolicy(OBS, ACT, sizes), onets.DDPGCritic(OBS, ACT, sizes)
  otp, otc = onets.D4PGPolicy(OBS, ACT, sizes), onets.DDPGCritic(OBS, ACT, sizes)
  for o, n_ in ((opol, policy), (otp, policy), (ocri, critic), (otc, critic)):
    o.load(n_.variables())
  ds = replay.ReplayDataset(table, B, seed=11, stratified=False)
  learner = d4pg.DDPGLearner(policy, critic, policy.clone(), critic.clone(), 0.99, target_update_period=2, dataset=ds,
                             logger=loggers.NoOpLogger(), use_cuda_graph=use_graph)
  ol = olearner.DDPGOracleLearner(opol, ocri, otp, otc, 0.99, 2)
  counter = torch.zeros(1, dtype=torch.int64, device='cuda')
  u_dev = torch.empty(B, device='cuda')
  lr = 1e-4
  for step in range(4):
    _capi.call('b200rl_uniform', u_dev.data_ptr(), B, 11, counter.data_ptr(), step, _capi.current_stream())
    keys, pos, prob = oracle.sample(u_dev.cpu().numpy(), False)
    ref = ol.step(*oracle.gather(pos))
    learner.step()
    torch.cuda.synchronize()
    np.testing.assert_array_equal(ds.idx.cpu().numpy(), pos)
    close(learner.td.cpu().numpy(), ref['td'], atol_scale=2e-5, name=f'td step {step}')
    close(learner.critic_loss_ps.cpu().numpy(), ref['per_sample'], rtol=1e-4, atol_scale=2e-5, name='0.5 td^2')
    close(learner.critic_loss.cpu().numpy()[0], ref['critic_loss'], rtol=1e-4)
    close(learner.dqda.cpu().numpy(), ref['dqda'], rtol=1e-3, atol_scale=1e-4, name='dq/da')
    close(learner.policy_loss.cpu().numpy()[0], ref['policy_loss'], rtol=1e-3)
    if step < 2:
      for net, onet, what in ((critic, ocri, 'critic'), (policy, opol, 'policy')):
        got = net.variables()
        for k, v in onet.numpy().items():
          bad = ~np.isclose(got[k], v, rtol=1e-4, atol=0.02 * lr)
          assert bad.mean() < 2e-3, f'{what} {k} step {step}: {bad.sum()} of {bad.size} outside 2% of lr'
  assert learner.num_steps == 4
  server.stop()
