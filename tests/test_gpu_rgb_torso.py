"""Convolutional torsos on frames of any channel count C in [1, 16] (RGB: 3; a stack of F RGB frames: 3 F).

conv1 reads uint8 pixels 4 channels at a time, so frames with C % 4 != 0 are copied into pixels of Cp = C rounded up to 4
channels by `b200rl_frames_pad_u8`, and conv1's filter is stored with Cp input channels whose padding columns are zero.
Checked here:
  * the padding kernel against NumPy, and its refusals;
  * the torso's forward features and all weight gradients against an fp64 autograd reference over the C real channels,
    at every precision;
  * the bf16 row-image layer calls (precisions 2 and 3: channel group Cp = 4, 8 or 16) against fp64, and their refusals;
  * K3's row gather (plain ring and frame-deduplicated ring) equals b200rl_conv2d_rows_bf16_from_u8 byte for byte;
  * the padding stays dead: after 20 learner updates the padded filter columns, their gradient, Adam moments, bf16
    shadow and target copy are exactly zero, and `variables()` exports [8, 8, C, 32];
  * D4PG / DDPG at B = 256 on 84 x 84 x 3 and 84 x 84 x 12 uint8 observations against tests/pixel_oracle.py for three
    updates, at the bounds of tests/test_gpu_visual_d4pg.py (TOL); measured errors go to
    $B200RL_PARITY_DIR/parity_rgb_<learner>_c<C>_<mode>.json when that variable is set;
  * DQN at 84 x 84 x 3 against oracle/learner.py at precision 2;
  * flattened frame stacks [H, W, 3 F] in a frame-deduplicated table give the same updates as the full-stack table;
  * the D4PG agent on RGB observations under the batched loop (num_envs = 16, frame_stack = 4) and at num_envs = 1."""
import json
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

HW, ACT, B = 84, 6, 256
TOL = {0: dict(value=2e-5, loss=1e-4, grad_rel_l2=1e-3), 3: dict(value=2e-5, loss=1e-4, grad_rel_l2=1e-3),
       1: dict(value=1e-2, loss=1e-2, grad_rel_l2=5e-2), 2: dict(value=2e-2, loss=2e-2, grad_rel_l2=1e-1)}
MODE = {0: 'fp32', 1: 'tf32', 2: 'bf16', 3: 'fp32x3'}


@pytest.fixture(autouse=True)
def _release():
  yield
  import gc
  import torch
  torch.cuda.synchronize()
  gc.collect()


def _t(x):
  import torch
  return torch.as_tensor(np.ascontiguousarray(x)).cuda()


def _rows_ok(C):
  return -(-C // 4) * 4 == 4


def _cp(C):
  return 4 if C <= 4 else 8 if C <= 8 else 16


# ------------------------------------------------------------------------------ the padding kernel
@pytest.mark.parametrize('C', [1, 2, 3, 5, 9, 12, 16])
def test_frames_pad_kernel(C):
  import torch
  from acme_b200 import _capi
  Cp = -(-C // 4) * 4
  for cp in sorted({Cp, 16}):
    x = np.random.default_rng(C).integers(0, 256, (3, 17, 13, C), dtype=np.uint8)
    out = torch.full((3, 17, 13, cp), 7, dtype=torch.uint8, device='cuda')
    _capi.call('b200rl_frames_pad_u8', _t(x).data_ptr(), 3 * 17 * 13, C, cp, out.data_ptr(), _capi.current_stream())
    want = np.zeros((3, 17, 13, cp), np.uint8)
    want[..., :C] = x
    np.testing.assert_array_equal(out.cpu().numpy(), want)


def test_frames_pad_kernel_rejects_bad_arguments():
  import torch
  from acme_b200 import _capi
  x = torch.zeros(1 << 12, dtype=torch.uint8, device='cuda')
  out = torch.zeros(1 << 14, dtype=torch.uint8, device='cuda')
  st = _capi.current_stream()
  for C, Cp in ((0, 4), (17, 20), (3, 6), (5, 4), (16, 32)):
    with pytest.raises(ValueError):
      _capi.call('b200rl_frames_pad_u8', x.data_ptr(), 16, C, Cp, out.data_ptr(), st)
  with pytest.raises(ValueError, match='aligned'):
    _capi.call('b200rl_frames_pad_u8', x.data_ptr(), 16, 3, 4, out.data_ptr() + 1, st)
  with pytest.raises(ValueError):
    _capi.call('b200rl_frames_pad_u8', None, 16, 3, 4, out.data_ptr(), st)


# ------------------------------------------------------------------------------ the torso against fp64
def _ref_torso(variables, frames, dz3):
  """fp64 autograd through the reference AtariTorso (TF SAME padding) on the C-channel frames; dz3: the gradient w.r.t.
  conv3's pre-activation (masked by the device's own ReLU, so that both sides back-propagate the same gradient)."""
  import torch
  from oracle import nets as onets
  x = torch.tensor(frames.astype(np.float64) / 255.0)
  v = {k: torch.tensor(w.astype(np.float64), requires_grad=True) for k, w in variables.items()}
  h = x
  for i, s in ((1, 4), (2, 2), (3, 1)):
    z = onets._conv_same(h, v[f'conv{i}/w'], v[f'conv{i}/b'], s)
    h = torch.relu(z)
  z.backward(torch.tensor(dz3.astype(np.float64)))
  return h.detach().numpy(), {k: t.grad.numpy() for k, t in v.items()}


@pytest.mark.parametrize('precision', [0, 1, 2, 3])
@pytest.mark.parametrize('C', [1, 3, 4, 9, 12, 16])
def test_torso_matches_fp64(C, precision):
  """Forward features and every weight gradient of AtariTorso(input_channels=C), conv1 on the frames (x_u8 = 1) and,
  where the precision builds one, on the row image of the padded frames (x_u8 = 2)."""
  import torch
  from acme_b200 import networks
  Bt = 32
  rng = np.random.default_rng(C)
  net = networks.AtariTorso(precision=precision, seed=3, input_channels=C)
  v = net.variables()
  assert v['conv1/w'].shape == (8, 8, C, 32)
  v['conv1/b'] = (rng.standard_normal(32) * 0.05).astype(np.float32)
  net.load_variables(v)
  frames = rng.integers(0, 256, (Bt, HW, HW, C), dtype=np.uint8)
  bufs, gbufs = net.make_buffers(Bt), net.make_grad_buffers(Bt)
  obs = _t(frames)
  y = net.forward(obs, bufs).float().cpu().numpy()
  mask = (y > 0)
  dy3 = rng.standard_normal(y.shape).astype(np.float32)
  gbufs['dy3'].copy_(_t(dy3 * mask))
  net.backward(obs, bufs, gbufs)
  torch.cuda.synchronize()
  ref_y, ref_g = _ref_torso(v, frames, dy3 * mask)
  tol = TOL[precision]
  assert np.abs(y - ref_y).max() <= tol['value'] * np.abs(ref_y).max()
  g = net.variables(grad=True)
  # Bounds of the paths the dispatcher takes: without a row image (C > 4) precision 1 runs conv1 on the loader-fed bf16
  # kernel (gemm_tc.cu), held to the bf16 bound; precision 3's torso gradients at the precision-1 bound, as in
  # test_gpu_visual_d4pg (cancelling batch sums amplify its per-element error, DESIGN.md "D4PG and DDPG from pixels")
  gtol = {0: TOL[0], 1: TOL[1] if _rows_ok(C) else TOL[2], 2: TOL[2], 3: TOL[1]}[precision]['grad_rel_l2']
  for k, want in ref_g.items():
    if not k.endswith('/w'):
      continue
    rel = np.linalg.norm(g[k].astype(np.float64) - want) / np.linalg.norm(want)
    assert rel <= gtol, (k, rel)
  Cp = net.in_cp
  if Cp != C:
    assert not net.params.view('conv1.w', grad=True)[..., C:].any(), 'padding columns got a gradient'
  # the same through an explicit prepare_frames() operand (row image or padded frames), built once for both passes
  rows = net.prepare_frames(obs, 'x')
  if rows is not None:
    y2 = net.forward(obs, bufs, rows=rows).float().cpu().numpy()
    np.testing.assert_array_equal(y2, y)


# ------------------------------------------------------------------------------ bf16 row-image layer calls
@pytest.mark.parametrize('C', [1, 3, 4, 9, 12, 16])
def test_bf16_row_conv1_matches_fp64(C):
  """b200rl_conv2d_rows_bf16_from_u8 + b200rl_conv2d_{fwd,wgrad}_bf16(x_rows=1) on C-channel frames, filter
  [32][8][8][Cp] with zero padding columns: y and dW against fp64 over the C real channels (bf16 bound), dW's padding
  columns exactly zero."""
  import torch
  from acme_b200 import _capi, networks
  from oracle import nets as onets
  Bt = 16
  rng = np.random.default_rng(100 + C)
  g = networks.AtariTorso(precision=2, input_channels=C).geom(0, Bt)
  assert g.C == C
  cp = _cp(C)
  frames = rng.integers(0, 256, (Bt, HW, HW, C), dtype=np.uint8)
  w = (rng.standard_normal((32, 8, 8, C)) / np.sqrt(64 * C)).astype(np.float32)
  wp = np.zeros((32, 8, 8, cp), np.float32)
  wp[..., :C] = w
  lib, st = _capi.load(), _capi.current_stream()
  import ctypes
  nbytes = int(lib.b200rl_conv2d_rows_bf16_bytes(ctypes.byref(g)))
  assert nbytes > 0
  rows = torch.zeros(nbytes + 128, dtype=torch.uint8, device='cuda')
  _capi.call('b200rl_conv2d_rows_bf16_from_u8', _t(frames).data_ptr(), g, rows.data_ptr(), nbytes, st)
  wb = torch.as_tensor(wp).cuda().to(torch.bfloat16)
  bias = torch.zeros(32, device='cuda')
  y = torch.empty((Bt, g.OH, g.OW, 32), device='cuda')
  ws = torch.empty(96 << 20, dtype=torch.uint8, device='cuda')
  _capi.call('b200rl_conv2d_fwd_bf16', rows.data_ptr(), 1, wb.data_ptr(), bias.data_ptr(), y.data_ptr(), 0, g, 0, ws.data_ptr(),
             ws.numel(), st)
  dy = rng.standard_normal((Bt, g.OH, g.OW, 32)).astype(np.float32)
  dyb = torch.as_tensor(dy).cuda().to(torch.bfloat16)
  dw = torch.full((32, 8, 8, cp), float('nan'), device='cuda')
  _capi.call('b200rl_conv2d_wgrad_bf16', rows.data_ptr(), 1, dyb.data_ptr(), dw.data_ptr(), None, g, ws.data_ptr(), ws.numel(), st)
  torch.cuda.synchronize()
  x = torch.tensor(frames.astype(np.float64) / 255.0)
  wt = torch.tensor(w.transpose(1, 2, 3, 0).astype(np.float64).copy(), requires_grad=True)
  wt_b = torch.tensor(wp.astype(np.float32)).to(torch.bfloat16).double()[..., :C].permute(1, 2, 3, 0).contiguous()
  ref = onets._conv_same(x, wt_b, torch.zeros(32, dtype=torch.float64), 4)
  err = float((y.cpu().double() - ref).abs().max() / ref.abs().max())
  assert err <= TOL[2]['value'], err
  out = onets._conv_same(x, wt, torch.zeros(32, dtype=torch.float64), 4)
  out.backward(torch.tensor(dyb.float().cpu().numpy().astype(np.float64)))
  want = wt.grad.numpy().transpose(3, 0, 1, 2)
  got = dw.cpu().numpy()
  assert not got[..., C:].any(), 'padding columns got a gradient'
  rel = np.linalg.norm(got[..., :C] - want) / np.linalg.norm(want)
  assert rel <= TOL[2]['grad_rel_l2'], rel
  # refusals: channel counts outside [1, 16], a too-small or misaligned image
  for bad in (0, 17):
    gb = networks.AtariTorso(precision=2, input_channels=C).geom(0, Bt)
    gb.C = bad
    assert int(lib.b200rl_conv2d_rows_bf16_bytes(ctypes.byref(gb))) == 0
    with pytest.raises(ValueError):
      _capi.call('b200rl_conv2d_rows_bf16_from_u8', _t(frames).data_ptr(), gb, rows.data_ptr(), nbytes, st)
    with pytest.raises(ValueError):
      _capi.call('b200rl_conv2d_fwd_bf16', rows.data_ptr(), 1, wb.data_ptr(), bias.data_ptr(), y.data_ptr(), 0, gb, 0,
                 ws.data_ptr(), ws.numel(), st)
  with pytest.raises(ValueError):
    _capi.call('b200rl_conv2d_rows_bf16_from_u8', _t(frames).data_ptr(), g, rows.data_ptr(), nbytes - 16, st)
  with pytest.raises(ValueError):
    _capi.call('b200rl_conv2d_rows_bf16_from_u8', _t(frames).data_ptr(), g, rows.data_ptr() + 16, nbytes, st)


@pytest.mark.parametrize('shape,frame_stack', [((HW, HW, 3), 0), ((HW, HW, 12), 0), ((HW, HW, 3, 4), 4), ((HW, HW, 12), 4),
                                               ((HW, HW, 1, 4), 4)])
def test_gather_rows_equals_rows_from_u8(shape, frame_stack):
  """K3's row gather writes the row image of the gathered frames byte for byte as b200rl_conv2d_rows_bf16_from_u8 does
  (padding channels and borders included), on the plain and the frame-deduplicated ring."""
  import ctypes
  import torch
  from acme_b200 import _capi, networks, replay
  C = int(np.prod(shape[2:]))
  table, server, _ = _replay(31, C, episodes=6, frame_stack=frame_stack, stack_shape=shape if len(shape) == 4 or frame_stack else None)
  Bt = 64
  net = networks.AtariTorso(precision=2, input_channels=C)
  ds = replay.ReplayDataset(table, Bt, seed=3, stratified=False)
  fb = net.rows_frame_bytes()
  buf = torch.zeros(2 * Bt * fb, dtype=torch.uint8, device='cuda')    # zeroed as rows_buffer() is (Atari frames: interior only)
  ds.sample_only(torch.as_tensor(np.random.default_rng(1).random(Bt, dtype=np.float32)).cuda())
  ds.gather_only((buf.data_ptr(), buf.data_ptr() + Bt * fb, net.geom(0, 1)))
  want = torch.full_like(buf, 0x5C)
  g = net.geom(0, Bt)
  st = _capi.current_stream()
  for half, o in ((0, ds.o_tm1), (1, ds.o_t)):
    _capi.call('b200rl_conv2d_rows_bf16_from_u8', o.data_ptr(), g, want.data_ptr() + half * Bt * fb, Bt * fb, st)
  torch.cuda.synchronize()
  assert torch.equal(buf, want)
  server.stop()


def test_torso_rejects_bad_channel_counts():
  from acme_b200 import networks
  for c in (0, 17, 2.5, -3):
    with pytest.raises(ValueError, match='input_channels'):
      networks.AtariTorso(precision=1, input_channels=c)
    with pytest.raises(ValueError, match='input_channels'):
      networks.DQNAtariNetwork(4, input_channels=c)
  net = networks.AtariTorso(precision=1, input_channels=3)
  with pytest.raises(ValueError, match='uint8'):
    net.forward(_t(np.zeros((4, HW, HW, 3), np.float32)), net.make_buffers(4))
  with pytest.raises(ValueError, match='input channels'):
    net.load_variables({k: (np.zeros((8, 8, 4, 32), np.float32) if k == 'conv1/w' else w) for k, w in net.variables().items()})


# ------------------------------------------------------------------------------ learners
def _replay(seed, C, episodes=12, frame_stack=0, stack_shape=None):
  """stack_shape: episodes of FrameStacker stacks of F = 4 frames ((HW, HW, c, F) or flattened (HW, HW, c F))."""
  import helpers
  from acme_b200 import dm_env
  rng = np.random.default_rng(seed)
  shape = stack_shape or (HW, HW, C)
  spec, table, server, adder, oracle = helpers.make_pair(shape, np.uint8, 0, 5, 0.99, 0.0, max_size=1000, act_dim=ACT,
                                                         frame_stack=frame_stack)
  for _ in range(episodes):
    T = int(rng.integers(20, 50))
    if stack_shape is None:
      helpers.feed_episode(rng, adder, oracle, T, 5, shape, np.uint8, 0, act_dim=ACT)
      continue
    F = 4
    fc = int(np.prod(stack_shape[2:])) // F
    frames = [np.zeros((HW, HW, fc), np.uint8)] * (F - 1)
    def obs():
      frames.append(rng.integers(0, 256, (HW, HW, fc), dtype=np.uint8))
      return np.stack(frames[-F:], axis=-1).reshape(stack_shape)
    adder.add_first(dm_env.restart(obs()))
    for k in range(1, T + 1):
      step = dm_env.StepType.LAST if k == T else dm_env.StepType.MID
      adder.add(rng.uniform(-1, 1, ACT).astype(np.float32),
                dm_env.TimeStep(step, np.float32(rng.choice([-1., 0., 1.])), np.float32(k < T), obs()))
  table.flush()
  return table, server, oracle


def _nets(kind, precision, C, seed=0):
  from acme_b200 import networks
  torso = networks.AtariTorso(precision=precision, seed=seed, input_channels=C)
  policy = networks.D4PGPolicy(torso.flat_dim, ACT, seed=1 + seed, precision=precision)
  critic = (networks.D4PGCritic if kind == 'd4pg' else networks.DDPGCritic)(torso.flat_dim, ACT, seed=2 + seed,
                                                                          precision=precision)
  pv = policy.variables()
  pv['out/w'] = (np.random.default_rng(3 + seed).standard_normal(pv['out/w'].shape) * 0.05).astype(np.float32)
  policy.load_variables(pv)
  return torso, policy, critic


def _learner(kind, torso, policy, critic, ds, use_graph, **kw):
  from acme_b200 import d4pg, loggers
  cls = d4pg.D4PGLearner if kind == 'd4pg' else d4pg.DDPGLearner
  return cls(policy, critic, policy.clone(), critic.clone(), 0.99, target_update_period=2, dataset=ds,
             logger=loggers.NoOpLogger(), use_cuda_graph=use_graph, observation_network=torso,
             target_observation_network=torso.clone(), **kw)


def _export(net, flat):
  saved = net.params.flat
  net.params.flat = flat
  try:
    return net.variables()
  finally:
    net.params.flat = saved


def _scale_err(got, want):
  got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
  return float(np.abs(got - want).max() / max(np.abs(want).max(), 1e-30))


@pytest.mark.parametrize('precision', [0, 1, 2, 3])
@pytest.mark.parametrize('C', [3, 12])
@pytest.mark.parametrize('kind', ['d4pg', 'ddpg'])
def test_rgb_learner_parity(kind, C, precision):
  """As test_gpu_visual_d4pg.test_pixel_learner_parity, on C-channel frames."""
  import torch
  import pixel_oracle
  from oracle import nets as onets
  from acme_b200 import replay
  tol = TOL[precision]
  table, server, oracle = _replay(21, C)
  torso, policy, critic = _nets(kind, precision, C)
  ds = replay.ReplayDataset(table, B, seed=11, stratified=False)
  learner = _learner(kind, torso, policy, critic, ds, use_graph=False)
  tpolicy, tcritic, ttorso = learner._tpolicy, learner._tcritic, learner._tobs_net
  F = torso.flat_dim
  ocls = onets.D4PGCritic if kind == 'd4pg' else onets.DDPGCritic
  opol, ocri, otp, otc = onets.D4PGPolicy(F, ACT), ocls(F, ACT), onets.D4PGPolicy(F, ACT), ocls(F, ACT)
  oto, otto = pixel_oracle.AtariTorso(in_c=C), pixel_oracle.AtariTorso(in_c=C)
  ol = (pixel_oracle.D4PGOracleLearner if kind == 'd4pg' else pixel_oracle.DDPGOracleLearner)(
      opol, ocri, otp, otc, 0.99, 2, obs_net=oto, target_obs_net=otto)
  nt = torso.params.size
  rng = np.random.default_rng(5)
  measured = []
  for step in range(3):
    for o, net in ((opol, policy), (ocri, critic), (otp, tpolicy), (otc, tcritic), (oto, torso), (otto, ttorso)):
      o.load(net.variables())
    ol.popt.m, ol.popt.v, ol.popt.t = _export(policy, learner._pm), _export(policy, learner._pv), step
    mom = []
    for buf in (learner._cm, learner._cv):
      d = _export(critic, buf[nt:])
      d.update({'obs/' + k: v for k, v in _export(torso, buf[:nt]).items()})
      mom.append(d)
    ol.copt.m, ol.copt.v, ol.copt.t = mom[0], mom[1], step
    ol.num_steps = step
    u = rng.random(B, dtype=np.float32)
    keys, pos, prob = oracle.sample(u, False)
    ref = ol.step(*oracle.gather(pos))
    learner.step(uniforms=torch.as_tensor(u).cuda())
    torch.cuda.synchronize()
    np.testing.assert_array_equal(ds.idx.cpu().numpy(), pos)
    cscale, pscale = float(learner._cscale.cpu()[0]), float(learner._pscale.cpu()[0])
    cg, pg, og = (_export(critic, critic.params.grad), _export(policy, policy.params.grad),
                  _export(torso, torso.params.grad))
    rel = lambda got, want: float(np.linalg.norm(got.astype(np.float64) - want) / max(np.linalg.norm(want), 1e-30))
    err = dict(step=step,
               critic_loss_per_sample=_scale_err(learner.critic_loss_ps.cpu().numpy(), ref['per_sample']),
               critic_loss=_scale_err(learner.critic_loss.cpu().numpy()[0], ref['critic_loss']),
               dqda=_scale_err(learner.dqda.cpu().numpy(), ref['dqda']),
               policy_loss=_scale_err(learner.policy_loss.cpu().numpy()[0], ref['policy_loss']),
               critic_norm=_scale_err(learner.critic_norm.cpu().numpy()[0], ref['critic_norm']),
               policy_norm=_scale_err(learner.policy_norm.cpu().numpy()[0], ref['policy_norm']),
               critic_grad_rel_l2={k: rel(cg[k] * cscale, g) for k, g in ref['critic_grads'].items()},
               torso_grad_rel_l2={k: rel(og[k[4:]] * cscale, g) for k, g in ref['obs_grads'].items()},
               policy_grad_rel_l2={k: rel(pg[k] * pscale, g) for k, g in ref['policy_grads'].items()})
    if kind == 'd4pg':
      err['target'] = _scale_err(learner.target.cpu().numpy(), ref['target'])
    else:
      err['td'] = _scale_err(learner.td.cpu().numpy(), ref['td'])
    measured.append(err)
  out = os.environ.get('B200RL_PARITY_DIR')
  if out:
    os.makedirs(out, exist_ok=True)
    with open(os.path.join(out, f'parity_rgb_{kind}_c{C}_{MODE[precision]}.json'), 'w') as f:
      json.dump(dict(learner=kind, mode=MODE[precision], B=B, obs=[HW, HW, C], act=ACT, n=5, tolerances=tol,
                     measured=measured), f, indent=1)
  for err in measured:
    for k, v in err.items():
      if k == 'step':
        continue
      # precision 3: the torso gradients and the critic norm at the precision-1 bound (DESIGN.md "D4PG and DDPG from
      # pixels"), as in test_gpu_visual_d4pg
      t = TOL[1] if precision == 3 and k in ('torso_grad_rel_l2', 'critic_norm') else tol
      if isinstance(v, dict):
        assert len(v) and max(v.values()) <= t['grad_rel_l2'], (k, err['step'], v)
      else:
        assert v <= t['loss' if 'loss' in k else 'value'], (k, err['step'], v)
  server.stop()


@pytest.mark.parametrize('precision', [0, 1, 2, 3])
def test_padding_stays_dead(precision):
  """20 updates on 3-channel frames: the padded filter column of conv1 is exactly zero in the parameters, gradient, Adam
  moments, bf16 shadow and target torso; variables() has Sonnet's [8, 8, 3, 32]; save -> restore resumes bit-identically."""
  import torch
  from acme_b200 import replay
  C = 3
  table, server, _ = _replay(22, C, episodes=8)
  torso, policy, critic = _nets('d4pg', precision, C)
  learner = _learner('d4pg', torso, policy, critic, replay.ReplayDataset(table, B, seed=11, stratified=False), True)
  for _ in range(20):
    learner.step(fetch_loss=False)
  torch.cuda.synchronize()
  off, shape = torso.params.entries['conv1.w']
  n = int(np.prod(shape))
  pad = lambda flat: flat[off:off + n].view(shape)[..., C:]
  tt = learner._tobs_net
  for what, t in (('param', torso.params.flat), ('grad', torso.params.grad), ('adam m', learner._cm),
                  ('adam v', learner._cv), ('target', tt.params.flat)):
    assert not pad(t).any(), what
  if torso.params.shadow is not None:
    assert not pad(torso.params.shadow).float().any(), 'shadow'
  assert torso.params.view('conv1.w')[..., :C].abs().sum() > 0
  got = learner.get_variables(['policy'])[0]
  assert got[0].shape == (8, 8, C, 32) and torso.variables()['conv1/w'].shape == (8, 8, C, 32)
  state = learner.save()
  torso2, policy2, critic2 = _nets('d4pg', precision, C, seed=10)
  other = _learner('d4pg', torso2, policy2, critic2, replay.ReplayDataset(table, B, seed=11, stratified=False), False)
  other.restore(state)
  rng = np.random.default_rng(9)
  for _ in range(2):
    u = torch.as_tensor(rng.random(B, dtype=np.float32)).cuda()
    learner.step(uniforms=u, fetch_loss=False)
    other.step(uniforms=u, fetch_loss=False)
  torch.cuda.synchronize()
  assert torch.equal(learner.critic_loss, other.critic_loss)
  for a, b in ((learner._cparams.flat, other._cparams.flat), (learner._cm, other._cm), (learner._cv, other._cv),
               (learner._policy.params.flat, other._policy.params.flat)):
    assert torch.equal(a, b)
  server.stop()


def test_flattened_stack_dedup_matches_full_stack():
  """[H, W, 12] flattened RGB stacks in a frame_stack=4 table give the updates of [H, W, 3, 4] stacks in a full-stack
  table, bit for bit (same bytes, so the same K3 rebuild, blank frames included)."""
  import torch
  from acme_b200 import replay
  rng = np.random.default_rng(3)
  us = [torch.as_tensor(rng.random(B, dtype=np.float32)).cuda() for _ in range(3)]
  results, batches = [], []
  for fs, shape in ((0, (HW, HW, 3, 4)), (4, (HW, HW, 12)), (4, (HW, HW, 3, 4))):
    table, server, _ = _replay(25, 12, frame_stack=fs, stack_shape=shape)
    torso, policy, critic = _nets('d4pg', 1, 12)
    ds = replay.ReplayDataset(table, B, seed=11, stratified=False)
    learner = _learner('d4pg', torso, policy, critic, ds, False)
    for u in us:
      learner.step(uniforms=u, fetch_loss=False)
    torch.cuda.synchronize()
    batches.append((ds.o_tm1.cpu().clone(), ds.o_t.cpu().clone()))
    results.append([learner._cparams.flat.clone(), learner._policy.params.flat.clone(), learner._cm.clone()])
    server.stop()
  for r, bt in zip(results[1:], batches[1:]):
    assert all(torch.equal(x.view(-1), y.view(-1)) for x, y in zip(bt, batches[0]))
    assert all(torch.equal(x, y) for x, y in zip(r, results[0]))


def test_dqn_rgb_matches_oracle_bf16():
  """DQN on 84 x 84 x 3 frames at precision 2 (K3 writes the 4-channel row image) against oracle/learner.py."""
  import torch
  import helpers
  from acme_b200 import _capi, dqn, loggers, networks, replay
  from oracle import learner as olearner
  from oracle import nets as onets
  rng = np.random.default_rng(0)
  shape, A, n, Bd = (HW, HW, 3), 4, 3, 64
  spec, table, server, adder, oracle = helpers.make_pair(shape, np.uint8, A, n, 0.99, 0.6, max_size=300)
  for _ in range(6):
    helpers.feed_episode(rng, adder, oracle, int(rng.integers(5, 25)), n, shape, np.uint8, A)
  table.flush()
  helpers.sync_oracle_leaves(table, oracle)
  net = networks.DQNAtariNetwork(A, seed=4, precision=_capi.PRECISION_BF16FLOW, input_channels=3)
  onet, otgt = onets.DQNAtariNetwork(A, in_c=3), onets.DQNAtariNetwork(A, in_c=3)
  for o in (onet, otgt):
    o.load(net.variables())
  ds = replay.ReplayDataset(table, Bd, seed=7)
  learner = dqn.DQNLearner(net, net.clone(), 0.99, 0.2, 1e-3, 100, ds, replay_client=replay.Client(server),
                           logger=loggers.NoOpLogger(), use_cuda_graph=False)
  assert learner._gather_rows is not None          # K3 writes the row image of the 3-channel frames
  ol = olearner.DQNOracleLearner(onet, otgt, 0.99, 0.2, 1e-3, 100)
  u = rng.random(Bd, dtype=np.float32)
  keys, pos, prob = oracle.sample(u, True)
  ref = ol.step(*oracle.gather(pos), prob)
  learner.step(uniforms=torch.as_tensor(u).cuda())
  torch.cuda.synchronize()
  np.testing.assert_array_equal(ds.idx.cpu().numpy(), pos)
  td_err = float(np.abs(learner.td.cpu().numpy() - ref['td']).max()) / float(np.abs(ref['td']).max())
  assert td_err <= 2e-2, td_err
  np.testing.assert_allclose(float(learner.loss), ref['loss'], rtol=2e-2)
  server.stop()


# ------------------------------------------------------------------------------ agents
def _rgb_env(shape, episode_length=12):
  from acme_b200 import specs, testing
  return testing.Environment(specs.EnvironmentSpec(
      observations=specs.BoundedArray(shape, np.uint8, 0, 255), actions=specs.BoundedArray((ACT,), np.float32, -1., 1.),
      rewards=specs.Array((), np.float32), discounts=specs.BoundedArray((), np.float32, 0., 1.)), episode_length=episode_length)


@pytest.mark.parametrize('num_envs,frame_stack,shape,precision', [(16, 4, (HW, HW, 3, 4), 1), (16, 4, (HW, HW, 12), 3),
                                                                  (1, 0, (HW, HW, 3), 2)])
def test_rgb_agent_runs(num_envs, frame_stack, shape, precision):
  import gc
  import torch
  from acme_b200 import d4pg, environment_loop, loggers, specs
  envs = [_rgb_env(shape) for _ in range(num_envs)]
  spec = specs.make_environment_spec(envs[0])
  C = int(np.prod(shape[2:]))
  torso, policy, critic = _nets('d4pg', precision, C)
  ag = d4pg.D4PG(spec, policy, critic, batch_size=32, samples_per_insert=8, min_replay_size=32, max_replay_size=2000,
                 logger=loggers.NoOpLogger(), num_envs=num_envs, observation_network=torso, frame_stack=frame_stack)
  gc.collect()
  if num_envs == 1:
    loop = environment_loop.EnvironmentLoop(envs[0], ag, logger=loggers.NoOpLogger())
  else:
    loop = environment_loop.BatchedEnvironmentLoop(envs, ag, logger=loggers.NoOpLogger())
  loop.run(num_episodes=2 * num_envs + 4)
  torch.cuda.synchronize()
  assert int(ag._learner._num_steps) > 0
  assert torch.isfinite(ag._learner.critic_loss).all()
  if num_envs == 1:
    a = ag.select_action(np.random.default_rng(0).integers(0, 256, shape, dtype=np.uint8))
    assert a.shape == (ACT,) and np.all(a >= -1) and np.all(a <= 1)
