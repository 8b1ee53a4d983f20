"""Precision 3: the `*_x3` layer entry points (fp32 operands split into three bf16 planes, six products on the bf16 tensor
cores) and the networks / learners that use them.

Every output element is held to the precision-0 bound of the fp32 layer suite (layer_check._check, c_op = 0):

    |got - ref| <= 2^-16 (|A|.|B|)_ij

against fp64 on the exact fp32 operands.  The operands are arbitrary fp32 values N(0.3, 1) with full mantissas (on neither
the bf16 nor the tf32 grid); their low 16 bits lie in [0x4000, 0x8000), so that RN-bf16 of an operand always moves it
towards zero by a quarter to a half of a bf16 ulp.  (Operands of one sign throughout are not used: the tcgen05 fp32
accumulation is not round-to-nearest, and on all-positive sums it exceeds the bound, 1.8e-5 .. 3.9e-5 of the sum.)  Every row proves that the bound REJECTS the result of the hi x hi product alone, i.e. what bf16
operands give, and rows with a reduction of 1024 or more also that it rejects the reference without one 64-deep block
of the reduction.  Each row names its path ((a) planes concatenated along the reduction + one bf16 GEMM, (b) one raw
launch per plane + the combine kernel, (c) the fp32 FFMA path) and checks it three ways: the kernels torch.profiler sees,
the b200rl_launch_count() delta, and a sentinel-filled workspace that nothing past b200rl_x3_ws_bytes may touch.
Outputs sit inside sentinel guards.  A test without a GPU checks the Python mirror of the path rule (x3_path) against
every row.

Measured on an NVIDIA B200 (1000 W power limit), max over the rows below of |err| / (|A|.|B|):
    linear_fwd 3.2e-06   linear_dgrad 7.5e-06   linear_wgrad 5.1e-06   (bias gradient 7.2e-08)
    conv2d_fwd 3.4e-06   conv2d_wgrad 4.7e-06   conv2d_dgrad 2.9e-06   (bias gradient 9.3e-08)
i.e. up to half the bound (FFMA: 4.7e-07); the hi x hi result exceeds the bound by 44x or more on every row, the
reference without one block of its reduction by 75x or more.
(Run with `-s`: each check prints its ratio, and each rejection its margin, as `bound ...`.)"""
import ctypes
import json
import os
import zlib

import numpy as np
import pytest
from layer_check import ELU, NONE, RELU, SENT, TANH, Out, _capi, _check, _assert_rejects, mask_factor, mask_values, run

LIN_FWD, LIN_DGRAD, LIN_WGRAD, CONV_FWD, CONV_WGRAD, CONV_DGRAD = range(6)
OPS = {LIN_FWD: 'linear_fwd', LIN_DGRAD: 'linear_dgrad', LIN_WGRAD: 'linear_wgrad', CONV_FWD: 'conv2d_fwd',
       CONV_WGRAD: 'conv2d_wgrad', CONV_DGRAD: 'conv2d_dgrad'}


# ------------------------------------------------------------------------------ the path rule (mirror of fp32x3.cu)
def _rup(a, m):
  return -(-a // m) * m


def rows_eligible(g):
  """the bf16 row image of the first layer (gemm_bf16.cu rows_eligible)"""
  return g['C'] == 4 and g['kw'] * g['C'] == 32 and g['Cout'] in (32, 64) and (g['stride'] * g['C'] * 2) % 16 == 0


def x3_path(op, M=0, N=0, K=0, g=None, x_u8=0):
  if op in (LIN_FWD, LIN_DGRAD, LIN_WGRAD):
    if M * N * K < 1 << 26:
      return 'c'
    ok = {LIN_FWD: 6 * _rup(K, 8) >= 64, LIN_DGRAD: K % 64 == 0 and 6 * _rup(N, 8) >= 64,
          LIN_WGRAD: N % 64 == 0 and K % 64 == 0}[op]
    return 'a' if ok else 'c'
  if op == CONV_FWD:
    if x_u8:
      return 'b' if rows_eligible(g) else 'c'
    return 'a' if g['Cout'] in (32, 64, 128) else 'c'
  if op == CONV_WGRAD:
    if x_u8:
      return 'a' if rows_eligible(g) else 'c'
    return 'a' if (g['C'] == 32 or g['C'] % 64 == 0) and g['Cout'] in (32, 64) else 'c'
  s = g['stride']
  return 'a' if s <= 2 and g['kh'] >= s and g['kw'] >= s and g['C'] in (32, 64, 128) else 'c'


def G(B, H, C, k, s, Cout):
  """TF-SAME geometry as a dict (networks.tf_same_pad)"""
  oh = -(-H // s)
  pad = max((oh - 1) * s + k - H, 0) // 2
  return dict(B=B, H=H, W=H, C=C, kh=k, kw=k, stride=s, pad_top=pad, pad_left=pad, OH=oh, OW=oh, Cout=Cout)


# rows: (id, op, shape, options, path).  Dense shape (M, N, K); conv shape = geometry dict.  Options: act, bias, mask
# (mask_act), lda / ldb (row strides of the first / second operand), ldo (of the output and mask), x_u8, db.
DQN = [(84, 4, 8, 4, 32), (21, 32, 4, 2, 64), (11, 64, 3, 1, 64)]   # (H, C, k, stride, Cout) of conv1..3 (atari.py:44)
ROWS = []
for B in (256, 512):
  for i, (H, C, k, s, Co) in enumerate(DQN):
    g = G(B, H, C, k, s, Co)
    if i == 0:
      ROWS += [(f'dqn{B}-conv1-fwd-u8', CONV_FWD, g, dict(x_u8=1, act=RELU, bias=1), 'b'),
               (f'dqn{B}-conv1-fwd-rows', CONV_FWD, g, dict(x_u8=2, act=RELU, bias=1), 'b'),
               (f'dqn{B}-conv1-wgrad-rows', CONV_WGRAD, g, dict(x_u8=2, db=1), 'a')]
      if B == 256:
        ROWS.append((f'dqn{B}-conv1-wgrad-u8', CONV_WGRAD, g, dict(x_u8=1, db=1), 'a'))
    else:
      ROWS += [(f'dqn{B}-conv{i + 1}-fwd', CONV_FWD, g, dict(act=RELU, bias=1), 'a'),
               (f'dqn{B}-conv{i + 1}-wgrad', CONV_WGRAD, g, dict(db=1), 'a'),
               (f'dqn{B}-conv{i + 1}-dgrad', CONV_DGRAD, g, dict(mask=RELU), 'a')]
  ROWS += [(f'dqn{B}-fc1-fwd', LIN_FWD, (B, 1024, 7744), dict(act=RELU, bias=1), 'a'),
           (f'dqn{B}-fc1-dgrad', LIN_DGRAD, (B, 1024, 7744), dict(mask=RELU), 'a'),
           (f'dqn{B}-fc1-wgrad', LIN_WGRAD, (B, 1024, 7744), dict(db=1), 'a')]
ROWS += [
    # D4PG / DDPG critic (67 + 21 inputs, 512-512-256, 51 atoms) and policy (67 inputs, 256-256-256, 21 actions) at B = 256
    ('d4pg-l0-fwd', LIN_FWD, (256, 512, 88), dict(bias=1), 'c'),
    ('d4pg-l1-fwd', LIN_FWD, (256, 512, 512), dict(act=ELU, bias=1), 'a'),
    ('d4pg-l1-dgrad', LIN_DGRAD, (256, 512, 512), dict(mask=None), 'a'),
    ('d4pg-l1-wgrad', LIN_WGRAD, (256, 512, 512), dict(db=1), 'a'),
    ('d4pg-l2-fwd', LIN_FWD, (256, 256, 512), dict(act=ELU, bias=1), 'c'),
    ('d4pg-l2-dgrad', LIN_DGRAD, (256, 256, 512), dict(mask=ELU), 'c'),
    ('d4pg-head-wgrad', LIN_WGRAD, (256, 51, 256), dict(db=1), 'c'),
    ('policy-l1-fwd', LIN_FWD, (256, 256, 256), dict(act=ELU, bias=1), 'c'),
    # ragged dimensions (padding of every plane), row strides, each activation and mask
    ('ragged-fwd-tanh', LIN_FWD, (400, 200, 1100), dict(act=TANH, bias=1, lda=1104, ldo=203), 'a'),
    ('ragged-fwd-elu', LIN_FWD, (129, 70, 9000), dict(act=ELU, bias=1), 'a'),
    ('ragged-dgrad-tanh', LIN_DGRAD, (300, 250, 1024), dict(mask=TANH, lda=257, ldo=1030), 'a'),
    ('ragged-dgrad-elu', LIN_DGRAD, (257, 13, 20480), dict(mask=ELU), 'a'),
    ('ragged-wgrad', LIN_WGRAD, (1000, 128, 576), dict(db=1, lda=131, ldb=580), 'a'),
    ('dense-uncovered-dgrad', LIN_DGRAD, (512, 512, 1000), dict(mask=RELU), 'c'),
    ('conv-fwd-c12-elu', CONV_FWD, G(16, 15, 12, 3, 1, 64), dict(act=ELU, bias=1), 'a'),
    ('conv-fwd-c96-tanh', CONV_FWD, G(8, 9, 96, 3, 2, 128), dict(act=TANH, bias=1), 'a'),
    ('conv-fwd-cout16', CONV_FWD, G(8, 9, 32, 3, 1, 16), dict(act=RELU, bias=1), 'c'),
    ('conv-wgrad-c64-cout32', CONV_WGRAD, G(10, 12, 64, 3, 2, 32), dict(db=1), 'a'),
    ('conv-wgrad-c12', CONV_WGRAD, G(4, 9, 12, 3, 1, 32), dict(db=1), 'c'),
    ('conv-dgrad-cout20-elu', CONV_DGRAD, G(6, 13, 32, 4, 2, 20), dict(mask=ELU), 'a'),
    ('conv-dgrad-c128-tanh', CONV_DGRAD, G(4, 7, 128, 3, 1, 64), dict(mask=TANH), 'a'),
    ('conv-dgrad-stride3', CONV_DGRAD, G(4, 12, 32, 3, 3, 32), dict(mask=RELU), 'c'),
    ('conv1-stride3-u8', CONV_FWD, G(4, 24, 4, 8, 3, 32), dict(x_u8=1, act=RELU, bias=1), 'c'),
]


def test_path_rule_mirror_agrees_with_every_row():
  assert len({r[0] for r in ROWS}) == len(ROWS)
  for rid, op, shape, opt, path in ROWS:
    if op <= LIN_WGRAD:
      got = x3_path(op, *shape)
    else:
      got = x3_path(op, g=shape, x_u8=opt.get('x_u8', 0))
    assert got == path, (rid, got, path)
  # every DQN-Atari layer op runs on the tensor cores at precision 3
  assert all(r[4] in 'ab' for r in ROWS if r[0].startswith('dqn'))


# ------------------------------------------------------------------------------ GPU rows
_KEEP = []


@pytest.fixture(autouse=True)
def _release():
  yield
  _KEEP.clear()


def full_fp32(rng, shape):
  """fp32 values N(0.3, 1) with full mantissas whose low 16 bits lie in [0x4000, 0x8000): RN-bf16 moves every one of them
  towards zero by a quarter to a half of a bf16 ulp, so the error of bf16 operands follows the sign of each product and
  does not cancel in the sums, and the bound's rejection of it does not depend on luck"""
  v = (rng.standard_normal(shape) + 0.3).astype(np.float32)
  bits = v.view(np.uint32) & np.uint32(0xFFFF0000)
  bits |= rng.integers(0x4000, 0x8000, size=shape, dtype=np.uint32) | np.uint32(0x101)
  return bits.view(np.float32)


def bf16_hi(x):
  import torch
  return torch.as_tensor(np.ascontiguousarray(x, np.float32)).to(torch.bfloat16).double().numpy()


def dev_mat(a, ld=None):
  """[rows][cols] fp32 device matrix with row stride ld (NaN padding)"""
  import torch
  a = np.asarray(a, np.float32).reshape(a.shape[0], -1)
  ld = ld or a.shape[1]
  t = torch.full((a.shape[0], ld), float('nan'), dtype=torch.float32, device='cuda')
  t[:, :a.shape[1]] = torch.as_tensor(a).cuda()
  _KEEP.append(t)
  return t


def geom_c(g):
  return _capi().ConvGeom(**g)


def ws_bytes(op, shape, x_u8=0):
  c = _capi()
  if op <= LIN_WGRAD:
    return int(c.load().b200rl_x3_ws_bytes(op, *shape, None, 0))
  return int(c.load().b200rl_x3_ws_bytes(op, 0, 0, 0, ctypes.byref(geom_c(shape)), x_u8))


class Ws:
  """a 256-byte aligned, sentinel-filled workspace of exactly `need` bytes followed by 1 MB of guard"""

  def __init__(self, need):
    import torch
    self.need = need
    self.buf = torch.full((need + (1 << 20),), SENT, dtype=torch.uint8, device='cuda')
    self.ptr = self.buf.data_ptr()

  def check(self, what):
    assert bool((self.buf[self.need:] == SENT).all()), f'{what}: workspace written past b200rl_x3_ws_bytes = {self.need}'


def assert_path(what, got, path):
  launches, names = got
  if names is not None:
    assert launches == len(names), (what, launches, names)
    x3 = [n for n in names if n.startswith('x3_')]
    tc = [n for n in names if n.startswith(('hgemm', 'hconv'))]
    if path == 'c':
      assert not x3 and not tc, (what, names)
    else:
      assert x3.count('x3_split_kernel') == 1 and tc, (what, names)
      assert ('x3_combine_kernel' in x3) == (path == 'b'), (what, names)
      assert len(tc) == (3 if path == 'b' else 1), (what, names)   # split-K finish kernels are not counted here


# references (fp64 torch): (value, |A|.|B|) for given operands
def _conv_refs():
  import test_gpu_fp32_layers as f
  return f


def _fwd_ref(op, shape, a, b, bias_v, opt):
  """pre-activation reference of an op on operands a, b (numpy fp64)"""
  f = _conv_refs()
  if op == LIN_FWD:
    return a @ b.T
  if op == LIN_DGRAD:
    return a @ b
  if op == LIN_WGRAD:
    return a.T @ b
  g = shape
  k, s, H, oh, pad = g['kh'], g['stride'], g['H'], g['OH'], g['pad_top']
  if op == CONV_FWD:
    return f.conv_fwd_ref(a, b, k, s, H, oh, pad)
  if op == CONV_WGRAD:
    return f.conv_wgrad_ref(a, b, k, s, H, oh, pad, g['C'])
  return f.conv_dgrad_ref(a, b, k, s, H, oh, pad)


def _drop_block(op, shape, a):
  """operand a without one 64-deep block of the reduction (the middle one); None when the reduction is < 1024"""
  a = a.copy()
  if op == LIN_FWD and shape[2] >= 1024:
    a[:, shape[2] // 2:shape[2] // 2 + 64] = 0
  elif op == LIN_DGRAD and shape[1] >= 1024:
    a[:, shape[1] // 2:shape[1] // 2 + 64] = 0
  elif op == LIN_WGRAD and shape[0] >= 1024:
    a[shape[0] // 2:shape[0] // 2 + 64] = 0
  elif op == CONV_FWD and shape['kh'] * shape['kw'] * shape['C'] >= 1024:
    a[..., :min(64, shape['C'])] = 0
  elif op == CONV_WGRAD and shape['B'] * shape['OH'] * shape['OW'] >= 1024:
    a[shape['B'] // 2] = 0
  elif op == CONV_DGRAD and shape['kh'] * shape['kw'] * shape['Cout'] >= 1024:
    a[..., :min(64, shape['Cout'])] = 0
  else:
    return None
  return a


def _operands(rng, op, shape, opt):
  """(a, b): the two operands of the op in the order of the entry point's arguments (uint8 frames for x_u8 rows)"""
  if op == LIN_FWD:
    M, N, K = shape
    return full_fp32(rng, (M, K)), full_fp32(rng, (N, K))
  if op == LIN_DGRAD:
    M, N, K = shape
    return full_fp32(rng, (M, N)), full_fp32(rng, (N, K))
  if op == LIN_WGRAD:
    M, N, K = shape
    return full_fp32(rng, (M, N)), full_fp32(rng, (M, K))
  g = shape
  if op == CONV_FWD:
    if opt.get('x_u8'):
      x = rng.integers(0, 256, (g['B'], g['H'], g['W'], g['C']), dtype=np.uint8)
    else:
      x = full_fp32(rng, (g['B'], g['H'], g['W'], g['C']))
    return x, full_fp32(rng, (g['Cout'], g['kh'], g['kw'], g['C']))
  if op == CONV_WGRAD:
    if opt.get('x_u8'):
      x = rng.integers(0, 256, (g['B'], g['H'], g['W'], g['C']), dtype=np.uint8)
    else:
      x = full_fp32(rng, (g['B'], g['H'], g['W'], g['C']))
    return x, full_fp32(rng, (g['B'], g['OH'], g['OW'], g['Cout']))
  return full_fp32(rng, (g['B'], g['OH'], g['OW'], g['Cout'])), full_fp32(rng, (g['Cout'], g['kh'], g['kw'], g['C']))


def _call(op, shape, opt, a_d, b_d, out, extra, ws):
  """issues the x3 call; a_d, b_d device operands (or the row image), extra = (bias / mask / db pointer)"""
  c = _capi()
  st = c.current_stream()
  lib = c.load()
  if op == LIN_FWD:
    M, N, K = shape
    return lib.b200rl_linear_fwd_x3(M, N, K, a_d.data_ptr(), a_d.shape[1], b_d.data_ptr(), extra, out.ptr, out.ld,
                                    opt.get('act', NONE), ws.ptr, ws.need, st)
  if op == LIN_DGRAD:
    M, N, K = shape
    return lib.b200rl_linear_dgrad_x3(M, N, K, a_d.data_ptr(), a_d.shape[1], b_d.data_ptr(), out.ptr, out.ld, extra,
                                      opt.get('mask') or 0, ws.ptr, ws.need, st)
  if op == LIN_WGRAD:
    M, N, K = shape
    return lib.b200rl_linear_wgrad_x3(M, N, K, a_d.data_ptr(), a_d.shape[1], b_d.data_ptr(), b_d.shape[1], out.ptr, extra,
                                      ws.ptr, ws.need, st)
  g = ctypes.byref(geom_c(shape))
  if op == CONV_FWD:
    return lib.b200rl_conv2d_fwd_x3(a_d.data_ptr(), opt.get('x_u8', 0), b_d.data_ptr(), extra, out.ptr, g, opt.get('act', NONE),
                                    ws.ptr, ws.need, st)
  if op == CONV_WGRAD:
    return lib.b200rl_conv2d_wgrad_x3(a_d.data_ptr(), opt.get('x_u8', 0), b_d.data_ptr(), out.ptr, extra, g, ws.ptr, ws.need, st)
  return lib.b200rl_conv2d_dgrad_x3(a_d.data_ptr(), b_d.data_ptr(), out.ptr, g, extra, opt.get('mask') or 0, ws.ptr, ws.need, st)


def _dev_operand(op, shape, opt, a, which):
  import torch
  if which == 'a' and op in (CONV_FWD, CONV_WGRAD) and opt.get('x_u8'):
    t = torch.as_tensor(a).cuda()
    _KEEP.append(t)
    if opt['x_u8'] == 1:
      return t
    c = _capi()
    g = geom_c(shape)
    n = int(c.load().b200rl_conv2d_rows_bf16_bytes(ctypes.byref(g)))
    rows = torch.zeros(n, dtype=torch.uint8, device='cuda')
    _KEEP.append(rows)
    c.call('b200rl_conv2d_rows_bf16_from_u8', t.data_ptr(), g, rows.data_ptr(), n, c.current_stream())
    return rows
  if op <= LIN_WGRAD:
    return dev_mat(a, opt.get('ld' + which))
  return dev_mat(a.reshape(-1, a.shape[-1]))


def _out_dims(op, shape, opt):
  """(rows, cols, ld) of the output"""
  if op == LIN_FWD:
    return shape[0], shape[1], opt.get('ldo')
  if op == LIN_DGRAD:
    return shape[0], shape[2], opt.get('ldo')
  if op == LIN_WGRAD:
    return shape[1], shape[2], None
  g = shape
  if op == CONV_FWD:
    return g['B'] * g['OH'] * g['OW'], g['Cout'], None
  if op == CONV_WGRAD:
    return g['Cout'], g['kh'] * g['kw'] * g['C'], None
  return g['B'] * g['H'] * g['W'], g['C'], None


@pytest.mark.gpu
@pytest.mark.parametrize('rid,op,shape,opt,path', ROWS, ids=[r[0] for r in ROWS])
def test_x3_layer_rows(rid, op, shape, opt, path):
  import torch
  c = _capi()
  rng = np.random.default_rng(zlib.crc32(rid.encode()))
  a, b = _operands(rng, op, shape, opt)
  u8 = opt.get('x_u8', 0)
  a64 = a.astype(np.float64) / 255. if u8 else a.astype(np.float64)
  b64 = b.astype(np.float64)
  pre = _fwd_ref(op, shape, a64, b64, None, opt)
  absr = _fwd_ref(op, shape, np.abs(a64), np.abs(b64), None, opt)
  rows, cols, ld = _out_dims(op, shape, opt)
  pre, absr = pre.reshape(rows, cols), absr.reshape(rows, cols)
  ahi = a64 if u8 else bf16_hi(a)
  broken = _fwd_ref(op, shape, ahi, bf16_hi(b), None, opt).reshape(rows, cols)
  dropped = _drop_block(op, shape, a64)
  dropped = None if dropped is None else _fwd_ref(op, shape, dropped, b64, None, opt).reshape(rows, cols)
  extra, ref, post = None, pre, lambda v: v
  act = opt.get('act', NONE)
  if opt.get('bias'):
    bias = rng.standard_normal(cols).astype(np.float32)
    bias_d = dev_mat(bias[None])
    extra = bias_d.data_ptr()
    absr = absr + np.abs(bias)[None]
    post = lambda v: v + bias.astype(np.float64)[None]
  mask = opt.get('mask')
  if mask:
    y = mask_values(rng, (rows, cols), mask).astype(np.float32)
    mask_d = dev_mat(y, ld)
    extra = mask_d.data_ptr()
    gfac, gabs = mask_factor(y.astype(np.float64), mask)
    absr = absr * gabs
    post = lambda v: v * gfac
  need = ws_bytes(op, shape, u8)
  assert need > 0
  ws = Ws(need)
  a_d, b_d = _dev_operand(op, shape, opt, a, 'a'), _dev_operand(op, shape, opt, b, 'b')
  out = Out(rows, cols, False, ld=ld)
  got = run(lambda: c.check(_call(op, shape, opt, a_d, b_d, out, extra, ws)))
  assert_path(rid, got, path)
  ws.check(rid)
  what = f'{OPS[op]} {rid}'
  from layer_check import act as act_fn
  # ReLU, ELU and tanh are 1-Lipschitz: the bound of the pre-activation holds for the activation
  _check(what, out.read(what), act_fn(post(pre), act), absr, False)
  _assert_rejects(what + ' (hi x hi only)', post(pre), post(broken), absr, False)
  if dropped is not None:
    _assert_rejects(what + ' (one block of the reduction lost)', post(pre), post(dropped), absr, False)
  first = out.bits()
  # bit-identical on a repeat
  out.reset()
  c.check(_call(op, shape, opt, a_d, b_d, out, extra, ws))
  torch.cuda.synchronize()
  assert bool((out.bits() == first).all()), f'{what}: a repeat differs'
  if opt.get('db'):
    dycols = shape[1] if op == LIN_WGRAD else shape['Cout']
    db = Out(1, dycols, False)
    out.reset()
    c.check(_call(op, shape, opt, a_d, b_d, out, db.ptr, ws))
    torch.cuda.synchronize()
    assert bool((out.bits() == first).all()), f'{what}: dw changed when db was requested'
    dy = (a if op == LIN_WGRAD else b).astype(np.float64).reshape(-1, dycols)
    _check(what + ' db', db.read(what + ' db')[0], dy.sum(0), np.abs(dy).sum(0), False)
    ws.check(rid + ' db')


# ------------------------------------------------------------------------------ rejected calls
@pytest.mark.gpu
def test_x3_rejects_small_workspace_misalignment_and_uncovered_shapes():
  import torch
  from layer_check import _rejects
  c = _capi()
  lib = c.load()
  st = c.current_stream()
  M, N, K = 256, 1024, 7744
  need = ws_bytes(LIN_FWD, (M, N, K))
  ws = torch.empty(need + 512, dtype=torch.uint8, device='cuda')
  x = torch.randn(M * K + 8, device='cuda')
  w = torch.randn(N * K + 8, device='cuda')
  out = Out(M, N, False)
  _rejects('workspace one byte short', 'b200rl_linear_fwd_x3', out, M, N, K, x.data_ptr(), K, w.data_ptr(), None, out.ptr, N, 0,
           ws.data_ptr(), need - 1, st)
  _rejects('unaligned workspace', 'b200rl_linear_fwd_x3', out, M, N, K, x.data_ptr(), K, w.data_ptr(), None, out.ptr, N, 0,
           ws.data_ptr() + 16, need, st)
  _rejects('ldx < K', 'b200rl_linear_fwd_x3', out, M, N, K, x.data_ptr(), K - 1, w.data_ptr(), None, out.ptr, N, 0, ws.data_ptr(),
           need, st)
  g = G(8, 21, 32, 4, 2, 64)
  gc = geom_c(g)
  wsb = ws_bytes(CONV_FWD, g)
  cws = torch.empty(wsb, dtype=torch.uint8, device='cuda')
  xin = torch.randn(8 * 21 * 21 * 32 + 8, device='cuda')
  wt = torch.randn(64 * 16 * 32 + 8, device='cuda')
  yo = Out(8 * 11 * 11, 64, False)
  _rejects('misaligned conv x', 'b200rl_conv2d_fwd_x3', yo, xin.data_ptr() + 4, 0, wt.data_ptr(), None, yo.ptr, ctypes.byref(gc), 0,
           cws.data_ptr(), wsb, st)
  _rejects('x_u8 = 3', 'b200rl_conv2d_fwd_x3', yo, xin.data_ptr(), 3, wt.data_ptr(), None, yo.ptr, ctypes.byref(gc), 0,
           cws.data_ptr(), wsb, st)
  _rejects('row image of a non-first-layer geometry', 'b200rl_conv2d_fwd_x3', yo, xin.data_ptr(), 2, wt.data_ptr(), None, yo.ptr,
           ctypes.byref(gc), 0, cws.data_ptr(), wsb, st)
  dgc = geom_c(G(8, 21, 32, 4, 2, 64))
  _rejects('misaligned conv dgrad w', 'b200rl_conv2d_dgrad_x3', yo, xin.data_ptr(), wt.data_ptr() + 4, yo.ptr, ctypes.byref(dgc),
           None, 0, cws.data_ptr(), wsb, st)
  bad = geom_c(dict(G(8, 21, 32, 4, 2, 64), C=30))
  _rejects('channels not a multiple of 4', 'b200rl_conv2d_fwd_x3', yo, xin.data_ptr(), 0, wt.data_ptr(), None, yo.ptr,
           ctypes.byref(bad), 0, cws.data_ptr(), wsb, st)
  assert lib.b200rl_x3_ws_bytes(6, 1, 1, 1, None, 0) == -1
  assert lib.b200rl_x3_ws_bytes(CONV_FWD, 0, 0, 0, ctypes.byref(bad), 0) == -1
  assert lib.b200rl_x3_ws_bytes(CONV_DGRAD, 0, 0, 0, ctypes.byref(dgc), 1) == -1


# ------------------------------------------------------------------------------ launch order
@pytest.mark.gpu
def test_x3_bit_identical_across_pdl_graph_and_streams():
  """fc1's forward (path a, split-K), conv1's forward on frames (path b) and conv2's data gradient: eager with and without
  programmatic dependent launch, CUDA-graph replay, and two concurrent calls on two streams with one workspace each."""
  import torch
  c = _capi()
  lib = c.load()
  rng = np.random.default_rng(3)
  calls = []
  for op, shape, opt in ((LIN_FWD, (256, 1024, 7744), dict(act=RELU, bias=1)), (CONV_FWD, G(256, 84, 4, 8, 4, 32), dict(x_u8=1, act=RELU)),
                         (CONV_DGRAD, G(256, 21, 32, 4, 2, 64), dict(mask=RELU))):
    a, b = _operands(rng, op, shape, opt)
    rows, cols, ld = _out_dims(op, shape, opt)
    extra = None
    if opt.get('bias'):
      extra = dev_mat(rng.standard_normal((1, cols)).astype(np.float32)).data_ptr()
    if opt.get('mask'):
      extra = dev_mat(mask_values(rng, (rows, cols), RELU).astype(np.float32)).data_ptr()
    a_d, b_d = _dev_operand(op, shape, opt, a, 'a'), _dev_operand(op, shape, opt, b, 'b')
    need = ws_bytes(op, shape, opt.get('x_u8', 0))
    calls.append((op, shape, opt, a_d, b_d, extra, [Ws(need), Ws(need)], [Out(rows, cols, False), Out(rows, cols, False)]))

  def issue(k):
    for op, shape, opt, a_d, b_d, extra, wss, outs in calls:
      c.check(_call(op, shape, opt, a_d, b_d, outs[k], extra, wss[k]))

  issue(0)
  torch.cuda.synchronize()
  ref = [cl[7][0].bits() for cl in calls]

  def same(what, k=0):
    torch.cuda.synchronize()
    for (op, shape, opt, *_rest), r in zip(calls, ref):
      assert bool((_rest[-1][k].bits() == r).all()), f'{what}: {OPS[op]} differs'
    for cl in calls:
      cl[7][k].reset()

  for cl in calls:
    cl[7][0].reset()
  lib.b200rl_debug_set_pdl(0)
  try:
    issue(0)
    same('PDL off')
  finally:
    lib.b200rl_debug_set_pdl(-1)
  issue(0)
  same('PDL on')
  s = torch.cuda.Stream()
  g = torch.cuda.CUDAGraph()
  with torch.cuda.graph(g, stream=s):
    issue(0)
  for cl in calls:
    cl[7][0].reset()
  g.replay()
  same('graph replay')
  s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
  torch.cuda.synchronize()
  with torch.cuda.stream(s1):
    issue(0)
  with torch.cuda.stream(s2):
    issue(1)
  torch.cuda.synchronize()
  same('stream 1', 0)
  same('stream 2', 1)


# ------------------------------------------------------------------------------ learners
@pytest.mark.gpu
@pytest.mark.parametrize('use_cuda_graph', [False, True], ids=['eager', 'graph'])
def test_dqn_learner_c2_shape_parity_x3(use_cuda_graph):
  """The C2 shape (84x84x4 uint8, A = 18, B = 256, n = 3) through the whole DQN learner at precision 3 against the oracle
  under the unchanged FP32_TOL of test_gpu_learner.py, three updates on injected uniforms (graph: four, on the learner's
  own Philox draws, the last two replaying the graph)."""
  import torch
  import helpers
  from test_gpu_learner import FP32_TOL, _export_flat, _scale_err
  from acme_b200 import dqn, loggers, networks, replay
  from oracle import learner as olearner
  from oracle import nets as onets
  c = _capi()
  tolv = FP32_TOL
  rng = np.random.default_rng(21)
  shape, A, n, B = (84, 84, 4), 18, 3, 256
  spec, table, server, adder, oracle = helpers.make_pair(shape, np.uint8, A, n, 0.99, 0.6, max_size=1500)
  for ep in range(12):
    helpers.feed_episode(rng, adder, oracle, int(rng.integers(60, 140)), n, shape, np.uint8, A)
  table.flush()
  helpers.sync_oracle_leaves(table, oracle)
  keys = np.arange(oracle.item_tail, oracle.item_head, dtype=np.uint64)
  pr = np.abs(rng.standard_normal(keys.shape[0])).astype(np.float32)
  replay.Client(server).update_priorities(table.name, keys, pr.astype(np.float64))
  oracle.update_priorities(keys, pr)
  torch.cuda.synchronize()
  helpers.sync_oracle_leaves(table, oracle)
  net = networks.DQNAtariNetwork(A, seed=5, precision=c.PRECISION_FP32X3)
  tgt = net.clone()
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
    if use_cuda_graph:
      c.call('b200rl_uniform', u_dev.data_ptr(), B, 7, counter.data_ptr(), step, c.current_stream())
      u = u_dev.cpu().numpy()
    else:
      u = rng.random(B, dtype=np.float32)
    keys, pos, prob = oracle.sample(u)
    ref = ol.step(*oracle.gather(pos), prob)
    learner.step(uniforms=None if use_cuda_graph else torch.as_tensor(u).cuda())
    torch.cuda.synchronize()
    np.testing.assert_array_equal(ds.idx.cpu().numpy(), pos)
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
    helpers.sync_oracle_leaves_loose(table, oracle, rtol=5e-3, atol=1e-4)
  out = os.environ.get('B200RL_PARITY_DIR')
  if out:
    os.makedirs(out, exist_ok=True)
    mode = 'fp32x3' + ('_graph' if use_cuda_graph else '')
    with open(os.path.join(out, f'parity_c2_{mode}.json'), 'w') as f:
      json.dump(dict(mode=mode, B=B, A=A, tolerances=tolv, measured=measured), f, indent=1)
  server.stop()


@pytest.mark.gpu
def test_dqn_learner_eager_and_graph_bit_identical_x3():
  """Precision 3, four updates on the learner's own device draws: eager and one CUDA graph give bit-identical parameters,
  Adam moments and losses."""
  import torch
  import helpers
  from acme_b200 import dqn, loggers, networks, replay
  c = _capi()
  shape, A, n, B = (84, 84, 4), 18, 3, 256
  runs = []
  for graph in (False, True):
    rng = np.random.default_rng(4)     # the same table for both runs (the learner writes priorities back)
    spec, table, server, adder, oracle = helpers.make_pair(shape, np.uint8, A, n, 0.99, 0.6, max_size=1500)
    for ep in range(8):
      helpers.feed_episode(rng, adder, oracle, int(rng.integers(60, 140)), n, shape, np.uint8, A)
    table.flush()
    net = networks.DQNAtariNetwork(A, seed=5, precision=c.PRECISION_FP32X3)
    tgt = net.clone()
    ds = replay.ReplayDataset(table, B, seed=7)
    learner = dqn.DQNLearner(net, tgt, 0.99, 0.2, 1e-3, target_update_period=2, dataset=ds, replay_client=replay.Client(server),
                             logger=loggers.NoOpLogger(), use_cuda_graph=graph)
    losses = []
    for _ in range(4):
      learner.step()
      losses.append(learner.loss.clone())
    torch.cuda.synchronize()
    runs.append((torch.cat(losses), net.params.flat.clone(), tgt.params.flat.clone(), learner._m.clone(), learner._v.clone()))
    server.stop()
  for name, x, y in zip(('losses', 'parameters', 'target parameters', 'Adam m', 'Adam v'), runs[0], runs[1]):
    assert torch.equal(x, y), f'eager vs graph: {name} differ'


# C3 bounds at precision 3: the FP32_TOL numbers per quantity (values as q / td, losses as loss, gradients as grad_rel_l2)
C3_X3_TOL = dict(value=2e-5, loss=1e-4, grad_rel_l2=1e-3)


@pytest.mark.gpu
@pytest.mark.parametrize('kind', ['d4pg', 'ddpg'])
def test_learner_c3_shape_parity_x3(kind):
  """D4PG / DDPG at the C3 shape (67 / 21, 51 atoms, B = 256) at precision 3 against the oracle: three updates on injected
  uniforms, the oracle adopting the device networks and Adam moments before each."""
  import torch
  from test_gpu_d4pg_bf16 import ACT, OBS, _export_flat, _learner, _nets, _replay, _scale_err
  from oracle import learner as olearner
  from oracle import nets as onets
  from acme_b200 import replay
  B = 256
  table, server, oracle = _replay(B, 12)
  policy, critic = _nets(kind, _capi().PRECISION_FP32X3)
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
    np.testing.assert_array_equal(ds.idx.cpu().numpy(), pos)
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
  out = os.environ.get('B200RL_PARITY_DIR')
  if out:
    os.makedirs(out, exist_ok=True)
    with open(os.path.join(out, f'parity_c3_{kind}_fp32x3.json'), 'w') as f:
      json.dump(dict(learner=kind, mode='fp32x3', B=B, obs=OBS, act=ACT, n=5, tolerances=C3_X3_TOL, measured=measured), f, indent=1)
  for err in measured:
    for k, v in err.items():
      if k == 'step':
        continue
      if isinstance(v, dict):
        assert max(v.values()) <= C3_X3_TOL['grad_rel_l2'], (k, err['step'], v)
      else:
        assert v <= C3_X3_TOL['loss' if k.endswith('loss') else 'value'], (k, err['step'], v)
  server.stop()
