"""bf16 dataflow kernels (gemm_bf16.cu) through the C ABI against an fp64 reference on the SAME bf16-rounded operands.

Every output element is held to its own bound (`_check`):

    |got - ref| <= C_ACC * (|A|.|B|)_ij + c_out * |ref_ij|

where |A|.|B| is the same product (or convolution) on absolute values, bias magnitude included, and c_out = 2^-8 for a
bf16 output (one round-to-nearest to 8 significant bits: < 2^-8 relative) and 0 for an fp32 one.  Every row with a
reduction of 1024 or more also proves that the bound REJECTS the reference recomputed without one 64-wide k-block, without
the last (possibly ragged) k-block and, for split-K rows, without one whole split (`_assert_rejects`).

C_ACC = 2^-16.  Measured on a B200 (1000 W power limit), max over the rows below of |err| / (|A|.|B|) on fp32 outputs
and split-K partials:
    linear_fwd_bf16 7.8e-07    linear_dgrad_bf16 3.9e-07    linear_wgrad_bf16 2.5e-07    colsum_bf16 1.1e-08
    conv2d_fwd_bf16 3.3e-07    conv2d_wgrad_bf16 4.4e-07 (row image: 4.4e-07)          conv2d_dgrad_bf16 2.6e-07
i.e. <= 2^-20, 20x below C_ACC.  The estimate it was first set from, 2^-12, left the rejection of a conv1 weight
gradient without its last 25-pixel k-block at only 2x; at 2^-16 the smallest rejection margin is 32x.  (Run with `-s`:
each check prints its ratio, and each rejection its margin, as `bound ...`.)

Each variant-table row names the launch signature the dispatcher (`launch_h`, gemm_bf16.cu) must produce: the kernels
seen by torch.profiler (template arguments KE, A mode, B mode, BN included), the change of b200rl_launch_count(), and
for split-K the number of [M][N] fp32 partial slabs written into a sentinel-filled workspace -- each slab is checked
against the fp64 partial sum of its own k-range, which pins the split boundaries.  A dispatcher change that moves a row
to another variant fails here and the row is updated on purpose.  Every output sits inside a sentinel-filled buffer
(lead bytes, ld padding, extra rows): a store outside the logical region fails the row."""
import ctypes

import numpy as np
import pytest
from layer_check import (ELU, NONE, RELU, SENT, TANH, WS_BYTES, Out, Workspace, _assert_rejects, _capi, _check, _rejects,
                         act, assert_sig, mask_factor, mask_values, run)

pytestmark = pytest.mark.gpu

_KEEP = []
SMS = 148


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
  """array rounded to bf16 (returned as float64, exact)."""
  import torch
  return torch.as_tensor(np.ascontiguousarray(x, np.float32)).to(torch.bfloat16).double().numpy()


def mat_dev(a, ld=None, bf16=True):
  """[rows][cols] device matrix with row stride ld; the padding columns hold NaN (a kernel that reads them poisons its
  sums)."""
  import torch
  rows, cols = a.shape
  ld = ld or cols
  t = torch.full((rows, ld), float('nan'), dtype=torch.bfloat16 if bf16 else torch.float32, device='cuda')
  t[:, :cols] = torch.as_tensor(np.ascontiguousarray(a, np.float32)).to(t.dtype).cuda()
  _KEEP.append(t)
  return t


def stream():
  return _capi().current_stream()



def split_plan(M, N, K, KE, BN, wsb, allow=True):
  """launch_h's split-K rule -> (splits, k-blocks per split)"""
  tiles = -(-M // 128) * -(-N // BN)
  kb = -(-K // KE)
  s = 1
  if allow and 2 * tiles <= SMS and kb >= 16:
    s = max(1, min(-(-SMS // tiles), kb // 8, 64))
    s = max(1, min(s, wsb // (M * N * 4) if wsb else 0))
  kps = -(-kb // s)
  return -(-kb // kps), kps


def check_partials(what, slabs, kps, KE, K, partial_ref):
  """slab s = the fp32 sum over k-blocks [s * kps, (s + 1) * kps): partial_ref(lo, hi) -> (ref, |ref| bound) over k-range
  [lo, hi)"""
  for s in range(slabs.shape[0]):
    lo, hi = s * kps * KE, min(K, (s + 1) * kps * KE)
    ref, absr = partial_ref(lo, hi)
    _check(f'{what} split {s} partial (k {lo}..{hi})', slabs[s], ref, absr, False)


def drop_ranges(K, KE, splits, kps):
  """k-ranges a broken kernel might lose: one 64-wide block in the middle, the last (ragged) block, one whole split"""
  kb = -(-K // KE)
  blk = 64 // KE
  mid = (kb // 2) // blk * blk
  out = [('one 64-wide k-block', mid * KE, min(K, (mid + blk) * KE)), ('the last k-block', (kb - 1) * KE, K)]
  if splits > 1:
    s = splits // 2
    out.append((f'split {s}', s * kps * KE, min(K, (s + 1) * kps * KE)))
  return out


# ------------------------------------------------------------------------------ dense layers
def lin_ref(x, w, b, lo=0, hi=None):
  """x @ w^T over k in [lo, hi) (+ b): (value, |x| @ |w|^T (+ |b|))"""
  hi = x.shape[1] if hi is None else hi
  xs, ws = x[:, lo:hi], w[:, lo:hi]
  v, a = xs @ ws.T, np.abs(xs) @ np.abs(ws).T
  if b is not None:
    v, a = v + b, a + np.abs(b)
  return v, a


# M, N, K, splits, options; splits from launch_h (min(ceil(148 / tiles), kblocks / 8, 64, ws / (M N 4)), then rounded
# through kps = ceil(kblocks / splits))
LINEAR_FWD = [
    (256, 1024, 7744, 10, {}),                        # the learner's target pass
    (512, 1024, 7744, 5, {}),                         # the online pass over [o_tm1; o_t]
    (768, 1024, 7744, 4, {}),
    (1, 1024, 7744, 14, {}),                          # 15 rounded to 14
    (64, 18, 7752, 14, {'acts': [NONE, TANH]}),       # BN = 32; ragged last k-block inside the last split
    (129, 100, 1024, 2, {'acts': [ELU, RELU]}),       # ragged M and N
    (300, 200, 136, 1, {'acts': [TANH, NONE]}),       # ragged N and K
    (100, 64, 64, 1, {'acts': [RELU, ELU]}),
    (33, 1, 512, 1, {'acts': [NONE, RELU], 'ldy': 9}),
    (256, 1024, 7744, 3, {'wsb': 3 * 256 * 1024 * 4}),   # the workspace caps the split count
    (256, 1024, 7744, 1, {'ws': None}),               # no workspace: no split
    (256, 512, 512, 1, {'ldx': 1024, 'ldy': 1024, 'acts': [RELU, TANH]}),
]


@pytest.mark.parametrize('M,N,K,splits,opt', LINEAR_FWD, ids=lambda v: None if not isinstance(v, dict) else
                         '-'.join(f'{k}{"" if k == "acts" else v[k]}' for k in v) or 'default')
def test_linear_fwd_bf16(M, N, K, splits, opt):
  import torch
  c = _capi()
  rng = np.random.default_rng(M * 7 + N * 3 + K)
  x, w = bf(rng.standard_normal((M, K))), bf(rng.standard_normal((N, K)) / np.sqrt(K))
  b = rng.standard_normal(N).astype(np.float32).astype(np.float64)
  ldx, acts = opt.get('ldx', K), opt.get('acts', [RELU, RELU])
  xd, wd, bd = mat_dev(x, ldx), mat_dev(w), dev(b.astype(np.float32))
  ws = Workspace()
  wsp, wsb = (ws.ptr, opt.get('wsb', ws.bytes)) if 'ws' not in opt else (None, 0)
  BN = 32 if N <= 32 else (64 if N <= 64 else 128)
  plan, kps = split_plan(M, N, K, 64, BN, wsb)
  assert plan == splits, f'split rule gives {plan}, the table says {splits}'
  pre, absr = lin_ref(x, w, b)
  want = [f'hgemm_kernel<64,0,0,{BN},'] + (['splitk_finish_kernel'] if splits > 1 else [])
  for i, (out_bf16, a) in enumerate(((0, acts[0]), (1, acts[1]))):
    y = Out(M, N, out_bf16, ld=opt.get('ldy', N))
    ws.reset()
    sig = run(lambda: c.call('b200rl_linear_fwd_bf16', M, N, K, xd.data_ptr(), ldx, wd.data_ptr(), bd.data_ptr(), y.ptr, y.ld,
                             out_bf16, a, wsp, wsb, stream()), profile=i == 0)
    what = f'linear fwd {M}x{N}x{K} {"bf16" if out_bf16 else "fp32"} out act {a}'
    assert_sig(what, sig, want)
    ref = act(pre, a)
    _check(what, y.read(what), ref, absr, out_bf16)
    if wsp:
      slabs = ws.slabs(what, M, N, splits)
      if i == 0 and splits > 1:
        check_partials(what, slabs, kps, 64, K, lambda lo, hi: lin_ref(x, w, None, lo, hi))
    if i == 0 and K >= 1024:
      for how, lo, hi in drop_ranges(K, 64, splits, kps):
        _assert_rejects(f'{what} without {how}', ref, act(pre - lin_ref(x, w, None, lo, hi)[0], a), absr, out_bf16)


# M, N (reduction), K, BN, lddy, lddx, [(dx_bf16, mask_bf16 or None = no mask, mask_act)]; never split
LINEAR_DGRAD = [
    (256, 1024, 7744, 64, 1024, 7744, [(1, 1, RELU), (0, 0, TANH)]),      # BN 128 -> 64: fewer than 148 tiles
    (512, 1024, 7744, 128, 1024, 7744, [(1, 1, RELU), (0, 1, ELU)]),
    (129, 100, 128, 64, 104, 136, [(1, 1, TANH), (0, 0, RELU), (1, 0, ELU), (0, None, NONE)]),   # ragged reduction
    (1, 64, 64, 64, 64, 64, [(1, 1, RELU), (0, 0, TANH)]),
]


@pytest.mark.parametrize('M,N,K,BN,lddy,lddx,cfgs', LINEAR_DGRAD, ids=lambda v: 'cfgs' if isinstance(v, list) else None)
def test_linear_dgrad_bf16(M, N, K, BN, lddy, lddx, cfgs):
  c = _capi()
  rng = np.random.default_rng(M + N + K)
  dy, w = bf(rng.standard_normal((M, N))), bf(rng.standard_normal((N, K)) / np.sqrt(N))
  dyd, wd = mat_dev(dy, lddy), mat_dev(w)
  ws = Workspace()
  acc, absr = dy @ w, np.abs(dy) @ np.abs(w)
  for i, (dx_bf16, mask_bf16, ma) in enumerate(cfgs):
    what = f'linear dgrad {M}x{N}x{K} dx {"bf16" if dx_bf16 else "fp32"} mask {mask_bf16} act {ma}'
    if mask_bf16 is None:
      mptr, g, ag = None, 1., 1.
    else:
      ym = mask_values(rng, (M, K), ma)
      ym = bf(ym) if mask_bf16 else ym.astype(np.float32).astype(np.float64)
      mptr = mat_dev(ym, lddx, bf16=bool(mask_bf16)).data_ptr()        # the mask shares dx's row stride
      g, ag = mask_factor(ym, ma)
    dx = Out(M, K, dx_bf16, ld=lddx)
    sig = run(lambda: c.call('b200rl_linear_dgrad_bf16', M, N, K, dyd.data_ptr(), lddy, wd.data_ptr(), dx.ptr, lddx, dx_bf16,
                             mptr, mask_bf16 or 0, ma, ws.ptr, ws.bytes, stream()), profile=i == 0)
    assert_sig(what, sig, [f'hgemm_kernel<64,0,1,{BN},'])
    ref = acc * g
    _check(what, dx.read(what), ref, absr * ag, dx_bf16)
    ws.slabs(what, M, K, 1)
    if i == 0 and N >= 1024:
      for how, lo, hi in drop_ranges(N, 64, 1, 1):
        _assert_rejects(f'{what} without {how}', ref, (acc - dy[:, lo:hi] @ w[lo:hi]) * g, absr * ag, dx_bf16)


# M (reduction), N, K, splits, lddy, ldx
LINEAR_WGRAD = [
    (256, 1024, 7744, 1, 1024, 7744),
    (4096, 64, 64, 8, 72, 64),
    (2000, 64, 128, 4, 64, 136),        # ragged reduction in the last split
    (33, 64, 128, 1, 72, 136),
    (1, 128, 64, 1, 128, 64),
]


@pytest.mark.parametrize('M,N,K,splits,lddy,ldx', LINEAR_WGRAD)
def test_linear_wgrad_bf16(M, N, K, splits, lddy, ldx):
  c = _capi()
  rng = np.random.default_rng(M + 2 * N + K)
  dy, x = bf(rng.standard_normal((M, N))), bf(rng.standard_normal((M, K)))
  dyd, xd = mat_dev(dy, lddy), mat_dev(x, ldx)
  ws = Workspace()
  BN = 128 if K >= 128 else 64
  plan, kps = split_plan(N, K, M, 64, BN, ws.bytes)
  assert plan == splits, f'split rule gives {plan}, the table says {splits}'
  what = f'linear wgrad {M}x{N}x{K}'
  ref, absr = dy.T @ x, np.abs(dy).T @ np.abs(x)
  dw = Out(N, K, False)
  hg = [f'hgemm_kernel<64,1,1,{BN},'] + (['splitk_finish_kernel'] if splits > 1 else [])
  assert_sig(what, run(lambda: c.call('b200rl_linear_wgrad_bf16', M, N, K, dyd.data_ptr(), lddy, xd.data_ptr(), ldx, dw.ptr, None,
                                      ws.ptr, ws.bytes, stream())), hg)
  _check(what, dw.read(what), ref, absr, False)
  slabs = ws.slabs(what, N, K, splits)
  if splits > 1:
    check_partials(what, slabs, kps, 64, M, lambda lo, hi: (dy[lo:hi].T @ x[lo:hi], np.abs(dy[lo:hi]).T @ np.abs(x[lo:hi])))
  if M >= 1024:
    for how, lo, hi in drop_ranges(M, 64, splits, kps):
      _assert_rejects(f'{what} without {how}', ref, ref - dy[lo:hi].T @ x[lo:hi], absr, False)
  # with the bias gradient: the same dw bit for bit, plus one column-sum launch
  first = dw.bits()
  dw.reset()
  db = Out(1, N, False)
  ws.reset()
  assert_sig(what + ' + db', run(lambda: c.call('b200rl_linear_wgrad_bf16', M, N, K, dyd.data_ptr(), lddy, xd.data_ptr(), ldx, dw.ptr,
                                                db.ptr, ws.ptr, ws.bytes, stream())), hg + ['colsum_vec_kernel<true>'])
  assert bool((dw.bits() == first).all()), f'{what}: dw changed when db was requested'
  _check(what + ' db', db.read(what + ' db')[0], dy.sum(0), np.abs(dy).sum(0), False)


# ------------------------------------------------------------------------------ convolutions
def _geom(B, H, C, k, s, Cout):
  from acme_b200 import networks
  oh, pad = networks.tf_same_pad(H, k, s)
  return _capi().ConvGeom(B=B, H=H, W=H, C=C, kh=k, kw=k, stride=s, pad_top=pad, pad_left=pad, OH=oh, OW=oh, Cout=Cout), oh, pad


def _padded(x, k, s, H, oh, pad):
  import torch
  import torch.nn.functional as F
  total = max((oh - 1) * s + k - H, 0)
  return F.pad(torch.from_numpy(np.ascontiguousarray(x)).permute(0, 3, 1, 2), (pad, total - pad, pad, total - pad))


def conv_fwd_ref(x, w, k, s, H, oh, pad):
  """TF-SAME convolution in fp64 (explicit asymmetric padding): NHWC x, OHWI w -> NHWC"""
  import torch.nn.functional as F
  import torch
  return F.conv2d(_padded(x, k, s, H, oh, pad), torch.from_numpy(np.ascontiguousarray(w)).permute(0, 3, 1, 2),
                  stride=s).permute(0, 2, 3, 1).numpy()


def conv_wgrad_ref(x, dy, k, s, H, oh, pad, C):
  """sum over pixels of patch x dy -> OHWI"""
  import torch
  xp = _padded(x, k, s, H, oh, pad)
  dyt = torch.from_numpy(np.ascontiguousarray(dy)).permute(0, 3, 1, 2)
  return torch.nn.grad.conv2d_weight(xp, (dy.shape[3], C, k, k), dyt, stride=s).permute(0, 2, 3, 1).numpy()


def conv_dgrad_ref(dy, w, k, s, H, oh, pad):
  import torch
  total = max((oh - 1) * s + k - H, 0)
  B, C = dy.shape[0], w.shape[3]
  dyt = torch.from_numpy(np.ascontiguousarray(dy)).permute(0, 3, 1, 2)
  dxp = torch.nn.grad.conv2d_input((B, C, H + total, H + total), torch.from_numpy(np.ascontiguousarray(w)).permute(0, 3, 1, 2),
                                   dyt, stride=s)
  return dxp[:, :, pad:pad + H, pad:pad + H].permute(0, 2, 3, 1).numpy()


def wk(w, lo, hi):
  """OHWI weights with only the flattened reduction indices [lo, hi) kept: (tap, channel) order = the kernels' k order"""
  f = np.zeros_like(w).reshape(w.shape[0], -1)
  f[:, lo:hi] = w.reshape(w.shape[0], -1)[:, lo:hi]
  return f.reshape(w.shape)


def wgrad_range(x, dy, lo, hi, k, s, H, oh, pad, C):
  """weight gradient (value, |x| |dy| bound) over the flattened output pixels [lo, hi) only -- the k-range of a weight
  gradient's split or k-block; computed on the images that range touches"""
  hw, Cout = oh * oh, dy.shape[-1]
  b0, b1 = lo // hw, (hi - 1) // hw + 1
  d = np.zeros(((b1 - b0) * hw, Cout))
  d[lo - b0 * hw:hi - b0 * hw] = dy.reshape(-1, Cout)[lo:hi]
  d = d.reshape(b1 - b0, oh, oh, Cout)
  return (conv_wgrad_ref(x[b0:b1], d, k, s, H, oh, pad, C), conv_wgrad_ref(np.abs(x[b0:b1]), np.abs(d), k, s, H, oh, pad, C))


# B, H, C, k, s, Cout, splits
CONV_FWD = [
    (1, 21, 32, 4, 2, 64, 2), (6, 21, 32, 4, 2, 64, 2), (256, 21, 32, 4, 2, 64, 1), (512, 21, 32, 4, 2, 64, 1),   # conv2
    (1, 11, 64, 3, 1, 64, 1), (40, 11, 64, 3, 1, 64, 1), (256, 11, 64, 3, 1, 64, 1), (512, 11, 64, 3, 1, 64, 1),  # conv3
    (6, 11, 64, 3, 1, 32, 1), (40, 21, 32, 4, 2, 128, 2), (6, 11, 128, 3, 1, 128, 2),
    (6, 13, 32, 4, 2, 64, 2),           # odd H: asymmetric SAME padding (1 top / left, 2 bottom / right)
]


@pytest.mark.parametrize('B,H,C,k,s,Cout,splits', CONV_FWD)
def test_conv_fwd_bf16(B, H, C, k, s, Cout, splits):
  c = _capi()
  rng = np.random.default_rng(B + H + C + Cout)
  g, oh, pad = _geom(B, H, C, k, s, Cout)
  K, M, KE = k * k * C, B * oh * oh, 32 if C == 32 else 64
  x = bf(np.maximum(rng.standard_normal((B, H, H, C)), 0))
  w = bf(rng.standard_normal((Cout, k, k, C)) / np.sqrt(K))
  b = (rng.standard_normal(Cout) * 0.1).astype(np.float32).astype(np.float64)
  xd, wd, bd = dev(x, _bf16()), dev(w, _bf16()), dev(b.astype(np.float32))
  acc, absr = conv_fwd_ref(x, w, k, s, H, oh, pad), conv_fwd_ref(np.abs(x), np.abs(w), k, s, H, oh, pad) + np.abs(b)
  pre = (acc + b).reshape(M, Cout)
  absr, acc = absr.reshape(M, Cout), acc.reshape(M, Cout)
  ws = Workspace()
  plan, kps = split_plan(M, Cout, K, KE, Cout, ws.bytes)
  assert plan == splits, f'split rule gives {plan}, the table says {splits}'
  want = [f'hgemm_kernel<{KE},0,0,{Cout},'] + (['splitk_finish_kernel'] if splits > 1 else [])
  a2 = (NONE, ELU, TANH)[(B + H) % 3]
  for i, (out_bf16, a) in enumerate(((1, RELU), (0, a2))):
    what = f'conv fwd B{B} H{H} C{C} k{k} s{s} Cout{Cout} {"bf16" if out_bf16 else "fp32"} out act {a}'
    y = Out(M, Cout, out_bf16)
    ws.reset()
    assert_sig(what, run(lambda: c.call('b200rl_conv2d_fwd_bf16', xd.data_ptr(), 0, wd.data_ptr(), bd.data_ptr(), y.ptr, out_bf16, g,
                                        a, ws.ptr, ws.bytes, stream()), profile=i == 0), want)
    ref = act(pre, a)
    _check(what, y.read(what), ref, absr, out_bf16)
    slabs = ws.slabs(what, M, Cout, splits)
    if i == 0 and splits > 1:
      check_partials(what, slabs, kps, KE, K, lambda lo, hi: (
          conv_fwd_ref(x, wk(w, lo, hi), k, s, H, oh, pad).reshape(M, Cout),
          conv_fwd_ref(np.abs(x), np.abs(wk(w, lo, hi)), k, s, H, oh, pad).reshape(M, Cout)))
    if i == 0 and K >= 1024:
      for how, lo, hi in drop_ranges(K, KE, splits, kps):
        lost = conv_fwd_ref(x, wk(w, lo, hi), k, s, H, oh, pad).reshape(M, Cout)
        _assert_rejects(f'{what} without {how}', ref, act(pre - lost, a), absr, out_bf16)


def _bf16():
  import torch
  return torch.bfloat16


# B, H, C, k, s, Cout, splits
CONV_WGRAD = [(B, H, C, k, s, Cout, sp) for (H, C, k, s) in ((21, 32, 4, 2), (11, 64, 3, 1)) for Cout in (32, 64)
              for B, sp in ((1, 1), (256, 35 if C == 32 else 29))]


@pytest.mark.parametrize('B,H,C,k,s,Cout,splits', CONV_WGRAD)
def test_conv_wgrad_bf16(B, H, C, k, s, Cout, splits):
  """all four (C, Cout) template pairs: <64,1,1,64>, <64,2,1,64>, <64,2,2,32>, <64,1,2,32>"""
  c = _capi()
  rng = np.random.default_rng(B + H + C + 3 * Cout)
  g, oh, pad = _geom(B, H, C, k, s, Cout)
  K, P = k * k * C, B * oh * oh
  x = bf(np.maximum(rng.standard_normal((B, H, H, C)), 0))
  dy = bf(rng.standard_normal((B, oh, oh, Cout)))
  xd, dyd = dev(x, _bf16()), dev(dy, _bf16())
  ws = Workspace()
  BN = Cout
  plan, kps = split_plan(K, Cout, P, 64, BN, ws.bytes)
  assert plan == splits, f'split rule gives {plan}, the table says {splits}'
  what = f'conv wgrad B{B} H{H} C{C} k{k} s{s} Cout{Cout}'
  wr = lambda lo, hi: wgrad_range(x, dy, lo, hi, k, s, H, oh, pad, C)
  ref, absr = (r.reshape(Cout, K) for r in wr(0, P))
  am, bm = 1 if C == 64 else 2, 1 if Cout == 64 else 2
  hg = [f'hgemm_kernel<64,{am},{bm},{BN},'] + (['splitk_finish_kernel'] if splits > 1 else [])
  dw = Out(Cout, K, False)
  assert_sig(what, run(lambda: c.call('b200rl_conv2d_wgrad_bf16', xd.data_ptr(), 0, dyd.data_ptr(), dw.ptr, None, g, ws.ptr,
                                      ws.bytes, stream())), hg)
  _check(what, dw.read(what), ref, absr, False)
  slabs = ws.slabs(what, K, Cout, splits)
  if splits > 1:   # partial slabs hold dW^T: [(tap, channel)][Cout]
    check_partials(what, slabs, kps, 64, P, lambda lo, hi: tuple(r.reshape(Cout, K).T for r in wr(lo, hi)))
  if P >= 1024:
    for how, lo, hi in drop_ranges(P, 64, splits, kps):
      _assert_rejects(f'{what} without {how}', ref, ref - wr(lo, hi)[0].reshape(Cout, K), absr, False)
  first = dw.bits()
  dw.reset()
  db = Out(1, Cout, False)
  ws.reset()
  assert_sig(what + ' + db', run(lambda: c.call('b200rl_conv2d_wgrad_bf16', xd.data_ptr(), 0, dyd.data_ptr(), dw.ptr, db.ptr, g,
                                                ws.ptr, ws.bytes, stream())), hg + ['colsum_vec_kernel<true>'])
  assert bool((dw.bits() == first).all()), f'{what}: dw changed when db was requested'
  d2 = dy.reshape(-1, Cout)
  _check(what + ' db', db.read(what + ' db')[0], d2.sum(0), np.abs(d2).sum(0), False)


# B, H, C, k, s, Cout, dx_bf16, mask_bf16 (None: no mask), mask_act
CONV_DGRAD = [
    (1, 21, 32, 4, 2, 64, 1, 1, RELU), (6, 21, 32, 4, 2, 64, 0, 0, RELU), (256, 21, 32, 4, 2, 64, 1, 1, RELU),   # conv2
    (6, 20, 32, 4, 2, 64, 1, 0, ELU),                                                                            # even H
    (1, 11, 64, 3, 1, 64, 0, 1, TANH), (6, 11, 64, 3, 1, 64, 1, None, NONE), (256, 11, 64, 3, 1, 64, 1, 1, RELU),  # conv3
    (6, 11, 128, 3, 1, 128, 0, 0, RELU), (6, 13, 64, 4, 2, 128, 1, 1, TANH), (1, 10, 128, 3, 2, 64, 1, 0, RELU),
    (256, 13, 32, 4, 2, 128, 0, 1, ELU),
]


@pytest.mark.parametrize('B,H,C,k,s,Cout,dx_bf16,mask_bf16,ma', CONV_DGRAD)
def test_conv_dgrad_bf16(B, H, C, k, s, Cout, dx_bf16, mask_bf16, ma):
  """one stride-1 sub-problem per stride phase; odd H gives the phases unequal pixel counts"""
  c = _capi()
  rng = np.random.default_rng(B + H + C + Cout + s)
  g, oh, pad = _geom(B, H, C, k, s, Cout)
  w = bf(rng.standard_normal((Cout, k, k, C)) / np.sqrt(k * k * Cout))
  dy = bf(rng.standard_normal((B, oh, oh, Cout)))
  wd, dyd = dev(w, _bf16()), dev(dy, _bf16())
  M = B * H * H
  if mask_bf16 is None:
    mptr, gm, ag = None, 1., 1.
  else:
    ym = mask_values(rng, (M, C), ma)
    ym = bf(ym) if mask_bf16 else ym.astype(np.float32).astype(np.float64)
    mptr = mat_dev(ym, bf16=bool(mask_bf16)).data_ptr()
    gm, ag = mask_factor(ym, ma)
  acc = conv_dgrad_ref(dy, w, k, s, H, oh, pad).reshape(M, C)
  absr = conv_dgrad_ref(np.abs(dy), np.abs(w), k, s, H, oh, pad).reshape(M, C) * ag
  ref = acc * gm
  what = f'conv dgrad B{B} H{H} C{C} k{k} s{s} Cout{Cout} dx {"bf16" if dx_bf16 else "fp32"} mask {mask_bf16} act {ma}'
  dx = Out(M, C, dx_bf16)
  assert_sig(what, run(lambda: c.call('b200rl_conv2d_dgrad_bf16', dyd.data_ptr(), wd.data_ptr(), dx.ptr, dx_bf16, g, mptr,
                                      mask_bf16 or 0, ma, stream())), [f'hconv_dgrad_kernel<{C}>'])
  _check(what, dx.read(what), ref, absr, dx_bf16)
  red = -(-k // s) ** 2 * Cout     # reduction length of the largest stride phase
  if red >= 1024:
    co = np.zeros_like(w)
    co[:64, k // 2, k // 2] = w[:64, k // 2, k // 2]      # one 64-wide k-block: 64 output channels of one tap
    lost = conv_dgrad_ref(dy, co, k, s, H, oh, pad).reshape(M, C)
    _assert_rejects(f'{what} without one 64-wide k-block', ref, (acc - lost) * gm, absr, dx_bf16)


# ------------------------------------------------------------------------------ first layer (uint8 frames, row image)
# B, H, Cout, forward persistent, weight-gradient splits
CONV1_ROWS = [
    (1, 84, 32, False, 1), (5, 84, 32, False, 4), (33, 84, 32, False, 26),
    (171, 84, 32, False, 63),   # 590 tiles: one tile per CTA
    (172, 84, 32, True, 63),    # 593 tiles >= 4 x 148: persistent CTAs with resident weights
    (256, 84, 32, True, 63),    # weight gradient: 64 splits (SPLITK_MAX) rounded to 63
    (512, 84, 32, True, 63),
    (33, 84, 64, False, 26),    # Cout = 64: weights too large to stay resident, never persistent
    (5, 20, 32, False, 1),
]


@pytest.mark.parametrize('B,H,Cout,pers,wsplits', CONV1_ROWS)
def test_conv1_rows_bf16(B, H, Cout, pers, wsplits):
  """First layer on uint8 frames (atari.py:44, atari_wrapper.py:303-304): integer-valued bf16 row image, 1/255 applied to
  the accumulator; forward, weight and bias gradients."""
  import torch
  c = _capi()
  rng = np.random.default_rng(B + H + Cout)
  C, k, s = 4, 8, 4
  g, oh, pad = _geom(B, H, C, k, s, Cout)
  K, M = k * k * C, B * oh * oh
  frames = rng.integers(0, 256, (B, H, H, C), dtype=np.uint8)
  w = bf(rng.standard_normal((Cout, k, k, C)) / np.sqrt(K))
  b = (rng.standard_normal(Cout) * 0.1).astype(np.float32).astype(np.float64)
  x = frames.astype(np.float64) / 255.
  nbytes = int(c.load().b200rl_conv2d_rows_bf16_bytes(ctypes.byref(g)))
  assert nbytes > 0
  rows = torch.empty(nbytes, dtype=torch.uint8, device='cuda')
  c.call('b200rl_conv2d_rows_bf16_from_u8', dev(frames).data_ptr(), g, rows.data_ptr(), nbytes, stream())
  wd, bd = dev(w, _bf16()), dev(b.astype(np.float32))
  ws = Workspace()
  # forward (never split: 8 k-blocks)
  what = f'conv1 fwd B{B} H{H} Cout{Cout}'
  acc = conv_fwd_ref(x, w, k, s, H, oh, pad).reshape(M, Cout)
  absr = conv_fwd_ref(x, np.abs(w), k, s, H, oh, pad).reshape(M, Cout) + np.abs(b)
  y = Out(M, Cout, True)
  want = ['hgemm_pers_kernel<32,0,32,' if pers else f'hgemm_kernel<32,0,0,{Cout},']
  assert_sig(what, run(lambda: c.call('b200rl_conv2d_fwd_bf16', rows.data_ptr(), 1, wd.data_ptr(), bd.data_ptr(), y.ptr, 1, g, RELU,
                                      ws.ptr, ws.bytes, stream())), want)
  _check(what, y.read(what), act(acc + b, RELU), absr, True)
  ws.slabs(what, M, Cout, 1)
  # weight gradient: dy of the bf16 dataflow
  dy = bf(rng.standard_normal((B, oh, oh, Cout)) * (acc.reshape(B, oh, oh, Cout) + b > 0))
  dyd = dev(dy, _bf16())
  plan, kps = split_plan(K, Cout, M, 64, Cout, ws.bytes)
  assert plan == wsplits, f'split rule gives {plan}, the table says {wsplits}'
  what = f'conv1 wgrad B{B} H{H} Cout{Cout}'
  wr = lambda lo, hi: wgrad_range(x, dy, lo, hi, k, s, H, oh, pad, C)
  ref, absr = (r.reshape(Cout, K) for r in wr(0, M))
  hg = [f'hgemm_kernel<64,2,{2 if Cout == 32 else 1},{Cout},'] + (['splitk_finish_kernel'] if wsplits > 1 else [])
  dw, db = Out(Cout, K, False), Out(1, Cout, False)
  ws.reset()
  assert_sig(what, run(lambda: c.call('b200rl_conv2d_wgrad_bf16', rows.data_ptr(), 1, dyd.data_ptr(), dw.ptr, None, g, ws.ptr,
                                      ws.bytes, stream())), hg)
  _check(what, dw.read(what), ref, absr, False)
  slabs = ws.slabs(what, K, Cout, wsplits)
  if wsplits > 1:   # raw integer-pixel sums: the 1/255 is applied when the partials are combined
    check_partials(what, slabs, kps, 64, M, lambda lo, hi: tuple(255. * r.reshape(Cout, K).T for r in wr(lo, hi)))
  if M >= 1024:
    for how, lo, hi in drop_ranges(M, 64, wsplits, kps):
      _assert_rejects(f'{what} without {how}', ref, ref - wr(lo, hi)[0].reshape(Cout, K), absr, False)
  first = dw.bits()
  dw.reset()
  ws.reset()
  assert_sig(what + ' + db', run(lambda: c.call('b200rl_conv2d_wgrad_bf16', rows.data_ptr(), 1, dyd.data_ptr(), dw.ptr, db.ptr, g,
                                                ws.ptr, ws.bytes, stream()), profile=False), hg + ['colsum_vec_kernel<true>'])
  assert bool((dw.bits() == first).all()), f'{what}: dw changed when db was requested'
  d2 = dy.reshape(-1, Cout)
  _check(what + ' db', db.read(what + ' db')[0], d2.sum(0), np.abs(d2).sum(0), False)


def test_conv1_wgrad_unaligned_workspace():
  """A split-K weight gradient of the first layer with a workspace that is only 4-byte aligned: the partial sums take the
  per-element store path, which must still write the raw partials (the 1/255 belongs to the combining pass)."""
  import torch
  c = _capi()
  rng = np.random.default_rng(3)
  B, H, C, k, s, Cout = 33, 84, 4, 8, 4, 32
  g, oh, pad = _geom(B, H, C, k, s, Cout)
  K, M = k * k * C, B * oh * oh
  frames = rng.integers(0, 256, (B, H, H, C), dtype=np.uint8)
  x = frames.astype(np.float64) / 255.
  nbytes = int(c.load().b200rl_conv2d_rows_bf16_bytes(ctypes.byref(g)))
  rows = torch.empty(nbytes, dtype=torch.uint8, device='cuda')
  c.call('b200rl_conv2d_rows_bf16_from_u8', dev(frames).data_ptr(), g, rows.data_ptr(), nbytes, stream())
  dy = bf(rng.standard_normal((B, oh, oh, Cout)))
  ws = Workspace(off=4)
  dw = Out(Cout, K, False)
  assert_sig('conv1 wgrad, unaligned workspace', run(lambda: c.call(
      'b200rl_conv2d_wgrad_bf16', rows.data_ptr(), 1, dev(dy, _bf16()).data_ptr(), dw.ptr, None, g, ws.ptr, ws.bytes, stream())),
      ['hgemm_kernel<64,2,2,32,', 'splitk_finish_kernel'])
  ref, absr = (r.reshape(Cout, K) for r in wgrad_range(x, dy, 0, M, k, s, H, oh, pad, C))
  _check('conv1 wgrad, unaligned workspace', dw.read('conv1 wgrad'), ref, absr, False)
  ws.slabs('conv1 wgrad, unaligned workspace', K, Cout, 26)




def test_fused_head_td_matches_unfused_kernels():
  """b200rl_dqn_head_td == duelling_head_fwd x3 + dqn_td + duelling_head_bwd (dh) bit for bit."""
  import torch
  from acme_b200 import _capi
  rng = np.random.default_rng(8)
  B, A, H = 256, 18, 512
  hs = [np.maximum(rng.standard_normal((B, 2 * H)), 0).astype(np.float32) for _ in range(3)]     # tm1, sel, tgt
  def head():
    return (rng.standard_normal(H).astype(np.float32) * 0.05, rng.standard_normal(1).astype(np.float32),
            rng.standard_normal((A, H)).astype(np.float32) * 0.05, rng.standard_normal(A).astype(np.float32))
  on, tg = head(), head()
  a = rng.integers(0, A, B).astype(np.int32)
  R = rng.choice([-1., 0., 1., 2.5], B).astype(np.float32)
  D = rng.choice([0., 0.9801, 1.0], B).astype(np.float32)
  prob = rng.uniform(1e-7, 1e-3, B).astype(np.float32)
  st = _capi.current_stream()
  f = lambda *s: torch.empty(s, device='cuda')
  hd = [dev(h) for h in hs]
  ond, tgd = [dev(x) for x in on], [dev(x) for x in tg]
  ad, Rd, Dd, pd = dev(a), dev(R), dev(D), dev(prob)
  # unfused reference
  qs = []
  for h, hp in ((hd[0], ond), (hd[2], tgd), (hd[1], ond)):
    q, val, adv = f(B, A), f(B, 1), f(B, A)
    _capi.call('b200rl_duelling_head_fwd', B, A, H, h.data_ptr(), 2 * H, hp[0].data_ptr(), hp[1].data_ptr(), hp[2].data_ptr(),
               hp[3].data_ptr(), val.data_ptr(), adv.data_ptr(), q.data_ptr(), st)
    qs.append(q)
  td, lps, w, pr, dq, lm = f(B), f(B), f(B), f(B), f(B, A), f(1)
  _capi.call('b200rl_dqn_td', B, A, qs[0].data_ptr(), qs[1].data_ptr(), qs[2].data_ptr(), ad.data_ptr(), Rd.data_ptr(), Dd.data_ptr(),
             pd.data_ptr(), 0.99, 1.0, 0.2, 1.0, None, 1.0 / B, td.data_ptr(), lps.data_ptr(), w.data_ptr(), pr.data_ptr(),
             dq.data_ptr(), lm.data_ptr(), 0, st)
  dval, dadv, dh = f(B, 1), f(B, A), f(B, 2 * H)
  gw = [f(H), f(1), f(A, H), f(A)]
  wsbuf = torch.empty(8 << 20, dtype=torch.uint8, device='cuda')
  _capi.call('b200rl_duelling_head_bwd', B, A, H, dq.data_ptr(), hd[0].data_ptr(), 2 * H, ond[0].data_ptr(), ond[2].data_ptr(),
             dval.data_ptr(), dadv.data_ptr(), dh.data_ptr(), 2 * H, gw[0].data_ptr(), gw[1].data_ptr(), gw[2].data_ptr(),
             gw[3].data_ptr(), wsbuf.data_ptr(), wsbuf.numel(), st)
  # fused
  wmax = torch.zeros(1, dtype=torch.float64, device='cuda')
  _capi.call('b200rl_is_weight_max', B, pd.data_ptr(), 0.2, wmax.data_ptr(), 0, st)
  q3 = f(3, B, A)
  td2, lps2, w2, pr2, dq2, dval2, dadv2, dh2 = f(B), f(B), f(B), f(B), f(B, A), f(B, 1), f(B, A), f(B, 2 * H)
  _capi.call('b200rl_dqn_head_td', B, A, H, hd[0].data_ptr(), hd[1].data_ptr(), hd[2].data_ptr(), 2 * H,
             ond[0].data_ptr(), ond[1].data_ptr(), ond[2].data_ptr(), ond[3].data_ptr(),
             tgd[0].data_ptr(), tgd[1].data_ptr(), tgd[2].data_ptr(), tgd[3].data_ptr(),
             ad.data_ptr(), Rd.data_ptr(), Dd.data_ptr(), pd.data_ptr(), 0.99, 1.0, 0.2, 1.0, wmax.data_ptr(), 1.0 / B, 0,
             q3[0].data_ptr(), q3[1].data_ptr(), q3[2].data_ptr(), td2.data_ptr(), lps2.data_ptr(), w2.data_ptr(), pr2.data_ptr(),
             dq2.data_ptr(), dval2.data_ptr(), dadv2.data_ptr(), dh2.data_ptr(), 2 * H, 0, st)
  torch.cuda.synchronize()
  for i in range(3):
    assert torch.equal(q3[i], qs[i]), f'q[{i}]'
  for name, x, y in (('td', td2, td), ('loss', lps2, lps), ('weight', w2, w), ('priority', pr2, pr), ('dq', dq2, dq),
                     ('dval', dval2, dval), ('dadv', dadv2, dadv), ('dh', dh2, dh)):
    assert torch.equal(x, y), name
  # head parameter gradients alone
  gw2 = [f(H), f(1), f(A, H), f(A)]
  _capi.call('b200rl_duelling_head_wgrad', B, A, H, dval2.data_ptr(), dadv2.data_ptr(), hd[0].data_ptr(), 2 * H, gw2[0].data_ptr(),
             gw2[1].data_ptr(), gw2[2].data_ptr(), gw2[3].data_ptr(), wsbuf.data_ptr(), wsbuf.numel(), st)
  mean = f(1)
  _capi.call('b200rl_mean', B, lps2.data_ptr(), mean.data_ptr(), st)
  torch.cuda.synchronize()
  for x, y in zip(gw2, gw):
    assert torch.equal(x, y)
  np.testing.assert_allclose(mean.cpu().numpy()[0], lps.cpu().numpy().astype(np.float64).mean(), rtol=1e-6)


@pytest.mark.parametrize('hw', [84, 20])
def test_gather_rows_equals_gather_plus_conversion(hw):
  """b200rl_replay_gather_rows == b200rl_replay_gather followed by b200rl_conv2d_rows_bf16_from_u8, byte for byte."""
  import ctypes
  import torch
  import helpers
  from acme_b200 import _capi, replay
  rng = np.random.default_rng(hw)
  shape, A, n, B = (hw, hw, 4), 4, 3, 32
  spec, table, server, adder, oracle = helpers.make_pair(shape, np.uint8, A, n, 0.99, 0.6, max_size=200)
  for ep in range(5):
    helpers.feed_episode(rng, adder, oracle, int(rng.integers(5, 30)), n, shape, np.uint8, A)
  table.flush()
  g1, oh, pad = _geom(1, hw, 4, 8, 4, 32)
  g2, _, _ = _geom(2 * B, hw, 4, 8, 4, 32)
  fb = int(_capi.load().b200rl_conv2d_rows_bf16_bytes(ctypes.byref(g1)))
  assert fb > 0 and fb % 128 == 0
  ds = replay.ReplayDataset(table, B, seed=1)
  ds.sample_only(torch.as_tensor(rng.random(B, dtype=np.float32)).cuda())
  rows = torch.zeros(2 * B * fb, dtype=torch.uint8, device='cuda')
  ds.gather_only((rows.data_ptr(), rows.data_ptr() + B * fb, g1))
  torch.cuda.synchronize()
  o_both, R, D, a = ds.o_both.clone(), ds.R.clone(), ds.D.clone(), ds.a_tm1.clone()
  ds.o_both.zero_()
  ds.gather_only()
  want = torch.full((2 * B * fb,), 0xAB, dtype=torch.uint8, device='cuda')
  _capi.call('b200rl_conv2d_rows_bf16_from_u8', ds.o_both.data_ptr(), g2, want.data_ptr(), want.numel(), _capi.current_stream())
  torch.cuda.synchronize()
  assert torch.equal(ds.o_both, o_both) and torch.equal(ds.R, R) and torch.equal(ds.D, D) and torch.equal(ds.a_tm1, a)
  assert torch.equal(rows, want)
  server.stop()


# ------------------------------------------------------------------------------ column sums, fp32 -> bf16
@pytest.mark.parametrize('M,N,ld', [(1, 32, 32), (121, 64, 72), (30976, 64, 64), (112896, 32, 40), (256, 1024, 1032),
                                    (30976, 4, 8)])
def test_colsum_bf16(M, N, ld):
  c = _capi()
  rng = np.random.default_rng(M + N)
  x = bf(rng.standard_normal((M, N)))
  xd = mat_dev(x, ld)
  ws = Workspace()
  out = Out(1, N, False)
  assert_sig(f'colsum {M}x{N}', run(lambda: c.call('b200rl_colsum_bf16', M, N, xd.data_ptr(), ld, out.ptr, ws.ptr, ws.bytes,
                                                   stream())), ['colsum_vec_kernel<true>'])
  _check(f'colsum {M}x{N} ld {ld}', out.read('colsum')[0], x.sum(0), np.abs(x).sum(0), False)


@pytest.mark.parametrize('n', [0, 8, 64, 8_000_000])
def test_bf16_from_f32_rounds_to_nearest_even(n):
  import torch
  c = _capi()
  rng = np.random.default_rng(n)
  src = (rng.standard_normal(n) * np.exp2(rng.integers(-140, 120, n))).astype(np.float32)
  # ties to even (up, down, negative), +-0, subnormals, +-Inf, FLT_MAX -> Inf, NaN; then below-tie, more subnormals, NaNs
  special = np.array([0x3F808000, 0x3F818000, 0x80000000, 0x00000001, 0x7F800000, 0xFF800000, 0x7F7FFFFF, 0x7FC00000,
                      0xBF808000, 0x3F807FFF, 0x00000000, 0x807FFFFF, 0x00408000, 0xFF7FFFFF, 0x7F7F8000, 0x7F800001],
                     np.uint32).view(np.float32)
  src[:min(n, special.size)] = special[:n]
  if not n:    # nothing to convert: no launch, nothing written
    s, out = dev(np.zeros(8, np.float32)), Out(1, 8, True)
    assert_sig('bf16_from_f32 n=0', run(lambda: c.call('b200rl_bf16_from_f32', 0, s.data_ptr(), out.ptr, stream())), [])
    assert bool((out.raw == SENT).all())
    return
  s = dev(src)
  out = Out(1, n, True)
  assert_sig(f'bf16_from_f32 n={n}', run(lambda: c.call('b200rl_bf16_from_f32', n, s.data_ptr(), out.ptr, stream())),
             ['f32_to_bf16_kernel'])
  got = out.read('bf16_from_f32')[0]
  want = torch.from_numpy(src).to(torch.bfloat16).double().numpy()
  nan = np.isnan(want)
  assert (np.isnan(got) == nan).all(), 'NaN-ness differs'
  assert (got[~nan].view(np.uint64) == want[~nan].view(np.uint64)).all(), \
      f'rounding differs at {np.flatnonzero(got[~nan].view(np.uint64) != want[~nan].view(np.uint64))[:8]}'


# ------------------------------------------------------------------------------ shapes outside the kernels
def test_shapes_outside_the_kernels_are_rejected():
  import torch
  c = _capi()
  ws = Workspace(nbytes=1 << 20)
  big = torch.zeros(1 << 20, dtype=torch.bfloat16, device='cuda')
  p = big.data_ptr()
  y = Out(64, 256, False)
  _rejects('linear fwd K < 64', 'b200rl_linear_fwd_bf16', y, 64, 64, 32, p, 32, p, None, y.ptr, 64, 0, RELU, ws.ptr, ws.bytes, None)
  _rejects('linear fwd ldx * 2 % 16 != 0', 'b200rl_linear_fwd_bf16', y, 64, 64, 64, p, 65, p, None, y.ptr, 64, 0, RELU, ws.ptr,
           ws.bytes, None)
  _rejects('linear dgrad K % 64 != 0', 'b200rl_linear_dgrad_bf16', y, 64, 64, 96, p, 64, p, y.ptr, 96, 0, None, 0, 0, ws.ptr,
           ws.bytes, None)
  _rejects('linear wgrad N % 64 != 0', 'b200rl_linear_wgrad_bf16', y, 64, 96, 64, p, 96, p, 64, y.ptr, None, ws.ptr, ws.bytes, None)
  _rejects('colsum N = 100', 'b200rl_colsum_bf16', y, 64, 100, p, 100, y.ptr, ws.ptr, ws.bytes, None)
  _rejects('bf16_from_f32 n % 8 != 0', 'b200rl_bf16_from_f32', y, 12, p, y.ptr, None)
  for what, geo, fn in (('conv fwd C = 16', (2, 11, 16, 3, 1, 64), 'fwd'), ('conv fwd Cout = 48', (2, 11, 64, 3, 1, 48), 'fwd'),
                        ('conv wgrad C = 16', (2, 11, 16, 3, 1, 64), 'wgrad'), ('conv dgrad stride 3', (2, 12, 64, 3, 3, 64), 'dgrad'),
                        ('conv dgrad Cout = 48', (2, 11, 64, 3, 1, 48), 'dgrad')):
    g, _, _ = _geom(*geo)
    if fn == 'fwd':
      _rejects(what, 'b200rl_conv2d_fwd_bf16', y, p, 0, p, None, y.ptr, 1, ctypes.byref(g), RELU, ws.ptr, ws.bytes, None)
    elif fn == 'wgrad':
      _rejects(what, 'b200rl_conv2d_wgrad_bf16', y, p, 0, p, y.ptr, None, ctypes.byref(g), ws.ptr, ws.bytes, None)
    else:
      _rejects(what, 'b200rl_conv2d_dgrad_bf16', y, p, p, y.ptr, 1, ctypes.byref(g), None, 0, 0, None)


# ------------------------------------------------------------------------------ launch ordering
def test_pdl_and_graph_capture_leave_results_bit_identical():
  """fc1 forward -> data gradient -> weight + bias gradient, then conv3 data gradient -> conv2 weight gradient on one
  stream: eager with programmatic dependent launch at its default, eager with it off, and captured in a CUDA graph
  (replayed twice) give the same bits.  Split-K combines its partials in a fixed order.  Then two split-K GEMMs on two
  streams at once, each with its own workspace, equal the two run one after the other."""
  import torch
  c = _capi()
  lib = c.load()
  rng = np.random.default_rng(11)
  M, N, K = 256, 1024, 7744
  x = dev(bf(rng.standard_normal((M, K))), _bf16())
  w = dev(bf(rng.standard_normal((N, K)) / 88.), _bf16())
  b = dev(rng.standard_normal(N).astype(np.float32))
  dy = dev(bf(rng.standard_normal((M, N))), _bf16())
  g3, _, _ = _geom(M, 11, 64, 3, 1, 64)
  g2, _, _ = _geom(M, 21, 32, 4, 2, 64)
  dy3 = dev(bf(rng.standard_normal((M, 11, 11, 64))), _bf16())
  w3 = dev(bf(rng.standard_normal((64, 3, 3, 64)) / 24.), _bf16())
  m3 = dev(bf(np.maximum(rng.standard_normal((M, 11, 11, 64)), 0)), _bf16())
  x2 = dev(bf(np.maximum(rng.standard_normal((M, 21, 21, 32)), 0)), _bf16())
  ws = torch.zeros(WS_BYTES, dtype=torch.uint8, device='cuda')
  outs = dict(y=torch.empty(M, N, dtype=torch.bfloat16, device='cuda'), dx=torch.empty(M, K, dtype=torch.bfloat16, device='cuda'),
              dw=torch.empty(N, K, device='cuda'), db=torch.empty(N, device='cuda'),
              dx3=torch.empty(M, 11, 11, 64, dtype=torch.bfloat16, device='cuda'), dw2=torch.empty(64, 4, 4, 32, device='cuda'),
              db2=torch.empty(64, device='cuda'))
  o = {k: v.data_ptr() for k, v in outs.items()}

  def chain():
    st = stream()
    c.call('b200rl_linear_fwd_bf16', M, N, K, x.data_ptr(), K, w.data_ptr(), b.data_ptr(), o['y'], N, 1, RELU, ws.data_ptr(), WS_BYTES, st)
    c.call('b200rl_linear_dgrad_bf16', M, N, K, dy.data_ptr(), N, w.data_ptr(), o['dx'], K, 1, x.data_ptr(), 1, RELU, ws.data_ptr(),
           WS_BYTES, st)
    c.call('b200rl_linear_wgrad_bf16', M, N, K, dy.data_ptr(), N, x.data_ptr(), K, o['dw'], o['db'], ws.data_ptr(), WS_BYTES, st)
    c.call('b200rl_conv2d_dgrad_bf16', dy3.data_ptr(), w3.data_ptr(), o['dx3'], 1, g3, m3.data_ptr(), 1, RELU, st)
    c.call('b200rl_conv2d_wgrad_bf16', x2.data_ptr(), 0, o['dx3'], o['dw2'], o['db2'], g2, ws.data_ptr(), WS_BYTES, st)

  def snapshot():
    torch.cuda.synchronize()
    res = {k: v.clone() for k, v in outs.items()}
    for v in outs.values():
      v.view(torch.uint8).fill_(SENT)
    return res

  def same(a, bb, what):
    for k in a:
      assert torch.equal(a[k].view(torch.uint8), bb[k].view(torch.uint8)), f'{k} differs: {what}'

  chain()
  ref = snapshot()
  try:
    lib.b200rl_debug_set_pdl(0)
    chain()
    same(ref, snapshot(), 'PDL off vs on')
  finally:
    lib.b200rl_debug_set_pdl(-1)
  graph = torch.cuda.CUDAGraph()
  with torch.cuda.graph(graph):
    chain()
  for i in range(2):
    graph.replay()
    same(ref, snapshot(), f'graph replay {i} vs eager')
  del graph
  # two split-K GEMMs concurrently on two streams
  shapes = ((256, 1024, 7744), (512, 1024, 7744))
  ins = [(dev(bf(rng.standard_normal((m, k))), _bf16()), dev(bf(rng.standard_normal((n, k)) / 88.), _bf16())) for m, n, k in shapes]
  ys = [torch.empty(m, n, device='cuda') for m, n, _ in shapes]
  wss = [torch.empty(WS_BYTES, dtype=torch.uint8, device='cuda') for _ in shapes]

  def gemm(i, st):
    (m, n, k), (xi, wi) = shapes[i], ins[i]
    c.call('b200rl_linear_fwd_bf16', m, n, k, xi.data_ptr(), k, wi.data_ptr(), None, ys[i].data_ptr(), n, 0, NONE, wss[i].data_ptr(),
           WS_BYTES, st)

  for i in range(2):
    gemm(i, stream())
  torch.cuda.synchronize()
  serial = [y.clone() for y in ys]
  for y in ys:
    y.fill_(float('nan'))
  streams = [torch.cuda.Stream() for _ in shapes]
  for i, s in enumerate(streams):
    s.wait_stream(torch.cuda.current_stream())
    gemm(i, s.cuda_stream)
  torch.cuda.synchronize()
  for i in range(2):
    assert torch.equal(ys[i], serial[i]), f'GEMM {shapes[i]} differs when run beside another split-K GEMM'
