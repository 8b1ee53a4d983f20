"""Checks shared by the layer-kernel suites (test_gpu_bf16_layers.py, test_gpu_fp32_layers.py): sentinel-guarded outputs
and workspaces, the per-element error bound against an fp64 reference, launch signatures seen by torch.profiler, and
rejected calls."""
import re

import numpy as np
import pytest

C_ACC = 2.0 ** -16
C_OUT_BF16 = 2.0 ** -8
WS_BYTES = 64 << 20
SENT = 0xFF                 # sentinel byte: 0xFFFF / 0xFFFFFFFF are NaNs no kernel computes
LEAD = 256                  # guard bytes before an output (keeps the output 256-byte aligned)
EINVAL = -1
NONE, RELU, ELU, TANH = 0, 1, 2, 3


def _capi():
  from acme_b200 import _capi as c
  return c


class Out:
  """An output of rows x cols elements (row stride ld) inside a sentinel-filled buffer: LEAD (+ off) guard bytes before
  it, ld - cols padding elements per row and `extra` whole rows after it."""

  def __init__(self, rows, cols, bf16, ld=None, extra=3, off=0):
    import torch
    self.rows, self.cols, self.ld, self.es = rows, cols, ld or cols, 2 if bf16 else 4
    self.lead = LEAD + off
    self.body = rows * self.ld * self.es
    self.raw = torch.full((self.lead + self.body + extra * self.ld * self.es + 64,), SENT, dtype=torch.uint8, device='cuda')
    self.ptr = self.raw.data_ptr() + self.lead

  def reset(self):
    self.raw.fill_(SENT)

  def read(self, what):
    """The logical region as float64; asserts every other byte still holds the sentinel."""
    h = self.raw.cpu().numpy()
    assert (h[:self.lead] == SENT).all() and (h[self.lead + self.body:] == SENT).all(), f'{what}: store outside the output rows'
    body = h[self.lead:self.lead + self.body].view(np.uint16 if self.es == 2 else np.uint32).reshape(self.rows, self.ld)
    assert (body[:, self.cols:] == (0xFFFF if self.es == 2 else 0xFFFFFFFF)).all(), f'{what}: store into the ld padding'
    v = np.ascontiguousarray(body[:, :self.cols])
    if self.es == 2:
      v = (v.astype(np.uint32) << 16).view(np.float32)
    else:
      v = v.view(np.float32)
    return v.astype(np.float64)

  def bits(self):
    return self.raw.clone()


def act(v, a):
  if a == RELU:
    return np.maximum(v, 0.)
  if a == ELU:
    return np.where(v > 0, v, np.expm1(np.minimum(v, 0.)))
  if a == TANH:
    return np.tanh(v)
  return v


def act_grad(y, a):
  """derivative from the activation's OUTPUT y (the mask of a data gradient)"""
  if a == RELU:
    return (y > 0).astype(np.float64)
  if a == ELU:
    return np.where(y > 0, 1., y + 1.)
  if a == TANH:
    return 1. - y * y
  return np.ones_like(y)


def mask_values(rng, shape, a):
  """a plausible producer output for activation `a`"""
  z = rng.standard_normal(shape)
  return np.maximum(z, 0.) if a == RELU else (np.tanh(z) if a == TANH else act(z, ELU))


def mask_factor(y, a):
  """(g, |g| for the bound): the bound carries |A|.|B| * 2^-4 on top of |g| for a computed (non-ReLU) derivative, whose
  fp32 evaluation (1 - y*y, y + 1) is exact only to ~2^-23 absolute"""
  g = act_grad(y, a)
  return g, np.abs(g) + (0. if a == RELU else 2. ** -4)


def _bound(ref, absr, out_bf16, c_acc, op):
  """op = (c_op, |operands| product): the operand term of rows whose operands are rounded by the kernel itself"""
  b = c_acc * absr + (C_OUT_BF16 if out_bf16 else 0.) * np.abs(ref)
  return b if op is None else b + op[0] * op[1]


def _check(what, got, ref, absr, out_bf16, c_acc=C_ACC, op=None):
  got = np.asarray(got, np.float64)
  assert got.shape == ref.shape, (what, got.shape, ref.shape)
  assert np.isfinite(got).all(), f'{what}: {int((~np.isfinite(got)).sum())} non-finite elements'
  err = np.abs(got - ref)
  bound = _bound(ref, absr, out_bf16, c_acc, op)
  acc_err = np.maximum(err - (C_OUT_BF16 * np.abs(ref) if out_bf16 else 0.), 0.)
  ratio = float((acc_err / np.maximum(absr, 1e-300)).max()) if err.size else 0.
  used = float((err / np.maximum(bound, 1e-300)).max()) if err.size else 0.
  print(f'bound {what}: |err|/(|A||B|) {ratio:.2e}, {used:.3f} of the bound')
  bad = err > bound
  if bad.any():
    i = np.unravel_index(int(np.argmax(err - bound)), err.shape)
    raise AssertionError(f'{what}: {int(bad.sum())} of {err.size} elements outside the bound; worst at {i}: got {got[i]!r} '
                         f'want {ref[i]!r} bound {bound[i]:.3e}')
  return ratio


def _assert_rejects(what, ref, broken, absr, out_bf16, c_acc=C_ACC, op=None):
  """the bound must fail a result that lost part of its reduction (by at least 2x somewhere, so the rounding noise of a
  real broken kernel cannot hide it)"""
  bound = _bound(ref, absr, out_bf16, c_acc, op)
  r = float((np.abs(broken - ref) / np.maximum(bound, 1e-300)).max())
  print(f'bound {what}: a broken kernel would exceed the bound {r:.1f}x')
  assert r >= 2., f'{what}: the bound would accept it (worst |diff| / bound = {r:.2f})'
  return r


# ------------------------------------------------------------------------------ launch signature
def _sig_name(name):
  """'void b200rl::k<b200rl::A<false>, b200rl::B, 64>(...)' -> 'k<A<false>,B,64>' (None for kernels of other libraries)"""
  m = re.search(r'b200rl::(\w+)', name)
  if not m:
    return None
  out, i = m.group(1), m.end()
  if i < len(name) and name[i] == '<':
    depth, j = 0, i
    while j < len(name):
      depth += {'<': 1, '>': -1}.get(name[j], 0)
      j += 1
      if depth == 0:
        break
    t = name[i:j].replace(' ', '').replace('b200rl::', '').replace('(bool)0', 'false').replace('(bool)1', 'true')
    out += t.replace('(int)', '')
  return out


def run(fn, profile=True):
  """(launch-count delta, sorted library kernel names seen by torch.profiler) of fn()"""
  import torch
  lib = _capi().load()
  torch.cuda.synchronize()
  if not profile:
    n0 = lib.b200rl_launch_count()
    fn()
    torch.cuda.synchronize()
    return lib.b200rl_launch_count() - n0, None
  from torch.profiler import ProfilerActivity, profile as prof_ctx
  for attempt in range(2):
    with prof_ctx(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
      n0 = lib.b200rl_launch_count()
      fn()
      torch.cuda.synchronize()
      n1 = lib.b200rl_launch_count()
    names = sorted(n for n in (_sig_name(e.name) for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA) if n)
    # a short capture now and then comes back without any device activity at all: capture the (deterministic) call again
    if names or n1 == n0:
      break
  return n1 - n0, names


def assert_sig(what, got, want):
  """want: kernel-name prefixes (template arguments up to BN, STAGES left out), one per launch"""
  launches, names = got
  assert launches == len(want), f'{what}: {launches} launches, expected {len(want)} ({want}); profiler saw {names}'
  if names is not None:
    assert len(names) == len(want) and all(any(n.startswith(w) for n in names) for w in want) and \
        all(any(n.startswith(w) for w in want) for n in names), f'{what}: kernels {names}, expected {want}'


class Workspace:
  """split-K workspace filled with the sentinel: `slabs(M, N)` = the number of leading [M][N] fp32 partial slabs that were
  written completely, asserting that nothing after them was touched"""

  def __init__(self, off=0, nbytes=WS_BYTES, head=0):
    import torch
    self.buf = torch.full((nbytes + off,), SENT, dtype=torch.uint8, device='cuda')
    self.off = off
    self.ptr, self.bytes = self.buf.data_ptr() + off, nbytes
    self.head = head    # bytes in front of the partial slabs (a row map, a row image)

  def reset(self):
    self.buf.fill_(SENT)

  def slabs(self, what, M, N, splits):
    import torch
    words = self.buf[self.off + self.head:self.off + self.bytes // 4 * 4].view(torch.int32)
    n = M * N
    used = splits * n if splits > 1 else 0
    assert not bool((words[used:] != -1).any()), f'{what}: workspace written past {splits} partial slab(s)'
    if splits > 1:
      assert bool((words[:used] != -1).all()), f'{what}: not all of the {splits} expected partial slabs were written'
      return words[:used].view(torch.float32).view(splits, M, N).double().cpu().numpy()
    return None


def _rejects(what, fn_name, out, *args):
  lib = _capi().load()
  n0 = lib.b200rl_launch_count()
  rc = getattr(lib, fn_name)(*args)
  import torch
  torch.cuda.synchronize()
  assert rc == EINVAL, f'{what}: rc {rc}, expected EINVAL'
  assert lib.b200rl_launch_count() == n0, f'{what}: launched a kernel'
  assert bool((out.raw == SENT).all()), f'{what}: output written'
  with pytest.raises(ValueError):
    _capi().check(rc)
