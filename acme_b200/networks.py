"""Q-network / critic / policy modules of the hot path, forward AND hand-written backward, as
sequences of calls into libb200rl (K6).  No autograd, no torch math: torch tensors are memory.

Mirrors (shapes, padding, activation placement, parameter set):
  DQNAtariNetwork   acme/tf/networks/atari.py:36-69 + duelling.py:27-59
  MLPQNetwork       examples/bsuite/run_dqn.py:46-49 (snt.Sequential([Flatten, MLP([50, 50, A])]))
  LayerNormMLP      acme/tf/networks/continuous.py:37-68
  D4PGCritic        multiplexers.py:58-80 + continuous.py:37-68 + distributional.py:36-67
  D4PGPolicy        continuous.py:30-68 + rescaling.py:55-74
Parameters live in ONE flat fp32 device buffer per network (so Adam, target copy and the NCCL
all-reduce are single passes); weights are stored [out][in] (conv: [Cout][kh][kw][Cin]) and are
exported in Sonnet's shapes (conv HWIO, linear [in, out]) by `variables()`.
"""

from __future__ import annotations

import math
from typing import Dict, List, Optional, Tuple

import numpy as np

from acme_b200 import _capi
from acme_b200._capi import ACT_ELU, ACT_NONE, ACT_RELU, ACT_TANH, ConvGeom


def tf_same_pad(size: int, k: int, s: int) -> Tuple[int, int]:
  """TF 'SAME': out = ceil(size/s); pad_before = total // 2 (the remainder goes after)."""
  out = -(-size // s)
  total = max((out - 1) * s + k - size, 0)
  return out, total // 2


def _truncated_normal(rng, shape, std):
  x = rng.standard_normal(shape)
  bad = np.abs(x) > 2
  while bad.any():
    x[bad] = rng.standard_normal(int(bad.sum()))
    bad = np.abs(x) > 2
  return (x * std).astype(np.float32)


class ParamStore:
  """Flat fp32 parameter buffer + named views; gradients / Adam moments mirror the layout."""

  def __init__(self, device: int):
    self.device = device
    self.entries: Dict[str, Tuple[int, Tuple[int, ...]]] = {}
    self.size = 0
    self.flat = None
    self.grad = None
    self.shadow = None

  def declare(self, name: str, shape):
    shape = tuple(int(s) for s in shape)
    self.entries[name] = (self.size, shape)
    n = int(np.prod(shape))
    self.size += -(-n // 8) * 8          # every tensor 32-byte aligned in fp32 and 16-byte aligned in the bf16 shadow

  def allocate(self):
    import torch
    dev = torch.device('cuda', self.device)
    self.flat = torch.zeros(self.size, dtype=torch.float32, device=dev)
    self.grad = torch.zeros(self.size, dtype=torch.float32, device=dev)

  def ensure_shadow(self):
    """bf16 copy of the parameters at the same element offsets (the weight operands of the bf16 dataflow).  Kept in
    step by the optimizer (`b200rl_adam(..., bf16_shadow)`) or `refresh_shadow()` after any other parameter write."""
    import torch
    if self.shadow is None:
      self.shadow = torch.zeros(self.size, dtype=torch.bfloat16, device=self.flat.device)
      self.refresh_shadow()
    return self.shadow

  def refresh_shadow(self, off: int = 0, n: Optional[int] = None):
    if self.shadow is None:
      return
    n = self.size - off if n is None else n
    assert off % 8 == 0 and n % 8 == 0
    _capi.call('b200rl_bf16_from_f32', n, self.flat.data_ptr() + 4 * off, self.shadow.data_ptr() + 2 * off,
               _capi.current_stream())

  def sp(self, name: str) -> int:
    """Device address of `name` in the bf16 shadow."""
    return self.shadow.data_ptr() + 2 * self.entries[name][0]

  def rebind(self, flat, grad):
    """Moves the parameters / gradients into caller-provided storage (the peer-mapped region of
    `parallel.PeerExchange`); call before any CUDA graph that uses them is captured."""
    assert flat.numel() == self.size and grad.numel() == self.size
    flat.copy_(self.flat)
    grad.copy_(self.grad)
    self.flat, self.grad = flat, grad

  def view(self, name: str, grad: bool = False):
    off, shape = self.entries[name]
    n = int(np.prod(shape))
    return (self.grad if grad else self.flat)[off:off + n].view(shape)

  def p(self, name: str) -> int:
    return self.flat.data_ptr() + 4 * self.entries[name][0]

  def g(self, name: str) -> int:
    return self.grad.data_ptr() + 4 * self.entries[name][0]

  def set(self, name: str, value: np.ndarray):
    import torch
    self.view(name).copy_(torch.as_tensor(np.ascontiguousarray(value, dtype=np.float32)))
    if self.shadow is not None:
      self.refresh_shadow()

  def get(self, name: str, grad: bool = False) -> np.ndarray:
    return self.view(name, grad).detach().cpu().numpy().copy()


class Marks:
  """tools/step_phases.py: global-timer stamps issued between kernels (also inside a captured step); name -> slot."""

  def __init__(self, device: int, slots: int = 128):
    import torch
    self.buf = torch.zeros(slots, dtype=torch.int64, device=torch.device('cuda', device))
    self.slots = {}

  def mark(self, name: str):
    import ctypes
    slot = self.slots.setdefault(name, len(self.slots))
    if slot < self.buf.numel():
      _capi.load().b200rl_debug_stamp(ctypes.c_void_p(self.buf.data_ptr()), slot, ctypes.c_void_p(_capi.current_stream()))

  def timeline(self):
    t = self.buf.cpu().numpy()
    ev = sorted((int(t[s]), n) for n, s in self.slots.items() if s < len(t) and t[s] > 0)
    t0 = ev[0][0] if ev else 0
    return [(n, (x - t0) / 1e3) for x, n in ev]


class Network:
  """Common plumbing: parameter store, workspace, precision."""
  marks: Optional[Marks] = None
  mark_prefix = ''

  def _mark(self, name: str):
    if self.marks is not None:
      self.marks.mark(self.mark_prefix + name)

  def __init__(self, device: int = 0, precision: int = _capi.PRECISION_FP32):
    self.device = device
    self.precision = precision
    self.params = ParamStore(device)
    self._ws = None

  @property
  def flow(self) -> bool:
    """precision 2: the bf16 dataflow"""
    return self.precision == _capi.PRECISION_BF16FLOW

  @property
  def x3(self) -> bool:
    """precision 3: fp32 tensors, every layer call through the `*_x3` entry points (split bf16 operands)"""
    return self.precision == _capi.PRECISION_FP32X3

  def _x3_calls(self, B: int):
    """(op, M, N, K, conv geometry, x_u8) of every `*_x3` layer call a pass at batch B makes."""
    raise NotImplementedError

  def _size_lanes(self, B: int):
    """Precision 3: grows the workspace lanes to the largest b200rl_x3_ws_bytes of the layer calls at batch B (in place,
    so that clones sharing the lanes see them).  Other precisions keep their fixed lanes."""
    import ctypes
    import torch
    if not self.x3:
      return
    lib = _capi.load()
    need = 0
    for op, M, N, K, g, x_u8 in self._x3_calls(B):
      n = int(lib.b200rl_x3_ws_bytes(op, M, N, K, ctypes.byref(g) if g is not None else None, x_u8))
      if n < 0:
        raise ValueError(f'precision 3: layer call {op} {(M, N, K)} has a shape no path takes')
      need = max(need, n)
    if need > self._ws_all[0].numel():
      dev = torch.device('cuda', self.device)
      self._ws_all[:] = [torch.empty(need, dtype=torch.uint8, device=dev) for _ in range(3)]

  def _finalize(self):
    import torch
    _capi.require_device(self.device)
    self.params.allocate()
    # one split-K / partial-sum workspace per concurrent stream (see Network.lanes)
    # (precision 3: sized by make_buffers from the layer calls at its batch, see _size_lanes)
    lane_bytes = 0 if self.x3 else 96 << 20
    self._ws_all = [torch.empty(lane_bytes, dtype=torch.uint8, device=torch.device('cuda', self.device)) for _ in range(3)]
    self._lane = 0

  @property
  def ws(self):
    w = self._ws_all[self._lane]
    return w.data_ptr(), w.numel()

  def lane(self, i: int):
    """Selects the workspace used by the following calls; kernels issued on different streams must use
    different lanes (0..2)."""
    self._lane = i
    return self

  def copy_params_from(self, other: 'Network'):
    self.params.flat.copy_(other.params.flat)
    self.params.refresh_shadow()

  def clone(self) -> 'Network':
    """Same architecture, separately stored copy of the parameters (copy.deepcopy(network),
    `acme/agents/tf/dqn/agent.py:127`).  The split-K workspace is shared (same stream)."""
    import copy
    other = copy.copy(self)
    other.params = ParamStore(self.device)
    other.params.entries = dict(self.params.entries)
    other.params.size = self.params.size
    other.params.allocate()
    other.params.flat.copy_(self.params.flat)
    if self.params.shadow is not None:
      other.params.ensure_shadow()
    if hasattr(self, '_rows'):
      other._rows = {}                  # row images are per network (their forwards may run concurrently)
    return other

  # --- Sonnet-shaped export / import (get_variables, checkpoints, parity tests)
  def variables(self, grad: bool = False) -> Dict[str, np.ndarray]:
    out = {}
    for sonnet_name, (name, kind) in self._export.items():
      a = self.params.get(name, grad)
      if kind == 'conv':      # OHWI -> HWIO
        a = a.transpose(1, 2, 3, 0)
      elif isinstance(kind, tuple) and kind[0] == 'conv':   # OHWI with padding input channels -> HWIO of the first kind[1]
        a = a.transpose(1, 2, 3, 0)[:, :, :kind[1], :]
      elif kind == 'linear':  # [out, in] -> [in, out]
        a = a.T
      elif isinstance(kind, tuple) and kind[0] == 'rows':   # rows [lo:hi] of a stacked [out, in]
        a = a[kind[1]:kind[2]].T if a.ndim == 2 else a[kind[1]:kind[2]]
      elif isinstance(kind, tuple) and kind[0] == 'cat':    # [out, in0] and [out, in1] stored apart: one [in0 + in1, out]
        a = np.concatenate([a, self.params.get(kind[1], grad)], axis=1).T
      out[sonnet_name] = np.ascontiguousarray(a)
    return out

  def load_variables(self, variables: Dict[str, np.ndarray]):
    staged: Dict[str, np.ndarray] = {}
    for sonnet_name, (name, kind) in self._export.items():
      v = np.asarray(variables[sonnet_name], np.float32)
      if kind == 'conv':
        staged[name] = v.transpose(3, 0, 1, 2)
      elif isinstance(kind, tuple) and kind[0] == 'conv':
        if v.shape[2] != kind[1]:
          raise ValueError(f'{sonnet_name}: expected {kind[1]} input channels, got shape {v.shape}')
        full = np.zeros(self.params.entries[name][1], np.float32)
        full[..., :kind[1]] = v.transpose(3, 0, 1, 2)
        staged[name] = full
      elif kind == 'linear':
        staged[name] = v.T
      elif isinstance(kind, tuple) and kind[0] == 'rows':
        full = staged.get(name)
        if full is None:
          full = self.params.get(name)
        full[kind[1]:kind[2]] = v.T if full.ndim == 2 else v
        staged[name] = full
      elif isinstance(kind, tuple) and kind[0] == 'cat':
        n0 = self.params.entries[name][1][1]
        staged[name], staged[kind[1]] = v.T[:, :n0], v.T[:, n0:]
      else:
        staged[name] = v
    for name, v in staged.items():
      self.params.set(name, v)


# fp32-tensor layer calls: precisions 0 / 1 through the fp32 entry points, precision 3 through the `*_x3` ones
def _linear(M, N, K, x, ldx, w, b, y, ldy, act, net: Network):
  ws, wsb = net.ws
  if net.x3:
    return _capi.call('b200rl_linear_fwd_x3', M, N, K, x, ldx, w, b, y, ldy, act, ws, wsb, _capi.current_stream())
  _capi.call('b200rl_linear_fwd', M, N, K, x, ldx, w, b, y, ldy, act, net.precision, ws, wsb,
             _capi.current_stream())


def _linear_dgrad(M, N, K, dy, lddy, w, dx, lddx, mask, mask_act, net: Network):
  ws, wsb = net.ws
  if net.x3:
    return _capi.call('b200rl_linear_dgrad_x3', M, N, K, dy, lddy, w, dx, lddx, mask, mask_act, ws, wsb,
                      _capi.current_stream())
  _capi.call('b200rl_linear_dgrad', M, N, K, dy, lddy, w, dx, lddx, mask, mask_act, net.precision, ws,
             wsb, _capi.current_stream())


def _linear_wgrad(M, N, K, dy, lddy, x, ldx, dw, db, net: Network):
  ws, wsb = net.ws
  if net.x3:
    return _capi.call('b200rl_linear_wgrad_x3', M, N, K, dy, lddy, x, ldx, dw, db, ws, wsb, _capi.current_stream())
  _capi.call('b200rl_linear_wgrad', M, N, K, dy, lddy, x, ldx, dw, db, net.precision, ws, wsb,
             _capi.current_stream())


def _conv_fwd(x, x_u8, w, b, y, g, act, net: Network):
  ws, wsb = net.ws
  if net.x3:
    return _capi.call('b200rl_conv2d_fwd_x3', x, x_u8, w, b, y, g, act, ws, wsb, _capi.current_stream())
  _capi.call('b200rl_conv2d_fwd', x, x_u8, w, b, y, g, act, net.precision, ws, wsb, _capi.current_stream())


def _conv_wgrad(x, x_u8, dy, dw, db, g, net: Network):
  ws, wsb = net.ws
  if net.x3:
    return _capi.call('b200rl_conv2d_wgrad_x3', x, x_u8, dy, dw, db, g, ws, wsb, _capi.current_stream())
  _capi.call('b200rl_conv2d_wgrad', x, x_u8, dy, dw, db, g, net.precision, ws, wsb, _capi.current_stream())


def _conv_dgrad(dy, w, dx, g, mask, mask_act, net: Network):
  ws, wsb = net.ws
  if net.x3:
    return _capi.call('b200rl_conv2d_dgrad_x3', dy, w, dx, g, mask, mask_act, ws, wsb, _capi.current_stream())
  _capi.call('b200rl_conv2d_dgrad', dy, w, dx, g, mask, mask_act, net.precision, ws, wsb, _capi.current_stream())


# =============================================================================== AtariTorso convolutions
class _ConvTorso(Network):
  """The AtariTorso convolutions (atari.py:36-52: three SAME-padded convs + ReLU, NHWC): geometry, parameters, row
  images and the layer calls of their forward and backward passes, shared by AtariTorso and DQNAtariNetwork."""

  def _declare_convs(self, input_hw: int, input_channels: int):
    """input_channels C in [1, 16] (4: the grayscale Atari stack; 3: an RGB frame; 3 F: a flattened stack of F RGB frames).
    conv1's filter is stored with Cp >= C input channels, the last Cp - C of them zero.  Precisions 2 and 3: Cp = 4, 8
    or 16, the channel group of the bf16 row image, which is written from the C-channel frames with zero padding
    channels.  Precisions 0 and 1: Cp = C rounded up to 4, the frames padded to Cp channels on the device
    (`b200rl_frames_pad_u8`).  Every padding product is exactly zero.  Their weight gradient is exactly zero too, so those columns stay zero under clip, Adam, the bf16 shadow,
    precision 3's split and the target copy; `variables()` exports and loads only the C real channels."""
    if isinstance(input_channels, bool) or int(input_channels) != input_channels or not 1 <= input_channels <= 16:
      raise ValueError(f'input_channels must be an integer in [1, 16], got {input_channels!r}')
    self.in_hw, self.in_c = input_hw, int(input_channels)
    # the filter's channel count: the bf16 row image's channel group 4, 8 or 16 at precisions 2 and 3 (built from the
    # C-channel frames directly), C rounded up to 4 at precisions 0 and 1 (the frames padded by b200rl_frames_pad_u8)
    c = self.in_c
    self.in_cp = (4 if c <= 4 else 8 if c <= 8 else 16) if self._bf16_rows else -(-c // 4) * 4
    self.convs = []  # (k, stride, cin, cout, in_hw, out_hw, pad); conv1's cin is the padded in_cp
    h, c = input_hw, self.in_cp
    for k, s, co in ((8, 4, 32), (4, 2, 64), (3, 1, 64)):
      oh, pad = tf_same_pad(h, k, s)
      self.convs.append((k, s, c, co, h, oh, pad))
      h, c = oh, co
    self.flat_dim = h * h * c
    for i, (k, s, ci, co, _, _, _) in enumerate(self.convs, 1):
      self.params.declare(f'conv{i}.w', (co, k, k, ci))
      self.params.declare(f'conv{i}.b', (co,))

  def _init_convs(self, rng):
    """Sonnet defaults: TruncatedNormal(stddev=1/sqrt(fan_in)) weights, zero biases."""
    for i, (k, s, ci, co, _, _, _) in enumerate(self.convs, 1):
      c = self.in_c if i == 1 else ci            # conv1: the real fan-in 8 * 8 * C; padding columns stay zero
      w = np.zeros((co, k, k, ci), np.float32)
      w[..., :c] = _truncated_normal(rng, (co, k, k, c), 1 / math.sqrt(k * k * c))
      self.params.set(f'conv{i}.w', w)

  def _conv_export(self, i: int):
    """`_export` kind of conv i's filter: HWIO, conv1's restricted to the frame's real channels."""
    return ('conv', self.in_c) if i == 1 and self.in_c != self.in_cp else 'conv'

  @property
  def pads_frames(self) -> bool:
    """Precisions 0 and 1 on frames whose channel count is not a multiple of 4: uint8 frames are padded to in_cp channels
    before conv1."""
    return self.in_c != self.in_cp and not self._bf16_rows

  def _padded_frames(self, obs, slot: str):
    """uint8 [B, H, W, C] -> the cached [B, H, W, in_cp] copy with zero padding channels (`b200rl_frames_pad_u8`)."""
    import torch
    if obs.dtype != torch.uint8:
      raise ValueError(f'frames with {self.in_c} channels (not a multiple of 4) must be uint8')
    B = obs.shape[0]
    if obs.numel() != B * self.in_hw * self.in_hw * self.in_c:
      raise ValueError(f'expected {B} frames of {self.in_hw} x {self.in_hw} x {self.in_c} bytes, got shape {tuple(obs.shape)}')
    cache = self.__dict__.setdefault('_rows', {})
    key = ('pad', slot, B)
    if key not in cache:
      cache[key] = torch.empty((B, self.in_hw, self.in_hw, self.in_cp), dtype=torch.uint8, device=torch.device('cuda', self.device))
    out = cache[key]
    _capi.call('b200rl_frames_pad_u8', obs.data_ptr(), B * self.in_hw * self.in_hw, self.in_c, self.in_cp, out.data_ptr(),
               _capi.current_stream())
    return out

  @property
  def _bf16_rows(self) -> bool:
    """conv1 reads the bf16 row image (precisions 2 and 3), whose entry points take the frames' own channel count."""
    return self.flow or self.x3

  def geom(self, i: int, B: int) -> ConvGeom:
    k, s, ci, co, h, oh, pad = self.convs[i]
    if i == 0 and self._bf16_rows:
      ci = self.in_c
    return ConvGeom(B=B, H=h, W=h, C=ci, kh=k, kw=k, stride=s, pad_top=pad, pad_left=pad, OH=oh, OW=oh, Cout=co)

  def _conv_x3_calls(self, B: int):
    X = _capi
    calls = []
    for i in range(3):
      g = self.geom(i, B)
      x_u8s = ((1, 2) if self.rows_frame_bytes() else (1,)) if i == 0 else (0,)   # conv1 on uint8 frames or their row image
      calls += [(op, 0, 0, 0, g, u) for u in x_u8s for op in (X.X3_CONV_FWD, X.X3_CONV_WGRAD)]
      if i > 0:
        calls.append((X.X3_CONV_DGRAD, 0, 0, 0, g, 0))
    return calls

  def _torso_forward(self, obs, bufs, rows=None) -> int:
    """The three convolutions: obs -> bufs['y1'..'y3']; returns the address of y3 (post-ReLU, bf16 in the bf16 dataflow).
    obs: uint8 or float32 [B, H, W, C] (NHWC); uint8 is read as float32(x)/255.  `rows`: the frames' row image from
    prepare_frames() (required in the bf16 dataflow; built here if absent)."""
    import torch
    B, P, st = bufs['B'], self.params, _capi.current_stream()
    ws, wsb = self.ws
    if self.flow:
      P.ensure_shadow()
      if rows is None:
        if obs.dtype != torch.uint8:
          raise ValueError('the bf16 dataflow reads uint8 frames')
        rows = self.prepare_frames(obs, 'fwd')
      x, x_rows = rows.data_ptr(), 1
      self._mark(f'fwd{B}.start')
      for i in range(3):
        y = bufs[f'y{i + 1}']
        _capi.call('b200rl_conv2d_fwd_bf16', x, x_rows, P.sp(f'conv{i + 1}.w'), P.p(f'conv{i + 1}.b'), y.data_ptr(), 1,
                   self.geom(i, B), ACT_RELU, ws, wsb, st)
        self._mark(f'fwd{B}.conv{i + 1}')
        x, x_rows = y.data_ptr(), 0
      return x
    if obs.dtype != torch.uint8 and self.in_c != self.in_cp:
      raise ValueError(f'frames of {self.in_c} channels (conv1 padded to {self.in_cp}) must be uint8')
    if rows is None and self.pads_frames:
      rows = self.prepare_frames(obs, 'fwd')
    x, x_u8 = obs.data_ptr(), int(obs.dtype == torch.uint8)
    if rows is not None:              # from prepare_frames(): the frames' row image, or the padded frames (4-D)
      x, x_u8 = rows.data_ptr(), 1 if rows.dim() == 4 else 2
    for i in range(3):
      y = bufs[f'y{i + 1}']
      _conv_fwd(x, x_u8, P.p(f'conv{i + 1}.w'), P.p(f'conv{i + 1}.b'), y.data_ptr(), self.geom(i, B), ACT_RELU, self)
      x, x_u8 = y.data_ptr(), 0
    return x

  def rows_frame_bytes(self) -> int:
    """Bytes of ONE frame in the bf16 row image (precisions 2 and 3): a batched image can be sliced per sample range."""
    import ctypes
    return int(_capi.load().b200rl_conv2d_rows_bf16_bytes(ctypes.byref(self.geom(0, 1)))) if self.flow or self.x3 else 0

  def rows_buffer(self, B: int, slot: str = 'x'):
    """The (cached, zero-initialised) row-image buffer of B frames; None if the geometry has no row image.  Zeroed because
    `b200rl_replay_gather_rows` writes only the frames' interior and relies on the padding staying zero."""
    import ctypes
    import torch
    cache = self.__dict__.setdefault('_rows', {})
    if (slot, B) not in cache:
      lib = _capi.load()
      fn = lib.b200rl_conv2d_rows_bf16_bytes if self.flow or self.x3 else lib.b200rl_conv2d_rows_bytes
      nbytes = int(fn(ctypes.byref(self.geom(0, B))))
      cache[(slot, B)] = (torch.zeros(nbytes, dtype=torch.uint8, device=torch.device('cuda', self.device)) if nbytes > 0 else None)
    return cache[(slot, B)]

  def prepare_frames(self, obs, slot: str = 'x'):
    """uint8 frames -> the row image that first-layer calls accept, built ONCE for all the passes over the same frames
    (two networks on o_t; forward + weight gradient on o_tm1).  Precision 1: zero-padded fp32 rows x/255
    (`b200rl_conv2d_rows_from_u8`); precisions 2 and 3: zero-padded bf16 rows of the integer pixel values
    (`b200rl_conv2d_rows_bf16_from_u8`, exact in bf16).  None when not applicable (fp32 mode, float frames, geometry not eligible):
    callers then pass the frames themselves.  Frames whose channel count is not a multiple of 4 are first padded
    (`_padded_frames`); without a row image the padded frames themselves ([B, H, W, in_cp] uint8) are returned."""
    import torch
    if self.pads_frames:
      obs = self._padded_frames(obs, slot)
    if obs.dtype != torch.uint8:
      return None
    if self.precision == _capi.PRECISION_FP32:
      return obs if self.pads_frames else None
    B = obs.shape[0]
    buf = self.rows_buffer(B, slot)
    if buf is None:
      if self.flow:
        raise ValueError(f'the bf16 dataflow needs the Atari first-layer geometry (kw * C = 32); frames of {self.in_c} '
                         'channels have no row image: use precision 0, 1 or 3')
      return obs if self.pads_frames else None
    name = 'b200rl_conv2d_rows_bf16_from_u8' if self.flow or self.x3 else 'b200rl_conv2d_rows_from_u8'
    _capi.call(name, obs.data_ptr(), self.geom(0, B), buf.data_ptr(), buf.numel(), _capi.current_stream())
    return buf

  def _conv_bias_grad(self, i, bufs, gbufs):
    """bf16 dataflow: db of conv layer i+1 = column sums of dy, as its own launch (so it can sit on another stream)."""
    B, P = bufs['B'], self.params
    ws, wsb = self.ws
    _, _, _, co, _, oh, _ = self.convs[i]
    _capi.call('b200rl_colsum_bf16', B * oh * oh, co, gbufs[f'dy{i + 1}'].data_ptr(), co, P.g(f'conv{i + 1}.b'), ws, wsb,
               _capi.current_stream())

  def _conv_wgrad(self, i, obs, bufs, gbufs, rows, bias: bool = True):
    import torch
    B, P = bufs['B'], self.params
    ws, wsb = self.ws
    g = self.geom(i, B)
    dy = gbufs[f'dy{i + 1}'].data_ptr()
    if self.flow:
      if i > 0:
        x, x_rows = bufs[f'y{i}'].data_ptr(), 0
      else:
        if rows is None:
          rows = self.prepare_frames(obs, 'bwd')
        x, x_rows = rows.data_ptr(), 1
      _capi.call('b200rl_conv2d_wgrad_bf16', x, x_rows, dy, P.g(f'conv{i + 1}.w'), P.g(f'conv{i + 1}.b') if bias else None, g,
                 ws, wsb, _capi.current_stream())
      return
    if i == 0 and rows is None and self.pads_frames:
      rows = self.prepare_frames(obs, 'bwd')
    if i > 0:
      x, x_u8 = bufs[f'y{i}'].data_ptr(), 0
    elif rows is not None:
      x, x_u8 = rows.data_ptr(), 1 if rows.dim() == 4 else 2
    else:
      x, x_u8 = obs.data_ptr(), int(obs.dtype == torch.uint8)
    _conv_wgrad(x, x_u8, dy, P.g(f'conv{i + 1}.w'), P.g(f'conv{i + 1}.b'), g, self)

  def _conv_dgrad(self, i, bufs, gbufs):
    B, P = bufs['B'], self.params
    ws, wsb = self.ws
    g = self.geom(i, B)
    dy = gbufs[f'dy{i + 1}'].data_ptr()
    if self.flow:
      _capi.call('b200rl_conv2d_dgrad_bf16', dy, P.sp(f'conv{i + 1}.w'), gbufs[f'dy{i}'].data_ptr(), 1, g,
                 bufs[f'y{i}'].data_ptr(), 1, ACT_RELU, _capi.current_stream())
    else:
      _conv_dgrad(dy, P.p(f'conv{i + 1}.w'), gbufs[f'dy{i}'].data_ptr(), g, bufs[f'y{i}'].data_ptr(), ACT_RELU, self)


# =============================================================================== DQN Atari network
class DQNAtariNetwork(_ConvTorso):
  """AtariTorso (3 SAME-padded convs + ReLU, NHWC) -> DuellingMLP([512]) (atari.py:36-69)."""

  def __init__(self, num_actions: int, device: int = 0, precision: int = _capi.PRECISION_FP32,
               seed: int = 0, input_hw: int = 84, input_channels: int = 4):
    super().__init__(device, precision)
    self.A = int(num_actions)
    self._declare_convs(input_hw, input_channels)
    P = self.params
    P.declare('fc1.w', (1024, self.flat_dim))   # rows 0..511 value stream, 512..1023 advantage stream
    P.declare('fc1.b', (1024,))
    P.declare('v2.w', (1, 512))
    P.declare('v2.b', (1,))
    P.declare('a2.w', (self.A, 512))
    P.declare('a2.b', (self.A,))
    self._export = {
        'conv1/w': ('conv1.w', self._conv_export(1)), 'conv1/b': ('conv1.b', None),
        'conv2/w': ('conv2.w', 'conv'), 'conv2/b': ('conv2.b', None),
        'conv3/w': ('conv3.w', 'conv'), 'conv3/b': ('conv3.b', None),
        'value/l0/w': ('fc1.w', ('rows', 0, 512)), 'value/l0/b': ('fc1.b', ('rows', 0, 512)),
        'value/l1/w': ('v2.w', 'linear'), 'value/l1/b': ('v2.b', None),
        'adv/l0/w': ('fc1.w', ('rows', 512, 1024)), 'adv/l0/b': ('fc1.b', ('rows', 512, 1024)),
        'adv/l1/w': ('a2.w', 'linear'), 'adv/l1/b': ('a2.b', None),
    }
    self._finalize()
    self.init(seed)

  def init(self, seed: int):
    """Sonnet defaults: TruncatedNormal(stddev=1/sqrt(fan_in)) weights, zero biases."""
    rng = np.random.default_rng(seed)
    P = self.params
    self._init_convs(rng)
    P.set('fc1.w', _truncated_normal(rng, (1024, self.flat_dim), 1 / math.sqrt(self.flat_dim)))
    P.set('v2.w', _truncated_normal(rng, (1, 512), 1 / math.sqrt(512)))
    P.set('a2.w', _truncated_normal(rng, (self.A, 512), 1 / math.sqrt(512)))

  # ---- buffers.  In the bf16 dataflow (precision 2) activations y1..y3 and the back-propagated gradients dh, dy1..dy3
  # are bf16; the hidden row h (consumed by the duelling head in fp32), q, value / advantage and everything the loss
  # touches stay fp32.
  def make_buffers(self, B: int):
    import torch
    dev = torch.device('cuda', self.device)
    f = lambda *shape: torch.empty(shape, dtype=torch.float32, device=dev)
    a = (lambda *shape: torch.empty(shape, dtype=torch.bfloat16, device=dev)) if self.flow else f
    bufs = dict(B=B, q=f(B, self.A), h=f(B, 1024), val=f(B, 1), adv=f(B, self.A))
    for i, (k, s, ci, co, h, oh, pad) in enumerate(self.convs, 1):
      bufs[f'y{i}'] = a(B, oh, oh, co)
    self._size_lanes(B)
    return bufs

  def _x3_calls(self, B: int):
    X = _capi
    return [(X.X3_LINEAR_FWD, B, 1024, self.flat_dim, None, 0), (X.X3_LINEAR_DGRAD, B, 1024, self.flat_dim, None, 0),
            (X.X3_LINEAR_WGRAD, B, 1024, self.flat_dim, None, 0)] + self._conv_x3_calls(B)

  def make_grad_buffers(self, B: int):
    import torch
    dev = torch.device('cuda', self.device)
    f = lambda *shape: torch.empty(shape, dtype=torch.float32, device=dev)
    a = (lambda *shape: torch.empty(shape, dtype=torch.bfloat16, device=dev)) if self.flow else f
    g = dict(dh=a(B, 1024), dval=f(B, 1), dadv=f(B, self.A))
    if self.flow:
      g['dh32'] = f(B, 1024)           # the unfused head backward writes fp32; converted for the bf16 GEMMs
    for i, (k, s, ci, co, h, oh, pad) in enumerate(self.convs, 1):
      g[f'dy{i}'] = a(B, oh, oh, co)
    return g

  def features(self, obs, bufs, before_fc1=None, rows=None):
    """The torso and the first dense layer of both streams: obs -> bufs['h'] (post-ReLU, fp32 [B, 1024]).
    obs: uint8 or float32 [B, H, W, C] (NHWC); uint8 is read as float32(x)/255.  `rows`: the frames' row image from
    prepare_frames() (required in the bf16 dataflow; built here if absent).  `before_fc1` (optional callable) runs after
    the torso has been issued and before the dense layer: the pipelined data-parallel learner makes the stream wait there
    for the fc1 + head parameters, which arrive while the convolutions run."""
    B, P, st = bufs['B'], self.params, _capi.current_stream()
    ws, wsb = self.ws
    x = self._torso_forward(obs, bufs, rows)
    if self.flow:
      if before_fc1 is not None:
        before_fc1()
      _capi.call('b200rl_linear_fwd_bf16', B, 1024, self.flat_dim, x, self.flat_dim, P.sp('fc1.w'), P.p('fc1.b'),
                 bufs['h'].data_ptr(), 1024, 0, ACT_RELU, ws, wsb, st)
      self._mark(f'fwd{B}.fc1')
      return bufs['h']
    if before_fc1 is not None:
      before_fc1()
    h = bufs['h']
    _linear(B, 1024, self.flat_dim, x, self.flat_dim, P.p('fc1.w'), P.p('fc1.b'), h.data_ptr(), 1024, ACT_RELU, self)
    return h

  def head_params(self):
    """(wv, bv, wa, ba) device addresses of the duelling head (fp32 master weights)."""
    P = self.params
    return P.p('v2.w'), P.p('v2.b'), P.p('a2.w'), P.p('a2.b')

  def forward(self, obs, bufs, before_fc1=None, rows=None) -> 'torch.Tensor':
    """features() followed by the duelling head (`duelling.py:37-59`): q [B, A]."""
    P, B = self.params, bufs['B']
    h = self.features(obs, bufs, before_fc1=before_fc1, rows=rows)
    _capi.call('b200rl_duelling_head_fwd', B, self.A, 512, h.data_ptr(), 1024, P.p('v2.w'), P.p('v2.b'), P.p('a2.w'),
               P.p('a2.b'), bufs['val'].data_ptr(), bufs['adv'].data_ptr(), bufs['q'].data_ptr(), _capi.current_stream())
    return bufs['q']

  def _head_backward(self, bufs, gbufs, dq):
    """Unfused duelling-head backward: dval, dadv, dh (masked by relu'(h)) and the head's four parameter gradients."""
    B, P = bufs['B'], self.params
    ws, wsb = self.ws
    dh = gbufs['dh32'] if self.flow else gbufs['dh']
    _capi.call('b200rl_duelling_head_bwd', B, self.A, 512, dq.data_ptr(), bufs['h'].data_ptr(), 1024, P.p('v2.w'), P.p('a2.w'),
               gbufs['dval'].data_ptr(), gbufs['dadv'].data_ptr(), dh.data_ptr(), 1024, P.g('v2.w'), P.g('v2.b'), P.g('a2.w'),
               P.g('a2.b'), ws, wsb, _capi.current_stream())
    if self.flow:
      _capi.call('b200rl_bf16_from_f32', B * 1024, dh.data_ptr(), gbufs['dh'].data_ptr(), _capi.current_stream())

  def head_wgrad(self, bufs, gbufs):
    """The head's parameter gradients from gbufs['dval'] / ['dadv'] (after the fused head + TD kernel)."""
    B, P = bufs['B'], self.params
    ws, wsb = self.ws
    _capi.call('b200rl_duelling_head_wgrad', B, self.A, 512, gbufs['dval'].data_ptr(), gbufs['dadv'].data_ptr(),
               bufs['h'].data_ptr(), 1024, P.g('v2.w'), P.g('v2.b'), P.g('a2.w'), P.g('a2.b'), ws, wsb, _capi.current_stream())

  # layer calls of the backward pass in either dataflow
  def _fc1_bias_grad(self, bufs, gbufs):
    """bf16 dataflow: d fc1.b = column sums of dh, as its own launch."""
    B, P = bufs['B'], self.params
    ws, wsb = self.ws
    _capi.call('b200rl_colsum_bf16', B, 1024, gbufs['dh'].data_ptr(), 1024, P.g('fc1.b'), ws, wsb, _capi.current_stream())

  def _fc1_wgrad(self, bufs, gbufs, bias: bool = True):
    B, P = bufs['B'], self.params
    ws, wsb = self.ws
    if self.flow:
      _capi.call('b200rl_linear_wgrad_bf16', B, 1024, self.flat_dim, gbufs['dh'].data_ptr(), 1024, bufs['y3'].data_ptr(),
                 self.flat_dim, P.g('fc1.w'), P.g('fc1.b') if bias else None, ws, wsb, _capi.current_stream())
    else:
      _linear_wgrad(B, 1024, self.flat_dim, gbufs['dh'].data_ptr(), 1024, bufs['y3'].data_ptr(), self.flat_dim, P.g('fc1.w'),
                    P.g('fc1.b'), self)

  def _fc1_dgrad(self, bufs, gbufs):
    B, P = bufs['B'], self.params
    ws, wsb = self.ws
    if self.flow:
      _capi.call('b200rl_linear_dgrad_bf16', B, 1024, self.flat_dim, gbufs['dh'].data_ptr(), 1024, P.sp('fc1.w'),
                 gbufs['dy3'].data_ptr(), self.flat_dim, 1, bufs['y3'].data_ptr(), 1, ACT_RELU, ws, wsb, _capi.current_stream())
    else:
      _linear_dgrad(B, 1024, self.flat_dim, gbufs['dh'].data_ptr(), 1024, P.p('fc1.w'), gbufs['dy3'].data_ptr(), self.flat_dim,
                    bufs['y3'].data_ptr(), ACT_RELU, self)

  def backward(self, obs, bufs, gbufs, dq, rows=None):
    """Accumulates nothing: overwrites params.grad with d(loss)/d(params) given dq [B, A].  `rows`: the row image of
    `obs` from prepare_frames(), if the caller has one.

    All on the current stream.  backward_dense_part followed by backward_conv_part is the same computation with the
    weight-gradient GEMMs on a side stream, concurrent with the data-gradient chain: the two are independent once a
    layer's dy exists, and each kernel alone is too latency-bound to fill the machine."""
    self._head_backward(bufs, gbufs, dq)
    self.backward_from_dh(obs, bufs, gbufs, rows)

  def backward_from_dh(self, obs, bufs, gbufs, rows=None):
    """fc1's and the torso's gradients from gbufs['dh'] (written by _head_backward or the fused head + TD kernel), on
    the current stream."""
    self._fc1_wgrad(bufs, gbufs)
    self._fc1_dgrad(bufs, gbufs)
    for i in (2, 1, 0):
      self._conv_wgrad(i, obs, bufs, gbufs, rows)
      if i > 0:
        self._conv_dgrad(i, bufs, gbufs)

  def backward_after_head(self, obs, bufs, gbufs, s1, s2, rows=None, on_dense_done=None):
    """Everything behind the fused head + TD kernel (which has produced gbufs['dh'] / ['dval'] / ['dadv']), scheduled on
    three streams: the data-gradient chain fc1 -> conv3 -> conv2 (+ conv1's weight gradient) on the current stream, the
    weight-gradient GEMMs on `s1`, the head's parameter gradients and (bf16 dataflow) the bias-gradient column sums on
    `s2`.  Workspace lanes 0 / 1 / 2.  `on_dense_done(event_list)` is called once fc1's and the head's gradients and fc1's
    data gradient (the last reader of fc1's weights) have been issued, with the events that mark their completion: a
    caller may start the optimizer update of that bucket there, underneath the convolution backward."""
    import torch
    main = torch.cuda.current_stream()
    flow = self.flow

    def fork(*streams):
      ev = torch.cuda.Event()
      ev.record(main)
      for st in streams:
        st.wait_event(ev)

    self._mark('bwd.start')
    fork(s1, s2)
    with torch.cuda.stream(s1):
      self.lane(1)
      self._fc1_wgrad(bufs, gbufs, bias=not flow)
      self._mark('bwd.s1.fc1_wgrad')
      ev_w = torch.cuda.Event()
      ev_w.record(s1)
    with torch.cuda.stream(s2):
      self.lane(2)
      self.head_wgrad(bufs, gbufs)
      if flow:
        self._fc1_bias_grad(bufs, gbufs)
      self._mark('bwd.s2.head_wgrad+fc1_db')
      ev_h = torch.cuda.Event()
      ev_h.record(s2)
    self.lane(0)
    self._fc1_dgrad(bufs, gbufs)
    self._mark('bwd.fc1_dgrad')
    if on_dense_done is not None:
      # fc1's data gradient READS fc1's weights: an optimizer update of that bucket must wait for it too
      ev_d = torch.cuda.Event()
      ev_d.record(main)
      on_dense_done([ev_w, ev_h, ev_d])
    for i in (2, 1):
      fork(s1, s2) if flow else fork(s1)
      with torch.cuda.stream(s1):
        self.lane(1)
        self._conv_wgrad(i, obs, bufs, gbufs, rows, bias=not flow)
        self._mark(f'bwd.s1.conv{i + 1}_wgrad')
      if flow:
        with torch.cuda.stream(s2):
          self.lane(2)
          self._conv_bias_grad(i, bufs, gbufs)
          self._mark(f'bwd.s2.conv{i + 1}_db')
      self.lane(0)
      self._conv_dgrad(i, bufs, gbufs)
      self._mark(f'bwd.conv{i + 1}_dgrad')
    if flow:
      fork(s2)
      with torch.cuda.stream(s2):
        self.lane(2)
        self._conv_bias_grad(0, bufs, gbufs)
    self.lane(0)
    self._conv_wgrad(0, obs, bufs, gbufs, rows, bias=not flow)
    self._mark('bwd.conv1_wgrad')
    for st in (s1, s2):
      ev = torch.cuda.Event()
      ev.record(st)
      main.wait_event(ev)

  def grad_buckets(self):
    """(offset, count) in floats of the gradient regions that become final after backward_dense_part
    (fc1 + heads: the tail of the flat buffer, 99% of the bytes) and after backward_conv_part (the convs)."""
    split = self.params.entries['fc1.w'][0]
    return (split, self.params.size - split), (0, split)

  def backward_dense_part(self, bufs, gbufs, dq, side):
    """Duelling head + fc1: parameter gradients of everything after the torso, and dy3.  dq = None: the fused head + TD
    kernel has already produced gbufs['dh'] / ['dval'] / ['dadv']; only the head's parameter gradients remain (side)."""
    import torch
    main = torch.cuda.current_stream()
    self.lane(0)
    if dq is not None:
      self._head_backward(bufs, gbufs, dq)
    ev = torch.cuda.Event()
    ev.record(main)
    side.wait_event(ev)
    with torch.cuda.stream(side):
      self.lane(1)
      if dq is None:
        self.head_wgrad(bufs, gbufs)
      self._fc1_wgrad(bufs, gbufs)
    self.lane(0)
    self._fc1_dgrad(bufs, gbufs)
    ev = torch.cuda.Event()
    ev.record(side)
    main.wait_event(ev)

  def backward_conv_part(self, obs, bufs, gbufs, side, rows=None):
    """The three convolutions: weight gradients on `side`, data gradients on the current stream."""
    import torch
    main = torch.cuda.current_stream()
    for i in (2, 1, 0):
      if i > 0:
        ev = torch.cuda.Event()
        ev.record(main)
        side.wait_event(ev)
        with torch.cuda.stream(side):
          self.lane(1)
          self._conv_wgrad(i, obs, bufs, gbufs, rows)
        self.lane(0)
        self._conv_dgrad(i, bufs, gbufs)
      else:   # conv1 has no data gradient: its weight gradient finishes the main chain
        if self.flow:   # ... and its bias gradient runs beside it
          ev = torch.cuda.Event()
          ev.record(main)
          side.wait_event(ev)
          with torch.cuda.stream(side):
            self.lane(1)
            self._conv_bias_grad(0, bufs, gbufs)
          self.lane(0)
        self._conv_wgrad(0, obs, bufs, gbufs, rows, bias=not self.flow)
    ev = torch.cuda.Event()
    ev.record(side)
    main.wait_event(ev)
    self.lane(0)


# =============================================================================== AtariTorso as an observation network
class AtariTorso(_ConvTorso):
  """AtariTorso (atari.py:36-52): three SAME-padded convolutions with ReLU, flattened in (H, W, C) order to `flat_dim`
  (7744 at 84 x 84) features.  The observation network of D4PG / DDPG from pixels (d4pg/learning.py:189-195): its
  output feeds the policy and the critic, whose first layers read it directly.  Features are fp32 at precisions 0, 1 and
  3, bf16 at precision 2 (the bf16 dataflow, which reads uint8 frames)."""

  def __init__(self, device: int = 0, precision: int = _capi.PRECISION_FP32, seed: int = 0, input_hw: int = 84,
               input_channels: int = 4):
    super().__init__(device, precision)
    self._declare_convs(input_hw, input_channels)
    self._export = {}
    for i in range(1, 4):
      self._export[f'conv{i}/w'] = (f'conv{i}.w', self._conv_export(i))
      self._export[f'conv{i}/b'] = (f'conv{i}.b', None)
    self._finalize()
    self._init_convs(np.random.default_rng(seed))
    if self.flow:
      self.params.ensure_shadow()

  def make_buffers(self, B: int):
    import torch
    dev = torch.device('cuda', self.device)
    dt = torch.bfloat16 if self.flow else torch.float32
    bufs = dict(B=B)
    for i, (k, s, ci, co, h, oh, pad) in enumerate(self.convs, 1):
      bufs[f'y{i}'] = torch.empty((B, oh, oh, co), dtype=dt, device=dev)
    self._size_lanes(B)
    return bufs

  def make_grad_buffers(self, B: int):
    import torch
    dev = torch.device('cuda', self.device)
    dt = torch.bfloat16 if self.flow else torch.float32
    return {f'dy{i}': torch.empty((B, oh, oh, co), dtype=dt, device=dev)
            for i, (k, s, ci, co, h, oh, pad) in enumerate(self.convs, 1)}

  def _x3_calls(self, B: int):
    return self._conv_x3_calls(B)

  def forward(self, obs, bufs, rows=None):
    """obs [B, H, W, C] -> the features bufs['y3'] [B, OH, OW, 64] (read as [B, flat_dim])."""
    self._torso_forward(obs, bufs, rows)
    return bufs['y3']

  def backward(self, obs, bufs, gbufs, rows=None):
    """Overwrites params.grad from gbufs['dy3'], the gradient w.r.t. conv3's pre-activation (the caller's data gradient
    of the features, already masked by conv3's ReLU): conv3 and conv2 data gradients and the three weight gradients."""
    for i in (2, 1, 0):
      self._conv_wgrad(i, obs, bufs, gbufs, rows)
      if i > 0:
        self._conv_dgrad(i, bufs, gbufs)


# =============================================================================== plain MLP Q-net
class MLPQNetwork(Network):
  """snt.Sequential([snt.Flatten(), snt.nets.MLP(sizes)]) with ReLU between layers."""

  def __init__(self, input_dim: int, sizes, device: int = 0, precision: int = _capi.PRECISION_FP32, seed: int = 0):
    super().__init__(device, precision)
    self.in_dim = int(input_dim)
    self.sizes = [int(s) for s in sizes]
    self.A = self.sizes[-1]
    d = self.in_dim
    self._export = {}
    for i, hdim in enumerate(self.sizes):
      self.params.declare(f'l{i}.w', (hdim, d))
      self.params.declare(f'l{i}.b', (hdim,))
      self._export[f'l{i}/w'] = (f'l{i}.w', 'linear')
      self._export[f'l{i}/b'] = (f'l{i}.b', None)
      d = hdim
    self._finalize()
    rng = np.random.default_rng(seed)
    d = self.in_dim
    for i, hdim in enumerate(self.sizes):
      self.params.set(f'l{i}.w', _truncated_normal(rng, (hdim, d), 1 / math.sqrt(d)))
      d = hdim

  def make_buffers(self, B: int):
    import torch
    dev = torch.device('cuda', self.device)
    bufs = dict(B=B)
    for i, hdim in enumerate(self.sizes):
      bufs[f'y{i}'] = torch.empty((B, hdim), dtype=torch.float32, device=dev)
    bufs['q'] = bufs[f'y{len(self.sizes) - 1}']
    self._size_lanes(B)
    return bufs

  def _x3_calls(self, B: int):
    dims = [self.in_dim] + self.sizes
    return [(op, B, dims[i + 1], dims[i], None, 0) for i in range(len(self.sizes))
            for op in (_capi.X3_LINEAR_FWD, _capi.X3_LINEAR_DGRAD, _capi.X3_LINEAR_WGRAD)]

  def make_grad_buffers(self, B: int):
    import torch
    dev = torch.device('cuda', self.device)
    return {f'dy{i}': torch.empty((B, hdim), dtype=torch.float32, device=dev) for i, hdim in enumerate(self.sizes)}

  def forward(self, obs, bufs):
    import torch
    if obs.dtype != torch.float32:
      raise ValueError('MLPQNetwork expects float32 observations')
    B, P = bufs['B'], self.params
    x, d = obs.data_ptr(), self.in_dim
    n = len(self.sizes)
    for i, hdim in enumerate(self.sizes):
      y = bufs[f'y{i}']
      _linear(B, hdim, d, x, d, P.p(f'l{i}.w'), P.p(f'l{i}.b'), y.data_ptr(), hdim,
              ACT_RELU if i + 1 < n else ACT_NONE, self)
      x, d = y.data_ptr(), hdim
    return bufs['q']

  def backward(self, obs, bufs, gbufs, dq):
    B, P = bufs['B'], self.params
    n = len(self.sizes)
    dy = dq.data_ptr()
    for i in range(n - 1, -1, -1):
      hdim = self.sizes[i]
      d = self.sizes[i - 1] if i > 0 else self.in_dim
      x = bufs[f'y{i - 1}'].data_ptr() if i > 0 else obs.data_ptr()
      _linear_wgrad(B, hdim, d, dy, hdim, x, d, P.g(f'l{i}.w'), P.g(f'l{i}.b'), self)
      if i > 0:
        dx = gbufs[f'dy{i - 1}'].data_ptr()
        _linear_dgrad(B, hdim, d, dy, hdim, P.p(f'l{i}.w'), dx, d, x, ACT_RELU, self)
        dy = dx


# =============================================================================== D4PG networks
class LayerNormMLP(Network):
  """Linear -> LayerNorm -> tanh -> [Linear -> ELU]* -> optional linear head (continuous.py:37-68).

  Precision 2 (bf16 dataflow): the first layer (K = the input width, whose bf16 rows are not 16-byte multiples) and its
  LayerNorm stay fp32; the LayerNorm also writes a bf16 copy of y0.  The hidden ELU layers read bf16 activations and the
  bf16 weight shadow and pass bf16 gradients back (tcgen05 kind::f16); the head's forward is a bf16 GEMM with an fp32
  output, its backward one `b200rl_dense_head_bwd_bf16` launch.  Weight gradients, biases and the master weights are fp32.
  """
  act_in = 0     # width of the first layer's separate action block (split_action_input), 0: none

  def __init__(self, input_dim: int, sizes, head_dim: int, head_name: str, head_scale: Optional[float],
               device: int, precision: int, seed: int):
    super().__init__(device, precision)
    self.in_dim, self.sizes, self.head_dim, self.head = int(input_dim), [int(s) for s in sizes], int(head_dim), head_name
    if self.flow:
      self._check_bf16_shapes()
    P = self.params
    d = self.in_dim
    self._export = {}
    for i, hdim in enumerate(self.sizes):
      P.declare(f'l{i}.w', (hdim, d))
      P.declare(f'l{i}.b', (hdim,))
      self._export[f'l{i}/w'] = (f'l{i}.w', 'linear')
      self._export[f'l{i}/b'] = (f'l{i}.b', None)
      if i == 0:
        P.declare('ln.scale', (hdim,))
        P.declare('ln.offset', (hdim,))
        self._export['ln/scale'] = ('ln.scale', None)
        self._export['ln/offset'] = ('ln.offset', None)
      d = hdim
    P.declare(f'{head_name}.w', (self.head_dim, d))
    P.declare(f'{head_name}.b', (self.head_dim,))
    self._export[f'{head_name}/w'] = (f'{head_name}.w', 'linear')
    self._export[f'{head_name}/b'] = (f'{head_name}.b', None)
    self._finalize()
    rng = np.random.default_rng(seed)
    d = self.in_dim
    for i, hdim in enumerate(self.sizes):
      lim = math.sqrt(3.0 * 0.333 / hdim)   # VarianceScaling(0.333, 'fan_out', 'uniform')
      P.set(f'l{i}.w', rng.uniform(-lim, lim, (hdim, d)).astype(np.float32))
      d = hdim
    P.set('ln.scale', np.ones(self.sizes[0], np.float32))
    if head_scale is None:
      P.set(f'{head_name}.w', _truncated_normal(rng, (self.head_dim, d), 1 / math.sqrt(d)))
    else:  # NearZeroInitializedLinear: VarianceScaling(scale) -> truncated normal over fan_in
      P.set(f'{head_name}.w', _truncated_normal(rng, (self.head_dim, d), math.sqrt(head_scale / d) / .87962566103423978))
    if self.flow:
      P.ensure_shadow()

  def _check_bf16_shapes(self):
    """The shapes the bf16 entry points accept (b200rl.h), checked before anything is allocated."""
    s = self.sizes
    if len(s) < 2:
      raise ValueError(f'precision 2 needs at least two hidden layers (the head reads a bf16 ELU layer); sizes = {s}')
    if s[0] % 64 != 0:
      raise ValueError(f'precision 2 needs the first hidden size to be a multiple of 64 (the K of the bf16 GEMMs); sizes = {s}')
    if any(h < 64 or h > 1024 or h & (h - 1) for h in s[1:]):
      raise ValueError(f'precision 2 needs hidden sizes after the first to be powers of two in [64, 1024] (bf16 GEMM N and '
                       f'the bf16 bias column sum); sizes = {s}')
    if not 1 <= self.head_dim <= 64:
      raise ValueError(f'precision 2 needs a head of 1 to 64 outputs (b200rl_dense_head_bwd_bf16); head_dim = {self.head_dim}')

  def make_buffers(self, B: int):
    import torch
    dev = torch.device('cuda', self.device)
    f = lambda *shape: torch.empty(shape, dtype=torch.float32, device=dev)
    h0 = self.sizes[0]
    bufs = dict(B=B, x=f(B, self.in_dim), z0=f(B, h0), y0=f(B, h0), xhat=f(B, h0), rstd=f(B), out=f(B, self.head_dim))
    a = (lambda *shape: torch.empty(shape, dtype=torch.bfloat16, device=dev)) if self.flow else f
    if self.flow:
      bufs['y0_bf16'] = a(B, h0)
    for i in range(1, len(self.sizes)):
      bufs[f'y{i}'] = a(B, self.sizes[i])
    self._size_lanes(B)
    return bufs

  def _x3_calls(self, B: int):
    dims = [self.in_dim] + self.sizes + [self.head_dim]
    return [(op, B, dims[i + 1], dims[i], None, 0) for i in range(len(dims) - 1)
            for op in (_capi.X3_LINEAR_FWD, _capi.X3_LINEAR_DGRAD, _capi.X3_LINEAR_WGRAD)]

  def make_grad_buffers(self, B: int):
    import torch
    dev = torch.device('cuda', self.device)
    f = lambda *shape: torch.empty(shape, dtype=torch.float32, device=dev)
    a = (lambda *shape: torch.empty(shape, dtype=torch.bfloat16, device=dev)) if self.flow else f
    g = dict(dz0=f(B, self.sizes[0]), dx=f(B, self.in_dim))
    if self.act_in:
      g['da'] = f(B, self.act_in)
    if self.flow:
      g['dz0_bf16'] = a(B, self.sizes[0])
    for i in range(len(self.sizes)):
      g[f'dy{i}'] = a(B, self.sizes[i]) if i > 0 else f(B, self.sizes[i])   # dy0 feeds the fp32 LayerNorm backward
    return g

  def _hidden_forward(self, bufs):
    """The layers after the first one's LayerNorm + tanh (bufs['y0'], or ['y0_bf16'] in the bf16 dataflow): the ELU
    layers and the head -> bufs['out']."""
    B, P, st = bufs['B'], self.params, _capi.current_stream()
    ws, wsb = self.ws
    h0 = self.sizes[0]
    if self.flow:
      x, d = bufs['y0_bf16'].data_ptr(), h0
      for i in range(1, len(self.sizes)):
        y = bufs[f'y{i}']
        _capi.call('b200rl_linear_fwd_bf16', B, self.sizes[i], d, x, d, P.sp(f'l{i}.w'), P.p(f'l{i}.b'), y.data_ptr(),
                   self.sizes[i], 1, ACT_ELU, ws, wsb, st)
        x, d = y.data_ptr(), self.sizes[i]
      _capi.call('b200rl_linear_fwd_bf16', B, self.head_dim, d, x, d, P.sp(f'{self.head}.w'), P.p(f'{self.head}.b'),
                 bufs['out'].data_ptr(), self.head_dim, 0, ACT_NONE, ws, wsb, st)
      return bufs['out']
    x, d = bufs['y0'].data_ptr(), h0
    for i in range(1, len(self.sizes)):
      y = bufs[f'y{i}']
      _linear(B, self.sizes[i], d, x, d, P.p(f'l{i}.w'), P.p(f'l{i}.b'), y.data_ptr(), self.sizes[i], ACT_ELU, self)
      x, d = y.data_ptr(), self.sizes[i]
    _linear(B, self.head_dim, d, x, d, P.p(f'{self.head}.w'), P.p(f'{self.head}.b'), bufs['out'].data_ptr(),
            self.head_dim, ACT_NONE, self)
    return bufs['out']

  def _hidden_backward(self, bufs, gbufs, dout_ptr: int, param_grads: bool) -> int:
    """Backward through the head and the ELU layers: returns the address of dy0, the fp32 gradient w.r.t. y0."""
    B, P, st = bufs['B'], self.params, _capi.current_stream()
    ws, wsb = self.ws
    n = len(self.sizes)
    d_last = self.sizes[-1]
    if self.flow:
      last = bufs[f'y{n - 1}'].data_ptr()
      dy = gbufs[f'dy{n - 1}'].data_ptr()
      _capi.call('b200rl_dense_head_bwd_bf16', B, self.head_dim, d_last, dout_ptr, self.head_dim, last, d_last,
                 P.sp(f'{self.head}.w'), dy, d_last, last, ACT_ELU, P.g(f'{self.head}.w') if param_grads else None,
                 P.g(f'{self.head}.b') if param_grads else None, ws, wsb, st)
      for i in range(n - 1, 0, -1):
        hdim, d = self.sizes[i], self.sizes[i - 1]
        x = bufs[f'y{i - 1}'].data_ptr() if i > 1 else bufs['y0_bf16'].data_ptr()
        if param_grads:
          _capi.call('b200rl_linear_wgrad_bf16', B, hdim, d, dy, hdim, x, d, P.g(f'l{i}.w'), P.g(f'l{i}.b'), ws, wsb, st)
        dx = gbufs[f'dy{i - 1}'].data_ptr()
        # into y0 (tanh(LN(.)), handled by the fp32 LayerNorm backward): fp32, no mask
        _capi.call('b200rl_linear_dgrad_bf16', B, hdim, d, dy, hdim, P.sp(f'l{i}.w'), dx, d, int(i > 1), x if i > 1 else None,
                   1, ACT_ELU, ws, wsb, st)
        dy = dx
      return dy
    last = bufs[f'y{n - 1}'] if n > 1 else bufs['y0']
    if param_grads:
      _linear_wgrad(B, self.head_dim, d_last, dout_ptr, self.head_dim, last.data_ptr(), d_last,
                    P.g(f'{self.head}.w'), P.g(f'{self.head}.b'), self)
    dy = gbufs[f'dy{n - 1}'].data_ptr()
    _linear_dgrad(B, self.head_dim, d_last, dout_ptr, self.head_dim, P.p(f'{self.head}.w'), dy, d_last,
                  last.data_ptr(), ACT_ELU if n > 1 else ACT_NONE, self)
    for i in range(n - 1, 0, -1):
      hdim, d = self.sizes[i], self.sizes[i - 1]
      x = bufs[f'y{i - 1}']
      if param_grads:
        _linear_wgrad(B, hdim, d, dy, hdim, x.data_ptr(), d, P.g(f'l{i}.w'), P.g(f'l{i}.b'), self)
      dx = gbufs[f'dy{i - 1}'].data_ptr()
      # y_{i-1} is ELU output for i-1 >= 1; for i-1 == 0 it is tanh(LN(.)), handled by the LN backward
      _linear_dgrad(B, hdim, d, dy, hdim, P.p(f'l{i}.w'), dx, d, x.data_ptr() if i - 1 >= 1 else None,
                    ACT_ELU, self)
      dy = dx
    return dy

  def _forward_flat_bf16(self, x_ptr: int, bufs):
    B, P, st = bufs['B'], self.params, _capi.current_stream()
    ws, wsb = self.ws
    h0 = self.sizes[0]
    _capi.call('b200rl_linear_fwd', B, h0, self.in_dim, x_ptr, self.in_dim, P.p('l0.w'), P.p('l0.b'), bufs['z0'].data_ptr(), h0,
               ACT_NONE, _capi.PRECISION_TC, ws, wsb, st)
    _capi.call('b200rl_layernorm_tanh_fwd_bf16', B, h0, bufs['z0'].data_ptr(), P.p('ln.scale'), P.p('ln.offset'), 1e-5,
               bufs['y0'].data_ptr(), bufs['y0_bf16'].data_ptr(), bufs['xhat'].data_ptr(), bufs['rstd'].data_ptr(), st)
    return self._hidden_forward(bufs)

  def _backward_flat_bf16(self, x_ptr: int, bufs, gbufs, dout_ptr: int, param_grads: bool, input_grad: bool):
    B, P, st = bufs['B'], self.params, _capi.current_stream()
    ws, wsb = self.ws
    dy = self._hidden_backward(bufs, gbufs, dout_ptr, param_grads)
    h0 = self.sizes[0]
    _capi.call('b200rl_layernorm_tanh_bwd', B, h0, dy, bufs['y0'].data_ptr(), bufs['xhat'].data_ptr(),
               bufs['rstd'].data_ptr(), P.p('ln.scale'), gbufs['dz0'].data_ptr(),
               P.g('ln.scale') if param_grads else None, P.g('ln.offset') if param_grads else None, st)
    dz0 = gbufs['dz0'].data_ptr()
    if param_grads:
      _capi.call('b200rl_linear_wgrad', B, h0, self.in_dim, dz0, h0, x_ptr, self.in_dim, P.g('l0.w'), P.g('l0.b'),
                 _capi.PRECISION_TC, ws, wsb, st)
    if input_grad:
      _capi.call('b200rl_linear_dgrad', B, h0, self.in_dim, dz0, h0, P.p('l0.w'), gbufs['dx'].data_ptr(), self.in_dim, None,
                 ACT_NONE, _capi.PRECISION_TC, ws, wsb, st)

  def forward_flat(self, x_ptr: int, bufs):
    if self.flow:
      return self._forward_flat_bf16(x_ptr, bufs)
    B, P, st = bufs['B'], self.params, _capi.current_stream()
    h0 = self.sizes[0]
    _linear(B, h0, self.in_dim, x_ptr, self.in_dim, P.p('l0.w'), P.p('l0.b'), bufs['z0'].data_ptr(), h0, ACT_NONE, self)
    _capi.call('b200rl_layernorm_tanh_fwd', B, h0, bufs['z0'].data_ptr(), P.p('ln.scale'), P.p('ln.offset'), 1e-5,
               bufs['y0'].data_ptr(), bufs['xhat'].data_ptr(), bufs['rstd'].data_ptr(), st)
    return self._hidden_forward(bufs)

  def backward_flat(self, x_ptr: int, bufs, gbufs, dout_ptr: int, param_grads: bool = True, input_grad: bool = False):
    """dout: gradient w.r.t. the head output.  Writes params.grad (if param_grads) and gbufs['dx']
    (if input_grad)."""
    if self.flow:
      return self._backward_flat_bf16(x_ptr, bufs, gbufs, dout_ptr, param_grads, input_grad)
    B, P, st = bufs['B'], self.params, _capi.current_stream()
    dy = self._hidden_backward(bufs, gbufs, dout_ptr, param_grads)
    h0 = self.sizes[0]
    _capi.call('b200rl_layernorm_tanh_bwd', B, h0, dy, bufs['y0'].data_ptr(), bufs['xhat'].data_ptr(),
               bufs['rstd'].data_ptr(), P.p('ln.scale'), gbufs['dz0'].data_ptr(),
               P.g('ln.scale') if param_grads else None, P.g('ln.offset') if param_grads else None, st)
    dz0 = gbufs['dz0'].data_ptr()
    if param_grads:
      _linear_wgrad(B, h0, self.in_dim, dz0, h0, x_ptr, self.in_dim, P.g('l0.w'), P.g('l0.b'), self)
    if input_grad:
      _linear_dgrad(B, h0, self.in_dim, dz0, h0, P.p('l0.w'), gbufs['dx'].data_ptr(), self.in_dim, None, ACT_NONE, self)

  # ---- over observation-network features (d4pg/learning.py:189-195): the first layer's feature block is a GEMM on the
  # features as the observation network wrote them (bf16 at precision 2), its action block (critics, after
  # split_action_input) and bias, LayerNorm and tanh one b200rl_feature_layer_fwd launch.
  def split_action_input(self):
    """Critic over observation-network features: stores the first layer as two blocks, w_f [h0][obs_dim] ('l0.w') and
    w_a [h0][act_dim] ('l0a.w'), instead of one matrix over the concatenated [obs, act] row, which at obs_dim = 7744 is
    neither 16-byte aligned (TMA) nor bf16.  Values and the Sonnet export (one `l0/w` [obs_dim + act_dim, h0], features
    first as CriticMultiplexer concatenates) are unchanged.  Call before buffers are made and graphs captured."""
    if self.act_in:
      return
    values = self.variables()
    old, P = self.params, ParamStore(self.device)
    for name, (_, shape) in old.entries.items():
      if name == 'l0.w':
        P.declare('l0.w', (shape[0], self.obs_dim))
        P.declare('l0a.w', (shape[0], self.act_dim))
      else:
        P.declare(name, shape)
    P.allocate()
    self.params, self.in_dim, self.act_in = P, self.obs_dim, self.act_dim
    self._export = dict(self._export, **{'l0/w': ('l0.w', ('cat', 'l0a.w'))})
    self.load_variables(values)
    if old.shadow is not None:
      P.ensure_shadow()

  def forward_features(self, feat_ptr: int, act_ptr, bufs):
    """feat [B, in_dim] (bf16 at precision 2, else fp32) and, after split_action_input(), act [B, act_dim] fp32 ->
    bufs['out']."""
    B, P, st = bufs['B'], self.params, _capi.current_stream()
    ws, wsb = self.ws
    h0, F = self.sizes[0], self.in_dim
    zf = bufs['z0'].data_ptr()
    if self.flow:
      _capi.call('b200rl_linear_fwd_bf16', B, h0, F, feat_ptr, F, P.sp('l0.w'), None, zf, h0, 0, ACT_NONE, ws, wsb, st)
    else:
      _linear(B, h0, F, feat_ptr, F, P.p('l0.w'), None, zf, h0, ACT_NONE, self)
    _capi.call('b200rl_feature_layer_fwd', B, h0, self.act_in, zf, act_ptr if self.act_in else None,
               P.p('l0a.w') if self.act_in else None, P.p('l0.b'), P.p('ln.scale'), P.p('ln.offset'), 1e-5,
               bufs['y0'].data_ptr(), bufs['y0_bf16'].data_ptr() if self.flow else None, bufs['xhat'].data_ptr(),
               bufs['rstd'].data_ptr(), st)
    return self._hidden_forward(bufs)

  def backward_features(self, feat_ptr: int, act_ptr, bufs, gbufs, dout_ptr: int, param_grads: bool = True,
                        action_grad: bool = False, feat_grad=None):
    """Backward of forward_features from dout (gradient w.r.t. bufs['out']).  param_grads: params.grad; action_grad:
    gbufs['da'] = d/d act (only the act_dim input columns); feat_grad = (dx_ptr, relu_y_ptr): the features' data
    gradient, multiplied by relu'(relu_y) (the observation network's last ReLU), written to dx_ptr in the features' type."""
    B, P, st = bufs['B'], self.params, _capi.current_stream()
    ws, wsb = self.ws
    h0, F, A = self.sizes[0], self.in_dim, self.act_in
    dy = self._hidden_backward(bufs, gbufs, dout_ptr, param_grads)
    pg = param_grads
    dz0, dz0_bf = gbufs['dz0'].data_ptr(), gbufs['dz0_bf16'].data_ptr() if self.flow else None
    _capi.call('b200rl_feature_layer_bwd', B, h0, A, dy, bufs['y0'].data_ptr(), bufs['xhat'].data_ptr(),
               bufs['rstd'].data_ptr(), P.p('ln.scale'), act_ptr if A else None, P.p('l0a.w') if A else None, dz0, dz0_bf,
               P.g('ln.scale') if pg else None, P.g('ln.offset') if pg else None, P.g('l0.b') if pg else None,
               P.g('l0a.w') if pg and A else None, gbufs['da'].data_ptr() if action_grad else None, ws, wsb, st)
    if pg:
      if self.flow:
        _capi.call('b200rl_linear_wgrad_bf16', B, h0, F, dz0_bf, h0, feat_ptr, F, P.g('l0.w'), None, ws, wsb, st)
      else:
        _linear_wgrad(B, h0, F, dz0, h0, feat_ptr, F, P.g('l0.w'), None, self)
    if feat_grad is not None:
      dx, relu_y = feat_grad
      if self.flow:
        _capi.call('b200rl_linear_dgrad_bf16', B, h0, F, dz0_bf, h0, P.sp('l0.w'), dx, F, 1, relu_y, 1, ACT_RELU, ws, wsb, st)
      else:
        _linear_dgrad(B, h0, F, dz0, h0, P.p('l0.w'), dx, F, relu_y, ACT_RELU, self)


class D4PGCritic(LayerNormMLP):
  """CriticMultiplexer() -> LayerNormMLP(sizes, activate_final=True) -> DiscreteValuedHead."""

  def __init__(self, obs_dim: int, act_dim: int, sizes=(512, 512, 256), vmin=-150., vmax=150., num_atoms=51,
               device: int = 0, precision: int = _capi.PRECISION_FP32, seed: int = 0):
    super().__init__(obs_dim + act_dim, sizes, num_atoms, 'head', None, device, precision, seed)
    self.obs_dim, self.act_dim = int(obs_dim), int(act_dim)
    self.vmin, self.vmax, self.K = float(vmin), float(vmax), int(num_atoms)

  def logits(self, obs, act, bufs):
    """obs f32 [B, obs_dim], act f32 [B, act_dim] -> logits [B, K] (input concat kept in bufs['x'])."""
    _capi.call('b200rl_concat2', bufs['B'], self.obs_dim, self.act_dim, obs.data_ptr(), act.data_ptr(),
               bufs['x'].data_ptr(), _capi.current_stream())
    return self.forward_flat(bufs['x'].data_ptr(), bufs)


class DDPGCritic(LayerNormMLP):
  """CriticMultiplexer(critic_network=LayerNormMLP(sizes + [1])) (`acme/agents/tf/ddpg/agent_test.py:46-47`): the scalar
  critic of DDPG -- the same torso as the D4PG critic with one linear output instead of the 51 atoms."""

  def __init__(self, obs_dim: int, act_dim: int, sizes=(512, 512, 256), device: int = 0,
               precision: int = _capi.PRECISION_FP32, seed: int = 0):
    super().__init__(obs_dim + act_dim, sizes, 1, 'q', None, device, precision, seed)
    self.obs_dim, self.act_dim, self.K = int(obs_dim), int(act_dim), 1

  def logits(self, obs, act, bufs):
    """q(obs, act) [B, 1] (named like D4PGCritic.logits so both critics drive the same learner plumbing)."""
    _capi.call('b200rl_concat2', bufs['B'], self.obs_dim, self.act_dim, obs.data_ptr(), act.data_ptr(),
               bufs['x'].data_ptr(), _capi.current_stream())
    return self.forward_flat(bufs['x'].data_ptr(), bufs)


class D4PGPolicy(LayerNormMLP):
  """LayerNormMLP(sizes, activate_final=True) -> NearZeroInitializedLinear(A) -> TanhToSpec."""

  def __init__(self, obs_dim: int, act_dim: int, sizes=(256, 256, 256), act_min=-1., act_max=1.,
               device: int = 0, precision: int = _capi.PRECISION_FP32, seed: int = 0):
    import torch
    super().__init__(obs_dim, sizes, act_dim, 'out', 1e-4, device, precision, seed)
    self.obs_dim, self.act_dim = int(obs_dim), int(act_dim)
    dev = torch.device('cuda', device)
    lo = np.broadcast_to(np.asarray(act_min, np.float32), (act_dim,))
    hi = np.broadcast_to(np.asarray(act_max, np.float32), (act_dim,))
    self.scale = torch.as_tensor(np.ascontiguousarray(hi - lo)).to(dev)
    self.offset = torch.as_tensor(np.ascontiguousarray(lo)).to(dev)

  def make_buffers(self, B: int):
    import torch
    bufs = super().make_buffers(B)
    bufs['a'] = torch.empty((B, self.act_dim), dtype=torch.float32, device=bufs['out'].device)
    bufs['dpre'] = torch.empty_like(bufs['a'])
    return bufs

  def _to_spec(self, pre, bufs):
    _capi.call('b200rl_tanh_to_spec_fwd', bufs['B'], self.act_dim, pre.data_ptr(), self.scale.data_ptr(),
               self.offset.data_ptr(), bufs['a'].data_ptr(), _capi.current_stream())
    return bufs['a']

  def _to_spec_bwd(self, bufs, da):
    _capi.call('b200rl_tanh_to_spec_bwd', bufs['B'], self.act_dim, da.data_ptr(), bufs['out'].data_ptr(),
               self.scale.data_ptr(), bufs['dpre'].data_ptr(), _capi.current_stream())

  def action(self, obs, bufs):
    return self._to_spec(self.forward_flat(obs.data_ptr(), bufs), bufs)

  def backward_action(self, obs, bufs, gbufs, da):
    self._to_spec_bwd(bufs, da)
    self.backward_flat(obs.data_ptr(), bufs, gbufs, bufs['dpre'].data_ptr(), param_grads=True, input_grad=False)

  def action_features(self, feat_ptr: int, bufs):
    """The action from observation-network features (see LayerNormMLP.forward_features)."""
    return self._to_spec(self.forward_features(feat_ptr, None, bufs), bufs)

  def backward_action_features(self, feat_ptr: int, bufs, gbufs, da):
    self._to_spec_bwd(bufs, da)
    self.backward_features(feat_ptr, None, bufs, gbufs, bufs['dpre'].data_ptr(), param_grads=True)
