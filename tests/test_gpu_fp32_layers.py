"""fp32-tensor layer kernels through the C ABI against an fp64 reference: precision 0 (the FFMA kernel, gemm_simt.cu) and
precision 1 (TMA-fed tf32 tcgen05 kernels, gemm_tma.cu; the loader-fed bf16 tcgen05 kernel, gemm_tc.cu, where TMA refuses
the operands; the FFMA kernel for dense layers below 2^26 multiply-adds).

Every output element is held to its own bound (layer_check._check):

    |got - ref| <= C_ACC * (|A|.|B|)_ij + c_op * (|A|.|B|)_ij

against fp64 on the exact operands, |A|.|B| being the same product (or convolution) on absolute values, bias included.
Precision 0 takes arbitrary fp32 operands and c_op = 0.  Precision-1 rows draw their operands on the grid their path
multiplies exactly (c_op = 0): bf16 values for the loader-fed kernel, tf32 values for TMA and FFMA rows.  The tf32 values
are chosen NOT to be bf16 values (mantissa bits 13..15 = 011), and every such row also proves that the bound rejects the
result of bf16-rounded operands: a row that silently took the bf16 path fails.  The first layer on uint8 frames cannot
have exact operands at precision 1 (x / 255 is on neither grid): its rows carry c_op = 2^-10 (tf32, truncated or rounded)
or 2^-9 (bf16, rounded) on the input side.  Every row with a reduction of 1024 or more proves that the bound rejects the
reference without one k-block of its kernel, without the last (ragged) k-block and, for split-K, without one split.

C_ACC = 2^-16.  Measured on an NVIDIA B200 (1000 W power limit), max over the rows below of |err| / (|A|.|B|) on outputs
and split-K partials:
    precision 0   linear_fwd 3.5e-07   linear_dgrad 4.7e-07   linear_wgrad 3.8e-07   (bias gradient 7.8e-08)
                  conv2d_fwd 4.3e-07   conv2d_wgrad 3.7e-07   conv2d_dgrad 3.6e-07
    precision 1   linear_fwd 1.0e-06   linear_dgrad 9.5e-07   linear_wgrad 5.0e-07   (bias gradient 1.4e-08)
                  conv2d_fwd 4.9e-07   conv2d_wgrad 8.0e-07   conv2d_dgrad 5.4e-07
                  first layer on frames 5.8e-04, inside its 2^-10 / 2^-9 operand term
i.e. <= 2^-19.9, 15x below C_ACC.  The smallest margin by which the bound rejects a lost k-block or split is 6.9x (conv
weight gradient, precision 1, B = 5, Cout = 16, without its last k-block).  The whole file, fp64 references included,
runs in 22 s on that card.  (Run with `-s`: each check prints its ratio, and each rejection its margin, as `bound ...`.)

Each table row names its launch signature: the kernels torch.profiler sees (template arguments included), the change of
b200rl_launch_count(), and for split-K the [M][N] fp32 partial slabs in a sentinel-filled workspace, each checked against
the fp64 sum of its own k-range (behind the first layer's row image where the workspace holds one; for the phase-wise
data gradient: the row map, then the slabs of the last phase that splits, as the phases share one slab region).  The
split counts and tiles of the tables are checked against Python mirrors of the dispatch rules (`simt_plan`, `tma_plan`,
`tc_plan`, `colsum_plan`, `small_dense`) by a test that needs no GPU.  Every output sits inside sentinel guard memory;
inputs with a row stride hold NaN in their padding."""
import ctypes
import math

import numpy as np
import pytest
from layer_check import (ELU, NONE, RELU, SENT, TANH, WS_BYTES, Out, Workspace, _assert_rejects, _capi, _check,
                         _rejects, act, assert_sig, mask_factor, mask_values, run)

SMS = 148
_KEEP = []
gpu = pytest.mark.gpu


def cdiv(a, b):
  return -(-a // b)


# ------------------------------------------------------------------------------ mirrors of the dispatch rules
def small_dense(precision, M, N, K):
  """layers_api.cu: dense layers below 2^26 multiply-adds run the FFMA kernel at precision 1"""
  return 0 if precision == 1 and M * N * K < (1 << 26) else precision


def simt_plan(M, N, K, wsb):
  """gemm_simt.cu launch_gemm -> (TM, TN, splits, k per split)"""
  tm = tn = 4
  if M >= 128 and N >= 128 and cdiv(M, 128) * cdiv(N, 128) >= SMS:
    tm = tn = 8
  elif M >= 128 and cdiv(M, 128) * cdiv(N, 64) >= SMS:
    tm = 8
  tiles = cdiv(M, 16 * tm) * cdiv(N, 16 * tn)
  s = 1
  if tiles < 2 * SMS and K >= 64:
    s = max(1, min(cdiv(2 * SMS, tiles), K // 32, 64, wsb // (M * N * 4) if wsb else 0))
  kps = cdiv(cdiv(K, s), 16) * 16
  return tm, tn, cdiv(K, kps), kps


def pick_bn(N):
  return 32 if N <= 32 else (64 if N <= 64 else 128)


def tma_dgrad_bn(M, K):
  """gemm_tma.cu tma_linear_dgrad: 128-wide tiles are halved when they leave SMs idle"""
  bn = pick_bn(K)
  return 64 if bn == 128 and cdiv(M, 128) * cdiv(K, 128) < SMS else bn


def tma_plan(M, N, K, BN, wsb):
  """gemm_tma.cu launch_tma_bn -> (splits, k per split)"""
  tiles, kb = cdiv(M, 128) * cdiv(N, BN), cdiv(K, 32)
  s = 1
  if 2 * tiles <= SMS and kb >= 16:
    s = max(1, min(cdiv(SMS, tiles), kb // 8, 64, wsb // (M * N * 4) if wsb else 0))
  kps = cdiv(kb, s)
  return cdiv(kb, kps), kps * 32


def tc_plan(M, N, K, wsb):
  """gemm_tc.cu launch_tc / launch_tc_bn -> (BN, splits, k per split)"""
  bn = pick_bn(N)
  tiles, kb = cdiv(M, 128) * cdiv(N, bn), cdiv(K, 64)
  s = 1
  if tiles < SMS and kb >= 8:
    s = max(1, min(cdiv(2 * SMS, tiles), kb // 4, 64, wsb // (M * N * 4) if wsb else 0))
  kps = cdiv(kb, s)
  return bn, cdiv(kb, kps), kps * 64


def colsum_plan(M, N, ld, aligned, wsb):
  """gemm_simt.cu launch_colsum -> (kernels, CTAs or row splits)"""
  if 4 <= N <= 1024 and N & (N - 1) == 0 and ld % 4 == 0 and aligned:
    blocks = max(1, min(int(math.floor(math.sqrt(M) + 0.5)), 2 * SMS))
    blocks = max(1, min(blocks, wsb // (N * 4) if wsb else 1))
    return ['colsum_vec_kernel<false>'], cdiv(M, cdiv(M, blocks))
  s = max(1, min(cdiv(M, 64), (2 * SMS) // cdiv(N, 32), 96))
  s = min(s, wsb // (N * 4) if wsb else 1)
  if s <= 1:
    return ['colsum_partial_kernel'], 1
  return ['colsum_partial_kernel', 'colsum_finish_kernel'], cdiv(M, cdiv(M, s))


def plan(path, M, N, K, wsb, bn=None):
  """(kernel tag, splits, k per split) of one GEMM launch: 's44' / 's84' / 's88', 't<BN>' (TMA), 'c<BN>' (loader-fed)"""
  if path == 'simt':
    tm, tn, s, kps = simt_plan(M, N, K, wsb)
    return f's{tm}{tn}', s, kps
  if path == 'tma':
    s, kps = tma_plan(M, N, K, bn or pick_bn(N), wsb)
    return f't{bn or pick_bn(N)}', s, kps
  b, s, kps = tc_plan(M, N, K, wsb)
  return f'c{b}', s, kps


# ------------------------------------------------------------------------------ operands
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
  if torch.cuda.is_available():
    torch.cuda.synchronize()
  _KEEP.clear()


def stream():
  return _capi().current_stream()


def on_grid(x, grid):
  """x on the grid of a path: 'f32' (any fp32), 'bf16', 'tf32' (10 mantissa bits, bits 13..15 = 011: never a bf16 value,
  and bf16 rounding always moves it down by 3/8 of a bf16 ulp)"""
  x = np.ascontiguousarray(x, np.float32)
  if grid == 'bf16':
    import torch
    return torch.from_numpy(x).to(torch.bfloat16).double().numpy()
  if grid == 'tf32':
    u = (x.view(np.uint32) & np.uint32(0xFFFF0000)) | np.uint32(0x6000)
    return u.view(np.float32).astype(np.float64)
  return x.astype(np.float64)


def bf(x):
  return on_grid(x, 'bf16')


def fmat(a, ld=None, off=0):
  """fp32 [rows][cols] device matrix with row stride ld, starting `off` floats into its allocation; padding = NaN"""
  import torch
  rows, cols = a.shape
  ld = ld or cols
  t = torch.full((rows * ld + off + 4,), float('nan'), dtype=torch.float32, device='cuda')
  t[off:off + rows * ld].view(rows, ld)[:, :cols] = torch.from_numpy(np.ascontiguousarray(a, np.float32)).cuda()
  _KEEP.append(t)
  return t.data_ptr() + 4 * off


def grid_of(precision, path):
  return 'f32' if precision == 0 else ('bf16' if path == 'tc' else 'tf32')


def drops(K, KE, splits, kps):
  """k-ranges a broken kernel might lose: one k-block of the kernel in the middle, the last (ragged) block, one split"""
  kb = cdiv(K, KE)
  out = [('one k-block', (kb // 2) * KE, min(K, (kb // 2 + 1) * KE)), ('the last k-block', (kb - 1) * KE, K)]
  if splits > 1:
    s = splits // 2
    out.append((f'split {s}', s * kps, min(K, (s + 1) * kps)))
  return out


KE = {'simt': 16, 'tma': 32, 'tc': 64}


def gemm_sig(path, tag, loaders):
  """kernel-name prefix of one GEMM launch; loaders = (simt A, simt B, TMA A MN-major, TMA B MN-major, tc A, tc B)"""
  if path == 'simt':
    return f'gemm_kernel<{loaders[0]},{loaders[1]},{tag[1]},{tag[2]},'.rstrip(',') + '>'
  if path == 'tma':
    return f'tma_gemm_kernel<{loaders[2]},{loaders[3]},{tag[1:]},'
  return f'tc_gemm_kernel<{loaders[4]},{loaders[5]},{tag[1:]}>'


def bf16_rejection(what, precision, path, ref_fn, ref, absr, op=None):
  """TMA and FFMA rows at precision 1: the bound must reject the result of bf16-rounded operands (not the first layer
  on frames: its operand term is as wide as a bf16 rounding; its row signature pins the path)"""
  if precision == 1 and path in ('tma', 'simt') and op is None:
    _assert_rejects(f'{what}: bf16-rounded operands', ref, ref_fn(bf), absr, False, op=op)


# ------------------------------------------------------------------------------ dense layers
LIN_LOADERS = {
    'fwd': ('DenseRed', 'DenseRed', 'false', 'false', 'RowMatK', 'RowMatK'),
    'dgrad': ('DenseRed', 'DenseOuter', 'false', 'true', 'RowMatK', 'RowMatMN'),
    'wgrad': ('DenseOuter', 'DenseOuter', 'true', 'true', 'RowMatMN', 'RowMatMN'),
}


def lin_product(entry, M, N, K):
  """(rows, cols, reduction) of the GEMM behind an entry point"""
  return {'fwd': (M, N, K), 'dgrad': (M, K, N), 'wgrad': (N, K, M)}[entry]


def lin_path(entry, precision, M, N, K, opt):
  """which kernel family the dispatcher picks (layers_api.cu + the TMA eligibility tests of gemm_tma.cu)"""
  if small_dense(precision, M, N, K) == 0:
    return 'simt'
  if opt.get('tma_off'):
    return 'tc'
  al = lambda name: opt.get('off_' + name, 0) % 4 == 0
  if entry == 'fwd':
    ok = al('x') and opt.get('ldx', K) % 4 == 0 and K % 4 == 0 and K >= 32
  elif entry == 'dgrad':
    ok = (opt.get('mask') is None or (al('mask') and al('dx'))) and opt.get('lddy', N) % 4 == 0 and K % 4 == 0 and N >= 32
  else:
    ok = opt.get('lddy', N) % 4 == 0 and opt.get('ldx', K) % 4 == 0 and M >= 32
  return 'tma' if ok else 'tc'


def lin_plan(entry, precision, M, N, K, opt):
  path = lin_path(entry, precision, M, N, K, opt)
  R, C, red = lin_product(entry, M, N, K)
  wsb = 0 if opt.get('ws', True) is None else opt.get('wsb', WS_BYTES)
  bn = tma_dgrad_bn(M, K) if entry == 'dgrad' and path == 'tma' else None
  return (path,) + plan(path, R, C, red, wsb, bn)


def _id(v):
  if isinstance(v, dict):
    return '-'.join(f'{k}{"" if isinstance(x, (list, tuple)) else x}' for k, x in v.items()) or 'default'
  return None


# precision, M, N, K, kernel tag, splits, options
LINEAR_FWD = [
    (0, 256, 512, 88, 's44', 2, {}),                                   # D4PG critic: k [0, 48) and [48, 88)
    (0, 256, 256, 67, 's44', 2, {'acts': [TANH, ELU]}),                # K % 4 != 0: scalar row loads
    (0, 256, 51, 256, 's44', 8, {'acts': [NONE, RELU]}),
    (0, 256, 21, 256, 's44', 8, {}),
    (0, 256, 1, 512, 's44', 16, {'acts': [TANH, NONE]}),
    (0, 256, 512, 7744, 's44', 10, {}),                                # fc1, fp32 mode
    (0, 512, 512, 7744, 's44', 5, {}),
    (0, 2048, 1280, 64, 's88', 2, {'acts': [ELU, RELU]}),              # 128 x 128 tiles
    (0, 1280, 960, 48, 's84', 1, {}),                                  # 128 x 64 tiles, K < 64: never split
    (0, 1, 64, 256, 's44', 8, {'acts': [TANH, RELU]}),
    (0, 300, 200, 48, 's44', 1, {'acts': [ELU, NONE]}),
    (0, 256, 512, 7744, 's44', 3, {'wsb': 3 * 256 * 512 * 4}),        # the workspace caps the split count
    (0, 256, 512, 7744, 's44', 1, {'ws': None}),                       # no workspace: no split
    (0, 100, 64, 300, 's44', 7, {'ldx': 301, 'ldy': 67, 'bias': False, 'acts': [RELU, TANH]}),
    (0, 256, 1024, 7744, 's44', 5, {}), (0, 10, 50, 50, 's44', 1, {'acts': [ELU, ELU]}),
    (0, 256, 18, 512, 's44', 16, {'acts': [ELU, ELU]}), (0, 33, 51, 256, 's44', 8, {'acts': [ELU, ELU]}),
    (0, 300, 200, 136, 's44', 3, {'acts': [ELU, ELU]}),
    (1, 256, 256, 1023, 's44', 16, {}),                                # 2^26 - 2^16 multiply-adds: FFMA
    (1, 256, 256, 1024, 't128', 4, {'acts': [ELU, TANH]}),             # 2^26: TMA
    (1, 256, 512, 512, 't128', 2, {}),                                 # the D4PG critic's middle layer, exactly 2^26
    (1, 4096, 32, 1024, 't32', 4, {'acts': [TANH, NONE]}),
    (1, 2048, 64, 1024, 't64', 4, {}),
    (1, 256, 1024, 7752, 't128', 10, {'acts': [NONE, ELU]}),            # ragged last k-block (8 of 32)
    (1, 256, 1024, 7744, 't128', 3, {'wsb': 3 * 256 * 1024 * 4}),
    (1, 256, 1024, 7744, 't128', 10, {'ldy': 1030, 'bias': False}),
    (1, 8192, 1024, 16, 'c128', 1, {}),                                # K < 32: loader-fed
    (1, 256, 1024, 1024, 'c128', 4, {'ldx': 1025}),                    # ldx % 4 != 0; split-K on the loader-fed kernel
    (1, 256, 1024, 1024, 'c128', 4, {'off_x': 1, 'acts': [TANH, ELU]}),   # x offset by 4 bytes
    (1, 256, 1024, 1024, 'c128', 4, {'tma_off': True}),                # b200rl_debug_set_tma(0)
    (1, 10, 50, 50, 's44', 1, {'acts': [ELU, ELU]}), (1, 256, 18, 512, 's44', 16, {'acts': [ELU, ELU]}),
    (1, 256, 1, 512, 's44', 16, {'acts': [ELU, ELU]}), (1, 33, 51, 256, 's44', 8, {'acts': [ELU, ELU]}),
    (1, 300, 200, 136, 's44', 3, {'acts': [ELU, ELU]}),
]

# precision, M, N (reduction), K, kernel tag, splits, options (mask: activation of the producer, None = no mask)
LINEAR_DGRAD = [
    (0, 256, 512, 88, 's44', 16, {'mask': RELU}),
    (0, 256, 256, 67, 's44', 8, {'mask': ELU}),                        # ragged 67-wide output: scalar loads of w
    (0, 256, 51, 256, 's44', 1, {'mask': TANH}),
    (0, 256, 512, 7744, 's84', 2, {'mask': RELU}),                     # fc1: 122 128 x 128 tiles < 148: 128 x 64
    (0, 256, 1024, 7744, 's84', 2, {}),
    (0, 1, 64, 256, 's44', 2, {'mask': TANH}),
    (0, 100, 300, 64, 's44', 7, {'lddy': 301, 'lddx': 70, 'mask': ELU}),
    (0, 10, 50, 50, 's44', 1, {}), (0, 256, 18, 512, 's44', 1, {}), (0, 256, 1, 512, 's44', 1, {}),
    (0, 33, 51, 256, 's44', 1, {}), (0, 300, 200, 136, 's44', 5, {}),
    (1, 256, 256, 1023, 's44', 4, {'mask': RELU}),
    (1, 256, 512, 512, 't64', 2, {'mask': ELU}),                      # 2^26; 2 x 4 tiles
    (1, 256, 1024, 7744, 't64', 1, {'mask': RELU}),                    # BN 128 -> 64
    (1, 2048, 1024, 1536, 't128', 1, {'mask': TANH}),                  # 16 x 12 tiles >= 148: BN stays 128
    (1, 512, 1024, 7744, 't128', 1, {}),
    (1, 8192, 16, 1024, 'c128', 1, {}),                                # N < 32: loader-fed
    (1, 256, 1024, 1024, 'c128', 4, {'mask': RELU, 'off_mask': 1}),    # mask not 16-byte aligned
    (1, 256, 1024, 1024, 'c128', 4, {'mask': ELU, 'off_dx': 1}),       # dx not 16-byte aligned
    (1, 256, 1024, 1024, 'c128', 4, {'lddy': 1025}),
    (1, 10, 50, 50, 's44', 1, {}), (1, 256, 18, 512, 's44', 1, {}), (1, 256, 1, 512, 's44', 1, {}),
    (1, 33, 51, 256, 's44', 1, {}), (1, 300, 200, 136, 's44', 5, {}),
]

# precision, M (reduction), N, K, kernel tag, splits, options (db: None = no bias gradient, else the colsum kernels)
LINEAR_WGRAD = [
    (0, 256, 512, 88, 's44', 8, {'db': ['colsum_vec_kernel<false>']}),     # vector colsum, 16 CTAs
    (0, 256, 256, 67, 's44', 8, {'db': ['colsum_vec_kernel<false>']}),
    (0, 256, 51, 256, 's44', 8, {'db': ['colsum_partial_kernel', 'colsum_finish_kernel']}),   # N not a power of two
    (0, 2048, 51, 1, 's44', 64, {'db': ['colsum_partial_kernel', 'colsum_finish_kernel']}),
    (0, 2048, 51, 1, 's44', 1, {'ws': None, 'db': ['colsum_partial_kernel']}),           # no workspace: one pass
    (0, 256, 512, 7744, 's88', 2, {'db': None}),
    (0, 1, 64, 256, 's44', 1, {'db': ['colsum_vec_kernel<false>']}),        # one CTA: no partial rows
    (0, 4096, 64, 64, 's44', 64, {'db': ['colsum_vec_kernel<false>'], 'lddy': 68, 'ldx': 65}),
    (0, 256, 1024, 7744, 's88', 1, {'db': ['colsum_vec_kernel<false>']}),
    (0, 10, 50, 50, 's44', 1, {'db': ['colsum_partial_kernel']}), (0, 256, 18, 512, 's44', 8, {'db': ['colsum_partial_kernel', 'colsum_finish_kernel']}),
    (0, 256, 1, 512, 's44', 8, {'db': ['colsum_partial_kernel', 'colsum_finish_kernel']}),
    (0, 33, 51, 256, 's44', 1, {'db': ['colsum_partial_kernel']}), (0, 300, 200, 136, 's44', 7, {'db': ['colsum_partial_kernel', 'colsum_finish_kernel']}),
    (1, 1023, 256, 256, 's44', 16, {'db': ['colsum_vec_kernel<false>']}),
    (1, 512, 256, 512, 't128', 2, {'db': ['colsum_vec_kernel<false>']}),
    (1, 4096, 64, 1024, 't128', 16, {'db': ['colsum_vec_kernel<false>']}),
    (1, 256, 1024, 7744, 't128', 1, {'db': ['colsum_vec_kernel<false>']}),
    (1, 16384, 256, 16, 't32', 64, {'db': None}),                      # K = 16: BN = 32, 64 splits
    (1, 4096, 1024, 32, 'c32', 16, {'ldx': 33, 'db': ['colsum_vec_kernel<false>']}),
    (1, 16, 2048, 2048, 'c128', 1, {'db': None}),                      # M < 32: loader-fed
    (1, 10, 50, 50, 's44', 1, {'db': ['colsum_partial_kernel']}), (1, 256, 18, 512, 's44', 8, {'db': ['colsum_partial_kernel', 'colsum_finish_kernel']}),
    (1, 256, 1, 512, 's44', 8, {'db': ['colsum_partial_kernel', 'colsum_finish_kernel']}),
    (1, 33, 51, 256, 's44', 1, {'db': ['colsum_partial_kernel']}), (1, 300, 200, 136, 's44', 7, {'db': ['colsum_partial_kernel', 'colsum_finish_kernel']}),
]


def test_tables_agree_with_the_dispatch_rules():
  """every row's kernel tag and split count is what the mirrored dispatch rules give (no GPU needed)"""
  for entry, table in (('fwd', LINEAR_FWD), ('dgrad', LINEAR_DGRAD), ('wgrad', LINEAR_WGRAD)):
    for precision, M, N, K, tag, splits, opt in table:
      path, t, s, _ = lin_plan(entry, precision, M, N, K, opt)
      assert (t, s) == (tag, splits), f'linear {entry} {(precision, M, N, K, opt)}: rules give {t} / {s} splits'
      if entry == 'wgrad' and opt.get('db') is not None:
        wsb = 0 if opt.get('ws', True) is None else WS_BYTES
        assert colsum_plan(M, N, opt.get('lddy', N), True, wsb)[0] == opt['db'], f'linear wgrad {(M, N, K)}: colsum'
  for row in CONV_FWD + CONV_WGRAD + CONV_DGRAD:
    assert conv_plan(row)[1:] == row[-2:], f'conv {row}: rules give {conv_plan(row)}'
  assert simt_plan(256, 512, 88, WS_BYTES)[3] == 48 and tma_plan(256, 1024, 7752, 128, WS_BYTES) == (10, 25 * 32)
  assert small_dense(1, 256, 512, 512) == 1 and small_dense(1, 256, 256, 1023) == 0 and small_dense(0, 8192, 8192, 8192) == 0


def _lin_setup(entry, precision, M, N, K, opt, seed):
  path = lin_path(entry, precision, M, N, K, opt)
  rng = np.random.default_rng(seed)
  g = grid_of(precision, path)
  return path, rng, g


@gpu
@pytest.mark.parametrize('precision,M,N,K,tag,splits,opt', LINEAR_FWD, ids=_id)
def test_linear_fwd(precision, M, N, K, tag, splits, opt):
  c = _capi()
  lib = c.load()
  path, rng, grid = _lin_setup('fwd', precision, M, N, K, opt, M * 7 + N * 3 + K)
  x, w = on_grid(rng.standard_normal((M, K)), grid), on_grid(rng.standard_normal((N, K)) / np.sqrt(K), grid)
  b = rng.standard_normal(N).astype(np.float32).astype(np.float64) if opt.get('bias', True) else None
  ldx, acts = opt.get('ldx', K), opt.get('acts', [RELU, RELU])
  xp, wp = fmat(x, ldx, opt.get('off_x', 0)), fmat(w)
  bp = dev(b.astype(np.float32)).data_ptr() if b is not None else None
  ws = Workspace()
  wsp, wsb = (ws.ptr, opt.get('wsb', ws.bytes)) if 'ws' not in opt else (None, 0)
  _, t, s, kps = lin_plan('fwd', precision, M, N, K, opt)
  assert (t, s) == (tag, splits)
  want = [gemm_sig(path, tag, LIN_LOADERS['fwd'])] + (['splitk_finish_kernel'] if splits > 1 else [])

  def ref_of(fn, lo=0, hi=K):
    xs, wt = fn(x)[:, lo:hi], fn(w)[:, lo:hi]
    return xs @ wt.T + (0. if b is None else b)
  pre = ref_of(lambda v: v)
  absr = np.abs(x) @ np.abs(w).T + (0. if b is None else np.abs(b))
  try:
    if opt.get('tma_off'):
      lib.b200rl_debug_set_tma(0)
    for i, a in enumerate(acts):
      y = Out(M, N, False, ld=opt.get('ldy', N))
      ws.reset()
      sig = run(lambda: c.call('b200rl_linear_fwd', M, N, K, xp, ldx, wp, bp, y.ptr, y.ld, a, precision, wsp, wsb, stream()),
                profile=i == 0)
      what = f'linear fwd p{precision} {M}x{N}x{K} act {a}'
      assert_sig(what, sig, want)
      ref = act(pre, a)
      _check(what, y.read(what), ref, absr, False)
      if wsp:
        slabs = ws.slabs(what, M, N, splits)
        if i == 0 and splits > 1:
          for j in range(splits):
            lo, hi = j * kps, min(K, (j + 1) * kps)
            _check(f'{what} split {j} partial (k {lo}..{hi})', slabs[j], x[:, lo:hi] @ w[:, lo:hi].T,
                   np.abs(x[:, lo:hi]) @ np.abs(w[:, lo:hi]).T, False)
      if i == 0:
        bf16_rejection(what, precision, path, lambda r: act(ref_of(r), a), ref, absr)
        if K >= 1024:
          for how, lo, hi in drops(K, KE[path], splits, kps):
            _assert_rejects(f'{what} without {how}', ref, act(pre - x[:, lo:hi] @ w[:, lo:hi].T, a), absr, False)
  finally:
    lib.b200rl_debug_set_tma(1)


@gpu
@pytest.mark.parametrize('precision,M,N,K,tag,splits,opt', LINEAR_DGRAD, ids=_id)
def test_linear_dgrad(precision, M, N, K, tag, splits, opt):
  c = _capi()
  path, rng, grid = _lin_setup('dgrad', precision, M, N, K, opt, M + N + K)
  dy, w = on_grid(rng.standard_normal((M, N)), grid), on_grid(rng.standard_normal((N, K)) / np.sqrt(N), grid)
  lddy, lddx, ma = opt.get('lddy', N), opt.get('lddx', K), opt.get('mask')
  dyp, wp = fmat(dy, lddy), fmat(w)
  if ma is None:
    mptr, gm, ag = None, 1., 1.
  else:
    ym = mask_values(rng, (M, K), ma).astype(np.float32).astype(np.float64)
    mptr = fmat(ym, lddx, opt.get('off_mask', 0))
    gm, ag = mask_factor(ym, ma)
  ws = Workspace()
  _, t, s, kps = lin_plan('dgrad', precision, M, N, K, opt)
  assert (t, s) == (tag, splits)
  want = [gemm_sig(path, tag, LIN_LOADERS['dgrad'])] + (['splitk_finish_kernel'] if splits > 1 else [])
  what = f'linear dgrad p{precision} {M}x{N}x{K} mask {ma}'
  dx = Out(M, K, False, ld=lddx, off=4 * opt.get('off_dx', 0))
  assert_sig(what, run(lambda: c.call('b200rl_linear_dgrad', M, N, K, dyp, lddy, wp, dx.ptr, lddx, mptr, ma or 0, precision,
                                      ws.ptr, ws.bytes, stream())), want)
  acc, absr = dy @ w, (np.abs(dy) @ np.abs(w)) * ag
  ref = acc * gm
  _check(what, dx.read(what), ref, absr, False)
  slabs = ws.slabs(what, M, K, splits)
  if splits > 1:
    for j in range(splits):
      lo, hi = j * kps, min(N, (j + 1) * kps)
      _check(f'{what} split {j} partial', slabs[j], dy[:, lo:hi] @ w[lo:hi], np.abs(dy[:, lo:hi]) @ np.abs(w[lo:hi]), False)
  bf16_rejection(what, precision, path, lambda r: (r(dy) @ r(w)) * gm, ref, absr)
  if N >= 1024:
    for how, lo, hi in drops(N, KE[path], splits, kps):
      _assert_rejects(f'{what} without {how}', ref, (acc - dy[:, lo:hi] @ w[lo:hi]) * gm, absr, False)


@gpu
@pytest.mark.parametrize('precision,M,N,K,tag,splits,opt', LINEAR_WGRAD, ids=_id)
def test_linear_wgrad(precision, M, N, K, tag, splits, opt):
  c = _capi()
  path, rng, grid = _lin_setup('wgrad', precision, M, N, K, opt, M + 2 * N + K)
  dy, x = on_grid(rng.standard_normal((M, N)), grid), on_grid(rng.standard_normal((M, K)), grid)
  lddy, ldx = opt.get('lddy', N), opt.get('ldx', K)
  dyp, xp = fmat(dy, lddy), fmat(x, ldx)
  ws = Workspace()
  wsp, wsb = (ws.ptr, ws.bytes) if 'ws' not in opt else (None, 0)
  _, t, s, kps = lin_plan('wgrad', precision, M, N, K, opt)
  assert (t, s) == (tag, splits)
  what = f'linear wgrad p{precision} {M}x{N}x{K}'
  gemm = [gemm_sig(path, tag, LIN_LOADERS['wgrad'])] + (['splitk_finish_kernel'] if splits > 1 else [])
  ref, absr = dy.T @ x, np.abs(dy).T @ np.abs(x)
  dw = Out(N, K, False)
  assert_sig(what, run(lambda: c.call('b200rl_linear_wgrad', M, N, K, dyp, lddy, xp, ldx, dw.ptr, None, precision, wsp, wsb,
                                      stream())), gemm)
  _check(what, dw.read(what), ref, absr, False)
  if wsp:
    slabs = ws.slabs(what, N, K, splits)
    if splits > 1:
      for j in range(splits):
        lo, hi = j * kps, min(M, (j + 1) * kps)
        _check(f'{what} split {j} partial', slabs[j], dy[lo:hi].T @ x[lo:hi], np.abs(dy[lo:hi]).T @ np.abs(x[lo:hi]), False)
  bf16_rejection(what, precision, path, lambda r: r(dy).T @ r(x), ref, absr)
  if M >= 1024:
    for how, lo, hi in drops(M, KE[path], splits, kps):
      _assert_rejects(f'{what} without {how}', ref, ref - dy[lo:hi].T @ x[lo:hi], absr, False)
  if opt.get('db') is None:
    return
  # with the bias gradient: the same dw bit for bit, plus the column-sum launches
  first = dw.bits()
  dw.reset()
  db = Out(1, N, False)
  assert_sig(what + ' + db', run(lambda: c.call('b200rl_linear_wgrad', M, N, K, dyp, lddy, xp, ldx, dw.ptr, db.ptr, precision,
                                                wsp, wsb, stream())), gemm + opt['db'])
  assert bool((dw.bits() == first).all()), f'{what}: dw changed when db was requested'
  _check(what + ' db', db.read(what + ' db')[0], dy.sum(0), np.abs(dy).sum(0), False)


# ------------------------------------------------------------------------------ convolutions
def geom(B, H, C, k, s, Cout):
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
  import torch
  import torch.nn.functional as F
  return F.conv2d(_padded(x, k, s, H, oh, pad), torch.from_numpy(np.ascontiguousarray(w)).permute(0, 3, 1, 2),
                  stride=s).permute(0, 2, 3, 1).numpy()


def conv_wgrad_ref(x, dy, k, s, H, oh, pad, C):
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
  """OHWI weights with only the flattened reduction indices [lo, hi) kept ((tap, channel) order)"""
  f = np.zeros_like(w).reshape(w.shape[0], -1)
  f[:, lo:hi] = w.reshape(w.shape[0], -1)[:, lo:hi]
  return f.reshape(w.shape)


def wgrad_range(x, dy, lo, hi, k, s, H, oh, pad, C):
  """weight gradient (value, |x| |dy| bound) over the flattened output pixels [lo, hi) only: the reduction range of one
  split; computed on the images that range touches"""
  hw, Cout = oh * oh, dy.shape[-1]
  b0, b1 = lo // hw, (hi - 1) // hw + 1
  d = np.zeros(((b1 - b0) * hw, Cout))
  d[lo - b0 * hw:hi - b0 * hw] = dy.reshape(-1, Cout)[lo:hi]
  d = d.reshape(b1 - b0, oh, oh, Cout)
  return (conv_wgrad_ref(x[b0:b1], d, k, s, H, oh, pad, C), conv_wgrad_ref(np.abs(x[b0:b1]), np.abs(d), k, s, H, oh, pad, C))


def dgrad_taps(dy, w, co, ky, kx, k, s, H, oh, pad):
  """data gradient (value, |dy| |w| bound) through the filter entries (co, ky, kx) only: one split's reduction range"""
  wm = np.zeros_like(w)
  wm[co, ky, kx] = w[co, ky, kx]
  M, C = dy.shape[0] * H * H, w.shape[3]
  return (conv_dgrad_ref(dy, wm, k, s, H, oh, pad).reshape(M, C),
          conv_dgrad_ref(np.abs(dy), np.abs(wm), k, s, H, oh, pad).reshape(M, C))


def phase_pixels(B, H, pad, s):
  """the input pixels of each non-empty stride phase in (b, iy, ix) order: the row map the FFMA data gradient builds"""
  ph = (np.arange(H) + pad) % s
  out = []
  for py in range(s):
    for px in range(s):
      ys, xs = np.flatnonzero(ph == py), np.flatnonzero(ph == px)
      if len(ys) and len(xs):
        out.append(((np.arange(B)[:, None, None] * H + ys[None, :, None]) * H + xs[None, None, :]).reshape(-1))
  return out


def rows_head(ws, x, B, H, k, s, oh, pad):
  """bytes of the workspace head taken by the first layer's fp32 row image (gemm_tma.cu rows_used): the overlapping view
  (the zero-padded image itself) when the driver accepted it, else the materialised one; rounded up to 1 KB"""
  pb = max((oh - 1) * s + k - H - pad, 0)
  img = np.pad(x.astype(np.float32), ((0, 0), (pad, pb), (pad, pb), (0, 0)))
  h = ws.buf[ws.off:ws.off + img.nbytes].cpu().numpy().view(np.float32)
  used = img.nbytes if np.array_equal(h, img.reshape(-1)) else B * (H + pad + pb) * oh * 32 * 4
  return (used + 1023) // 1024 * 1024


def conv_path(row):
  """the dispatcher's choice for a conv table row: (entry, precision, B, H, C, k, s, Cout, opt, tag, splits)"""
  entry, precision, B, H, C, k, s, Cout, opt = row[:9]
  if precision == 0:
    return 'simt'
  if opt.get('tma_off'):
    return 'tc'
  u8 = opt.get('u8', 0)
  g, oh, _ = geom(B, H, C, k, s, Cout)
  M = B * oh * oh
  wide = C == 4 and k * C == 32 and Cout % 8 == 0 and Cout <= 128
  big_x = B * H * H * C * 4 >= 131072
  rows_fit = opt.get('ws_bytes', WS_BYTES) >= rows_bytes(B, H, k, s) and opt.get('ws_off', 0) % 128 == 0
  if entry == 'fwd':
    if u8:
      return 'tma' if wide and M * Cout * 4 >= 131072 and rows_fit else 'tc'
    return 'tma' if C % 32 == 0 and big_x else 'tc'
  if entry == 'wgrad':
    if u8:
      return 'tma' if wide and Cout % 32 == 0 and M * Cout * 4 >= 131072 and M >= 32 and rows_fit else 'tc'
    return 'tma' if C % 32 == 0 and big_x and M >= 32 else 'tc'
  ok = s <= 2 and k >= s and Cout % 32 == 0 and C in (32, 64, 128) and M * Cout * 4 >= 131072
  return 'tma' if ok else 'tc'


def rows_bytes(B, H, k, s):
  """tma_rows_bytes for the 4-channel first layer: the larger of the overlapping and the materialised row image"""
  from acme_b200 import networks
  oh, pad = networks.tf_same_pad(H, k, s)
  pb = max((oh - 1) * s + k - H - pad, 0)
  hp = H + pad + pb
  return max(B * hp * (H + pad + pb) * 4 * 4, B * hp * oh * 32 * 4)


def conv_plan(row):
  """(path, kernel tag, splits) of the main GEMM of a conv row (the data gradient's phase path: of its largest phase)"""
  entry, precision, B, H, C, k, s, Cout, opt = row[:9]
  path = conv_path(row)
  g, oh, _ = geom(B, H, C, k, s, Cout)
  M, K = B * oh * oh, k * k * C
  wsb = 0 if opt.get('ws', True) is None else opt.get('ws_bytes', WS_BYTES)
  if entry == 'fwd':
    return (path,) + plan(path, M, Cout, K, wsb)[:2]
  if entry == 'wgrad':
    if path == 'simt':
      return (path,) + plan(path, Cout, K, M, wsb)[:2]
    return (path,) + plan(path, K, Cout, M, wsb, pick_bn(Cout))[:2]
  if path == 'tma':
    return path, f't{C}', 1
  if path == 'simt' and phased(s, k, wsb, B * H * H):
    _, _, Mp, Rp = phases(B, H, C, k, s, Cout)[0]
    return (path,) + plan(path, Mp, C, Rp, wsb - map_bytes(B * H * H))[:2]
  return (path,) + plan(path, B * H * H, C, k * k * Cout, wsb)[:2]


def map_bytes(Min):
  return (Min * 4 + 255) // 256 * 256


def phased(s, k, wsb, Min):
  return 1 < s <= k and wsb > map_bytes(Min)


def phases(B, H, C, k, s, Cout):
  """(py, px, pixels, reduction) of each non-empty stride phase of the FFMA data gradient, in launch order"""
  _, oh, pad = geom(B, H, C, k, s, Cout)
  first = lambda p: ((p - pad) % s + s) % s
  count = lambda p: (H - first(p) + s - 1) // s if first(p) < H else 0
  out = []
  for py in range(s):
    for px in range(s):
      Mp = B * count(py) * count(px)
      Rp = ((k - py + s - 1) // s) * ((k - px + s - 1) // s) * Cout
      if Mp > 0:
        out.append((py, px, Mp, Rp))
  return out


# entry, precision, B, H, C, k, s, Cout, options, kernel tag, splits
CONV_FWD = [
    ('fwd', 0, 2, 84, 4, 8, 4, 32, {'u8': 1}, 's44', 8),                          # conv1: im2col straight from the frames
    ('fwd', 0, 256, 21, 32, 4, 2, 64, {}, 's84', 2), ('fwd', 0, 5, 21, 32, 4, 2, 64, {}, 's44', 16),    # conv2
    ('fwd', 0, 256, 11, 64, 3, 1, 64, {}, 's84', 2), ('fwd', 0, 5, 11, 64, 3, 1, 64, {}, 's44', 18),   # conv3
    ('fwd', 0, 5, 13, 32, 4, 2, 64, {}, 's44', 16),                                # odd H: 1 / 2 padding
    ('fwd', 0, 5, 12, 8, 3, 2, 16, {}, 's44', 2), ('fwd', 0, 13, 20, 32, 5, 2, 32, {}, 's44', 13),
    ('fwd', 0, 11, 17, 64, 3, 2, 96, {}, 's44', 9), ('fwd', 0, 5, 84, 4, 8, 4, 32, {'u8': 1}, 's44', 8),
    ('fwd', 1, 2, 84, 4, 8, 4, 32, {'u8': 1}, 'c32', 1),                          # y < 128 KB: loader-fed u8
    ('fwd', 1, 3, 84, 4, 8, 4, 32, {'u8': 1}, 't32', 1),                          # row image in the workspace
    ('fwd', 1, 3, 84, 4, 8, 4, 32, {'u8': 1, 'ws_bytes': 1 << 16}, 'c32', 1),     # workspace too small for it
    ('fwd', 1, 3, 84, 4, 8, 4, 32, {'u8': 1, 'ws_off': 64}, 'c32', 1),            # workspace not 128-byte aligned
    ('fwd', 1, 5, 84, 4, 8, 4, 16, {'u8': 1}, 't32', 1),                          # Cout = 16: row image
    ('fwd', 1, 5, 84, 4, 8, 4, 32, {'u8': 1}, 't32', 1),
    ('fwd', 1, 256, 21, 32, 4, 2, 64, {}, 't64', 1), ('fwd', 1, 5, 21, 32, 4, 2, 64, {}, 't64', 2),
    ('fwd', 1, 256, 11, 64, 3, 1, 64, {}, 't64', 1), ('fwd', 1, 5, 11, 64, 3, 1, 64, {}, 't64', 2),
    ('fwd', 1, 1, 11, 64, 3, 1, 64, {}, 'c64', 2),                                # x < 128 KB: loader-fed
    ('fwd', 1, 5, 13, 32, 4, 2, 64, {}, 'c64', 2),
    ('fwd', 1, 5, 12, 8, 3, 2, 16, {}, 'c32', 1), ('fwd', 1, 13, 20, 32, 5, 2, 32, {}, 't32', 3),
    ('fwd', 1, 11, 17, 64, 3, 2, 96, {}, 't128', 2),
    ('fwd', 1, 256, 21, 32, 4, 2, 64, {'tma_off': True}, 'c64', 1),
]
CONV_WGRAD = [
    ('wgrad', 0, 2, 84, 4, 8, 4, 32, {'u8': 1}, 's44', 19),
    ('wgrad', 0, 256, 21, 32, 4, 2, 64, {}, 's44', 37), ('wgrad', 0, 5, 21, 32, 4, 2, 64, {}, 's44', 13),
    ('wgrad', 0, 256, 11, 64, 3, 1, 64, {}, 's44', 33), ('wgrad', 0, 7, 11, 64, 3, 1, 64, {'ws': None}, 's44', 1),
    ('wgrad', 0, 5, 13, 32, 4, 2, 64, {}, 's44', 6),
    ('wgrad', 0, 5, 12, 8, 3, 2, 16, {}, 's44', 4), ('wgrad', 0, 13, 20, 32, 5, 2, 32, {}, 's44', 21),
    ('wgrad', 0, 11, 17, 64, 3, 2, 96, {}, 's44', 14), ('wgrad', 0, 5, 84, 4, 8, 4, 32, {'u8': 1}, 's44', 46),
    ('wgrad', 1, 2, 84, 4, 8, 4, 32, {'u8': 1}, 'c32', 3),
    ('wgrad', 1, 3, 84, 4, 8, 4, 32, {'u8': 1}, 't32', 5),
    ('wgrad', 1, 5, 84, 4, 8, 4, 16, {'u8': 1}, 'c32', 7),                       # Cout = 16: no row image
    ('wgrad', 1, 5, 84, 4, 8, 4, 32, {'u8': 1}, 't32', 8),
    ('wgrad', 1, 256, 21, 32, 4, 2, 64, {}, 't64', 36), ('wgrad', 1, 5, 21, 32, 4, 2, 64, {}, 't64', 2),
    ('wgrad', 1, 256, 11, 64, 3, 1, 64, {}, 't64', 30), ('wgrad', 1, 5, 11, 64, 3, 1, 64, {}, 't64', 2),
    ('wgrad', 1, 5, 12, 8, 3, 2, 16, {}, 'c32', 1), ('wgrad', 1, 13, 20, 32, 5, 2, 32, {}, 't32', 5),
    ('wgrad', 1, 11, 17, 64, 3, 2, 96, {}, 't128', 3),
]
CONV_DGRAD = [
    ('dgrad', 0, 256, 21, 32, 4, 2, 64, {'mask': RELU}, 's84', 2),               # phases at stride 2
    ('dgrad', 0, 5, 21, 32, 4, 2, 64, {'mask': ELU}, 's44', 8),                  # split-K inside a phase
    ('dgrad', 0, 3, 84, 4, 8, 4, 32, {'mask': TANH}, 's44', 4),                   # stride 4, k = 8
    ('dgrad', 0, 256, 11, 64, 3, 1, 64, {'mask': RELU}, 's84', 2),                # stride 1: gather form
    ('dgrad', 0, 5, 11, 64, 3, 1, 64, {}, 's44', 18),
    ('dgrad', 0, 5, 21, 32, 4, 2, 64, {'ws': None}, 's44', 1),                    # no workspace: gather form
    ('dgrad', 0, 5, 13, 64, 1, 2, 32, {'mask': ELU}, 's44', 1),                   # kh < stride: gather form
    ('dgrad', 0, 5, 12, 8, 3, 2, 16, {}, 's44', 2), ('dgrad', 0, 13, 20, 32, 5, 2, 32, {'mask': TANH}, 's44', 9),
    ('dgrad', 0, 11, 17, 64, 3, 2, 96, {}, 's44', 12),
    ('dgrad', 1, 5, 21, 32, 4, 2, 64, {'mask': RELU}, 't32', 1),
    ('dgrad', 1, 5, 11, 64, 3, 1, 64, {'mask': ELU}, 't64', 1),
    ('dgrad', 1, 5, 11, 128, 3, 1, 128, {'mask': TANH}, 't128', 1),
    ('dgrad', 1, 256, 11, 64, 3, 1, 64, {'mask': RELU}, 't64', 1),
    ('dgrad', 1, 5, 12, 8, 3, 2, 16, {}, 'c32', 1), ('dgrad', 1, 5, 12, 16, 3, 2, 32, {'mask': TANH}, 'c32', 1),
    ('dgrad', 1, 5, 12, 32, 3, 3, 32, {'mask': ELU}, 'c32', 1),                   # stride 3: loader-fed
    ('dgrad', 1, 13, 20, 32, 5, 2, 32, {}, 't32', 1), ('dgrad', 1, 11, 17, 64, 3, 2, 96, {}, 't64', 1),
]


def _conv_id(row):
  entry, precision, B, H, C, k, s, Cout, opt = row[:9]
  return f'p{precision}-B{B}-H{H}-C{C}-k{k}-s{s}-Cout{Cout}' + ''.join(f'-{a}{v}' for a, v in opt.items())


def _conv_inputs(row, rng):
  entry, precision, B, H, C, k, s, Cout, opt = row[:9]
  path = conv_path(row)
  grid = grid_of(precision, path)
  if opt.get('u8'):
    frames = rng.integers(0, 256, (B, H, H, C), dtype=np.uint8)
    x = frames.astype(np.float32) / np.float32(255.)          # what the kernels compute from the frames (exact fp32)
    xd = dev(frames).data_ptr()
    c_op = 0. if precision == 0 else (2. ** -9 if path == 'tc' else 2. ** -10)
    return path, grid, x.astype(np.float64), xd, c_op
  x = on_grid(rng.standard_normal((B, H, H, C)), grid)
  return path, grid, x, fmat(x.reshape(-1, C)), 0.


def _conv_ws(opt):
  if opt.get('ws', True) is None:
    return None, None, 0
  ws = Workspace(off=opt.get('ws_off', 0), nbytes=opt.get('ws_bytes', WS_BYTES))
  return ws, ws.ptr, ws.bytes


def _conv_sig(row, path, tag, splits):
  entry, precision, B, H, C, k, s, Cout, opt = row[:9]
  u8 = bool(opt.get('u8'))
  if entry == 'fwd':
    lo = ('Im2colRows', 'DenseRed', 'false', 'false', f'Im2colRowsK<{"true" if u8 else "false"}>', 'RowMatK')
  elif entry == 'wgrad':
    lo = ('DenseOuter', 'Im2colCols', 'true', 'true', f'Im2colPixelsMN<{"true" if u8 else "false"}>', 'RowMatMN')
  else:
    lo = ('DgradRows', 'DgradWeights', '', '', 'DgradRowsK', 'DgradWMN')
  if entry == 'dgrad' and path == 'tma':
    return [f'tma_conv_dgrad_kernel<{C}>']
  want = [gemm_sig(path, tag, lo)] + (['splitk_finish_kernel'] if splits > 1 else [])
  if path == 'tma' and u8:
    want = ['u8_rows_to_f32_kernel'] + want
  if entry == 'dgrad' and path == 'simt':
    _, oh, _ = geom(B, H, C, k, s, Cout)
    wsb = 0 if opt.get('ws', True) is None else WS_BYTES
    if phased(s, k, wsb, B * H * H):
      want = ['dgrad_row_map_kernel']
      for _, _, Mp, Rp in phases(B, H, C, k, s, Cout):
        t, sp, _ = plan('simt', Mp, C, Rp, wsb - map_bytes(B * H * H))
        want += [f'gemm_kernel<DgradPhaseRows,DgradPhaseWeights,{t[1]},{t[2]}>'] + (['splitk_finish_kernel'] if sp > 1 else [])
  return want


@gpu
@pytest.mark.parametrize('row', CONV_FWD, ids=_conv_id)
def test_conv_fwd(row):
  entry, precision, B, H, C, k, s, Cout, opt, tag, splits = row
  c = _capi()
  lib = c.load()
  rng = np.random.default_rng(B + H + C + Cout + precision)
  g, oh, pad = geom(B, H, C, k, s, Cout)
  path, grid, x, xd, c_op = _conv_inputs(row, rng)
  K, M = k * k * C, B * oh * oh
  w = on_grid(rng.standard_normal((Cout, k, k, C)) / np.sqrt(K), grid)
  b = (rng.standard_normal(Cout) * 0.1).astype(np.float32).astype(np.float64)
  wd, bd = fmat(w.reshape(Cout, K)), dev(b.astype(np.float32)).data_ptr()
  ws, wsp, wsb = _conv_ws(opt)
  assert conv_plan(row) == (path, tag, splits)
  acc = conv_fwd_ref(x, w, k, s, H, oh, pad).reshape(M, Cout)
  absr = conv_fwd_ref(np.abs(x), np.abs(w), k, s, H, oh, pad).reshape(M, Cout) + np.abs(b)
  op = (c_op, absr) if c_op else None
  a = (RELU, ELU, TANH, NONE)[(B + H + precision) % 4]
  what = f'conv fwd p{precision} B{B} H{H} C{C} k{k} s{s} Cout{Cout} act {a}'
  y = Out(M, Cout, False)
  try:
    if opt.get('tma_off'):
      lib.b200rl_debug_set_tma(0)
    assert_sig(what, run(lambda: c.call('b200rl_conv2d_fwd', xd, opt.get('u8', 0), wd, bd, y.ptr, g, a, precision, wsp, wsb,
                                        stream())), _conv_sig(row, path, tag, splits))
  finally:
    lib.b200rl_debug_set_tma(1)
  ref = act(acc + b, a)
  _check(what, y.read(what), ref, absr, False, op=op)
  if ws is not None:
    if path == 'tma' and opt.get('u8'):
      ws.head = rows_head(ws, x, B, H, k, s, oh, pad)
    slabs = ws.slabs(what, M, Cout, splits)
    kps = plan(path, M, Cout, K, wsb)[2]
    for j in range(splits if splits > 1 else 0):
      lo, hi = j * kps, min(K, (j + 1) * kps)
      _check(f'{what} split {j} partial', slabs[j], conv_fwd_ref(x, wk(w, lo, hi), k, s, H, oh, pad).reshape(M, Cout),
             conv_fwd_ref(np.abs(x), np.abs(wk(w, lo, hi)), k, s, H, oh, pad).reshape(M, Cout), False, op=op)
  bf16_rejection(what, precision, path, lambda r: act(conv_fwd_ref(r(x), r(w), k, s, H, oh, pad).reshape(M, Cout) + b, a),
                 ref, absr, op)


@gpu
@pytest.mark.parametrize('row', CONV_WGRAD, ids=_conv_id)
def test_conv_wgrad(row):
  entry, precision, B, H, C, k, s, Cout, opt, tag, splits = row
  c = _capi()
  rng = np.random.default_rng(B + H + C + 3 * Cout + precision)
  g, oh, pad = geom(B, H, C, k, s, Cout)
  path, grid, x, xd, c_op = _conv_inputs(row, rng)
  K, P = k * k * C, B * oh * oh
  dy = on_grid(rng.standard_normal((B, oh, oh, Cout)), grid)
  dyd = fmat(dy.reshape(P, Cout))
  ws, wsp, wsb = _conv_ws(opt)
  assert conv_plan(row) == (path, tag, splits)
  ref = conv_wgrad_ref(x, dy, k, s, H, oh, pad, C).reshape(Cout, K)
  absr = conv_wgrad_ref(np.abs(x), np.abs(dy), k, s, H, oh, pad, C).reshape(Cout, K)
  op = (c_op, absr) if c_op else None
  what = f'conv wgrad p{precision} B{B} H{H} C{C} k{k} s{s} Cout{Cout}'
  want = _conv_sig(row, path, tag, splits)
  dw = Out(Cout, K, False)
  assert_sig(what, run(lambda: c.call('b200rl_conv2d_wgrad', xd, opt.get('u8', 0), dyd, dw.ptr, None, g, precision, wsp, wsb,
                                      stream())), want)
  _check(what, dw.read(what), ref, absr, False, op=op)
  kps = plan(path, Cout if path == 'simt' else K, K if path == 'simt' else Cout, P, wsb, pick_bn(Cout))[2]
  if ws is not None:
    # partial slabs of the product the path computes: [Cout][K] (FFMA), dW^T = [K][Cout] (tensor cores, stored untransposed)
    if path == 'tma' and opt.get('u8'):
      ws.head = rows_head(ws, x, B, H, k, s, oh, pad)
    slabs = ws.slabs(what, Cout, K, splits) if path == 'simt' else ws.slabs(what, K, Cout, splits)
    for j in range(splits if splits > 1 else 0):
      lo, hi = j * kps, min(P, (j + 1) * kps)
      pr, pa = (r.reshape(Cout, K) for r in wgrad_range(x, dy, lo, hi, k, s, H, oh, pad, C))
      if path != 'simt':
        pr, pa = pr.T, pa.T
      # FFMA sums exact x / 255; the tensor-core paths see the frames through their operand term, raw (unscaled) on the
      # loader-fed u8 kernel and through the row image on TMA
      _check(f'{what} split {j} partial (pixels {lo}..{hi})', slabs[j], pr, pa, False, op=(c_op, pa) if c_op else None)
  bf16_rejection(what, precision, path, lambda r: conv_wgrad_ref(r(x), r(dy), k, s, H, oh, pad, C).reshape(Cout, K), ref, absr, op)
  if P >= 1024:
    for how, lo, hi in drops(P, KE[path], splits, kps):
      d = np.zeros_like(dy).reshape(P, Cout)
      d[lo:hi] = dy.reshape(P, Cout)[lo:hi]
      lost = conv_wgrad_ref(x, d.reshape(dy.shape), k, s, H, oh, pad, C).reshape(Cout, K)
      _assert_rejects(f'{what} without {how}', ref, ref - lost, absr, False, op=op)
  # with the bias gradient: the same dw bit for bit, plus the column sum
  first = dw.bits()
  dw.reset()
  db = Out(1, Cout, False)
  cs = colsum_plan(P, Cout, Cout, True, wsb)[0]
  assert_sig(what + ' + db', run(lambda: c.call('b200rl_conv2d_wgrad', xd, opt.get('u8', 0), dyd, dw.ptr, db.ptr, g, precision,
                                                wsp, wsb, stream())), want + cs)
  assert bool((dw.bits() == first).all()), f'{what}: dw changed when db was requested'
  d2 = dy.reshape(P, Cout)
  _check(what + ' db', db.read(what + ' db')[0], d2.sum(0), np.abs(d2).sum(0), False)


@gpu
@pytest.mark.parametrize('row', CONV_DGRAD, ids=_conv_id)
def test_conv_dgrad(row):
  entry, precision, B, H, C, k, s, Cout, opt, tag, splits = row
  c = _capi()
  rng = np.random.default_rng(B + H + C + Cout + s + precision)
  g, oh, pad = geom(B, H, C, k, s, Cout)
  path = conv_path(row)
  grid = grid_of(precision, path)
  w = on_grid(rng.standard_normal((Cout, k, k, C)) / np.sqrt(k * k * Cout), grid)
  dy = on_grid(rng.standard_normal((B, oh, oh, Cout)), grid)
  wd, dyd = fmat(w.reshape(Cout, -1)), fmat(dy.reshape(-1, Cout))
  M = B * H * H
  ma = opt.get('mask')
  if ma is None:
    mptr, gm, ag = None, 1., 1.
  else:
    ym = mask_values(rng, (M, C), ma).astype(np.float32).astype(np.float64)
    mptr = fmat(ym)
    gm, ag = mask_factor(ym, ma)
  ws, wsp, wsb = _conv_ws(opt)
  assert conv_plan(row) == (path, tag, splits)
  acc = conv_dgrad_ref(dy, w, k, s, H, oh, pad).reshape(M, C)
  absr = conv_dgrad_ref(np.abs(dy), np.abs(w), k, s, H, oh, pad).reshape(M, C) * ag
  ref = acc * gm
  what = f'conv dgrad p{precision} B{B} H{H} C{C} k{k} s{s} Cout{Cout} mask {ma}'
  dx = Out(M, C, False)
  assert_sig(what, run(lambda: c.call('b200rl_conv2d_dgrad', dyd, wd, dx.ptr, g, mptr, ma or 0, precision, wsp, wsb, stream())),
             _conv_sig(row, path, tag, splits))
  _check(what, dx.read(what), ref, absr, False)
  if ws is not None:
    check_dgrad_workspace(what, ws, row, path, dy, w, oh, pad)
  bf16_rejection(what, precision, path, lambda r: conv_dgrad_ref(r(dy), r(w), k, s, H, oh, pad).reshape(M, C) * gm, ref, absr)
  red = cdiv(k, s) ** 2 * Cout     # reduction length of the largest stride phase
  if red >= 1024:
    co = np.zeros_like(w)
    co[:32, k // 2, k // 2] = w[:32, k // 2, k // 2]      # one 32-wide k-block: 32 output channels of one tap
    lost = conv_dgrad_ref(dy, co, k, s, H, oh, pad).reshape(M, C)
    _assert_rejects(f'{what} without one k-block', ref, (acc - lost) * gm, absr, False)


def check_dgrad_workspace(what, ws, row, path, dy, w, oh, pad):
  """TMA: the workspace is not used.  Gather form: [splits][pixels][C] partial slabs over the reduction (ky, kx, co).
  Stride phases: the row map at the head, then the slabs of the phase GEMMs, which all reuse one region: nothing past
  the largest of them is written, and the last phase that splits leaves its own slabs there, rows in row-map order."""
  import torch
  entry, precision, B, H, C, k, s, Cout, opt, tag, splits = row
  M = B * H * H
  if path == 'tma':
    ws.slabs(what, M, C, 1)
    return
  if not (path == 'simt' and phased(s, k, ws.bytes, M)):
    slabs = ws.slabs(what, M, C, splits)
    kps = plan(path, M, C, k * k * Cout, ws.bytes)[2]
    for j in range(splits if splits > 1 else 0):
      r = np.arange(j * kps, min(k * k * Cout, (j + 1) * kps))
      ref, absr = dgrad_taps(dy, w, r % Cout, r // Cout // k, r // Cout % k, k, s, H, oh, pad)
      _check(f'{what} split {j} partial', slabs[j], ref, absr, False)
    return
  words = ws.buf[ws.off:ws.off + ws.bytes].view(torch.int32).cpu().numpy()
  pix, head = phase_pixels(B, H, pad, s), map_bytes(M) // 4
  assert np.array_equal(words[:M], np.concatenate(pix)), f'{what}: row map'
  assert (words[M:head] == -1).all(), f'{what}: written between the row map and the partial slabs'
  plans = [(py, px, Mp, Rp) + plan('simt', Mp, C, Rp, ws.bytes - map_bytes(M))[1:] for py, px, Mp, Rp in phases(B, H, C, k, s, Cout)]
  assert [p[2] for p in plans] == [len(q) for q in pix], f'{what}: phase sizes'
  used = max([sp * Mp * C for _, _, Mp, _, sp, _ in plans if sp > 1], default=0)
  assert (words[head + used:] == -1).all(), f'{what}: workspace written past the partial slabs'
  split = [(p, q) for p, q in zip(plans, pix) if p[4] > 1]
  if not split:
    return
  (py, px, Mp, Rp, sp, kps), rows = split[-1]
  slabs = words[head:head + sp * Mp * C].view(np.float32).astype(np.float64).reshape(sp, Mp, C)
  ntx = cdiv(k - px, s)
  for j in range(sp):
    r = np.arange(j * kps, min(Rp, (j + 1) * kps))
    t2 = r // Cout
    ref, absr = dgrad_taps(dy, w, r % Cout, py + s * (t2 // ntx), px + s * (t2 % ntx), k, s, H, oh, pad)
    _check(f'{what} phase ({py}, {px}) split {j} partial', slabs[j], ref[rows], absr[rows], False)


@gpu
def test_conv1_row_image():
  """b200rl_conv2d_rows_from_u8 + x_u8 = 2 runs the TMA kernels on a shared row image and gives the bits of x_u8 = 1"""
  import torch
  c = _capi()
  lib = c.load()
  B, H, C, k, s, Cout = 5, 84, 4, 8, 4, 32
  g, oh, pad = geom(B, H, C, k, s, Cout)
  rng = np.random.default_rng(5)
  frames = dev(rng.integers(0, 256, (B, H, H, C), dtype=np.uint8)).data_ptr()
  w = on_grid(rng.standard_normal((Cout, k * k * C)) / 16., 'tf32')
  wd, bd = fmat(w), dev(rng.standard_normal(Cout).astype(np.float32)).data_ptr()
  P = B * oh * oh
  dyd = fmat(on_grid(rng.standard_normal((P, Cout)), 'tf32'))
  nbytes = int(lib.b200rl_conv2d_rows_bytes(ctypes.byref(g)))
  assert nbytes == rows_bytes(B, H, k, s)
  rows = torch.full((nbytes,), SENT, dtype=torch.uint8, device='cuda')
  assert_sig('rows_from_u8', run(lambda: c.call('b200rl_conv2d_rows_from_u8', frames, g, rows.data_ptr(), nbytes, stream())),
             ['u8_rows_to_f32_kernel'])
  ws = Workspace()
  outs = []
  for x, u8 in ((frames, 1), (rows.data_ptr(), 2)):
    y, dw, db = Out(P, Cout, False), Out(Cout, k * k * C, False), Out(1, Cout, False)
    assert_sig(f'conv1 fwd x_u8 {u8}', run(lambda: c.call('b200rl_conv2d_fwd', x, u8, wd, bd, y.ptr, g, RELU, 1, ws.ptr, ws.bytes,
                                                          stream())),
               (['u8_rows_to_f32_kernel'] if u8 == 1 else []) + ['tma_gemm_kernel<false,false,32,'])
    assert_sig(f'conv1 wgrad x_u8 {u8}', run(lambda: c.call('b200rl_conv2d_wgrad', x, u8, dyd, dw.ptr, db.ptr, g, 1, ws.ptr,
                                                            ws.bytes, stream())),
               (['u8_rows_to_f32_kernel'] if u8 == 1 else []) + ['tma_gemm_kernel<true,true,32,', 'splitk_finish_kernel',
                                                                 'colsum_vec_kernel<false>'])
    outs.append([o.read('conv1') for o in (y, dw, db)])
  for a, b in zip(*outs):
    assert np.array_equal(a, b), 'row image and frames give different results'


# ------------------------------------------------------------------------------ calls outside the kernels
@gpu
def test_misaligned_and_unsupported_calls_are_rejected():
  """EINVAL, nothing launched, output untouched.  The conv loaders read fp32 x, dy and w as 16-byte vectors and uint8
  frames as 4-byte pixels: a pointer off that alignment is refused at the entry point, for every precision."""
  import torch
  buf = torch.zeros(1 << 22, dtype=torch.float32, device='cuda')
  p = buf.data_ptr()
  ws = Workspace(nbytes=1 << 24)
  y = Out(4096, 256, False)
  lib = _capi().load()
  g1, _, _ = geom(2, 84, 4, 8, 4, 32)
  g2, _, _ = geom(2, 21, 32, 4, 2, 64)
  for precision in (0, 1):
    for off in (4, 8):
      _rejects(f'conv fwd p{precision} x + {off} B', 'b200rl_conv2d_fwd', y, p + off, 0, p, None, y.ptr, ctypes.byref(g2), RELU,
               precision, ws.ptr, ws.bytes, None)
      _rejects(f'conv wgrad p{precision} x + {off} B', 'b200rl_conv2d_wgrad', y, p + off, 0, p, y.ptr, None, ctypes.byref(g2),
               precision, ws.ptr, ws.bytes, None)
      _rejects(f'conv dgrad p{precision} dy + {off} B', 'b200rl_conv2d_dgrad', y, p + off, p, y.ptr, ctypes.byref(g2), None, 0,
               precision, ws.ptr, ws.bytes, None)
      _rejects(f'conv dgrad p{precision} w + {off} B', 'b200rl_conv2d_dgrad', y, p, p + off, y.ptr, ctypes.byref(g2), None, 0,
               precision, ws.ptr, ws.bytes, None)
    _rejects(f'conv1 fwd p{precision} frames + 2 B', 'b200rl_conv2d_fwd', y, p + 2, 1, p, None, y.ptr, ctypes.byref(g1), RELU,
             precision, ws.ptr, ws.bytes, None)
    _rejects(f'conv1 wgrad p{precision} frames + 1 B', 'b200rl_conv2d_wgrad', y, p + 1, 1, p, y.ptr, None, ctypes.byref(g1),
             precision, ws.ptr, ws.bytes, None)
  _rejects('rows_from_u8 frames + 2 B', 'b200rl_conv2d_rows_from_u8', y, p + 2, ctypes.byref(g1), y.ptr, 1 << 22, None)
  _rejects('row image at precision 0', 'b200rl_conv2d_fwd', y, p, 2, p, None, y.ptr, ctypes.byref(g1), RELU, 0, ws.ptr, ws.bytes,
           None)
  _rejects('row image wgrad at precision 0', 'b200rl_conv2d_wgrad', y, p, 2, p, y.ptr, None, ctypes.byref(g1), 0, ws.ptr,
           ws.bytes, None)
  g3, _, _ = geom(2, 12, 12, 3, 2, 32)
  _rejects('p1 conv dgrad C % 8 != 0', 'b200rl_conv2d_dgrad', y, p, p, y.ptr, ctypes.byref(g3), None, 0, 1, ws.ptr, ws.bytes, None)
  g4, _, _ = geom(2, 20, 16, 8, 2, 32)   # 8 x 8 x 32 = 2048 taps x channels > the 1024-entry tap table
  _rejects('p1 conv dgrad tap table', 'b200rl_conv2d_dgrad', y, p, p, y.ptr, ctypes.byref(g4), None, 0, 1, ws.ptr, ws.bytes, None)
  for precision in (2, 3, -1):
    _rejects(f'precision {precision}', 'b200rl_linear_fwd', y, 64, 64, 64, p, 64, p, None, y.ptr, 64, RELU, precision, ws.ptr,
             ws.bytes, None)
    _rejects(f'conv precision {precision}', 'b200rl_conv2d_fwd', y, p, 0, p, None, y.ptr, ctypes.byref(g2), RELU, precision,
             ws.ptr, ws.bytes, None)


# ------------------------------------------------------------------------------ launch order
@gpu
@pytest.mark.parametrize('precision', [0, 1])
def test_pdl_and_graph_capture_leave_results_bit_identical(precision):
  """fc1 forward -> data gradient -> weight + bias gradient, then conv3 data gradient -> conv2 weight + bias gradient on
  one stream: eager with programmatic dependent launch at its default, eager with it off, and captured in a CUDA graph
  (replayed twice) give the same bits.  Then two weight + bias gradients on two streams at once, each with its own
  workspace (the column sums take per-stream tickets), equal the two run one after the other."""
  import torch
  c = _capi()
  lib = c.load()
  rng = np.random.default_rng(11 + precision)
  M, N, K = 256, 1024 if precision else 512, 7744
  f = lambda *s: torch.empty(s, device='cuda')
  t = lambda a: dev(on_grid(a, 'tf32').astype(np.float32))
  x, w, b, dy = t(rng.standard_normal((M, K))), t(rng.standard_normal((N, K)) / 88.), t(rng.standard_normal(N)), \
      t(rng.standard_normal((M, N)))
  g3, _, _ = geom(M, 11, 64, 3, 1, 64)
  g2, _, _ = geom(M, 21, 32, 4, 2, 64)
  dy3, w3 = t(rng.standard_normal((M, 11, 11, 64))), t(rng.standard_normal((64, 3, 3, 64)) / 24.)
  m3, x2 = t(np.maximum(rng.standard_normal((M, 11, 11, 64)), 0)), t(np.maximum(rng.standard_normal((M, 21, 21, 32)), 0))
  ws = torch.zeros(WS_BYTES, dtype=torch.uint8, device='cuda')
  outs = dict(y=f(M, N), dx=f(M, K), dw=f(N, K), db=f(N), dx3=f(M, 11, 11, 64), dw2=f(64, 4, 4, 32), db2=f(64))
  o = {k: v.data_ptr() for k, v in outs.items()}

  def chain():
    st = stream()
    c.call('b200rl_linear_fwd', M, N, K, x.data_ptr(), K, w.data_ptr(), b.data_ptr(), o['y'], N, RELU, precision, ws.data_ptr(),
           WS_BYTES, st)
    c.call('b200rl_linear_dgrad', M, N, K, dy.data_ptr(), N, w.data_ptr(), o['dx'], K, x.data_ptr(), RELU, precision,
           ws.data_ptr(), WS_BYTES, st)
    c.call('b200rl_linear_wgrad', M, N, K, dy.data_ptr(), N, x.data_ptr(), K, o['dw'], o['db'], precision, ws.data_ptr(),
           WS_BYTES, st)
    c.call('b200rl_conv2d_dgrad', dy3.data_ptr(), w3.data_ptr(), o['dx3'], g3, m3.data_ptr(), RELU, precision, ws.data_ptr(),
           WS_BYTES, st)
    c.call('b200rl_conv2d_wgrad', x2.data_ptr(), 0, o['dx3'], o['dw2'], o['db2'], g2, precision, ws.data_ptr(), WS_BYTES, st)

  def snapshot():
    torch.cuda.synchronize()
    res = {k: v.clone() for k, v in outs.items()}
    for v in outs.values():
      v.view(torch.uint8).fill_(SENT)
    return res

  def same(a, bb, what):
    for k in a:
      assert torch.equal(a[k].view(torch.int32), bb[k].view(torch.int32)), f'{k} differs: {what}'

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
  # two weight + bias gradients concurrently on two streams (vector column sums with many CTAs each)
  shapes = ((4096, 64, 512), (8192, 128, 256))
  ins = [(t(rng.standard_normal((m, n))), t(rng.standard_normal((m, k)))) for m, n, k in shapes]
  dws, dbs = [f(n, k) for _, n, k in shapes], [f(n) for _, n, _ in shapes]
  wss = [torch.empty(WS_BYTES, dtype=torch.uint8, device='cuda') for _ in shapes]

  def wgrad(i, st):
    (m, n, k), (dyi, xi) = shapes[i], ins[i]
    c.call('b200rl_linear_wgrad', m, n, k, dyi.data_ptr(), n, xi.data_ptr(), k, dws[i].data_ptr(), dbs[i].data_ptr(), precision,
           wss[i].data_ptr(), WS_BYTES, st)

  for i in range(2):
    wgrad(i, stream())
  torch.cuda.synchronize()
  serial = [(a.clone(), bb.clone()) for a, bb in zip(dws, dbs)]
  for a in dws + dbs:
    a.fill_(float('nan'))
  streams = [torch.cuda.Stream() for _ in shapes]
  for i, st in enumerate(streams):
    st.wait_stream(torch.cuda.current_stream())
    wgrad(i, st.cuda_stream)
  torch.cuda.synchronize()
  for i in range(2):
    assert torch.equal(dws[i], serial[i][0]) and torch.equal(dbs[i], serial[i][1]), \
        f'wgrad {shapes[i]} differs when run beside another one'
