#!/usr/bin/env python
"""bench.py — the reference's headline metric on B200: DQN learner updates/s (and PER samples/s) on
the Atari-shaped workload of BASELINE.json configs[1]:
  uint8 84x84x4 observations, prioritized replay of 1,000,000 steps (alpha 0.6), batch 256, n-step 3,
  DQNAtariNetwork(18), Adam 1e-3, IS exponent 0.2, target period 100, synthetic data, random init.

One "step" = one full learner update (K1 sample -> K3 gather/n-step -> 3 forwards -> K4 -> backward ->
K7 Adam -> K2 priority write-back -> target copy) over one batch per rank.

  python bench.py [--gpus N --steps K --warmup W]          our arm (one rank per GPU under torchrun)
  python bench.py --impl reference [...]                  the reference's CPU path (oracle port), host cores
  python bench.py --dump-outputs DIR [...]                also write what the last timed update computed, DIR/<name>.npy

Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for what each key means.
"""

from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
  sys.path.insert(0, ROOT)

METRIC = 'learner_updates_per_sec_dqn_atari_b256'
UNIT = 'updates/s (one update = 256 transitions; N ranks do N x 256 per data-parallel step)'
OBS_SHAPE = (84, 84, 4)
NUM_ACTIONS = 18
STEP_FLOPS = 5 * 2 * 19_977_728 * 256     # 3 fwd + bwd(2x) of 19.98 MMAC/sample at B=256 (SURVEY App. B)


def peaks():
  p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
  if os.path.exists(p):
    d = json.load(open(p))
    return dict(hbm=d['hbm_gbs'], tf_burst=d['bf16_tflops'], tf_sustained=d['bf16_tflops_sustained'], src='measured')
  return dict(hbm=6650.0, tf_burst=1590.0, tf_sustained=1400.0, src='fallback')


# ------------------------------------------------------------------------------ synthetic workload
class SynthStream:
  """Host-side scalars of a synthetic actor stream (SURVEY §8d, C2): actions U{0..17}, rewards in
  {-1,0,1} w.p. {.05,.9,.05}, env discount 1 except 0 w.p. 1/1000, geometric episode lengths (mean
  ~1000 steps).  Element i is one observation slot; first/last mark episode boundaries and stay
  consistent across chunk boundaries."""

  def __init__(self, seed, mean_episode=1000):
    self.rng = np.random.default_rng(seed)
    self.mean = mean_episode
    self.left = 0          # slots left in the current episode (0 = next slot starts a new one)

  def chunk(self, n):
    rng = self.rng
    act = rng.integers(0, NUM_ACTIONS, n).astype(np.int32)
    rew = rng.choice(np.array([-1., 0., 1.], np.float32), n, p=[.05, .9, .05]).astype(np.float32)
    disc = np.where(rng.random(n) < 1e-3, 0., 1.).astype(np.float32)
    first, last = np.zeros(n, np.uint8), np.zeros(n, np.uint8)
    i = 0
    while i < n:
      if self.left == 0:
        self.left = int(rng.geometric(1.0 / self.mean)) + 1      # T steps -> T+1 slots, T >= 1
        first[i] = 1
      take = min(self.left, n - i)
      self.left -= take
      i += take
      if self.left == 0:
        last[i - 1] = 1
    return act, rew, disc, first, last


def fill_replay(table, steps, n_step, seed, chunk=32768, single_frames=False):
  """Fills the HBM ring with `steps` synthetic timesteps (observations generated on the device:
  setup only, not timed) and then sets priorities to |N(0,1)| like SURVEY §8d."""
  import ctypes as C
  import torch
  from acme_b200 import _capi
  stream = SynthStream(seed)
  wid = C.c_int32()
  _capi.call('b200rl_writer_open', table.handle, C.byref(wid))
  gen = torch.Generator(device='cuda')
  gen.manual_seed(seed)
  done = 0
  while done < steps:
    n = min(chunk, steps - done)
    act, rew, disc, first, last = stream.chunk(n)
    # frame-deduplicated table: the ring stores one 84x84 frame per step; feed it single frames (obs_on_device = 2)
    shape = (n, OBS_SHAPE[0] * OBS_SHAPE[1]) if single_frames else (n,) + OBS_SHAPE
    obs = torch.randint(0, 256, shape, dtype=torch.uint8, device='cuda', generator=gen)
    _capi.call('b200rl_writer_append_stream', table.handle, wid.value, n, obs.data_ptr(), 2 if single_frames else 1, act.ctypes.data,
               rew.ctypes.data, disc.ctypes.data, first.ctypes.data, last.ctypes.data, n_step, 1.0,
               _capi.current_stream())
    torch.cuda.synchronize()
    del obs
    done += n
  info = table.info()
  size, tail = info['size'], info['tail_key']
  keys = (torch.arange(size, dtype=torch.int64, device='cuda') + tail).view(torch.uint64)
  pr = torch.randn(size, device='cuda', generator=gen).abs_()
  table.update_priorities_device(keys, pr)
  torch.cuda.synchronize()
  return info


def fill_replay_control(table, steps, n_step, seed, obs_dim, act_dim, chunk=65536):
  """C3 (SURVEY §8d): obs f32[obs_dim] ~ N(0,1), act f32[act_dim] ~ U(-1,1), reward ~ U(0,1), env discount 1 except 0
  w.p. 1/1000, ~1000-step episodes; observations generated on the device (set-up, not timed)."""
  import ctypes as C
  import torch
  from acme_b200 import _capi
  stream = SynthStream(seed)
  wid = C.c_int32()
  _capi.call('b200rl_writer_open', table.handle, C.byref(wid))
  gen = torch.Generator(device='cuda')
  gen.manual_seed(seed)
  rng = np.random.default_rng(seed)
  done = 0
  while done < steps:
    n = min(chunk, steps - done)
    _, _, disc, first, last = stream.chunk(n)
    act = rng.uniform(-1, 1, (n, act_dim)).astype(np.float32)
    rew = rng.random(n, dtype=np.float32)
    obs = torch.randn((n, obs_dim), dtype=torch.float32, device='cuda', generator=gen)
    _capi.call('b200rl_writer_append_stream', table.handle, wid.value, n, obs.data_ptr(), 1, act.ctypes.data, rew.ctypes.data,
               disc.ctypes.data, first.ctypes.data, last.ctypes.data, n_step, 1.0, _capi.current_stream())
    torch.cuda.synchronize()
    done += n
  return table.info()


# ------------------------------------------------------------------------------ clocks sampler
class ClockSampler:
  """nvidia-smi sampler (the recipe's clocks line).  It is started before the warm-up and samples every 50 ms;
  `mark()` brackets the timed region so only samples taken inside it are summarised (if the region is shorter
  than the sampling period, the samples nearest to it are used)."""
  Q = ('timestamp,index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
       'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
       'clocks_event_reasons.sw_power_cap')

  def __init__(self, gpu_index=0):
    self.f = tempfile.NamedTemporaryFile('w+', suffix='.csv', delete=False)
    self.p = None
    self.t0 = self.t1 = None
    try:
      self.p = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits', '-lms', '50',
                                 '-i', str(gpu_index)], stdout=self.f, stderr=subprocess.DEVNULL)
    except Exception:  # noqa: BLE001
      self.p = None

  def mark(self):
    if self.t0 is None:
      self.t0 = time.time()
    else:
      self.t1 = time.time()

  def stop(self):
    import datetime
    if self.p is None:
      return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
    time.sleep(0.12)
    self.p.terminate()
    self.p.wait()
    self.f.flush()
    rows = [r.strip().split(', ') for r in open(self.f.name) if r.strip()]
    os.unlink(self.f.name)
    samples = []
    for r in rows:
      try:
        ts = datetime.datetime.strptime(r[0].strip(), '%Y/%m/%d %H:%M:%S.%f').timestamp()
        samples.append((ts, float(r[2]), float(r[3]), [v.strip().lower().startswith('active') for v in r[6:10]]))
      except Exception:  # noqa: BLE001
        continue
    if not samples:
      return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['no samples']}
    t0, t1 = self.t0 or samples[0][0], self.t1 or samples[-1][0]
    inside = [x for x in samples if t0 - 0.05 <= x[0] <= t1 + 0.05]
    if not inside:   # region shorter than the sampling period: take the two samples nearest to it
      inside = sorted(samples, key=lambda x: abs(x[0] - 0.5 * (t0 + t1)))[:2]
    names = ('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap')
    reasons = sorted({n for x in inside for n, on in zip(names, x[3]) if on})
    return {'sm_mhz': float(np.median([x[1] for x in inside])), 'sm_max_mhz': float(max(x[2] for x in inside)),
            'reasons': reasons, 'samples': len(inside)}


# ------------------------------------------------------------------------------ CPU baseline / reference arm
class CpuReferencePath:
  """The reference's CPU path restated (BASELINE.md §3): binary f64 sum-tree sample + update
  (Reverb Prioritized-like), NumPy gather + n-step, PyTorch-CPU DQN learner step (oracle.learner).
  Bounded sample of the workload: same tree size (1M priorities), same batch/network, observation
  ring of `ring` steps (28 KB/step makes a 1M-step host ring impractical)."""

  def __init__(self, items=1_000_000, ring=16384, batch=256, n_step=3, seed=0, threads=None):
    import torch
    from oracle import learner as olearner
    from oracle import nets as onets
    from oracle import sumtree
    self.threads = threads or os.cpu_count()
    torch.set_num_threads(self.threads)
    rng = np.random.default_rng(seed)
    self.rng, self.B, self.n, self.ring, self.items = rng, batch, n_step, ring, items
    self.tree = sumtree.BinarySumTreeF64(items)
    self.tree.build(np.abs(rng.standard_normal(items))**0.6)
    self.obs = rng.integers(0, 256, (ring,) + OBS_SHAPE, dtype=np.uint8)
    self.act, self.rew, self.disc, _, _ = SynthStream(seed).chunk(ring)
    net, tgt = onets.DQNAtariNetwork(NUM_ACTIONS, seed=seed), onets.DQNAtariNetwork(NUM_ACTIONS, seed=seed)
    tgt.copy_from(net)
    self.learner = olearner.DQNOracleLearner(net, tgt, 0.99, 0.2, 1e-3, 100)
    self.g = np.float32(0.99)

  def step(self):
    u = self.rng.random(self.B)
    idx, prob = self.tree.sample(u)                       # 256 root-to-leaf walks
    s = idx % (self.ring - self.n - 1)
    R = self.rew[s].copy()
    D = self.disc[s].copy()
    for j in range(1, self.n):                            # transition.py:135-145, vectorised over the batch
      D = D * self.g
      R = R + self.rew[s + j] * D
      D = D * self.disc[s + j]
    out = self.learner.step(self.obs[s], self.act[s], R, D, self.obs[s + self.n], prob.astype(np.float32))
    self.tree.set(idx, out['priority']**0.6)              # update_priorities
    return float(out['loss'])


D4PG_METRIC = 'learner_updates_per_sec_d4pg_control_b256'
D4PG_UNIT = 'updates/s (one update = 256 transitions; N ranks do N x 256 per data-parallel step)'
D4PG_WORKLOAD = 'D4PG control-suite humanoid-shaped 67-d obs / 21-d act, C51 critic (51 atoms), uniform replay 1M items, batch 256, n=5 (BASELINE configs[2])'
OBS_DIM, ACT_DIM, ATOMS = 67, 21, 51
# MACs per sample (SURVEY App. B): critic 451,328, policy 153,600; step = 3 critic fwd + 2 policy fwd + critic bwd (2x) +
# critic dgrad-only (1x) + policy bwd (2x)
D4PG_STEP_FLOPS = 2 * (3 * 451_328 + 2 * 153_600 + 2 * 451_328 + 451_328 + 2 * 153_600) * 256
TREE_METRIC = 'per_samples_per_sec_sumtree_sweep'
TREE_UNIT = 'prioritized samples/s (K1 draws, whole job; one step = one stratified draw of B per rank + the priority update of the drawn items)'


class CpuD4PGPath:
  """The reference's CPU path of C3 restated: NumPy gather + n-step over a host ring, PyTorch-CPU D4PG learner
  (oracle.learner.D4PGOracleLearner: dense l2_project, CE, DPG with dq/da clipping, global-norm clip, two Adams)."""

  def __init__(self, ring=65536, batch=256, n_step=5, seed=0, threads=None):
    import torch
    from oracle import learner as olearner
    from oracle import nets as onets
    self.threads = threads or os.cpu_count()
    torch.set_num_threads(self.threads)
    rng = np.random.default_rng(seed)
    self.rng, self.B, self.n, self.ring = rng, batch, n_step, ring
    self.obs = rng.standard_normal((ring, OBS_DIM)).astype(np.float32)
    self.act = rng.uniform(-1, 1, (ring, ACT_DIM)).astype(np.float32)
    self.rew = rng.random(ring, dtype=np.float32)
    self.disc = np.where(rng.random(ring) < 1e-3, 0., 1.).astype(np.float32)
    pol, cri = onets.D4PGPolicy(OBS_DIM, ACT_DIM, seed=seed), onets.D4PGCritic(OBS_DIM, ACT_DIM, seed=seed + 1)
    tp, tc = onets.D4PGPolicy(OBS_DIM, ACT_DIM, seed=seed), onets.D4PGCritic(OBS_DIM, ACT_DIM, seed=seed + 1)
    self.learner = olearner.D4PGOracleLearner(pol, cri, tp, tc, 0.99, 100)
    self.g = np.float32(0.99)

  def step(self):
    s = self.rng.integers(0, self.ring - self.n - 1, self.B)       # uniform table
    R, D = self.rew[s].copy(), self.disc[s].copy()
    for j in range(1, self.n):
      D = D * self.g
      R = R + self.rew[s + j] * D
      D = D * self.disc[s + j]
    out = self.learner.step(self.obs[s], self.act[s], R, D, self.obs[s + self.n])
    return float(out['critic_loss'])


class CpuTreePath:
  """Reverb-Prioritized-like binary f64 sum tree on the host: B root-to-leaf walks + B leaf updates per step."""

  def __init__(self, items, batch, seed=0):
    from oracle import sumtree
    self.rng = np.random.default_rng(seed)
    self.tree = sumtree.BinarySumTreeF64(items)
    self.tree.build(np.abs(self.rng.standard_normal(items))**0.6)
    self.B = batch
    self.threads = 1

  def step(self):
    idx, _ = self.tree.sample(self.rng.random(self.B))
    self.tree.set(idx, np.abs(self.rng.standard_normal(self.B))**0.6)


def parity_record(precision: int):
  """The bench line's `parity` object: which arithmetic mode was timed, the tolerance stated (and asserted) for it by
  `tests/test_gpu_learner.py::test_dqn_learner_c2_shape_parity` against the fp32 oracle at the benchmarked shapes (B=256,
  A=18, three updates on injected uniforms), and the largest error that test measured on B200 (committed
  `profiles/parity_c2_<mode>.json`, written by the test itself; not re-measured in this run -- bench.py's own arm never
  executes the oracle)."""
  mode = {0: 'fp32', 1: 'tf32', 2: 'bf16'}[precision]
  rec = {'mode': mode, 'oracle': 'oracle/learner.py (fp32 restatement of dqn/learning.py:121-154)',
         'sampled_indices_and_nstep_bookkeeping': 'bit-exact (all modes)', 'tol': None, 'max_rel_err_td': None, 'source': None}
  path = os.path.join(ROOT, 'profiles', f'parity_c2_{mode}.json')
  try:
    d = json.load(open(path))
    runs = d['measured']
    worst = lambda k: max(float(r[k]) for r in runs)
    rec.update(tol=d['tolerances'], max_rel_err_td=worst('td'), max_rel_err_loss=worst('loss'), max_rel_err_priority=worst('priority'),
               max_grad_rel_l2=max(max(float(v) for v in r['grad_rel_l2'].values()) for r in runs),
               shape={'B': d['B'], 'A': d['A'], 'updates': len(runs)},
               source=f'profiles/parity_c2_{mode}.json (tests/test_gpu_learner.py, measured on B200; errors are relative to the tensor scale)')
  except (OSError, KeyError, ValueError, TypeError):
    pass
  return rec


def _cpu_model():
  cpu = open('/proc/cpuinfo').read()
  return next((l.split(':', 1)[1].strip() for l in cpu.splitlines() if l.startswith('model name')), 'unknown')


def run_reference_other(args):
  """Reference arm of the d4pg / sumtree workloads (rank 0 only): the CPU restatement on the host cores."""
  if int(os.environ.get('RANK', '0')) != 0:
    return
  t0 = time.time()
  if args.workload == 'd4pg':
    ref, metric, unit, workload, per_step = CpuD4PGPath(seed=1234), D4PG_METRIC, D4PG_UNIT, D4PG_WORKLOAD, 1.0
    sample = (f'{args.steps} full D4PG learner updates (B=256, critic (512,512,256)+51 atoms, policy (256,256,256)), NumPy n-step over a '
              f'{ref.ring}-step host ring, PyTorch-CPU, {ref.threads} threads, {_cpu_model()}')
  else:
    Bt = min(args.tree_batch, 1 << 16)      # bounded sample: the host tree walks ~1e5 samples/s
    ref, metric, unit, per_step = CpuTreePath(min(args.items, 4_000_000), Bt, seed=1234), TREE_METRIC, TREE_UNIT, float(Bt)
    workload = f'sum-tree sweep point: {args.items:,} items per rank, {args.tree_batch:,} draws + updates per step (BASELINE configs[3])'
    sample = (f'{args.steps} steps of {Bt:,} draws + {Bt:,} updates on a binary f64 NumPy sum tree over {ref.tree.n if hasattr(ref.tree, "n") else min(args.items, 4_000_000):,} '
              f'priorities (bounded: the GPU arm uses {args.items:,} items and {args.tree_batch:,} draws per step), 1 thread, {_cpu_model()}')
  for _ in range(args.warmup):
    ref.step()
  t1 = time.time()
  for _ in range(args.steps):
    ref.step()
  dt = (time.time() - t1) / max(args.steps, 1)
  value = per_step / dt
  print(json.dumps({
      'impl': 'reference', 'metric': metric, 'value': value, 'unit': unit, 'n_gpus': args.gpus, 'steps': args.steps,
      'warmup': args.warmup, 'ms_per_step': dt * 1e3, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
      'dtype': 'f32' if args.workload == 'd4pg' else 'f64', 'data': 'synthetic',
      'config': {'workload': workload, 'note': 'reference arm = CPU restatement (oracle port); Acme TF/JAX + Reverb are not installable offline'},
      'cpu_baseline': {'value': value, 'unit': unit.split(' (')[0], 'cores': ref.threads, 'kind': 'port', 'sample': sample},
      'e2e': {'value': value, 'unit': unit.split(' (')[0], 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
      'setup_s': t1 - t0,
  }))


def run_reference(args):
  rank = int(os.environ.get('RANK', '0'))
  if rank != 0:
    return
  t0 = time.time()
  ref = CpuReferencePath(seed=1234)
  for _ in range(args.warmup):
    ref.step()
  t1 = time.time()
  for _ in range(args.steps):
    ref.step()
  dt = (time.time() - t1) / max(args.steps, 1)
  cpu = open('/proc/cpuinfo').read()
  model = next((l.split(':', 1)[1].strip() for l in cpu.splitlines() if l.startswith('model name')), 'unknown')
  value = 1.0 / dt
  sample = (f'{args.steps} full learner updates (B=256, DQNAtariNetwork(18), binary f64 sum-tree over 1M priorities, '
            f'{ref.ring}-step uint8 observation ring), PyTorch-CPU + NumPy, {ref.threads} threads, {model}')
  print(json.dumps({
      'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': args.steps,
      'warmup': args.warmup, 'ms_per_step': dt * 1e3, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
      'dtype': 'f32', 'data': 'synthetic',
      'config': {'workload': 'DQN Atari-shaped 84x84x4 uint8, PER 1M items, batch 256, n=3 (BASELINE configs[1])',
                 'items_per_rank': ref.items, 'batch_per_rank': ref.B, 'n_step': ref.n, 'alpha': 0.6, 'beta': 0.2,
                 'network': 'DQNAtariNetwork(18), 8,018,611 params', 'optimizer': 'Adam 1e-3',
                 'replay_ring': f'host ring of {ref.ring} uint8 84x84x4 steps under the 1M-priority tree (bounded sample: a 1M-step '
                                'host ring would be 28 GB)',
                 'parallelism': 'host cores of rank 0', 'cuda_graph': False,
                 'note': 'reference arm = CPU restatement (oracle port); Acme TF/JAX + Reverb are not installable offline'},
      'cpu_baseline': {'value': value, 'unit': 'updates/s', 'cores': ref.threads, 'kind': 'port', 'sample': sample},
      'e2e': {'value': value, 'unit': 'updates/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
      'setup_s': t1 - t0,
  }))


# ------------------------------------------------------------------------------ our arm
def time_stage(fn, iters, torch):
  """Average device time of fn() over `iters` calls, CUDA events on the current stream."""
  fn()
  torch.cuda.synchronize()
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  e0.record()
  for _ in range(iters):
    fn()
  e1.record()
  torch.cuda.synchronize()
  return e0.elapsed_time(e1) / iters * 1e-3


DUMP_BUDGET = 64_000_000
DUMP_SAMPLE = 1 << 20


def dump_outputs(out_dir, arrays):
  """Writes each array as `out_dir/<name>.npy` for output-by-output comparison of two builds.  Floating-point arrays
  are stored as float32, integer arrays (indices, keys) as float64, which holds them exactly below 2**53."""
  arrays = {k: np.asarray(v) for k, v in arrays.items()}
  arrays = {k: v.astype(np.float64 if v.dtype.kind in 'iub' else np.float32) for k, v in arrays.items()}
  total = sum(v.nbytes for v in arrays.values())
  if total > DUMP_BUDGET:
    raise ValueError(f'--dump-outputs: {total} bytes exceed the {DUMP_BUDGET} byte budget')
  os.makedirs(out_dir, exist_ok=True)
  for name, v in arrays.items():
    np.save(os.path.join(out_dir, f'{name}.npy'), v)


def dqn_outputs(learner, ds, net, tgt):
  """What the last DQN update handed its caller: loss, TD errors, importance weights, the priorities written back,
  the sampled items and q(o_tm1), plus the updated state (online parameters in full; target parameters and Adam
  moments as a fixed, seeded sample of DUMP_SAMPLE positions, which keeps the dump inside DUMP_BUDGET; the update
  count)."""
  import torch
  torch.cuda.synchronize()
  pick = torch.as_tensor(np.sort(np.random.default_rng(0).choice(net.params.size, DUMP_SAMPLE, replace=False)),
                         device=net.params.flat.device)
  host = lambda t: t.detach().cpu().numpy()
  return {
      'loss': host(learner.loss), 'td_error': host(learner.td), 'importance_weight': host(learner.weight),
      'priority': host(learner.priority), 'q_tm1': host(learner.q_values()[0]),
      'sample_index': host(ds.idx), 'sample_key': host(ds.keys.view(torch.int64)), 'sample_prob': host(ds.prob),
      'online_params': host(net.params.flat), 'target_params_sample': host(tgt.params.flat[pick]),
      'adam_m_sample': host(learner._m[pick]), 'adam_v_sample': host(learner._v[pick]),
      'num_steps': host(learner._num_steps),
  }


def run_ours(args):
  import torch
  import torch.distributed as dist
  from acme_b200 import _capi, adders, dm_env, dqn, loggers, networks, replay, specs

  rank, world, local = int(os.environ.get('RANK', '0')), int(os.environ.get('WORLD_SIZE', '1')), int(os.environ.get('LOCAL_RANK', '0'))
  torch.cuda.set_device(local)
  _capi.require_device(local)
  pg = None
  if world > 1:
    dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    pg = dist.group.WORLD
  P = peaks()
  B, n_step, items = 256, 3, args.items
  precision = {'fp32': _capi.PRECISION_FP32, 'tf32': _capi.PRECISION_TC, 'tc': _capi.PRECISION_TC,
               'bf16': _capi.PRECISION_BF16FLOW}[args.precision]

  spec = specs.EnvironmentSpec(specs.Array(OBS_SHAPE, np.uint8), specs.DiscreteArray(NUM_ACTIONS),
                               specs.Array((), np.float32), specs.BoundedArray((), np.float32, 0., 1.))
  table = replay.Table(replay.DEFAULT_PRIORITY_TABLE, replay.selectors.Prioritized(0.6), replay.selectors.Fifo(),
                       max_size=items, rate_limiter=replay.rate_limiters.MinSize(1),
                       signature=adders.NStepTransitionAdder.signature(spec), max_window=n_step, discount=0.99,
                       device=local, slot_capacity=items + 4096, shard_count=world, shard_rank=rank, stage_slots=4096,
                       frame_stack=4 if args.frame_dedup else 0)
  server = replay.Server([table])
  t_setup = time.time()
  info = fill_replay(table, items, n_step, seed=1234 + rank, single_frames=args.frame_dedup)
  net = networks.DQNAtariNetwork(NUM_ACTIONS, device=local, precision=precision, seed=1234)   # replicated init
  tgt = net.clone()
  ds = replay.ReplayDataset(table, B, seed=1234 + rank)
  client = replay.Client(server)
  learner = dqn.DQNLearner(net, tgt, 0.99, 0.2, 1e-3, 100, ds, replay_client=client, logger=loggers.NoOpLogger(),
                           process_group=pg, use_cuda_graph=not args.no_graph)
  adder = adders.NStepTransitionAdder(client, n_step=n_step, discount=0.99)
  t_setup = time.time() - t_setup
  lib = _capi.load()

  def barrier():
    if world > 1:
      dist.barrier()
    torch.cuda.synchronize()

  # ---- device-resident timing (value)
  clocks = ClockSampler(local)
  for _ in range(max(args.warmup, 3)):
    learner.step(fetch_loss=False)
  barrier()
  launches0 = lib.b200rl_launch_count()
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  barrier()
  clocks.mark()
  if args.profile:
    torch.cuda.profiler.start()     # ncu --profile-from-start off: only the timed learner steps are captured
  e0.record()
  for _ in range(args.steps):
    learner.step(fetch_loss=False)
  learner.flush()                   # pipelined data-parallel exchange: the last update is applied inside the timed region
  e1.record()
  barrier()
  if args.profile:
    torch.cuda.profiler.stop()
  clocks.mark()
  dev_s = e0.elapsed_time(e1) * 1e-3
  clk = clocks.stop()
  if world > 1:
    tt = torch.tensor([dev_s], device='cuda')
    dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    dev_s = float(tt)
  ms_per_step = dev_s / args.steps * 1e3
  value = world * args.steps / dev_s
  if args.dump_outputs and rank == 0:     # before the end-to-end leg below moves the learner on
    dump_outputs(args.dump_outputs, dqn_outputs(learner, ds, net, tgt))

  if args.profile:
    if rank == 0:
      print(json.dumps({'metric': METRIC, 'value': value, 'ms_per_step': ms_per_step, 'profile_run': True}))
    server.stop()
    if world > 1:
      dist.destroy_process_group()
    return

  # ---- end to end through the public API with host buffers: the reference loop's cadence is 8
  #      environment steps inserted per learner step (batch 256 / samples_per_insert 32, dqn/agent.py:158-162)
  rng = np.random.default_rng(99 + rank)
  host_obs = [rng.integers(0, 256, OBS_SHAPE, dtype=np.uint8) for _ in range(64)]
  inserts_per_step = 8
  adder.add_first(dm_env.restart(host_obs[0]))

  def e2e_step(i):
    for j in range(inserts_per_step):
      o = host_obs[(i * inserts_per_step + j + 1) % 64]
      adder.add(np.int32(j % NUM_ACTIONS), dm_env.transition(np.float32(0.), o, np.float32(1.)))
    # flush (H2D of the staged steps) + update + D2H of the loss into pinned memory; the loss of update i is consumed
    # (logged) when update i+1 has been issued, so the host-side inserts overlap the device step
    learner.step(fetch_loss='async')

  for i in range(10):   # warm-up: pinned staging, both staging sets, the async-loss ring
    e2e_step(i)
  barrier()
  t0 = time.perf_counter()
  e2e_steps = args.steps
  for i in range(e2e_steps):
    e2e_step(i + 3)
  learner.flush()
  last_loss = learner.drain()            # the final update's loss, read inside the timed region
  assert last_loss is not None and np.isfinite(last_loss)
  barrier()
  e2e_s = time.perf_counter() - t0
  if world > 1:
    tt = torch.tensor([e2e_s], device='cuda')
    dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    e2e_s = float(tt)
  e2e_value = world * e2e_steps / e2e_s
  obs_h2d = int(np.prod(OBS_SHAPE)) // (4 if args.frame_dedup else 1)       # a frame-deduplicated table uploads one frame per step
  h2d = inserts_per_step * (obs_h2d + 4 + 4 + 4 + 4) + inserts_per_step * 24 + 16
  d2h = 4

  # ---- per-stage device times (eager launches, CUDA events) and the roofline of the dominant kernel
  stages = {}
  if rank == 0:
    it = 20
    u = torch.rand(B, device='cuda')
    stages['k1_sample'] = time_stage(lambda: table.sample_into(u, ds.idx, ds.keys, ds.prob, True), it, torch)
    stages['k3_gather_nstep'] = time_stage(lambda: table.gather_into(ds.idx, ds.o_tm1, ds.a_tm1, ds.R, ds.D, ds.o_t), it, torch)
    # the network group exactly as the step runs it: target pass beside the batched online pass, then the fused
    # head + K4 kernel and the backward (weight gradients beside data gradients), recorded into ONE graph and replayed,
    # so the figure is the in-step time of the group, not a sum of serialised eager launches
    def join_tail():     # B200RL_SPLIT_ADAM=1 forks the fc1 + head optimizer update inside the backward: rejoin for the capture
      if getattr(learner, '_tail_done', None) is not None:
        torch.cuda.current_stream().wait_event(learner._tail_done)
        learner._tail_done = None
    g_fwd = learner._capture(learner._forwards)
    g_bwd = learner._capture(lambda: (learner._loss_backward(), join_tail()))
    g_net = learner._capture(lambda: (learner._forwards(), learner._loss_backward(), join_tail()))
    stages['k6_forwards_in_graph'] = time_stage(g_fwd.replay, it, torch)
    stages['k4_k6_loss_backward_in_graph'] = time_stage(g_bwd.replay, it, torch)
    stages['k6_network_group_in_graph'] = time_stage(g_net.replay, it, torch)
    Pn = net.params
    scratch_p, scratch_m, scratch_v = torch.zeros_like(Pn.flat), torch.zeros_like(Pn.flat), torch.zeros_like(Pn.flat)
    stages['k7_adam'] = time_stage(lambda: _capi.call(
        'b200rl_adam', Pn.size, scratch_p.data_ptr(), Pn.grad.data_ptr(), scratch_m.data_ptr(), scratch_v.data_ptr(),
        learner._num_steps.data_ptr(), 1e-3, 0.9, 0.999, 1e-8, 0, None, None, _capi.current_stream()), it, torch)
    stages['k2_update_priorities'] = time_stage(lambda: table.update_priorities_device(ds.keys, learner.priority), it, torch)
    del scratch_p, scratch_m, scratch_v
  net_s = stages.get('k6_network_group_in_graph', 0)

  # ---- PER sampling throughput (sample + gather), batch 256 and a large-batch sweep point
  per = {}
  if rank == 0:
    per['samples_per_sec_b256_sample_gather'] = B / (stages['k1_sample'] + stages['k3_gather_nstep'])
    Bl = 1 << 16
    ul = torch.rand(Bl, device='cuda')
    il = torch.empty(Bl, dtype=torch.int64, device='cuda')
    kl = torch.empty(Bl, dtype=torch.uint64, device='cuda')
    pl = torch.empty(Bl, device='cuda')
    t_l = time_stage(lambda: table.sample_into(ul, il, kl, pl, True), 20, torch)
    L, F, S = table.tree_levels()
    per['sample_only_b65536'] = {'samples_per_sec': Bl / t_l, 'us': t_l * 1e6,
                                 'alg_bytes_per_sample': (L - min(S + 1, L)) * F * 4 + 24, 'levels': L, 'fanout': F}

  # ---- CPU baseline beside it (rank 0, N=1 only, bounded)
  cpu_baseline = None
  if rank == 0 and world == 1 and not args.no_cpu_baseline:
    ref = CpuReferencePath(seed=1234, ring=8192)
    ref.step()
    t0 = time.time()
    n_cpu = 0
    while n_cpu < 3 or (time.time() - t0 < 12 and n_cpu < 30):
      ref.step()
      n_cpu += 1
    cdt = (time.time() - t0) / n_cpu
    cpu_baseline = {'value': 1.0 / cdt, 'unit': 'updates/s', 'cores': ref.threads, 'kind': 'port',
                    'sample': f'{n_cpu} full learner updates of the same workload on the host (oracle port: binary f64 '
                              f'sum-tree over 1M priorities, 8192-step uint8 ring, PyTorch-CPU DQNAtariNetwork(18) B=256)'}

  if rank == 0:
    gpu_launches = int(learner.kernel_launches_per_step or 0) * args.steps
    if not gpu_launches:
      gpu_launches = int(lib.b200rl_launch_count() - launches0)
    kname = {0: 'k6_network_gemm_conv (3 forwards + 1 backward, fp32 SIMT FFMA)',
             1: 'k6_network_gemm_conv (3 forwards + 1 backward; tcgen05 kind::tf32, TMA-fed, fp32 tensors)',
             2: 'k6_network_gemm_conv (3 forwards + 1 backward; tcgen05 kind::f16 on bf16 activations / weight shadows / '
                'gradients, TMA-fed: im2col for the convolutions incl. conv1 on uint8 frames via an integer-valued bf16 row image)'}[precision]
    achieved = STEP_FLOPS / net_s / 1e12 if net_s > 0 else None
    traffic = None    # dram bytes of the same kernel group from the committed `ncu --set full` capture (tensor-core mode)
    prof_name = {1: 'ncu_full_r01_tc_layers_summary.json', 2: 'ncu_full_r02c_bf16_step_summary.json'}.get(precision)
    prof = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'profiles', prof_name or 'none')
    traffic_source = None
    if os.path.exists(prof):
      traffic = json.load(open(prof)).get('step_group_dram_bytes')
      traffic_source = f'profiles/{prof_name} (committed ncu --set full capture of the same kernels; not measured in this run)'
    out = {
        'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps, 'warmup': max(args.warmup, 3),
        'ms_per_step': ms_per_step, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': {0: 'f32', 1: 'tf32 tensor-core operands, f32 accumulate, f32 master weights and optimizer',
                  2: 'bf16 tensor-core operands (activations, weight shadows, back-propagated gradients), f32 accumulate, '
                     'f32 master weights, weight gradients and optimizer'}[precision],
        'data': 'synthetic',
        'config': {'workload': 'DQN Atari-shaped 84x84x4 uint8, PER 1M items, batch 256, n=3 (BASELINE configs[1])',
                   'items_per_rank': info['size'], 'batch_per_rank': B, 'n_step': n_step, 'alpha': 0.6, 'beta': 0.2,
                   'network': 'DQNAtariNetwork(18), 8,018,611 params', 'optimizer': 'Adam 1e-3',
                   'replay_ring': ('frame-deduplicated: one 84x84 uint8 frame per step, stacks rebuilt by K3 '
                                   f'({(items + 4096) * 7056 / 1e9:.1f} GB)') if args.frame_dedup else
                                  f'one 84x84x4 uint8 stack per step ({(items + 4096) * 28224 / 1e9:.1f} GB)',
                   'parallelism': (f'dp{world}: per-rank replay shard; gradient mean + Adam + parameter broadcast over NVLink '
                                   f'peer memory (torso bucket: one fused SM kernel; fc1 + head bucket: reduce='
                                   f'{getattr(learner, "_dp_reduce", "sm")}, broadcast={getattr(learner, "_dp_bcast", None) or "same kernel"}; '
                                   'NCCL for set-up only)') if world > 1 else 'single GPU',
                   'cuda_graph': not args.no_graph,
                   'update_order': ('pipelined: the optimizer half of update t is issued at the start of step t+1\'s graph beside '
                                    'K1 / K3 / the target forward (same values as the serial order; the last update is flushed '
                                    'inside the timed region)') if getattr(learner, '_pipeline', False) else 'serial (one graph per step)',
                   'l2_policy': 'inputs larger than L2: 28 GB ring sampled at random + 160 MB of params/moments/grads per step'},
        'clocks': clk,
        'e2e': {'value': e2e_value, 'unit': 'updates/s', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
                'what': f'{inserts_per_step} adder.add() calls from host numpy (pinned staging -> H2D) + learner.step() '
                        "with every update's loss copied to pinned host memory and consumed one update later (fetch_loss='async'; the last one "
                        'inside the timed region), per update (the reference loop cadence)', 'steps': e2e_steps},
        'gpu_launches': gpu_launches,
        'roofline': {'kernel': kname, 'bound': 'tensor', 'achieved': achieved, 'peak': P['tf_sustained'], 'unit': 'TFLOP/s',
                     'frac': (achieved / P['tf_sustained']) if achieved else None, 'traffic': traffic,
                     'peak_source': f"{P['src']} (sustained bf16 dense peak: the group is timed inside a long run; "
                                    'tf32 runs at half that rate)',
                     'traffic_source': traffic_source, 'alg_flops_per_launch_group': STEP_FLOPS, 'group_seconds': net_s,
                     'group_timing': 'CUDA events around replays of the captured network group (forwards + head/K4 + backward)'},
        'cpu_baseline': cpu_baseline,
        'parity': parity_record(precision),
        'stages_us': {k: v * 1e6 for k, v in stages.items()},
        'hbm_kernels': {
            'k3_gather_nstep': {'alg_bytes': B * 112_944, 'GBps': B * 112_944 / stages['k3_gather_nstep'] / 1e9,
                                'frac_of_hbm_peak': B * 112_944 / stages['k3_gather_nstep'] / 1e9 / P['hbm']},
            'k7_adam': {'alg_bytes': net.params.size * 28, 'GBps': net.params.size * 28 / stages['k7_adam'] / 1e9,
                        'frac_of_hbm_peak': net.params.size * 28 / stages['k7_adam'] / 1e9 / P['hbm']},
        },
        'per': per,
        'setup_s': t_setup,
    }
    print(json.dumps(out))
  if world > 1:   # replicas must not have diverged (identical Adam on identical averaged gradients)
    learner._dp.assert_replicated(net.params.flat, 'online parameters')
  server.stop()
  if world > 1:
    dist.destroy_process_group()


def _dist_setup():
  import torch
  import torch.distributed as dist
  rank, world, local = int(os.environ.get('RANK', '0')), int(os.environ.get('WORLD_SIZE', '1')), int(os.environ.get('LOCAL_RANK', '0'))
  torch.cuda.set_device(local)
  pg = None
  if world > 1:
    dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    pg = dist.group.WORLD
  return rank, world, local, pg


def _max_over_ranks(x, world):
  import torch
  import torch.distributed as dist
  if world == 1:
    return x
  t = torch.tensor([x], device='cuda')
  dist.all_reduce(t, op=dist.ReduceOp.MAX)
  return float(t)


def run_d4pg(args):
  """BASELINE configs[2]: D4PG learner updates/s on control-suite-humanoid-shaped transitions (SURVEY §8d C3)."""
  import torch
  import torch.distributed as dist
  from acme_b200 import _capi, adders, d4pg, dm_env, loggers, networks, replay, specs
  rank, world, local, pg = _dist_setup()
  _capi.require_device(local)
  P = peaks()
  B, n_step, items = 256, 5, args.items
  spec = specs.EnvironmentSpec(specs.Array((OBS_DIM,), np.float32), specs.BoundedArray((ACT_DIM,), np.float32, -1., 1.),
                               specs.Array((), np.float32), specs.BoundedArray((), np.float32, 0., 1.))
  table = replay.Table(replay.DEFAULT_PRIORITY_TABLE, replay.selectors.Uniform(), replay.selectors.Fifo(), max_size=items,
                       rate_limiter=replay.rate_limiters.MinSize(1), signature=adders.NStepTransitionAdder.signature(spec),
                       max_window=n_step, discount=0.99, device=local, slot_capacity=items + 4096, shard_count=world,
                       shard_rank=rank, stage_slots=4096)
  server = replay.Server([table])
  t_setup = time.time()
  info = fill_replay_control(table, items, n_step, 1234 + rank, OBS_DIM, ACT_DIM)
  precision = _capi.PRECISION_FP32 if args.precision == 'fp32' else _capi.PRECISION_TC
  policy = networks.D4PGPolicy(OBS_DIM, ACT_DIM, device=local, precision=precision, seed=1)
  critic = networks.D4PGCritic(OBS_DIM, ACT_DIM, device=local, precision=precision, seed=2)
  ds = replay.ReplayDataset(table, B, seed=1234 + rank, stratified=False)
  client = replay.Client(server)
  learner = d4pg.D4PGLearner(policy, critic, policy.clone(), critic.clone(), 0.99, 100, ds, logger=loggers.NoOpLogger(),
                             process_group=pg, use_cuda_graph=not args.no_graph)
  adder = adders.NStepTransitionAdder(client, n_step=n_step, discount=0.99)
  t_setup = time.time() - t_setup
  lib = _capi.load()

  def barrier():
    if world > 1:
      dist.barrier()
    torch.cuda.synchronize()

  clocks = ClockSampler(local)
  for _ in range(max(args.warmup, 3)):
    learner.step(fetch_loss=False)
  barrier()
  launches0 = lib.b200rl_launch_count()
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  barrier()
  clocks.mark()
  e0.record()
  for _ in range(args.steps):
    learner.step(fetch_loss=False)
  e1.record()
  barrier()
  clocks.mark()
  clk = clocks.stop()
  dev_s = _max_over_ranks(e0.elapsed_time(e1) * 1e-3, world)
  value = world * args.steps / dev_s
  gpu_launches = int(lib.b200rl_launch_count() - launches0) if args.no_graph else None

  # ---- end to end: 8 adder.add() from host numpy per update (batch 256 / samples_per_insert 32, d4pg/agent.py:176-180)
  rng = np.random.default_rng(99 + rank)
  host_obs = rng.standard_normal((64, OBS_DIM)).astype(np.float32)
  host_act = rng.uniform(-1, 1, (64, ACT_DIM)).astype(np.float32)
  inserts = 8
  adder.add_first(dm_env.restart(host_obs[0]))

  def e2e_step(i):
    for j in range(inserts):
      k = (i * inserts + j + 1) % 64
      adder.add(host_act[k], dm_env.transition(np.float32(0.5), host_obs[k], np.float32(1.)))
    learner.step(fetch_loss='async')

  for i in range(3):
    e2e_step(i)
  barrier()
  t0 = time.perf_counter()
  e2e_steps = args.steps
  for i in range(e2e_steps):
    e2e_step(i + 3)
  last = learner.drain()
  assert last is not None and np.isfinite(last['critic_loss'])
  barrier()
  e2e_s = _max_over_ranks(time.perf_counter() - t0, world)
  e2e_value = world * e2e_steps / e2e_s
  h2d = inserts * (OBS_DIM * 4 + ACT_DIM * 4 + 4 + 4 + 4) + inserts * 24 + 16
  d2h = 8

  stages, k5 = {}, None
  if rank == 0:
    it = 30
    stages['k1_sample_uniform'] = time_stage(ds.sample_only, it, torch)
    stages['k3_gather_nstep'] = time_stage(ds.gather_only, it, torch)
    g_half = torch.cuda.CUDAGraph()
    torch.cuda.synchronize()
    with torch.cuda.graph(g_half):
      learner._gradient_half(None)
    stages['gradient_half_in_graph (K1, K3, 5 MLP passes, K5, DPG)'] = time_stage(g_half.replay, it, torch)
    K = critic.K
    t5 = time_stage(lambda: _capi.call(
        'b200rl_c51_loss', B, K, critic.vmin, critic.vmax, learner._c_train['out'].data_ptr(), learner._c_tgt['out'].data_ptr(),
        ds.R.data_ptr(), ds.D.data_ptr(), 0.99, 1.0 / B, learner.target.data_ptr(), learner.critic_loss_ps.data_ptr(),
        learner.dlogits.data_ptr(), None, _capi.current_stream()), it, torch)
    stages['k5_c51_project_ce'] = t5
    k5 = {'alg_bytes': B * 828, 'us': t5 * 1e6, 'GBps': B * 828 / t5 / 1e9, 'frac_of_hbm_peak': B * 828 / t5 / 1e9 / P['hbm'],
          'note': 'launch-latency bound at B = 256 (212 KB per launch); the HBM regime is tools/ncu_hbm_kernels.py (B = 65,536)'}

  cpu_baseline = None
  if rank == 0 and world == 1 and not args.no_cpu_baseline:
    ref = CpuD4PGPath(seed=1234)
    ref.step()
    t0 = time.time()
    n_cpu = 0
    while n_cpu < 3 or (time.time() - t0 < 12 and n_cpu < 200):
      ref.step()
      n_cpu += 1
    cdt = (time.time() - t0) / n_cpu
    cpu_baseline = {'value': 1.0 / cdt, 'unit': 'updates/s', 'cores': ref.threads, 'kind': 'port',
                    'sample': f'{n_cpu} full D4PG learner updates of the same workload on the host (oracle port: NumPy n-step over a '
                              f'{ref.ring}-step ring, PyTorch-CPU critic/policy, dense l2_project, B=256)'}
  if rank == 0:
    grp = stages.get('gradient_half_in_graph (K1, K3, 5 MLP passes, K5, DPG)', 0)
    achieved = D4PG_STEP_FLOPS / grp / 1e12 if grp else None
    print(json.dumps({
        'metric': D4PG_METRIC, 'value': value, 'unit': D4PG_UNIT, 'n_gpus': world, 'steps': args.steps, 'warmup': max(args.warmup, 3),
        'ms_per_step': dev_s / args.steps * 1e3, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'f32 (dense layers below 0.13 GFLOP take the exact FFMA path; larger ones tf32/bf16 tensor-core operands)' if precision else 'f32',
        'data': 'synthetic',
        'config': {'workload': D4PG_WORKLOAD, 'items_per_rank': info['size'], 'batch_per_rank': B, 'n_step': n_step,
                   'networks': 'critic LayerNormMLP(512,512,256) + DiscreteValuedHead(51), policy LayerNormMLP(256,256,256) + tanh',
                   'optimizer': 'Adam 1e-4 x2, global-norm clip 40',
                   'parallelism': f'dp{world}: per-rank replay shard, NCCL all-reduce(mean) of both gradient sets' if world > 1 else 'single GPU',
                   'cuda_graph': not args.no_graph,
                   'l2_policy': 'the 628 MB transition ring is sampled uniformly at random; parameters and activations (< 10 MB) are L2-resident by nature of the workload'},
        'clocks': clk,
        'e2e': {'value': e2e_value, 'unit': 'updates/s', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h, 'steps': e2e_steps,
                'what': f"{inserts} adder.add() calls from host numpy (pinned staging -> H2D) + learner.step(fetch_loss='async') per update, "
                        'both losses copied to pinned host memory every update'},
        'gpu_launches': gpu_launches if gpu_launches is not None else 'captured graph (count with --no-graph)',
        'roofline': {'kernel': 'critic / policy MLP group of the gradient half (3 critic + 2 policy forwards, critic backward, dq/da, policy backward)',
                     'bound': 'tensor', 'achieved': achieved, 'peak': P['tf_sustained'], 'unit': 'TFLOP/s',
                     'frac': achieved / P['tf_sustained'] if achieved else None, 'traffic': None,
                     'peak_source': f"{P['src']} (sustained bf16 dense peak)", 'alg_flops_per_launch_group': D4PG_STEP_FLOPS,
                     'group_seconds': grp,
                     'note': '1.7 GFLOP per step over ~100 small launches: launch- and latency-bound, not tensor-bound'},
        'hbm_kernels': {'k5_c51_project_ce': k5},
        'cpu_baseline': cpu_baseline,
        'stages_us': {k: v * 1e6 for k, v in stages.items()},
        'setup_s': t_setup,
    }))
  server.stop()
  if world > 1:
    dist.destroy_process_group()


def run_sumtree(args):
  """BASELINE configs[3]: prioritized sampling / update sweep point, one shard of `--items` priorities per rank, each rank
  drawing `--tree-batch` items locally per step; probabilities normalised by the GLOBAL priority mass (all-reduce of the
  shard masses, SURVEY §8e)."""
  import torch
  import torch.distributed as dist
  from acme_b200 import _capi, parallel, replay
  rank, world, local, pg = _dist_setup()
  _capi.require_device(local)
  P = peaks()
  N, B = args.items, args.tree_batch
  gen = torch.Generator(device='cuda')
  gen.manual_seed(1234 + rank)
  table = replay.Table.priorities_only('t', 0.6, N, device=local, shard_count=world, shard_rank=rank)
  w = torch.randn(N, device='cuda', generator=gen).abs_() * (1.0 + 0.1 * rank)      # shards of unequal mass
  table.set_weights(w)
  del w
  dp = parallel.DataParallel(pg)
  total = dp.refresh_global_mass(table)
  L, F, S_small = table.tree_levels()
  u = torch.rand(B, device='cuda', generator=gen)
  idx = torch.empty(B, dtype=torch.int64, device='cuda')
  keys = torch.empty(B, dtype=torch.uint64, device='cuda')
  prob = torch.empty(B, device='cuda')
  pr = torch.randn(B, device='cuda', generator=gen).abs_()

  def step():
    table.sample_into(u, idx, keys, prob, True)            # K1: local draws, probabilities = weight / sum_r M_r
    table.update_priorities_device(keys, pr)               # K2
    dp.refresh_global_mass(table, total)                   # one scalar all-reduce(SUM): the new global mass

  def barrier():
    if world > 1:
      dist.barrier()
    torch.cuda.synchronize()

  clocks = ClockSampler(local)
  for _ in range(max(args.warmup, 3)):
    step()
  barrier()
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  barrier()
  clocks.mark()
  e0.record()
  for _ in range(args.steps):
    step()
  e1.record()
  barrier()
  clocks.mark()
  clk = clocks.stop()
  dev_s = _max_over_ranks(e0.elapsed_time(e1) * 1e-3, world)
  value = world * args.steps * B / dev_s
  # sanity: with the global mass installed the probabilities of ALL shards' items sum to one
  masses = dp.gather_scalars(table.mass_tensor())
  ts = time_stage(lambda: table.sample_into(u, idx, keys, prob, True), 10, torch)
  tu = time_stage(lambda: table.update_priorities_device(keys, pr), 10, torch)
  # end to end: uniforms from pinned host memory in, sampled keys + probabilities back to pinned host memory, every step
  hu = torch.rand(B).pin_memory()
  hk, hp = torch.empty(B, dtype=torch.int64).pin_memory(), torch.empty(B).pin_memory()
  barrier()
  t0 = time.perf_counter()
  e2e_steps = args.steps
  for _ in range(e2e_steps):
    u.copy_(hu, non_blocking=True)
    step()
    hk.copy_(keys.view(torch.int64), non_blocking=True)
    hp.copy_(prob, non_blocking=True)
    torch.cuda.current_stream().synchronize()
  barrier()
  e2e_s = _max_over_ranks(time.perf_counter() - t0, world)
  staged = 0
  used = 0
  budget = (160 if B >= 16384 else 16) * 1024
  for l in range(1, L + 1):
    wl = len(table.read_tree_level(l)) * 4 if l < L else N * 4
    if used + wl > budget:
      break
    used += wl
    staged = l
  sample_bytes = (L - staged) * F * 4 + 28
  cpu_baseline = None
  if rank == 0 and world == 1 and not args.no_cpu_baseline:
    Bt = min(B, 1 << 15)
    ref = CpuTreePath(min(N, 4_000_000), Bt, seed=1234)
    t0 = time.time()
    n_cpu = 0
    while n_cpu < 2 or (time.time() - t0 < 10 and n_cpu < 50):
      ref.step()
      n_cpu += 1
    cdt = (time.time() - t0) / n_cpu
    cpu_baseline = {'value': Bt / cdt, 'unit': 'samples/s', 'cores': 1, 'kind': 'port',
                    'sample': f'{n_cpu} steps of {Bt:,} draws + {Bt:,} updates on a binary f64 NumPy sum tree over {min(N, 4_000_000):,} priorities'}
  if rank == 0:
    m = masses.cpu().numpy().astype(np.float64)
    print(json.dumps({
        'metric': TREE_METRIC, 'value': value, 'unit': TREE_UNIT, 'n_gpus': world, 'steps': args.steps, 'warmup': max(args.warmup, 3),
        'ms_per_step': dev_s / args.steps * 1e3, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32',
        'data': 'synthetic',
        'config': {'workload': f'sum-tree sweep point: {N:,} items per rank, {B:,} draws + updates per step (BASELINE configs[3])',
                   'levels': L, 'fanout': F, 'staged_levels': staged, 'alpha': 0.6,
                   'parallelism': (f'{world} shards, one per GPU; local sampling; global-priority-mass normalisation by one scalar '
                                   'all-reduce(SUM) per step') if world > 1 else 'single shard',
                   'l2_policy': f'tree of {N:,} leaves = {8 * N / 1e6:.0f} MB of values + prefix lines, sampled at random (larger than L2 for N >= 2^24)'},
        'clocks': clk,
        'shard_masses': m.tolist(), 'mass_imbalance_max_over_mean': float(m.max() / m.mean()), 'global_mass': float(total.item()),
        'e2e': {'value': world * e2e_steps * B / e2e_s, 'unit': 'samples/s', 'h2d_bytes_per_step': 4 * B, 'd2h_bytes_per_step': 12 * B,
                'steps': e2e_steps, 'what': 'uniforms from pinned host memory, sampled keys and probabilities copied back to pinned host memory, every step'},
        'gpu_launches': 'see stages',
        'roofline': {'kernel': 'k1 sample_kernel', 'bound': 'hbm', 'achieved': B * sample_bytes / ts / 1e9, 'peak': P['hbm'], 'unit': 'GB/s',
                     'frac': B * sample_bytes / ts / 1e9 / P['hbm'], 'traffic': None, 'peak_source': P['src'],
                     'alg_bytes_per_sample': sample_bytes,
                     'note': 'algorithmic bytes per SURVEY §8d: (L - S) * 128 + 28; DRAM bytes of the N = 1e8, B = 2^20 point are in profiles/ncu_full_r02_hbm_kernels.csv'},
        'stages_us': {'k1_sample': ts * 1e6, 'k2_update': tu * 1e6},
        'update': {'updates_per_sec_per_gpu': B / tu, 'alg_bytes_per_item': 4 + L * (F * 4 + 4) + 12},
        'cpu_baseline': cpu_baseline,
    }))
  table.close()
  if world > 1:
    dist.destroy_process_group()


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--gpus', type=int, default=1)
  ap.add_argument('--steps', type=int, default=None,
                  help='timed steps of every timed leg (default 2000; sumtree 100; reference arm 10, sumtree 3)')
  ap.add_argument('--warmup', type=int, default=None, help='default 50; sumtree 5; reference arm 2, sumtree 1')
  ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
  ap.add_argument('--precision', default=os.environ.get('B200RL_PRECISION', 'bf16'), choices=['fp32', 'tf32', 'tc', 'bf16'],
                  help="'bf16' (default): bf16 dataflow on tcgen05 (kind::f16); 'tf32' ('tc'): fp32 tensors with tf32 operands; "
                       "both with the stated tolerances of tests/test_gpu_learner.py; 'fp32': SIMT FFMA, 1e-5 parity with the oracle")
  ap.add_argument('--workload', default='dqn', choices=['dqn', 'd4pg', 'sumtree'],
                  help='dqn (default): BASELINE configs[1], the headline metric; d4pg: configs[2]; sumtree: a point of the configs[3] sweep')
  ap.add_argument('--items', type=int, default=None, help='items per rank (default 1M; sumtree: 100M)')
  ap.add_argument('--tree-batch', type=int, default=1 << 20, help='sumtree: draws (and updates) per rank per step')
  ap.add_argument('--frame-dedup', action='store_true',
                  help='dqn: store one frame per step in the HBM ring and rebuild the 4-stacks at gather time (SURVEY 8f-1)')
  ap.add_argument('--no-graph', action='store_true')
  ap.add_argument('--no-cpu-baseline', action='store_true')
  ap.add_argument('--profile', action='store_true', help='only warm-up + timed steps (for ncu captures)')
  ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                  help='dqn workload of our arm: after the timed steps, write what the last one computed as DIR/<name>.npy '
                       '(float32 / float64, at most 64 MB; the inputs are seeded, so two builds can be compared)')
  args = ap.parse_args()
  if args.items is None:
    args.items = 100_000_000 if args.workload == 'sumtree' else 1_000_000
  # a sumtree step is 2^20 draws + updates, and the reference arm runs on the host: shorter default runs
  if args.impl == 'reference':
    steps, warmup = (10, 2) if args.workload != 'sumtree' else (3, 1)
  else:
    steps, warmup = (2000, 50) if args.workload != 'sumtree' else (100, 5)
  args.steps = steps if args.steps is None else args.steps
  args.warmup = warmup if args.warmup is None else args.warmup
  if args.steps < 1:
    ap.error('--steps must be at least 1')
  if args.dump_outputs and (args.impl != 'ours' or args.workload != 'dqn'):
    ap.error('--dump-outputs is implemented for the dqn workload of our arm')
  if args.impl == 'reference':
    (run_reference if args.workload == 'dqn' else run_reference_other)(args)
  elif args.workload == 'd4pg':
    run_d4pg(args)
  elif args.workload == 'sumtree':
    run_sumtree(args)
  else:
    run_ours(args)


if __name__ == '__main__':
  main()
