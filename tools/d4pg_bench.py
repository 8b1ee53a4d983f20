"""D4PG learner updates/s on the control-suite-humanoid shape (67-d obs, 21-d act, C51 critic), batch 256, n=5
(BASELINE.json configs[2]); device-resident timing with CUDA events, whole step as a CUDA graph.

  python tools/d4pg_bench.py --precision tf32,bf16 [--replay uniform,prioritized] --steps 300 --reps 3 [--out DIR]

Several precisions (fp32 = 0, tf32 = 1, bf16 = 2, the network `precision` modes) are timed in one process, alternating
per repetition, so that they share the GPU's state.  Each line reports ms per step for every repetition, kernel launches
per eager step (`b200rl_launch_count`), and the GPU's name and power limit read in the same run.  `bench.py --workload
d4pg` keeps measuring precision 1.

`--replay prioritized` adds the opt-in prioritized learner (a Prioritized(0.6) table, importance_sampling_exponent 0.4,
priorities written back every step) beside the uniform one; the two arms read separate tables with identical contents
and alternate with the precisions.  Its results go to d4pg_bench_<precision>_prioritized.json.

`--observation atari` times D4PG from pixels instead: uint8 84 x 84 x 4 frames through an AtariTorso observation network,
6-d actions, critic (512, 512, 256) with 51 atoms, policy (256, 256, 256), batch 256, n = 5, at any of fp32, tf32, bf16,
fp32x3.  Each line adds the step's FLOP count (computed from the shapes by `pixel_step_flop`) and the achieved TFLOP/s.
`--channels 4,3,12` times frames of those channel counts side by side; C = 4 writes
d4pg_bench_pixels_<precision>.json as before, other counts d4pg_bench_pixels_c<C>_<precision>.json.
Results go to d4pg_bench_pixels_<precision>.json."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch

from acme_b200 import _capi, adders, d4pg, dm_env, loggers, networks, replay, specs

PRECISIONS = {'fp32': _capi.PRECISION_FP32, 'tf32': _capi.PRECISION_TC, 'bf16': _capi.PRECISION_BF16FLOW,
              'fp32x3': _capi.PRECISION_FP32X3}


def gpu_info():
  name = torch.cuda.get_device_name(0)
  try:
    limit = subprocess.run(['nvidia-smi', '-i', '0', '--query-gpu=power.limit', '--format=csv,noheader'], capture_output=True,
                           text=True, timeout=30).stdout.strip() or None
  except (OSError, subprocess.SubprocessError):
    limit = None
  return name, limit


ALPHA, BETA = 0.6, 0.4


def fill_table(OBS, ACT, n, items, sampler=None):
  rng = np.random.default_rng(0)
  spec = specs.EnvironmentSpec(specs.Array((OBS,), np.float32), specs.BoundedArray((ACT,), np.float32, -1., 1.),
                               specs.Array((), np.float32), specs.BoundedArray((), np.float32, 0., 1.))
  table = replay.Table(replay.DEFAULT_PRIORITY_TABLE, sampler or replay.selectors.Uniform(), replay.selectors.Fifo(), max_size=items,
                       rate_limiter=replay.rate_limiters.MinSize(1), signature=adders.NStepTransitionAdder.signature(spec),
                       max_window=n, discount=0.99, stage_slots=4096)
  server = replay.Server([table])
  adder = adders.NStepTransitionAdder(replay.Client(server), n_step=n, discount=0.99)
  steps = 0
  while steps < 20_000:     # 20k synthetic control steps through the product adder (setup, not timed)
    adder.add_first(dm_env.restart(rng.standard_normal(OBS).astype(np.float32)))
    T = 200
    for t in range(T):
      ts = dm_env.termination if t == T - 1 else dm_env.transition
      args = (np.float32(rng.random()), rng.standard_normal(OBS).astype(np.float32))
      adder.add(rng.uniform(-1, 1, ACT).astype(np.float32), ts(*args) if t == T - 1 else ts(args[0], args[1], np.float32(1.)))
      steps += 1
    table.flush()
  return table, server


def pixel_step_flop(B, torso, A, critic_sizes, K, policy_sizes):
  """Multiply-adds x 2 of one pixel learner update: online torso forward + three weight gradients + conv3 / conv2 data
  gradients, target torso forward; the critic's feature block in three forwards + weight and data gradient, the policy's
  in two forwards + weight gradient; the remaining critic layers in 3 forwards + 2 (train) + 1 (dq/da) backward GEMMs,
  the policy's in 2 forwards + 2 backward GEMMs."""
  conv = [oh * oh * co * k * k * ci for (k, s, ci, co, h, oh, pad) in torso.convs]
  F = torso.flat_dim
  rest = lambda sizes, out: sum(a * b for a, b in zip(sizes, list(sizes[1:]) + [out]))
  mac = (2 * sum(conv) + conv[2] + conv[1] + sum(conv) + 5 * F * critic_sizes[0] + 3 * F * policy_sizes[0] +
         6 * (rest(critic_sizes, K) + A * critic_sizes[0]) + 4 * rest(policy_sizes, A))
  return 2 * B * mac


def fill_pixel_table(A, n, items, C=4):
  rng = np.random.default_rng(0)
  spec = specs.EnvironmentSpec(specs.Array((84, 84, C), np.uint8), specs.BoundedArray((A,), np.float32, -1., 1.),
                               specs.Array((), np.float32), specs.BoundedArray((), np.float32, 0., 1.))
  table = replay.Table(replay.DEFAULT_PRIORITY_TABLE, replay.selectors.Uniform(), replay.selectors.Fifo(), max_size=items,
                       rate_limiter=replay.rate_limiters.MinSize(1), signature=adders.NStepTransitionAdder.signature(spec),
                       max_window=n, discount=0.99, stage_slots=256)
  server = replay.Server([table])
  adder = adders.NStepTransitionAdder(replay.Client(server), n_step=n, discount=0.99)
  frames = rng.integers(0, 256, (64, 84, 84, C), dtype=np.uint8)
  steps = 0
  while steps < items:
    adder.add_first(dm_env.restart(frames[steps % 64]))
    for t in range(100):
      o = frames[(steps + t * 7) % 64]
      a = rng.uniform(-1, 1, A).astype(np.float32)
      adder.add(a, dm_env.termination(np.float32(rng.random()), o) if t == 99 else
                dm_env.transition(np.float32(rng.random()), o, np.float32(1.)))
    steps += 100
    table.flush()
  return table, server


def main_pixels(args, precisions, channels):
  """One learner per (channel count, precision), timed alternately; C = 4 keeps the names it always had."""
  B, A, n, K = 256, 6, 5, 51
  tables = {C: fill_pixel_table(A, n, 20_000, C) for C in channels}
  lib = _capi.load()
  learners, launches, flop = {}, {}, {}
  arms = [(C, p) for C in channels for p in precisions]
  for arm in arms:
    C, p = arm
    table = tables[C][0]
    torso = networks.AtariTorso(precision=PRECISIONS[p], seed=0, input_channels=C)
    policy = networks.D4PGPolicy(torso.flat_dim, A, seed=1, precision=PRECISIONS[p])
    critic = networks.D4PGCritic(torso.flat_dim, A, seed=2, precision=PRECISIONS[p])
    flop[arm] = pixel_step_flop(B, torso, A, critic.sizes, K, policy.sizes)
    ds = replay.ReplayDataset(table, B, seed=11, stratified=False)
    L = d4pg.D4PGLearner(policy, critic, policy.clone(), critic.clone(), 0.99, target_update_period=100, dataset=ds,
                         logger=loggers.NoOpLogger(), observation_network=torso, target_observation_network=torso.clone())
    L.step(fetch_loss=False)
    torch.cuda.synchronize()
    n0 = lib.b200rl_launch_count()
    L.step(fetch_loss=False)
    torch.cuda.synchronize()
    launches[arm] = int(lib.b200rl_launch_count() - n0)
    for _ in range(args.warmup):
      L.step(fetch_loss=False)
    torch.cuda.synchronize()
    learners[arm] = L
  ms = {arm: [] for arm in arms}
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  for _ in range(args.reps):
    for arm in arms:
      L = learners[arm]
      torch.cuda.synchronize()
      e0.record()
      for _ in range(args.steps):
        L.step(fetch_loss=False)
      e1.record()
      torch.cuda.synchronize()
      ms[arm].append(e0.elapsed_time(e1) / args.steps)
  gpu, power_limit = gpu_info()
  for arm in arms:
    C, p = arm
    med = float(np.median(ms[arm]))
    # gflop_per_step counts the MMA work done: conv1 over the filter's padded channel count (networks._ConvTorso)
    out = {'workload': f'D4PG from pixels: uint8 84x84x{C}, AtariTorso, 6-d actions, critic (512, 512, 256) C51, policy '
                       '(256, 256, 256), batch 256, n=5', 'channels': C, 'precision': p, 'precision_mode': PRECISIONS[p],
           'steps_per_rep': args.steps, 'ms_per_step_reps': ms[arm], 'ms_per_step': med, 'updates_per_s': 1e3 / med,
           'launches_per_eager_step': launches[arm], 'gflop_per_step': flop[arm] / 1e9,
           'achieved_tflop_s': flop[arm] / (med * 1e-3) / 1e12, 'gpu': gpu, 'power_limit': power_limit}
    print(json.dumps(out))
    if args.out:
      os.makedirs(args.out, exist_ok=True)
      name = f'd4pg_bench_pixels_{p}.json' if C == 4 else f'd4pg_bench_pixels_c{C}_{p}.json'
      with open(os.path.join(args.out, name), 'w') as f:
        json.dump(out, f, indent=1)
  for _, server in tables.values():
    server.stop()


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--precision', default='tf32', help='comma-separated subset of fp32, tf32, bf16')
  ap.add_argument('--replay', default='uniform', help='comma-separated subset of uniform, prioritized')
  ap.add_argument('--steps', type=int, default=300, help='timed updates per repetition')
  ap.add_argument('--warmup', type=int, default=20)
  ap.add_argument('--reps', type=int, default=3)
  ap.add_argument('--out', default=None, help='directory for d4pg_bench_<precision>.json')
  ap.add_argument('--observation', default='state', choices=['state', 'atari'],
                  help='state: flat 67-d observations; atari: uint8 frames through an AtariTorso observation network')
  ap.add_argument('--channels', default='4',
                  help='--observation atari: comma-separated frame channel counts in [1, 16] (4: grayscale stack, 3: RGB)')
  args = ap.parse_args()
  channels = [int(c) for c in args.channels.split(',') if c.strip()]
  if any(not 1 <= c <= 16 for c in channels) or (channels != [4] and args.observation != 'atari'):
    ap.error('--channels takes counts in [1, 16] with --observation atari')
  precisions = [p.strip() for p in args.precision.split(',') if p.strip()]
  for p in precisions:
    if p not in PRECISIONS or (p == 'fp32x3' and args.observation == 'state'):
      ap.error(f'unknown precision {p!r} (fp32, tf32, bf16; fp32x3 with --observation atari)')
  if args.observation == 'atari':
    return main_pixels(args, precisions, channels)
  arms = [r.strip() for r in args.replay.split(',') if r.strip()]
  for r in arms:
    if r not in ('uniform', 'prioritized'):
      ap.error(f'unknown replay {r!r} (uniform, prioritized)')
  # one run per (precision, replay); a uniform run keeps the name it always had
  names = [p if r == 'uniform' else f'{p}_{r}' for p in precisions for r in arms]
  B, OBS, ACT, n = 256, 67, 21, 5
  tables = {r: fill_table(OBS, ACT, n, 100_000, replay.selectors.Prioritized(ALPHA) if r == 'prioritized' else None)
            for r in arms}
  lib = _capi.load()
  learners, launches = {}, {}
  for name in names:
    p, prio = name.split('_')[0], name.endswith('_prioritized')
    table, server = tables['prioritized' if prio else 'uniform']
    policy = networks.D4PGPolicy(OBS, ACT, seed=1, precision=PRECISIONS[p])
    critic = networks.D4PGCritic(OBS, ACT, seed=2, precision=PRECISIONS[p])
    ds = replay.ReplayDataset(table, B, seed=11, stratified=False)
    extra = dict(importance_sampling_exponent=BETA, replay_client=replay.Client(server)) if prio else {}
    L = d4pg.D4PGLearner(policy, critic, policy.clone(), critic.clone(), 0.99, target_update_period=100, dataset=ds,
                         logger=loggers.NoOpLogger(), **extra)
    L.step(fetch_loss=False)
    torch.cuda.synchronize()
    n0 = lib.b200rl_launch_count()
    L.step(fetch_loss=False)          # the second update is still eager; the graph is captured at the third
    torch.cuda.synchronize()
    launches[name] = int(lib.b200rl_launch_count() - n0)
    for _ in range(args.warmup):
      L.step(fetch_loss=False)
    torch.cuda.synchronize()
    learners[name] = L
  ms = {p: [] for p in names}
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  for _ in range(args.reps):
    for p in names:
      L = learners[p]
      torch.cuda.synchronize()
      e0.record()
      for _ in range(args.steps):
        L.step(fetch_loss=False)
      e1.record()
      torch.cuda.synchronize()
      ms[p].append(e0.elapsed_time(e1) / args.steps)
  gpu, power_limit = gpu_info()
  for name in names:
    p = name.split('_')[0]
    med = float(np.median(ms[name]))
    out = {'workload': 'D4PG humanoid-shaped 67/21, C51 (51 atoms), batch 256, n=5', 'precision': p,
           'precision_mode': PRECISIONS[p], 'steps_per_rep': args.steps, 'ms_per_step_reps': ms[name], 'ms_per_step': med,
           'updates_per_s': 1e3 / med, 'launches_per_eager_step': launches[name], 'gpu': gpu, 'power_limit': power_limit}
    if name.endswith('_prioritized'):
      out.update(replay=f'prioritized (alpha {ALPHA}, importance_sampling_exponent {BETA}, priorities written back)',
                 items=100_000)
      if p in ms:   # the uniform arm of the same run
        out.update(uniform_ms_per_step=float(np.median(ms[p])), uniform_launches_per_eager_step=launches[p])
    print(json.dumps(out))
    if args.out:
      os.makedirs(args.out, exist_ok=True)
      with open(os.path.join(args.out, f'd4pg_bench_{name}.json'), 'w') as f:
        json.dump(out, f, indent=1)
  for _, server in tables.values():
    server.stop()


if __name__ == '__main__':
  main()
