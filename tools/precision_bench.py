"""DQN learner step (the C2 shape: 84x84x4 uint8 frames, 18 actions, batch 256, n = 3, prioritized replay) in several
network precisions, device-resident, whole step as a CUDA graph.

  python tools/precision_bench.py --precision fp32,fp32x3,bf16 --steps 300 --reps 3 [--out DIR]

The precisions (fp32 = 0, tf32 = 1, bf16 = 2, fp32x3 = 3, the network `precision` modes) are timed in one process,
alternating per repetition, so that they share the GPU's state.  The result reports, per precision, the median ms per
step and its range over the repetitions, kernel launches per eager step (`b200rl_launch_count`), and the GPU's name and
power limit read in the same run.  `bench.py` keeps measuring its own fixed precision."""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))
import numpy as np
import torch

from acme_b200 import _capi, adders, dqn, loggers, networks, replay, specs
from bench import NUM_ACTIONS, OBS_SHAPE, fill_replay
from d4pg_bench import gpu_info

PRECISIONS = {'fp32': _capi.PRECISION_FP32, 'tf32': _capi.PRECISION_TC, 'bf16': _capi.PRECISION_BF16FLOW,
              'fp32x3': _capi.PRECISION_FP32X3}


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--precision', default='fp32,fp32x3,bf16', help='comma-separated subset of fp32, tf32, bf16, fp32x3')
  ap.add_argument('--steps', type=int, default=300, help='timed updates per repetition')
  ap.add_argument('--warmup', type=int, default=20)
  ap.add_argument('--reps', type=int, default=3)
  ap.add_argument('--items', type=int, default=200_000, help='replay items')
  ap.add_argument('--out', default=None, help='directory for precision_bench_c2.json')
  args = ap.parse_args()
  names = [p.strip() for p in args.precision.split(',') if p.strip()]
  for p in names:
    if p not in PRECISIONS:
      ap.error(f'unknown precision {p!r} ({", ".join(PRECISIONS)})')
  _capi.require_device(0)
  B, n = 256, 3
  spec = specs.EnvironmentSpec(specs.Array(OBS_SHAPE, np.uint8), specs.DiscreteArray(NUM_ACTIONS),
                               specs.Array((), np.float32), specs.BoundedArray((), np.float32, 0., 1.))
  table = replay.Table(replay.DEFAULT_PRIORITY_TABLE, replay.selectors.Prioritized(0.6), replay.selectors.Fifo(),
                       max_size=args.items, rate_limiter=replay.rate_limiters.MinSize(1),
                       signature=adders.NStepTransitionAdder.signature(spec), max_window=n, discount=0.99,
                       slot_capacity=args.items + 4096, stage_slots=4096)
  server = replay.Server([table])
  fill_replay(table, args.items, n, seed=1234)
  lib = _capi.load()
  learners, launches = {}, {}
  for p in names:
    net = networks.DQNAtariNetwork(NUM_ACTIONS, precision=PRECISIONS[p], seed=1234)
    tgt = net.clone()
    ds = replay.ReplayDataset(table, B, seed=1234)
    L = dqn.DQNLearner(net, tgt, 0.99, 0.2, 1e-3, 100, ds, replay_client=replay.Client(server), logger=loggers.NoOpLogger())
    L.step(fetch_loss=False)
    torch.cuda.synchronize()
    n0 = lib.b200rl_launch_count()
    L.step(fetch_loss=False)          # the second update is still eager; the graph is captured at the third
    torch.cuda.synchronize()
    launches[p] = int(lib.b200rl_launch_count() - n0)
    for _ in range(args.warmup):
      L.step(fetch_loss=False)
    torch.cuda.synchronize()
    learners[p] = L
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
  out = {'workload': 'DQN learner step, C2 shape: 84x84x4 uint8, 18 actions, batch 256, n=3, prioritized replay, CUDA graph',
         'steps_per_rep': args.steps, 'reps': args.reps, 'gpu': gpu, 'power_limit': power_limit, 'precisions': {}}
  for p in names:
    med = float(np.median(ms[p]))
    out['precisions'][p] = {'precision_mode': PRECISIONS[p], 'ms_per_step': med, 'ms_per_step_min': min(ms[p]),
                            'ms_per_step_max': max(ms[p]), 'ms_per_step_reps': ms[p], 'updates_per_s': 1e3 / med,
                            'launches_per_eager_step': launches[p]}
  print(json.dumps(out))
  if args.out:
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, 'precision_bench_c2.json'), 'w') as f:
      json.dump(out, f, indent=1)
  server.stop()


if __name__ == '__main__':
  main()
