"""Acting throughput: environment steps per second of the batch-1 policies against the batched actor, and of the whole DQN
agent loop, on synthetic environments that serve observations from a pre-generated seeded pool (the host environment
costs next to nothing, so the numbers are the actor's and the learner's).

  (a) batch-1:   EpsilonGreedyPolicy (C2: DQNAtariNetwork(18), precision 2, uint8 84x84x4) and GaussianNoisePolicy
                 (C3: D4PGPolicy(67 -> 21), precision 1), one observation per call;
  (b) batched:   BatchedActor at N in --num-envs, `select_actions` alone on a fixed batch, and `select_actions` + the
                 environments' steps + `observe` (one append_multi per step) through BatchedEnvironmentLoop;
  (c) agent:     DQN(num_envs=N, batch_size 256, samples_per_insert 32) under BatchedEnvironmentLoop once the learner
                 runs: environment steps and learner updates per second.

Variants alternate within each repetition; the JSON has the median and range over --reps, the GPU name and its power
limit.  Usage: python tools/acting_bench.py --out profiles/acting_bench_c2.json
"""

import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))

from acme_b200 import _capi, actors, adders, d4pg, dm_env, dqn, environment_loop, loggers, networks, replay, specs  # noqa: E402
from d4pg_bench import gpu_info  # noqa: E402


class PoolEnv(dm_env.Environment):
  """Observations drawn round-robin from a shared pre-generated pool; fixed-length episodes, reward 1, discount 1."""

  def __init__(self, pool, spec, offset, episode_length):
    self._pool, self._spec, self._i, self._L, self._t = pool, spec, offset, episode_length, 0

  def _obs(self):
    self._i = (self._i + 1) % len(self._pool)
    return self._pool[self._i]

  def reset(self):
    self._t = 0
    return dm_env.restart(self._obs())

  def step(self, action):
    self._t += 1
    if self._t == self._L:
      return dm_env.termination(1.0, self._obs())
    return dm_env.transition(1.0, self._obs())

  def observation_spec(self):
    return self._spec.observations

  def action_spec(self):
    return self._spec.actions

  def reward_spec(self):
    return self._spec.rewards

  def discount_spec(self):
    return self._spec.discounts


def c2_spec():
  return specs.EnvironmentSpec(specs.Array((84, 84, 4), np.uint8), specs.DiscreteArray(18), specs.Array((), np.float32),
                               specs.BoundedArray((), np.float32, 0., 1.))


def c3_spec():
  return specs.EnvironmentSpec(specs.Array((67,), np.float32), specs.BoundedArray((21,), np.float32, -1., 1.),
                               specs.Array((), np.float32), specs.BoundedArray((), np.float32, 0., 1.))


def table_for(spec, items, frame_stack=0):
  return replay.Table(replay.DEFAULT_PRIORITY_TABLE, replay.selectors.Prioritized(0.6), replay.selectors.Fifo(), items,
                      replay.rate_limiters.MinSize(1), signature=adders.NStepTransitionAdder.signature(spec), max_window=5,
                      frame_stack=frame_stack)


def rate(fn, steps_per_call, seconds):
  """Environment steps per second of `fn` (each call ends in a device synchronise) over at least `seconds`."""
  fn()
  calls, t0 = 0, time.perf_counter()
  while True:
    fn()
    calls += 1
    el = time.perf_counter() - t0
    if el >= seconds:
      return calls * steps_per_call / el


def summary(xs):
  return dict(median=float(np.median(xs)), min=float(np.min(xs)), max=float(np.max(xs)), reps=[float(x) for x in xs])


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--num-envs', default='16,64,256')
  ap.add_argument('--reps', type=int, default=3)
  ap.add_argument('--seconds', type=float, default=2.0, help='timed window of each variant in each repetition')
  ap.add_argument('--agent-iterations', type=int, default=150, help='timed lockstep steps of the agent loop')
  ap.add_argument('--out', default=None)
  args = ap.parse_args()
  _capi.require_device(0)
  torch.cuda.set_device(0)
  Ns = [int(n) for n in args.num_envs.split(',')]
  rng = np.random.default_rng(0)
  s2, s3 = c2_spec(), c3_spec()
  pool2 = rng.integers(0, 256, (4096, 84, 84, 4), dtype=np.uint8)
  pool3 = rng.standard_normal((4096, 67)).astype(np.float32)
  net = networks.DQNAtariNetwork(18, seed=0, precision=_capi.PRECISION_BF16FLOW)
  pol = networks.D4PGPolicy(67, 21, seed=0, precision=_capi.PRECISION_TC)

  # (a) batch-1 policies
  eg = actors.EpsilonGreedyPolicy(net, 0.05, seed=0)
  gn = d4pg.GaussianNoisePolicy(pol, 0.3, -1., 1., seed=0)
  it2, it3 = iter(range(1 << 62)), iter(range(1 << 62))
  variants = {
      'batch1_c2_epsilon_greedy': (lambda: eg(pool2[next(it2) % 4096]), 1),
      'batch1_c3_gaussian': (lambda: gn(pool3[next(it3) % 4096]), 1),
  }
  # (b) batched actors: selection alone, and selection + environment steps + insert through the loop
  loops = {}
  for N in Ns:
    for name, spec, pool, policy, fs in (('c2', s2, pool2, actors.BatchedEpsilonGreedy(net, 0.05, seed=0), 4),
                                         ('c3', s3, pool3, actors.BatchedGaussianNoise(pol, 0.3, -1., 1., seed=0), 0)):
      sel = actors.BatchedActor(policy, table_for(spec, 1000, fs), N, 5)
      batch = pool[rng.integers(0, 4096, N)]
      variants[f'batched_{name}_select_n{N}'] = ((lambda a=sel, b=batch: a.select_actions(b)), N)
      policy2 = (actors.BatchedEpsilonGreedy(net, 0.05, seed=1) if name == 'c2' else
                 actors.BatchedGaussianNoise(pol, 0.3, -1., 1., seed=1))
      ins = actors.BatchedActor(policy2, table_for(spec, 100000, fs), N, 5)
      envs = [PoolEnv(pool, spec, 16 * i, 400 + i) for i in range(N)]
      loop = environment_loop.BatchedEnvironmentLoop(envs, ins, logger=loggers.NoOpLogger())
      loops[(name, N)] = loop
      variants[f'batched_{name}_select_insert_n{N}'] = ((lambda lp=loop: (lp.run(num_steps=1), torch.cuda.synchronize())), N)

  results = {k: [] for k in variants}
  agent_rates = {N: dict(env_steps_per_s=[], updates_per_s=[]) for N in Ns}
  agents = {}
  for N in Ns:   # (c) the whole DQN agent loop: learner at the reference defaults, frames deduplicated in the ring
    anet = networks.DQNAtariNetwork(18, seed=1, precision=_capi.PRECISION_BF16FLOW)
    ag = dqn.DQN(s2, anet, batch_size=256, samples_per_insert=32.0, min_replay_size=1000, max_replay_size=100000,
                 logger=loggers.NoOpLogger(), frame_stack=4, num_envs=N)
    envs = [PoolEnv(pool2, s2, 16 * i, 400 + i) for i in range(N)]
    loop = environment_loop.BatchedEnvironmentLoop(envs, ag, logger=loggers.NoOpLogger())
    loop.run(num_steps=max(3000, 20 * N))        # past min_replay_size, learner graph captured
    torch.cuda.synchronize()
    agents[N] = (ag, loop)

  for rep in range(args.reps):
    for k, (fn, per) in variants.items():
      results[k].append(rate(fn, per, args.seconds))
    for N, (ag, loop) in agents.items():
      u0 = int(ag._learner._num_steps)
      t0 = time.perf_counter()
      loop.run(num_steps=args.agent_iterations * N)
      torch.cuda.synchronize()
      el = time.perf_counter() - t0
      agent_rates[N]['env_steps_per_s'].append(args.agent_iterations * N / el)
      agent_rates[N]['updates_per_s'].append((int(ag._learner._num_steps) - u0) / el)
    print(f'rep {rep}: ' + ', '.join(f'{k} {v[-1]:.0f}' for k, v in results.items()), flush=True)

  name, limit = gpu_info()
  out = dict(gpu=name, power_limit=limit, unit='environment steps per second', reps=args.reps, seconds=args.seconds,
             variants={k: summary(v) for k, v in results.items()},
             dqn_agent_loop={f'n{N}': dict(env_steps_per_s=summary(r['env_steps_per_s']),
                                           updates_per_s=summary(r['updates_per_s']),
                                           batch_size=256, samples_per_insert=32.0, iterations=args.agent_iterations)
                             for N, r in agent_rates.items()})
  text = json.dumps(out, indent=1)
  print(text)
  if args.out:
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
      f.write(text + '\n')


if __name__ == '__main__':
  main()
