"""EnvironmentLoop: drives an environment through the Actor seam (`acme/environment_loop.py:29-144`).

Contract kept from the reference (pinned by tests/test_wiring.py and tests/test_gpu_agents.py):
  * per environment step the actor sees `select_action -> (env.step) -> observe -> update`, after one `observe_first`;
  * an episode reports `episode_length`, `episode_return`, `steps_per_second` plus the shared counter's totals
    (`episodes`, `steps`), and the counter advances once per episode;
  * `run` stops after `num_episodes` episodes or once at least `num_steps` steps were taken (the episode in progress is
    always finished); giving both is an error; giving neither runs forever.
"""

import time
from typing import Iterator, Optional

from acme_b200 import core, counting, loggers


class EnvironmentLoop(core.Worker):

  def __init__(self, environment, actor: core.Actor, counter: counting.Counter = None,
               logger: loggers.Logger = None, label: str = 'environment_loop'):
    self._environment = environment
    self._actor = actor
    self._counter = counter or counting.Counter()
    self._logger = logger or loggers.make_default_logger(label)

  def _play(self) -> Iterator:
    """One episode, one yielded reward per environment step."""
    env, actor = self._environment, self._actor
    ts = env.reset()
    actor.observe_first(ts)
    while not ts.last():
      action = actor.select_action(ts.observation)
      ts = env.step(action)
      actor.observe(action, next_timestep=ts)
      actor.update()
      yield ts.reward

  def run_episode(self):
    began = time.time()
    length, total = 0, 0
    for reward in self._play():
      length += 1
      total += reward
    elapsed = max(time.time() - began, 1e-9)
    report = dict(episode_length=length, episode_return=total, steps_per_second=length / elapsed)
    report.update(self._counter.increment(episodes=1, steps=length))
    return report

  def run(self, num_episodes: Optional[int] = None, num_steps: Optional[int] = None):
    if num_episodes is not None and num_steps is not None:
      raise ValueError('Either "num_episodes" or "num_steps" should be None.')
    limit, unit = (num_episodes, 'episodes') if num_episodes is not None else (num_steps, 'steps')
    spent = {'episodes': 0, 'steps': 0}
    while limit is None or spent[unit] < limit:
      report = self.run_episode()
      spent['episodes'] += 1
      spent['steps'] += report['episode_length']
      self._logger.write(report)


class BatchedEnvironmentLoop(core.Worker):
  """Steps N ordinary dm_env environments in lockstep through a batched actor (`actors.BatchedActor`,
  `agent.BatchedAgent`): per step `select_actions(N observations) -> N x env.step -> observe -> update`.

  * every environment is reset on its own when its episode ends; each finished episode is reported with the keys
    EnvironmentLoop writes (`episode_length`, `episode_return`, `steps_per_second` and the counter's totals);
  * `run` counts episodes finished and steps taken over all environments and stops at the first step of the N
    environments that reaches `num_episodes` or `num_steps`; giving both is an error, neither runs forever;
  * unfinished episodes stay open: the next `run` continues them.
  """

  def __init__(self, environments, actor, counter: counting.Counter = None, logger: loggers.Logger = None,
               label: str = 'environment_loop'):
    self._environments = list(environments)
    if len(self._environments) != actor.num_envs:
      raise ValueError(f'{len(self._environments)} environments for an actor of num_envs = {actor.num_envs}')
    self._actor = actor
    self._counter = counter or counting.Counter()
    self._logger = logger or loggers.make_default_logger(label)
    self._timesteps = None

  def _begin(self, i: int):
    self._length[i], self._return[i], self._began[i] = 0, 0, time.time()

  def run(self, num_episodes: Optional[int] = None, num_steps: Optional[int] = None):
    if num_episodes is not None and num_steps is not None:
      raise ValueError('Either "num_episodes" or "num_steps" should be None.')
    envs, actor, N = self._environments, self._actor, len(self._environments)
    if self._timesteps is None:
      self._timesteps = [env.reset() for env in envs]
      self._length, self._return, self._began = [0] * N, [0] * N, [0.0] * N
      for i in range(N):
        self._begin(i)
      actor.observe_first(self._timesteps)
    limit, unit = (num_episodes, 'episodes') if num_episodes is not None else (num_steps, 'steps')
    spent = {'episodes': 0, 'steps': 0}
    while limit is None or spent[unit] < limit:
      actions = actor.select_actions([ts.observation for ts in self._timesteps])
      next_timesteps = [env.step(a) for env, a in zip(envs, actions)]
      actor.observe(actions, next_timesteps)
      actor.update()
      spent['steps'] += N
      for i, ts in enumerate(next_timesteps):
        self._length[i] += 1
        self._return[i] += ts.reward
        if ts.last():
          elapsed = max(time.time() - self._began[i], 1e-9)
          report = dict(episode_length=self._length[i], episode_return=self._return[i],
                        steps_per_second=self._length[i] / elapsed)
          report.update(self._counter.increment(episodes=1, steps=self._length[i]))
          self._logger.write(report)
          spent['episodes'] += 1
          ts = envs[i].reset()
          self._begin(i)
        self._timesteps[i] = ts
