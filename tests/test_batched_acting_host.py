"""Host logic of batched acting (no GPU): BatchedAgent's learner schedule against Agent's, and BatchedEnvironmentLoop's
reports, counters, stop rule and continuation with a fake batched actor."""
import numpy as np
import pytest

from acme_b200 import agent, counting, dm_env, environment_loop, loggers


class _Learner:

  def __init__(self):
    self.steps = 0

  def step(self):
    self.steps += 1


class _FakeBatchedActor:
  """Records the protocol calls; acts with the environment index."""

  def __init__(self, num_envs):
    self.num_envs, self.calls, self.updates = num_envs, [], 0

  def observe_first(self, timesteps):
    assert all(ts.first() for ts in timesteps)
    self.calls.append(('first', len(timesteps)))

  def select_actions(self, observations):
    assert len(observations) == self.num_envs
    return np.arange(self.num_envs, dtype=np.int32)

  def observe(self, actions, next_timesteps):
    self.calls.append(('observe', [ts.step_type for ts in next_timesteps]))

  def update(self):
    self.updates += 1


class _SerialActor(_FakeBatchedActor):

  def select_action(self, observation):
    return 0

  def observe(self, action, next_timestep):
    pass


class _CountingEnv(dm_env.Environment):
  """Episodes of `length` steps; reward = the step index within the episode."""

  def __init__(self, length):
    self.length, self.t, self.resets = length, 0, 0

  def reset(self):
    self.t, self.resets = 0, self.resets + 1
    return dm_env.restart(np.float32(0))

  def step(self, action):
    self.t += 1
    if self.t == self.length:
      return dm_env.termination(reward=float(self.t), observation=np.float32(self.t))
    return dm_env.transition(reward=float(self.t), observation=np.float32(self.t))

  def observation_spec(self):
    raise NotImplementedError

  def action_spec(self):
    raise NotImplementedError


def _ts(last):
  return dm_env.termination(0., np.float32(0)) if last else dm_env.transition(0., np.float32(0))


@pytest.mark.parametrize('num_envs', [1, 3, 64])
@pytest.mark.parametrize('warmup, ratio', [(10, 4.0), (7, 1.0), (0, 2.5), (5, 0.25), (33, 0.5)])
def test_batched_agent_runs_the_updates_agent_runs(num_envs, warmup, ratio):
  single_learner, batched_learner = _Learner(), _Learner()
  single = agent.Agent(_SerialActor(1), single_learner, warmup, ratio)
  batched = agent.BatchedAgent(_FakeBatchedActor(num_envs), batched_learner, warmup, ratio)
  for it in range(40):
    for _ in range(num_envs):
      single.observe(0, _ts(False))
      single.update()
    batched.observe(np.zeros(num_envs, np.int32), [_ts(False)] * num_envs)
    batched.update()
    assert batched_learner.steps == single_learner.steps, it
  assert batched_learner.steps > 0


def test_batched_loop_reports_counts_and_continues():
  lengths = [2, 3, 5]
  envs = [_CountingEnv(n) for n in lengths]
  actor = _FakeBatchedActor(len(envs))
  log = loggers.InMemoryLogger()
  counter = counting.Counter()
  loop = environment_loop.BatchedEnvironmentLoop(envs, actor, counter=counter, logger=log)
  loop.run(num_steps=6)                      # two lockstep steps (6 environment steps): env 0 finishes once
  assert actor.calls[0] == ('first', 3) and actor.updates == 2
  assert [d['episode_length'] for d in log.data] == [2]
  assert log.data[0]['episode_return'] == 1 + 2 and log.data[0]['episodes'] == 1 and log.data[0]['steps'] == 2
  assert set(log.data[0]) >= {'episode_length', 'episode_return', 'steps_per_second', 'episodes', 'steps'}
  loop.run(num_episodes=3)                   # continues the open episodes: no new observe_first
  assert sum(c[0] == 'first' for c in actor.calls) == 1
  # steps 3, 4, 5: env0 ends at step 4, env1 at step 3, env2 at step 5 -> 3 episodes after step 5; stop there
  assert actor.updates == 5
  assert [d['episode_length'] for d in log.data] == [2, 3, 2, 5]
  assert log.data[-1]['episodes'] == 4 and log.data[-1]['steps'] == 12
  assert [e.resets for e in envs] == [3, 2, 2]
  # the step types the actor was shown: LAST exactly where an episode ended
  observed = [c[1] for c in actor.calls if c[0] == 'observe']
  assert [[t == dm_env.StepType.LAST for t in s] for s in observed] == [
      [False, False, False], [True, False, False], [False, True, False], [True, False, False], [False, False, True]]


def test_batched_loop_stops_at_the_first_step_boundary_reaching_the_limit():
  envs = [_CountingEnv(4) for _ in range(4)]
  actor = _FakeBatchedActor(4)
  loop = environment_loop.BatchedEnvironmentLoop(envs, actor, logger=loggers.NoOpLogger())
  loop.run(num_steps=5)                      # 4 < 5 -> a second step; 8 >= 5 -> stop
  assert actor.updates == 2
  loop.run(num_episodes=1)                   # all four end together at step 4: the limit is passed, not cut
  assert actor.updates == 4


def test_batched_loop_checks_the_environment_count_and_arguments():
  with pytest.raises(ValueError):
    environment_loop.BatchedEnvironmentLoop([_CountingEnv(2)] * 2, _FakeBatchedActor(3), logger=loggers.NoOpLogger())
  loop = environment_loop.BatchedEnvironmentLoop([_CountingEnv(2)], _FakeBatchedActor(1), logger=loggers.NoOpLogger())
  with pytest.raises(ValueError):
    loop.run(num_episodes=1, num_steps=1)
