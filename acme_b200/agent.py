"""Acting + learning behind one Actor facade, and the schedule that decides when the learner runs.

Behaviour contract (SURVEY App. A.3, from `acme/agents/agent.py:45-89`; pinned by tests/test_wiring.py):
  * `observe_first` never counts; every `observe` counts one observation;
  * nothing is learned before `min_observations` observations;
  * afterwards, each time `update()` finds the count on a multiple of the period, the count restarts and the learner
    runs `burst` updates, then the actor refreshes its variables;
  * `observations_per_step >= 1` -> period = int(ratio), burst = 1; a ratio below one -> period = 1, burst = int(1/ratio).
"""

from typing import Dict, List, Tuple

from acme_b200 import core


class LearnerSchedule:
  """Counts observations and answers "how many learner updates are due now?"."""

  def __init__(self, warmup: int, observations_per_step: float):
    self.period, self.burst = self._split_ratio(observations_per_step)
    self._since = -int(warmup)          # negative while the replay is still warming up

  @staticmethod
  def _split_ratio(ratio: float) -> Tuple[int, int]:
    return (int(ratio), 1) if ratio >= 1.0 else (1, int(1.0 / ratio))

  def saw_observation(self):
    self._since += 1

  def due(self) -> int:
    """Updates to run at this `update()` call; a non-zero answer restarts the count."""
    if self._since < 0 or self._since % self.period:
      return 0
    self._since = 0
    return self.burst


class Agent(core.Actor, core.VariableSource):
  """An Actor that forwards acting calls to `actor` and drives `learner.step()` on a LearnerSchedule."""

  def __init__(self, actor: core.Actor, learner: core.Learner, min_observations: int, observations_per_step: float):
    self._actor, self._learner = actor, learner
    self._schedule = LearnerSchedule(min_observations, observations_per_step)

  # acting: plain delegation
  def select_action(self, observation):
    return self._actor.select_action(observation)

  def observe_first(self, timestep):
    self._actor.observe_first(timestep)

  def observe(self, action, next_timestep):
    self._schedule.saw_observation()
    self._actor.observe(action, next_timestep)

  # learning
  def update(self):
    n = self._schedule.due()
    if n == 0:
      return
    for _ in range(n):
      self._learner.step()
    self._actor.update()

  def get_variables(self, names: List[str]):
    return self._learner.get_variables(names)


class BatchedAgent(Agent):
  """An Agent whose actor acts for N environments at once (`actors.BatchedActor`), driven by
  `environment_loop.BatchedEnvironmentLoop`.  After each step of the N environments, `update()` runs exactly the learner
  updates `Agent` would run for the same N observations fed one at a time with an `update()` after each: every
  observation is counted and the schedule's `due()` summed (a single `due()` per step would skip periods)."""

  _due = 0

  @property
  def num_envs(self) -> int:
    return self._actor.num_envs

  def select_actions(self, observations):
    return self._actor.select_actions(observations)

  def observe_first(self, timesteps):
    self._actor.observe_first(timesteps)

  def observe(self, actions, next_timesteps):
    for _ in next_timesteps:
      self._schedule.saw_observation()
      self._due += self._schedule.due()
    self._actor.observe(actions, next_timesteps)

  def update(self):
    n, self._due = self._due, 0
    if n == 0:
      return
    for _ in range(n):
      self._learner.step()
    self._actor.update()

  _variants: Dict[type, type] = {}

  @classmethod
  def variant_of(cls, agent_cls: type) -> type:
    """`agent_cls` (an Agent subclass whose constructor builds the actor) with the batched acting protocol."""
    if issubclass(agent_cls, cls):
      return agent_cls
    if agent_cls not in cls._variants:
      cls._variants[agent_cls] = type(f'Batched{agent_cls.__name__}', (cls, agent_cls), {'__module__': agent_cls.__module__})
    return cls._variants[agent_cls]
