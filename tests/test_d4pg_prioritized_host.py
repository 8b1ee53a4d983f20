"""Prioritized D4PG / DDPG without a GPU: the argument rules of the learners and agents, and the oracle's weighted
critic step (tests/prioritized_oracle.py) against the uniform oracle and the DQN oracle's importance weights."""
import numpy as np
import pytest


@pytest.mark.parametrize('cls', ['D4PGLearner', 'DDPGLearner'])
def test_learner_rejects_forbidden_combinations(cls):
  from acme_b200 import d4pg
  learner = getattr(d4pg, cls)
  args = (None, None, None, None, 0.99, 100, None)
  with pytest.raises(ValueError, match='importance_sampling_exponent'):
    learner(*args, replay_client=object())
  with pytest.raises(ValueError, match='data-parallel'):
    learner(*args, importance_sampling_exponent=0.4, process_group=object())
  with pytest.raises(ValueError, match='>= 0'):
    learner(*args, importance_sampling_exponent=-0.1)


@pytest.mark.parametrize('cls', ['D4PG', 'DDPG'])
@pytest.mark.parametrize('num_envs', [1, 16])
def test_agent_needs_both_exponents(cls, num_envs):
  from acme_b200 import d4pg
  agent = getattr(d4pg, cls)
  for kw in (dict(priority_exponent=0.6), dict(importance_sampling_exponent=0.4)):
    with pytest.raises(ValueError, match='both'):
      agent(None, None, None, num_envs=num_envs, **kw)


def test_importance_weights_are_the_dqn_oracles():
  import prioritized_oracle as po
  from oracle import losses as L
  rng = np.random.default_rng(0)
  B = 64
  prob = rng.uniform(1e-4, 1e-2, B).astype(np.float32)
  z = np.zeros((B, 2), np.float32)
  ref = L.dqn_loss(z, z, z, np.zeros(B, np.int64), np.zeros(B, np.float32), np.zeros(B, np.float32), prob, 0.99,
                   is_exponent=0.4)
  np.testing.assert_array_equal(po.importance_weights(prob, 0.4), ref['weight'])


def _pair(kind, seed=0):
  import prioritized_oracle as po
  from oracle import learner as olearner
  from oracle import nets as onets
  obs, act = 5, 3
  rng = np.random.default_rng(seed)
  out = []
  for cls in ((olearner.D4PGOracleLearner, po.D4PGOracleLearner) if kind == 'd4pg' else
              (olearner.DDPGOracleLearner, po.DDPGOracleLearner)):
    ccls = onets.D4PGCritic if kind == 'd4pg' else onets.DDPGCritic
    nets = [onets.D4PGPolicy(obs, act, sizes=(16, 16)), ccls(obs, act, sizes=(16, 16))]
    out.append((cls(nets[0], nets[1], onets.D4PGPolicy(obs, act, sizes=(16, 16)), ccls(obs, act, sizes=(16, 16)), 0.99, 2), nets))
  (a, na), (b, nb) = out
  for x, y in zip(na, nb):
    y.load(x.numpy())
  B = 8
  batch = (rng.standard_normal((B, obs)).astype(np.float32), rng.uniform(-1, 1, (B, act)).astype(np.float32),
           rng.standard_normal(B).astype(np.float32), np.ones(B, np.float32), rng.standard_normal((B, obs)).astype(np.float32))
  return a, b, batch


@pytest.mark.parametrize('kind', ['d4pg', 'ddpg'])
def test_weighted_oracle_with_equal_probabilities_is_the_uniform_oracle(kind):
  a, b, batch = _pair(kind)
  B = batch[0].shape[0]
  ra = a.step(*batch)
  rb = b.step(*batch, prob=np.full(B, 0.01, np.float32), beta=0.4)
  assert np.all(rb['weight'] == 1)
  np.testing.assert_array_equal(rb['per_sample'], ra['per_sample'])
  np.testing.assert_array_equal(rb['critic_loss'], ra['critic_loss'])
  for k in ra['critic_grads']:
    np.testing.assert_array_equal(rb['critic_grads'][k], ra['critic_grads'][k])
  want = ra['per_sample'] if kind == 'd4pg' else np.abs(ra['td'])
  np.testing.assert_array_equal(rb['priority'], want)


@pytest.mark.parametrize('kind', ['d4pg', 'ddpg'])
def test_weighted_oracle_scales_the_critic_loss(kind):
  """Unequal probabilities: the per-sample loss is w * the unweighted one, the batch loss their mean, the policy step
  unweighted."""
  a, b, batch = _pair(kind, seed=1)
  B = batch[0].shape[0]
  prob = np.linspace(0.001, 0.01, B).astype(np.float32)
  ra = a.step(*batch)
  rb = b.step(*batch, prob=prob, beta=0.5)
  w = rb['weight']
  assert w.max() == 1 and w.min() < 1
  np.testing.assert_array_equal(rb['per_sample'], (ra['per_sample'] * w).astype(np.float32))
  np.testing.assert_allclose(rb['critic_loss'], rb['per_sample'].astype(np.float64).mean(), rtol=1e-6)
  np.testing.assert_array_equal(rb['dqda'], ra['dqda'])
  for k in ra['policy_grads']:
    np.testing.assert_array_equal(rb['policy_grads'][k], ra['policy_grads'][k])
