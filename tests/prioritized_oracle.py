"""The prioritized D4PG / DDPG critic update in the oracle's terms (test infrastructure, NumPy / PyTorch-CPU).

`oracle.learner.D4PGOracleLearner` / `DDPGOracleLearner` restate the reference's uniform step; the learners' opt-in
prioritized form only changes the critic loss, so these subclasses override that one piece:

  weight    w_b = f32(f64 (1 / prob_b)^beta / max_b f64 (1 / prob_b)^beta)    (acme/agents/tf/dqn/learning.py:138-143)
  D4PG      critic loss = mean_b(w_b * CE_b)          priority_b = CE_b (the unweighted per-sample cross-entropy)
  DDPG      critic loss = mean_b(w_b * 0.5 td_b^2)    priority_b = |td_b|

The critic's gradient comes from autograd through the weighted loss; the DPG policy loss is unweighted, as in the learner.
`step(..., prob=None)` is the parent's uniform step."""
from __future__ import annotations

import numpy as np
import torch

from oracle import learner as olearner
from oracle import losses as L

f32 = np.float32


def importance_weights(prob, beta):
  """The TF DQN learner's f64 importance weights, normalised by their batch maximum and cast to f32."""
  w64 = (1.0 / np.asarray(prob, np.float64))**np.float64(beta)
  return (w64 / np.max(w64)).astype(f32)


class _Weighted:

  _weight = None

  def step(self, o_tm1, a_tm1, R, D, o_t, prob=None, beta=None):
    self._weight = None if prob is None else importance_weights(prob, beta)
    out = super().step(o_tm1, a_tm1, R, D, o_t)
    if self._weight is not None:
      out.update(weight=self._weight, priority=self._priority)
    return out


class D4PGOracleLearner(_Weighted, olearner.D4PGOracleLearner):

  def _critic_loss(self, logits_tm1, logits_t, Rn, Dg):
    ref, loss = super()._critic_loss(logits_tm1, logits_t, Rn, Dg)
    if self._weight is None:
      return ref, loss
    w = self._weight
    target = torch.tensor(ref['target'])
    ce = -(target * torch.log_softmax(logits_tm1, dim=-1)).sum(dim=-1)
    self._priority = ref['loss']
    ref = dict(ref, loss=(ref['loss'] * w).astype(f32), dlogits_tm1=(ref['dlogits_tm1'] * w[:, None]).astype(f32))
    return ref, (torch.tensor(w) * ce).mean()


class DDPGOracleLearner(_Weighted, olearner.DDPGOracleLearner):

  def _critic_loss(self, q_tm1, q_t, Rn, Dg):
    ref, loss = super()._critic_loss(q_tm1, q_t, Rn, Dg)
    if self._weight is None:
      return ref, loss
    w = self._weight
    td = (torch.tensor(Rn) + torch.tensor(Dg) * q_t[:, 0]) - q_tm1[:, 0]
    self._priority = np.abs(ref['td']).astype(f32)
    ref = dict(ref, loss=(ref['loss'] * w).astype(f32), dv_tm1=(-ref['td'] * w / f32(len(w))).astype(f32))
    return ref, (torch.tensor(w) * (0.5 * td * td)).mean()

