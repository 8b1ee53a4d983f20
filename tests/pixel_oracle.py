"""D4PG / DDPG from pixels in the oracle's terms (test infrastructure, PyTorch-CPU fp32).

`AtariTorso` restates acme/tf/networks/atari.py:36-52 with the convolutions of `oracle.nets.DQNAtariNetwork` (same
initialisation draws, TF SAME padding, flattened in (h, w, c) order): the observation network.

`D4PGOracleLearner` / `DDPGOracleLearner` are the oracle's uniform step (`oracle.learner`) with an observation network in
front (acme/agents/tf/d4pg/learning.py:189-195; the semantics are the decision recorded in DESIGN.md §5):
  * o_tm1 -> obs_net, trained by the critic loss only; o_t -> target_obs_net once, without gradient, read by the target
    chain and by the DPG chain (so the policy loss does not reach the torso);
  * obs_net's variables join the critic's under one clip_by_global_norm(40) and the critic's Adam (moments keyed
    'obs/<name>');
  * the periodic target copy covers obs_net.
The critic loss is the parent's (`_critic_loss`: categorical for D4PG, td_learning for DDPG)."""
from __future__ import annotations

import math

import numpy as np
import torch

from oracle import learner as olearner
from oracle import losses as L
from oracle import nets as onets


class AtariTorso(onets._Net):

  def __init__(self, seed=0, in_hw=84, in_c=4):
    super().__init__()
    rng = np.random.default_rng(seed)
    h = in_hw
    for i, (k, s, ci, co) in enumerate([(8, 4, in_c, 32), (4, 2, 32, 64), (3, 1, 64, 64)], 1):
      self._add(f'conv{i}/w', onets.truncated_normal(rng, (k, k, ci, co), 1 / math.sqrt(k * k * ci)))
      self._add(f'conv{i}/b', np.zeros(co, np.float32))
      h = onets.tf_same_pad(h, k, s)[0]
    self.flat = h * h * 64

  def __call__(self, obs_nhwc_f32: torch.Tensor) -> torch.Tensor:
    x = obs_nhwc_f32
    for i, s in ((1, 4), (2, 2), (3, 1)):
      x = torch.relu(onets._conv_same(x, self.vars[f'conv{i}/w'], self.vars[f'conv{i}/b'], s))
    return x.reshape(x.shape[0], -1)


class _Pixels:

  def __init__(self, *args, obs_net, target_obs_net, **kwargs):
    super().__init__(*args, **kwargs)
    self.obs_net, self.tobs_net = obs_net, target_obs_net

  def step(self, o_tm1, a_tm1, R, D, o_t):
    if self.num_steps % self.period == 0:
      self.tpolicy.copy_from(self.policy)
      self.tcritic.copy_from(self.critic)
      self.tobs_net.copy_from(self.obs_net)
    self.num_steps += 1
    f0 = self.obs_net(torch.tensor(olearner.preprocess_obs(o_tm1)))
    with torch.no_grad():
      f1 = self.tobs_net(torch.tensor(olearner.preprocess_obs(o_t)))
    a0 = torch.tensor(np.asarray(a_tm1, np.float32))
    Rn = np.asarray(R, np.float32)
    Dg = (self.discount * np.asarray(D, np.float32)).astype(np.float32)

    logits_tm1 = self.critic.logits(f0, a0)
    with torch.no_grad():
      logits_t = self.tcritic.logits(f1, self.tpolicy.action(f1))
    ref, critic_loss = self._critic_loss(logits_tm1, logits_t, Rn, Dg)

    a_t = self.policy.action(f1)
    a_leaf = a_t.detach().clone().requires_grad_(True)
    q = self.critic.mean(f1, a_leaf)
    dqda = torch.autograd.grad(q.sum(), a_leaf)[0].numpy()
    da, dqda_clipped = L.dpg_action_grad(dqda, 1.0 if self.clipping else None, self.clipping)
    policy_loss = np.float32(0.5 * (dqda_clipped**2).sum(axis=-1).mean())

    on, cn, pn = self.obs_net.names(), self.critic.names(), self.policy.names()
    g = torch.autograd.grad(critic_loss, [self.obs_net.vars[k] for k in on] + [self.critic.vars[k] for k in cn])
    og = {'obs/' + k: x.numpy() for k, x in zip(on, g[:len(on)])}
    cg = {k: x.numpy() for k, x in zip(cn, g[len(on):])}
    pg = torch.autograd.grad(a_t, [self.policy.vars[k] for k in pn], grad_outputs=torch.tensor(da))
    pg = {k: x.numpy() for k, x in zip(pn, pg)}
    cnorm = pnorm = None
    if self.clipping:
      lst, pnorm = L.clip_by_global_norm([pg[k] for k in pn], 40.)
      pg = dict(zip(pn, lst))
      keys = list(og) + cn
      lst, cnorm = L.clip_by_global_norm([og[k] if k in og else cg[k] for k in keys], 40.)
      og, cg = dict(zip(keys[:len(og)], lst[:len(og)])), dict(zip(cn, lst[len(og):]))
    self.policy.load(self.popt.apply(pg, self.policy.numpy()))
    params = dict(self.critic.numpy(), **{'obs/' + k: v for k, v in self.obs_net.numpy().items()})
    new = self.copt.apply(dict(cg, **og), params)
    self.critic.load({k: new[k] for k in cn})
    self.obs_net.load({k: new['obs/' + k] for k in on})
    return dict(critic_loss=np.float32(critic_loss.item()), policy_loss=policy_loss,
                target=ref.get('target'), per_sample=ref['loss'], td=ref.get('td'),
                logits_tm1=logits_tm1.detach().numpy(), logits_t=logits_t.numpy(), dqda=dqda,
                critic_grads=cg, obs_grads=og, policy_grads=pg, critic_norm=cnorm, policy_norm=pnorm)


class D4PGOracleLearner(_Pixels, olearner.D4PGOracleLearner):
  pass


class DDPGOracleLearner(_Pixels, olearner.DDPGOracleLearner):
  pass
