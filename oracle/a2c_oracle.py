"""TEST INFRASTRUCTURE ONLY — CPU restatement (torch-CPU autograd) of Stable-Baselines3 2.9.0's A2C.train.  The product
path never imports this module.

PARITY UNPINNED: SB3 is not installed in this image (see oracle/ppo_oracle.py's header); this restates SB3's published
a2c.py on top of the PPO restatement's policy (A.1), GAE (A.3) and rollout conventions:
    rollout_buffer.get(batch_size=None)  -> the whole rollout is ONE batch, one gradient step per rollout
    advantages normalised only when normalize_advantage (default False): (adv - mean) / (std + 1e-8), std unbiased
    policy_loss = -(advantages * log_prob).mean();  value_loss = mse(returns, values);  entropy_loss = -mean(entropy)
    loss = policy_loss + ent_coef * entropy_loss + vf_coef * value_loss
    clip_grad_norm_(max_grad_norm);  torch.optim.RMSprop(lr, alpha=0.99, eps=rms_prop_eps=1e-5, weight_decay=0)
Defaults (A2C.__init__): learning_rate 7e-4, n_steps 5, gamma 0.99, gae_lambda 1.0, ent_coef 0.0, vf_coef 0.5,
max_grad_norm 0.5, rms_prop_eps 1e-5, use_rms_prop True, normalize_advantage False.
"""
from __future__ import annotations

import numpy as np
import torch

from . import ppo_oracle as po

RMSPROP_ALPHA = 0.99


def a2c_loss(logits, values, actions, advantages, returns, *, ent_coef=0.0, vf_coef=0.5, normalize=False):
    """A2C.train's loss for the whole batch (torch, differentiable). Returns (loss, stats dict)."""
    adv = advantages
    if normalize and adv.numel() > 1:
        adv = (adv - adv.mean()) / (adv.std() + 1e-8)
    logp, entropy = po.categorical(logits, actions)
    policy_loss = -(adv * logp).mean()
    value_loss = torch.nn.functional.mse_loss(returns, values)
    entropy_loss = -entropy.mean()
    loss = policy_loss + ent_coef * entropy_loss + vf_coef * value_loss
    stats = {k: float(v.detach()) for k, v in (("policy_loss", policy_loss), ("value_loss", value_loss), ("entropy_loss", entropy_loss),
                                                  ("loss", loss))}
    return loss, stats


def rmsprop_reference(p, g, sq, *, lr, alpha=RMSPROP_ALPHA, eps=1e-5):
    """torch.optim.RMSprop's rule written out (not centred, no momentum): float32 NumPy, eps added after the square root."""
    p, g, sq = (np.asarray(x, np.float32) for x in (p, g, sq))
    sq = (np.float32(alpha) * sq + np.float32(1.0 - alpha) * g * g).astype(np.float32)
    return (p - np.float32(lr) * (g / (np.sqrt(sq) + np.float32(eps)))).astype(np.float32), sq


class OracleA2C:
    """Flat-parameter A2C learner: evaluate -> loss -> backward -> clip_grad_norm_ -> RMSprop(alpha 0.99, eps 1e-5)."""

    def __init__(self, obs_dim, n_actions, seed=1, lr=7e-4, max_grad_norm=0.5, ent_coef=0.0, vf_coef=0.5, rms_prop_eps=1e-5,
                 normalize_advantage=False, params=None):
        self.obs_dim, self.n_actions = obs_dim, n_actions
        p = po.init_params(obs_dim, n_actions, seed) if params is None else np.asarray(params, np.float32)
        self.flat = torch.nn.Parameter(torch.from_numpy(p.copy()))
        self.opt = torch.optim.RMSprop([self.flat], lr=lr, alpha=RMSPROP_ALPHA, eps=rms_prop_eps, weight_decay=0)
        self.max_grad_norm, self.ent_coef, self.vf_coef = max_grad_norm, ent_coef, vf_coef
        self.normalize_advantage = normalize_advantage

    def evaluate(self, obs):
        with torch.no_grad():
            return po.forward(self.flat, torch.as_tensor(obs, dtype=torch.float32), self.obs_dim, self.n_actions)

    def gradient(self, obs, actions, advantages, returns):
        """Loss gradient of one batch (no step): (grad, stats)."""
        t = lambda x, dt=torch.float32: torch.as_tensor(np.asarray(x), dtype=dt)
        logits, values = po.forward(self.flat, t(obs), self.obs_dim, self.n_actions)
        loss, stats = a2c_loss(logits, values, t(actions, torch.int64), t(advantages), t(returns), ent_coef=self.ent_coef,
                               vf_coef=self.vf_coef, normalize=self.normalize_advantage)
        self.opt.zero_grad()
        loss.backward()
        return self.flat.grad.detach().clone().numpy(), stats

    def step(self, obs, actions, advantages, returns):
        """One A2C.train call on the whole rollout: (stats, pre-clip gradient)."""
        grad, stats = self.gradient(obs, actions, advantages, returns)
        stats["grad_norm"] = float(torch.nn.utils.clip_grad_norm_([self.flat], self.max_grad_norm))
        self.opt.step()
        return stats, grad
