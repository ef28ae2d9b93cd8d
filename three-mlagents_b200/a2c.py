"""CudaA2C — SB3-compatible A2C front-end on the same device-resident pipeline as CudaPPO.

SB3 2.9.0's A2C shares OnPolicyAlgorithm.collect_rollouts, RolloutBuffer, GAE and ActorCriticPolicy with PPO, so this
class inherits the rollout (tmla_rollout: sampling, timeout bootstrap, GAE), predict / evaluate, the learn loop and the
data-parallel set-up from CudaPPO.  What differs is A2C.train:
  * ONE gradient step per rollout over all n_steps x n_envs rows (rollout_buffer.get(batch_size=None)); the row order does
    not matter for a single batch, so the buffers are read in place (no permutation);
  * the loss is the plain policy gradient -(adv * log_prob).mean() + ent_coef * entropy_loss + vf_coef * value_loss
    (tmla_a2c_batch_bf16 fused, tmla_a2c_loss on the three-call path), advantages normalised only on request;
  * the optimizer is torch.optim.RMSprop(alpha=0.99, eps=rms_prop_eps) after clip_grad_norm_, one launch
    (tmla_rmsprop_clip_fused, or tmla_rmsprop_clip_allreduce with the gradient exchange fused in at world_size > 1).
"""
from __future__ import annotations

from typing import Any

import torch
from torch.cuda import nvtx

from . import ops
from .distributed import allreduce_sum_
from .ppo import CudaPPO, _on_device
from .vec_env import CudaVecEnv

RMSPROP_ALPHA = 0.99


class CudaA2C(CudaPPO):
    algorithm = "a2c"
    _log_interval = 100               # SB3 A2C.learn's default: its iterations are a few steps long
    _row_every_iteration = False
    _HYPER_KEYS = ("learning_rate", "n_steps", "gamma", "gae_lambda", "ent_coef", "vf_coef", "max_grad_norm", "rms_prop_eps",
                   "normalize_advantage")

    def __init__(self, policy: str, env: CudaVecEnv, *, seed: int = 1, learning_rate: float = 7e-4, n_steps: int = 5,
                 gamma: float = 0.99, gae_lambda: float = 1.0, ent_coef: float = 0.0, vf_coef: float = 0.5,
                 max_grad_norm: float = 0.5, rms_prop_eps: float = 1e-5, use_rms_prop: bool = True,
                 normalize_advantage: bool = False, policy_kwargs: dict | None = None, tensorboard_log: str | None = None,
                 verbose: int = 0, mlp_impl: str = "auto", fused_update: bool = True, rollout_impl: str = "fused",
                 _params: torch.Tensor | None = None):
        if not use_rms_prop:
            raise ValueError("CudaA2C implements A2C's RMSprop optimizer only (use_rms_prop=True)")
        pk = dict(policy_kwargs or {})
        pk.pop("optimizer_class", None)               # what SB3 stores for use_rms_prop; the optimizer is fixed here
        pk.pop("optimizer_kwargs", None)
        # the whole rollout is one batch: CudaPPO's buffers are sized for a minibatch of n_steps * n_envs rows
        super().__init__(policy, env, seed=seed, learning_rate=learning_rate, n_steps=n_steps, batch_size=n_steps * env.num_envs,
                         n_epochs=1, gamma=gamma, gae_lambda=gae_lambda, clip_range=0.0, ent_coef=ent_coef, vf_coef=vf_coef,
                         max_grad_norm=max_grad_norm, normalize_advantage=normalize_advantage, policy_kwargs=pk or None,
                         tensorboard_log=tensorboard_log, verbose=verbose, mlp_impl=mlp_impl, fused_update=fused_update,
                         rollout_impl=rollout_impl, _params=_params)
        self.rms_prop_eps = float(rms_prop_eps)
        self.use_rms_prop = True
        self.m = self.v = None                        # Adam state of the base class: unused
        self.sq_avg = torch.zeros_like(self.params)   # RMSprop square_avg
        self._opt_step = 0                            # optimizer steps (the exchange sequence number at world_size > 1)
        if self._comm is not None:
            self.allreduce_impl = "peer-memory one-shot, fused with clip+RMSprop (csrc/comm.cu)"

    @_on_device
    def train(self):
        """A2C.train: one forward + loss + backward over the whole rollout, clip_grad_norm_, RMSprop.step."""
        T, N, D, A = self.n_steps, self.n_envs, self.obs_dim, self.n_actions
        total = T * N
        self._alloc()
        obs_flat = self.obs[:T].reshape(total, D)
        nvtx.range_push("update")
        sums = None
        if self.normalize_advantage and total * self.world > 1:
            sums = ops.adv_stats(self.adv, None, total, self.adv_sums[0])
            allreduce_sum_(self.adv_sums)
        common = dict(rows=total, global_rows=total * self.world, adv_sums=sums, normalize=sums is not None, ent_coef=self.ent_coef,
                      vf_coef=self.vf_coef)
        if self.fused_update:              # the optimizer step below leaves the gradient zeroed
            ops.a2c_batch(self.params, self.wpack, obs_flat, D, A, self.act, self.adv, self.ret, grads=self.grads,
                          scratch=self.scratch_mb, stats=self.stats_acc, grads_zeroed=True, **common)
        else:
            ops.mlp_forward(self.params, obs_flat, D, A, rows=total, logits=self.logits_mb, values=self.values_mb,
                            act_cache=self.cache_mb, wpack=self.wpack)
            ops.a2c_loss(self.logits_mb, self.values_mb, self.act, self.adv, self.ret, dlogits=self.dlogits, dvalues=self.dvalues,
                         stats=self.stats_acc, **common)
            ops.mlp_backward(self.params, obs_flat, D, A, self.cache_mb, self.dlogits, self.dvalues, rows=total, grads=self.grads,
                             scratch=self.scratch_mb, wpack=self.wpack)
        self._opt_step += 1
        opt = dict(max_grad_norm=self.max_grad_norm, lr=self.lr, alpha=RMSPROP_ALPHA, eps=self.rms_prop_eps, norm_out=self.norm_out,
                   zero_grads=True)
        if self._comm is not None:
            nvtx.range_push("allreduce+rmsprop")
            ops.rmsprop_clip_allreduce(self._comm, self.params, self.grads, self.sq_avg, self._opt_step, **opt)
            nvtx.range_pop()
        else:
            if self.world > 1:
                nvtx.range_push("allreduce")
                self._allreduce_grads(self.grads)
                nvtx.range_pop()
            ops.rmsprop_clip(self.params, self.grads, self.sq_avg, **opt)
        self._repack()                     # one step per rollout: the full repack serves the next rollout and update
        self.n_updates += 1
        if self._comm is not None:
            self._comm.check()
        nvtx.range_pop()
        return 1

    def _log_row(self, n_mb: int, t_roll: float, t_train: float, t0: float) -> dict[str, Any]:
        """SB3 A2C's logger keys: train/policy_loss, value_loss, entropy_loss, explained_variance, n_updates, learning_rate."""
        row = super()._log_row(n_mb, t_roll, t_train, t0)
        row["train/policy_loss"] = row.pop("train/policy_gradient_loss")
        for k in ("train/approx_kl", "train/clip_fraction", "train/loss", "train/clip_range"):
            row.pop(k)
        return row

    def _load_optimizer_state(self, z: dict, meta: dict) -> None:
        if z.get("sq_avg") is not None:
            self.sq_avg.copy_(z["sq_avg"])
        self._opt_step = int(meta.get("opt_step", z.get("opt_step", 0)))


def smoke_update() -> None:
    """A few A2C iterations on cuda:0: parameters move and stay finite."""
    import math

    env = CudaVecEnv("ball3d", 256, seed=1)
    model = CudaA2C("MlpPolicy", env, seed=1, ent_coef=0.01)
    before = model.params.clone()
    model.learn(256 * 5 * 4)
    torch.cuda.synchronize()
    row = model.logger_rows[-1]
    assert torch.isfinite(model.params).all() and not torch.equal(before, model.params)
    assert math.isfinite(row["train/policy_loss"]) and row["train/n_updates"] == 4
    env.close()
