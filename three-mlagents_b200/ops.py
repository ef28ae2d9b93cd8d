"""Torch-tensor wrappers over the PPO and A2C entry points of libtmla.so (include/tmla.h).

Each function takes CUDA tensors, checks dtype/contiguity/device, and enqueues the kernel on
torch's current stream.  torch is plumbing here (memory + streams); the arithmetic is in csrc/.
"""
from __future__ import annotations

import torch

from . import native
from .native import lib, check, ptr

HIDDEN = 256


def _chk(t, dtype, name):
    if t is None:
        return
    if not t.is_cuda:
        raise ValueError(f"{name} must be a CUDA tensor (this backend has no CPU path)")
    if t.dtype != dtype:
        raise TypeError(f"{name} must be {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise ValueError(f"{name} must be contiguous")


def _s():
    return native.current_stream()


def num_params(obs_dim: int, n_actions: int) -> int:
    n = lib.tmla_mlp_num_params(obs_dim, HIDDEN, n_actions)
    if n < 0:
        raise ValueError("unsupported MLP shape")
    return int(n)


def gae(rewards, values, dones, last_values, gamma: float, gae_lambda: float, advantages=None, returns=None):
    """RolloutBuffer.compute_returns_and_advantage on [T,n] buffers."""
    T, n = rewards.shape
    _chk(rewards, torch.float32, "rewards"); _chk(values, torch.float32, "values")
    _chk(dones, torch.uint8, "dones"); _chk(last_values, torch.float32, "last_values")
    if advantages is None:
        advantages = torch.empty_like(rewards)
    if returns is None:
        returns = torch.empty_like(rewards)
    check(lib.tmla_gae(ptr(rewards), ptr(values), ptr(dones), ptr(last_values), float(gamma), float(gae_lambda),
                       int(T), int(n), ptr(advantages), ptr(returns), _s()))
    return advantages, returns


def permutation(seed: int, epoch: int, T: int, n: int, out=None, device="cuda"):
    total = T * n
    if out is None:
        out = torch.empty(total, dtype=torch.int32, device=device)
    _chk(out, torch.int32, "out")
    check(lib.tmla_permutation(int(seed) & (2**64 - 1), int(epoch), total, int(T), int(n), ptr(out), _s()))
    return out


def mlp_pack(params, obs_dim, n_actions, wpack=None):
    """bf16 copies {pi.W2, pi.W2^T, vf.W2, vf.W2^T, pi.W2 image, vf.W2 image} for the tensor-core path (refresh after
    every optimizer step)."""
    if wpack is None:
        wpack = torch.empty((6, HIDDEN, HIDDEN), dtype=torch.bfloat16, device=params.device)
    _chk(wpack, torch.bfloat16, "wpack")
    check(lib.tmla_mlp_pack_bf16(ptr(params), obs_dim, HIDDEN, n_actions, ptr(wpack), _s()))
    return wpack


def mlp_forward(params, x, obs_dim, n_actions, *, index=None, rows=None, rows_dev=None, logits=None, values=None,
                want_logits=True, want_values=True, act_cache=None, wpack=None, keep_act=True):
    """ActorCriticPolicy.forward.  wpack=None: float32 CUDA-core path; wpack=bf16 pack: tcgen05 path
    (act_cache is then bf16 [4,rows,256])."""
    _chk(params, torch.float32, "params"); _chk(x, torch.float32, "x"); _chk(index, torch.int32, "index")
    if rows is None:
        rows = index.numel() if index is not None else x.shape[0]
    dev = params.device
    act_dtype = torch.float32 if wpack is None else torch.bfloat16
    if want_logits and logits is None:
        logits = torch.empty((rows, n_actions), dtype=torch.float32, device=dev)
    if want_values and values is None:
        values = torch.empty(rows, dtype=torch.float32, device=dev)
    if wpack is not None and not keep_act and obs_dim <= 6:
        act_cache = None            # fused tower kernel, inference only: no activation workspace
    elif act_cache is None:
        act_cache = torch.empty((4, rows, HIDDEN), dtype=act_dtype, device=dev)
    _chk(act_cache, act_dtype, "act_cache")
    lg, vl = (ptr(logits) if want_logits else None), (ptr(values) if want_values else None)
    if wpack is None:
        check(lib.tmla_mlp_forward(ptr(params), obs_dim, HIDDEN, n_actions, ptr(x), ptr(index), int(rows), ptr(rows_dev),
                                   lg, vl, ptr(act_cache), _s()))
    else:
        check(lib.tmla_mlp_forward_bf16(ptr(params), ptr(wpack), obs_dim, HIDDEN, n_actions, ptr(x), ptr(index), int(rows),
                                        ptr(rows_dev), lg, vl, ptr(act_cache), _s()))
    return logits, values, act_cache


def mlp_backward(params, x, obs_dim, n_actions, act_cache, dlogits, dvalues, *, index=None, rows=None, grads=None,
                 scratch=None, wpack=None):
    if rows is None:
        rows = index.numel() if index is not None else x.shape[0]
    dev = params.device
    act_dtype = torch.float32 if wpack is None else torch.bfloat16
    if grads is None:
        grads = torch.empty_like(params)
    if scratch is None:
        scratch = torch.empty(lib.tmla_mlp_backward_scratch(obs_dim, HIDDEN, n_actions, rows), dtype=act_dtype, device=dev)
    _chk(dlogits, torch.float32, "dlogits"); _chk(dvalues, torch.float32, "dvalues")
    _chk(act_cache, act_dtype, "act_cache"); _chk(scratch, act_dtype, "scratch")
    if wpack is None:
        check(lib.tmla_mlp_backward(ptr(params), obs_dim, HIDDEN, n_actions, ptr(x), ptr(index), int(rows), ptr(act_cache),
                                    ptr(dlogits), ptr(dvalues), ptr(grads), ptr(scratch), _s()))
    else:
        check(lib.tmla_mlp_backward_bf16(ptr(params), ptr(wpack), obs_dim, HIDDEN, n_actions, ptr(x), ptr(index), int(rows),
                                         ptr(act_cache), ptr(dlogits), ptr(dvalues), ptr(grads), ptr(scratch), _s()))
    return grads


def adv_stats(advantages, index, rows, sums=None):
    if sums is None:
        sums = torch.empty(3, dtype=torch.float64, device=advantages.device)
    check(lib.tmla_adv_stats(ptr(advantages), ptr(index), int(rows), ptr(sums), _s()))
    return sums


def adv_stats_batched(advantages, index, total, mb_rows, sums=None):
    """(sum, sum of squares, count) of the advantages of every minibatch of an epoch: double[n_mb, 3]."""
    n_mb = (total + mb_rows - 1) // mb_rows
    if sums is None:
        sums = torch.empty((n_mb, 3), dtype=torch.float64, device=advantages.device)
    _chk(sums, torch.float64, "sums")
    check(lib.tmla_adv_stats_batched(ptr(advantages), ptr(index), int(total), int(mb_rows), ptr(sums), _s()))
    return sums


def ppo_loss(logits, values, actions, advantages, old_logp, returns, *, index=None, rows=None, global_rows=None,
             adv_sums=None, normalize=True, clip_range=0.2, ent_coef=0.01, vf_coef=0.5, dlogits=None, dvalues=None,
             stats=None):
    if rows is None:
        rows = logits.shape[0]
    n_actions = logits.shape[1]
    dev = logits.device
    _chk(actions, torch.int32, "actions"); _chk(index, torch.int32, "index")
    if dlogits is None:
        dlogits = torch.empty_like(logits)
    if dvalues is None:
        dvalues = torch.empty(rows, dtype=torch.float32, device=dev)
    if stats is None:
        stats = torch.empty(8, dtype=torch.float32, device=dev)
    if normalize and adv_sums is None:
        adv_sums = adv_stats(advantages, index, rows)
    check(lib.tmla_ppo_loss(ptr(logits), ptr(values), ptr(actions), ptr(advantages), ptr(old_logp), ptr(returns),
                            ptr(index), int(rows), int(global_rows or rows), int(n_actions), ptr(adv_sums),
                            1 if normalize else 0, float(clip_range), float(ent_coef), float(vf_coef), ptr(dlogits),
                            ptr(dvalues), ptr(stats), _s()))
    return dlogits, dvalues, stats


def a2c_loss(logits, values, actions, advantages, returns, *, index=None, rows=None, global_rows=None, adv_sums=None,
             normalize=False, ent_coef=0.0, vf_coef=0.5, dlogits=None, dvalues=None, stats=None):
    """A2C.train's loss head (tmla_a2c_loss): ppo_loss without old_logp and clip_range; normalisation off by default (SB3's A2C)."""
    if rows is None:
        rows = logits.shape[0]
    n_actions = logits.shape[1]
    dev = logits.device
    _chk(actions, torch.int32, "actions"); _chk(index, torch.int32, "index")
    if dlogits is None:
        dlogits = torch.empty_like(logits)
    if dvalues is None:
        dvalues = torch.empty(rows, dtype=torch.float32, device=dev)
    if stats is None:
        stats = torch.empty(8, dtype=torch.float32, device=dev)
    if normalize and adv_sums is None:
        adv_sums = adv_stats(advantages, index, rows)
    check(lib.tmla_a2c_loss(ptr(logits), ptr(values), ptr(actions), ptr(advantages), ptr(returns), ptr(index), int(rows),
                            int(global_rows or rows), int(n_actions), ptr(adv_sums), 1 if normalize else 0, float(ent_coef),
                            float(vf_coef), ptr(dlogits), ptr(dvalues), ptr(stats), _s()))
    return dlogits, dvalues, stats


def ppo_minibatch_supported(obs_dim: int, n_actions: int) -> bool:
    return bool(lib.tmla_ppo_minibatch_supported(obs_dim, HIDDEN, n_actions))


def ppo_minibatch(params, wpack, obs, obs_dim, n_actions, actions, advantages, old_logp, returns, *, index=None, rows=None,
                  global_rows=None, adv_sums=None, normalize=True, clip_range=0.2, ent_coef=0.01, vf_coef=0.5, grads=None,
                  scratch=None, stats=None, logits=None, values=None, grads_zeroed=False, accumulate_stats=False):
    """One PPO.train minibatch, forward + loss + backward fused (tmla_ppo_minibatch_bf16): returns (grads, stats).
    grads_zeroed: `grads` is known to be all zeros (adam_clip(zero_grads=True) left it so) — skips the memset launch;
    accumulate_stats: add to `stats` instead of overwriting it."""
    _chk(params, torch.float32, "params"); _chk(wpack, torch.bfloat16, "wpack"); _chk(obs, torch.float32, "obs")
    _chk(index, torch.int32, "index"); _chk(actions, torch.int32, "actions"); _chk(advantages, torch.float32, "advantages")
    _chk(old_logp, torch.float32, "old_logp"); _chk(returns, torch.float32, "returns")
    if rows is None:
        rows = index.numel() if index is not None else obs.shape[0]
    dev = params.device
    if grads is None:
        grads = torch.empty_like(params)
    if scratch is None:
        scratch = torch.empty(lib.tmla_ppo_minibatch_scratch(HIDDEN, rows), dtype=torch.bfloat16, device=dev)
    if stats is None:
        stats = torch.empty(8, dtype=torch.float32, device=dev)
    _chk(scratch, torch.bfloat16, "scratch"); _chk(grads, torch.float32, "grads"); _chk(stats, torch.float32, "stats")
    _chk(logits, torch.float32, "logits"); _chk(values, torch.float32, "values")
    if normalize and adv_sums is None:
        adv_sums = adv_stats(advantages, index, rows)
    check(lib.tmla_ppo_minibatch_bf16(ptr(params), ptr(wpack), obs_dim, HIDDEN, n_actions, ptr(obs), ptr(index), int(rows),
                                      int(global_rows or rows), ptr(actions), ptr(advantages), ptr(old_logp), ptr(returns),
                                      ptr(adv_sums), 1 if normalize else 0, float(clip_range), float(ent_coef),
                                      float(vf_coef), ptr(grads), ptr(scratch), ptr(stats), ptr(logits), ptr(values),
                                      (1 if grads_zeroed else 0) | (2 if accumulate_stats else 0), _s()))
    return grads, stats


def a2c_batch(params, wpack, obs, obs_dim, n_actions, actions, advantages, returns, *, index=None, rows=None, global_rows=None,
              adv_sums=None, normalize=False, ent_coef=0.0, vf_coef=0.5, grads=None, scratch=None, stats=None, logits=None,
              values=None, grads_zeroed=False, accumulate_stats=False):
    """One A2C.train step's forward + loss + backward over the whole rollout, fused (tmla_a2c_batch_bf16): returns (grads, stats).
    Flags as ppo_minibatch."""
    _chk(params, torch.float32, "params"); _chk(wpack, torch.bfloat16, "wpack"); _chk(obs, torch.float32, "obs")
    _chk(index, torch.int32, "index"); _chk(actions, torch.int32, "actions"); _chk(advantages, torch.float32, "advantages")
    _chk(returns, torch.float32, "returns")
    if rows is None:
        rows = index.numel() if index is not None else obs.shape[0]
    dev = params.device
    if grads is None:
        grads = torch.empty_like(params)
    if scratch is None:
        scratch = torch.empty(lib.tmla_ppo_minibatch_scratch(HIDDEN, rows), dtype=torch.bfloat16, device=dev)
    if stats is None:
        stats = torch.empty(8, dtype=torch.float32, device=dev)
    _chk(scratch, torch.bfloat16, "scratch"); _chk(grads, torch.float32, "grads"); _chk(stats, torch.float32, "stats")
    _chk(logits, torch.float32, "logits"); _chk(values, torch.float32, "values")
    if normalize and adv_sums is None:
        adv_sums = adv_stats(advantages, index, rows)
    check(lib.tmla_a2c_batch_bf16(ptr(params), ptr(wpack), obs_dim, HIDDEN, n_actions, ptr(obs), ptr(index), int(rows),
                                  int(global_rows or rows), ptr(actions), ptr(advantages), ptr(returns), ptr(adv_sums),
                                  1 if normalize else 0, float(ent_coef), float(vf_coef), ptr(grads), ptr(scratch), ptr(stats),
                                  ptr(logits), ptr(values), (1 if grads_zeroed else 0) | (2 if accumulate_stats else 0), _s()))
    return grads, stats


def adam_clip(params, grads, m, v, step, *, grad_scale=1.0, max_grad_norm=0.5, lr=3e-4, beta1=0.9, beta2=0.999,
              eps=1e-5, norm_out=None, zero_grads=False, wpack=None, obs_dim=0, n_actions=0):
    """clip_grad_norm_ + Adam.step.  zero_grads: clear `grads` once consumed.  wpack (+ obs_dim, n_actions): also refresh the bf16
    operand images of the hidden-layer weights inside `wpack` (what the fused minibatch kernel reads)."""
    if norm_out is None:
        norm_out = torch.zeros(132, dtype=torch.float32, device=params.device)
    _chk(wpack, torch.bfloat16, "wpack")
    check(lib.tmla_adam_clip_fused(ptr(params), ptr(grads), ptr(m), ptr(v), params.numel(), float(grad_scale),
                                   float(max_grad_norm), float(lr), float(beta1), float(beta2), float(eps), int(step),
                                   ptr(norm_out), 1 if zero_grads else 0, ptr(wpack), int(obs_dim), HIDDEN, int(n_actions), _s()))
    return norm_out


def adam_clip_allreduce(comm, params, grads, m, v, step, *, grad_scale=1.0, max_grad_norm=0.5, lr=3e-4, beta1=0.9, beta2=0.999,
                        eps=1e-5, norm_out=None, zero_grads=False, wpack=None, obs_dim=0, n_actions=0):
    """grads <- sum over ranks (one-shot all-reduce over NVLink peer memory, rank order), then adam_clip — two launches, no NCCL."""
    if norm_out is None:
        norm_out = torch.zeros(132, dtype=torch.float32, device=params.device)
    _chk(wpack, torch.bfloat16, "wpack"); _chk(grads, torch.float32, "grads")
    check(lib.tmla_adam_clip_allreduce(comm.handle, ptr(params), ptr(grads), ptr(m), ptr(v), params.numel(), float(grad_scale),
                                       float(max_grad_norm), float(lr), float(beta1), float(beta2), float(eps), int(step),
                                       ptr(norm_out), 1 if zero_grads else 0, ptr(wpack), int(obs_dim), HIDDEN, int(n_actions), _s()))
    return norm_out


def rmsprop_clip(params, grads, sq_avg, *, grad_scale=1.0, max_grad_norm=0.5, lr=7e-4, alpha=0.99, eps=1e-5, norm_out=None,
                 zero_grads=False, wpack=None, obs_dim=0, n_actions=0):
    """clip_grad_norm_ + torch.optim.RMSprop.step in one launch (tmla_rmsprop_clip_fused); flags as adam_clip."""
    if norm_out is None:
        norm_out = torch.zeros(132, dtype=torch.float32, device=params.device)
    _chk(wpack, torch.bfloat16, "wpack"); _chk(grads, torch.float32, "grads"); _chk(sq_avg, torch.float32, "sq_avg")
    check(lib.tmla_rmsprop_clip_fused(ptr(params), ptr(grads), ptr(sq_avg), params.numel(), float(grad_scale), float(max_grad_norm),
                                      float(lr), float(alpha), float(eps), ptr(norm_out), 1 if zero_grads else 0, ptr(wpack),
                                      int(obs_dim), HIDDEN, int(n_actions), _s()))
    return norm_out


def rmsprop_clip_allreduce(comm, params, grads, sq_avg, step, *, grad_scale=1.0, max_grad_norm=0.5, lr=7e-4, alpha=0.99, eps=1e-5,
                           norm_out=None, zero_grads=False, wpack=None, obs_dim=0, n_actions=0):
    """grads <- sum over ranks over NVLink peer memory, then rmsprop_clip, in the same launch; `step` = exchange sequence number."""
    if norm_out is None:
        norm_out = torch.zeros(132, dtype=torch.float32, device=params.device)
    _chk(wpack, torch.bfloat16, "wpack"); _chk(grads, torch.float32, "grads"); _chk(sq_avg, torch.float32, "sq_avg")
    check(lib.tmla_rmsprop_clip_allreduce(comm.handle, ptr(params), ptr(grads), ptr(sq_avg), params.numel(), float(grad_scale),
                                          float(max_grad_norm), float(lr), float(alpha), float(eps), int(step), ptr(norm_out),
                                          1 if zero_grads else 0, ptr(wpack), int(obs_dim), HIDDEN, int(n_actions), _s()))
    return norm_out


def bootstrap_add(rew_buf, trunc_count, trunc_index, trunc_values, gamma: float):
    check(lib.tmla_bootstrap_add(ptr(rew_buf), ptr(trunc_count), ptr(trunc_index), ptr(trunc_values), float(gamma),
                                 int(trunc_index.numel()), _s()))


def step_policy(env, logits, row_index, obs_next, act, logp, rew, done, *, deterministic=False, trunc_count=None,
                trunc_index=None, trunc_obs=None, ep_stats=None, step_base=None):
    cap = 0 if trunc_index is None else int(trunc_index.numel())
    check(lib.tmla_step_policy(env.handle, ptr(logits), 1 if deterministic else 0, int(row_index), ptr(obs_next),
                               ptr(act), ptr(logp), ptr(rew), ptr(done), ptr(trunc_count), ptr(trunc_index),
                               ptr(trunc_obs), cap, ptr(ep_stats), ptr(step_base), _s()))
