"""Torch-tensor wrappers over the PPO and A2C entry points of libtmla.so (include/tmla.h).

Each function takes CUDA tensors, checks dtype/contiguity/device, and enqueues the kernel on
torch's current stream.  torch is plumbing here (memory + streams); the arithmetic is in csrc/.
"""
from __future__ import annotations

import torch

from . import native
from .native import lib, check, ptr

HIDDEN = 256          # default width; 64 and 128 run on the float32 kernels of csrc/mlp_small.cu (wpack=None only)


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


def num_params(obs_dim: int, n_actions: int, hidden: int = HIDDEN) -> int:
    n = lib.tmla_mlp_num_params(obs_dim, hidden, n_actions)
    if n < 0:
        raise ValueError(f"unsupported MLP shape (obs_dim {obs_dim}, hidden {hidden}, n_actions {n_actions}): hidden is 64, 128 or 256")
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
                want_logits=True, want_values=True, act_cache=None, wpack=None, keep_act=True, hidden=HIDDEN):
    """ActorCriticPolicy.forward.  wpack=None: float32 CUDA-core path; wpack=bf16 pack: tcgen05 path
    (act_cache is then bf16 [4,rows,256]).  hidden 64 / 128: float32 only; keep_act=False keeps no activations."""
    if wpack is not None and hidden != HIDDEN:
        raise ValueError(f"the bf16 tensor-core path covers hidden = {HIDDEN} only (got {hidden})")
    _chk(params, torch.float32, "params"); _chk(x, torch.float32, "x"); _chk(index, torch.int32, "index")
    if rows is None:
        rows = index.numel() if index is not None else x.shape[0]
    dev = params.device
    act_dtype = torch.float32 if wpack is None else torch.bfloat16
    if want_logits and logits is None:
        logits = torch.empty((rows, n_actions), dtype=torch.float32, device=dev)
    if want_values and values is None:
        values = torch.empty(rows, dtype=torch.float32, device=dev)
    if not keep_act and ((wpack is not None and obs_dim <= 6) or hidden != HIDDEN):
        act_cache = None            # fused tower kernel / small widths, inference only: no activation workspace
    elif act_cache is None:
        act_cache = torch.empty((4, rows, hidden), dtype=act_dtype, device=dev)
    _chk(act_cache, act_dtype, "act_cache")
    lg, vl = (ptr(logits) if want_logits else None), (ptr(values) if want_values else None)
    if wpack is None:
        check(lib.tmla_mlp_forward(ptr(params), obs_dim, hidden, n_actions, ptr(x), ptr(index), int(rows), ptr(rows_dev),
                                   lg, vl, ptr(act_cache), _s()))
    else:
        check(lib.tmla_mlp_forward_bf16(ptr(params), ptr(wpack), obs_dim, HIDDEN, n_actions, ptr(x), ptr(index), int(rows),
                                        ptr(rows_dev), lg, vl, ptr(act_cache), _s()))
    return logits, values, act_cache


def det_scratch_bytes(obs_dim: int, n_actions: int, rows: int, hidden: int = HIDDEN) -> int:
    """Bytes of the deterministic-mode partials (tmla_det_scratch_bytes) for calls of up to `rows` rows: the `partials` of
    mlp_backward / ppo_loss / a2c_loss, and what ppo_minibatch / a2c_batch(deterministic=True) add to their scratch."""
    n = lib.tmla_det_scratch_bytes(obs_dim, hidden, n_actions, int(rows))
    if n < 0:
        raise ValueError(native.last_error())
    return int(n)


def fused_scratch_elems(obs_dim: int, n_actions: int, rows: int, deterministic: bool = False) -> int:
    """bf16 elements of the scratch of ppo_minibatch / a2c_batch: the tile images, plus the partials when deterministic."""
    n = lib.tmla_ppo_minibatch_scratch(HIDDEN, int(rows))
    return n + ((det_scratch_bytes(obs_dim, n_actions, rows) + 1) // 2 if deterministic else 0)


def _partials(partials, name="partials"):
    if partials is not None and (not partials.is_cuda or not partials.is_contiguous()):
        raise ValueError(f"{name} must be a contiguous CUDA tensor")


def mlp_backward(params, x, obs_dim, n_actions, act_cache, dlogits, dvalues, *, index=None, rows=None, grads=None,
                 scratch=None, wpack=None, hidden=HIDDEN, partials=None):
    """Gradient of ActorCriticPolicy.forward (flat, overwritten).  hidden 64 / 128: scratch holds per-chunk partial gradients,
    summed in a fixed order (bit-identical across calls).  partials (bf16 path, det_scratch_bytes bytes): the deterministic
    form, tmla_mlp_backward_bf16_det."""
    if wpack is not None and hidden != HIDDEN:
        raise ValueError(f"the bf16 tensor-core path covers hidden = {HIDDEN} only (got {hidden})")
    if rows is None:
        rows = index.numel() if index is not None else x.shape[0]
    dev = params.device
    act_dtype = torch.float32 if wpack is None else torch.bfloat16
    if grads is None:
        grads = torch.empty_like(params)
    if scratch is None:
        size = lib.tmla_mlp_backward_scratch(obs_dim, hidden, n_actions, rows)
        if size < 0:
            raise ValueError(native.last_error())
        scratch = torch.empty(size, dtype=act_dtype, device=dev)
    _chk(dlogits, torch.float32, "dlogits"); _chk(dvalues, torch.float32, "dvalues")
    _chk(act_cache, act_dtype, "act_cache"); _chk(scratch, act_dtype, "scratch")
    _partials(partials)
    if wpack is None:
        check(lib.tmla_mlp_backward(ptr(params), obs_dim, hidden, n_actions, ptr(x), ptr(index), int(rows), ptr(act_cache),
                                    ptr(dlogits), ptr(dvalues), ptr(grads), ptr(scratch), _s()))
    elif partials is not None:
        check(lib.tmla_mlp_backward_bf16_det(ptr(params), ptr(wpack), obs_dim, HIDDEN, n_actions, ptr(x), ptr(index), int(rows),
                                             ptr(act_cache), ptr(dlogits), ptr(dvalues), ptr(grads), ptr(scratch), ptr(partials), _s()))
    else:
        check(lib.tmla_mlp_backward_bf16(ptr(params), ptr(wpack), obs_dim, HIDDEN, n_actions, ptr(x), ptr(index), int(rows),
                                         ptr(act_cache), ptr(dlogits), ptr(dvalues), ptr(grads), ptr(scratch), _s()))
    return grads


def adv_stats(advantages, index, rows, sums=None):
    if sums is None:
        sums = torch.empty(3, dtype=torch.float64, device=advantages.device)
    check(lib.tmla_adv_stats(ptr(advantages), ptr(index), int(rows), ptr(sums), _s()))
    return sums


def adv_stats_batched(advantages, index, total, mb_rows, sums=None, partials=None):
    """(sum, sum of squares, count) of the advantages of every minibatch of an epoch: double[n_mb, 3].  partials
    (adv_det_scratch_bytes bytes): the deterministic form, per-block sums added in block order."""
    n_mb = (total + mb_rows - 1) // mb_rows
    if sums is None:
        sums = torch.empty((n_mb, 3), dtype=torch.float64, device=advantages.device)
    _chk(sums, torch.float64, "sums")
    _partials(partials)
    if partials is not None:
        check(lib.tmla_adv_stats_batched_det(ptr(advantages), ptr(index), int(total), int(mb_rows), ptr(sums), ptr(partials), _s()))
    else:
        check(lib.tmla_adv_stats_batched(ptr(advantages), ptr(index), int(total), int(mb_rows), ptr(sums), _s()))
    return sums


def adv_det_scratch_bytes(total: int, mb_rows: int) -> int:
    n = lib.tmla_adv_stats_det_scratch_bytes(int(total), int(mb_rows))
    if n < 0:
        raise ValueError(native.last_error())
    return int(n)


def ppo_loss(logits, values, actions, advantages, old_logp, returns, *, index=None, rows=None, global_rows=None,
             adv_sums=None, normalize=True, clip_range=0.2, ent_coef=0.01, vf_coef=0.5, dlogits=None, dvalues=None,
             stats=None, partials=None):
    """PPO's loss head (tmla_ppo_loss); partials (det_scratch_bytes bytes): statistics summed in block order (tmla_ppo_loss_det)."""
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
    _partials(partials)
    args = (ptr(logits), ptr(values), ptr(actions), ptr(advantages), ptr(old_logp), ptr(returns), ptr(index), int(rows),
            int(global_rows or rows), int(n_actions), ptr(adv_sums), 1 if normalize else 0, float(clip_range), float(ent_coef),
            float(vf_coef), ptr(dlogits), ptr(dvalues), ptr(stats))
    if partials is not None:
        check(lib.tmla_ppo_loss_det(*args, ptr(partials), _s()))
    else:
        check(lib.tmla_ppo_loss(*args, _s()))
    return dlogits, dvalues, stats


def a2c_loss(logits, values, actions, advantages, returns, *, index=None, rows=None, global_rows=None, adv_sums=None,
             normalize=False, ent_coef=0.0, vf_coef=0.5, dlogits=None, dvalues=None, stats=None, partials=None):
    """A2C.train's loss head (tmla_a2c_loss): ppo_loss without old_logp and clip_range; normalisation off by default (SB3's A2C).
    partials: as ppo_loss (tmla_a2c_loss_det)."""
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
    _partials(partials)
    args = (ptr(logits), ptr(values), ptr(actions), ptr(advantages), ptr(returns), ptr(index), int(rows), int(global_rows or rows),
            int(n_actions), ptr(adv_sums), 1 if normalize else 0, float(ent_coef), float(vf_coef), ptr(dlogits), ptr(dvalues), ptr(stats))
    if partials is not None:
        check(lib.tmla_a2c_loss_det(*args, ptr(partials), _s()))
    else:
        check(lib.tmla_a2c_loss(*args, _s()))
    return dlogits, dvalues, stats


TMLA_MB_GRADS_ZEROED, TMLA_MB_ACCUMULATE_STATS, TMLA_MB_DETERMINISTIC = 1, 2, 4      # include/tmla.h


def _mb_flags(grads_zeroed: bool, accumulate_stats: bool, deterministic: bool) -> int:
    return ((TMLA_MB_GRADS_ZEROED if grads_zeroed else 0) | (TMLA_MB_ACCUMULATE_STATS if accumulate_stats else 0)
            | (TMLA_MB_DETERMINISTIC if deterministic else 0))


def ppo_minibatch_supported(obs_dim: int, n_actions: int, hidden: int = HIDDEN) -> bool:
    return bool(lib.tmla_ppo_minibatch_supported(obs_dim, hidden, n_actions))


def ppo_minibatch(params, wpack, obs, obs_dim, n_actions, actions, advantages, old_logp, returns, *, index=None, rows=None,
                  global_rows=None, adv_sums=None, normalize=True, clip_range=0.2, ent_coef=0.01, vf_coef=0.5, grads=None,
                  scratch=None, stats=None, logits=None, values=None, grads_zeroed=False, accumulate_stats=False, deterministic=False):
    """One PPO.train minibatch, forward + loss + backward fused (tmla_ppo_minibatch_bf16): returns (grads, stats).
    grads_zeroed: `grads` is known to be all zeros (adam_clip(zero_grads=True) left it so) — skips the memset launch;
    accumulate_stats: add to `stats` instead of overwriting it; deterministic: TMLA_MB_DETERMINISTIC (bit-reproducible sums,
    scratch of fused_scratch_elems(..., deterministic=True))."""
    _chk(params, torch.float32, "params"); _chk(wpack, torch.bfloat16, "wpack"); _chk(obs, torch.float32, "obs")
    _chk(index, torch.int32, "index"); _chk(actions, torch.int32, "actions"); _chk(advantages, torch.float32, "advantages")
    _chk(old_logp, torch.float32, "old_logp"); _chk(returns, torch.float32, "returns")
    if rows is None:
        rows = index.numel() if index is not None else obs.shape[0]
    dev = params.device
    if grads is None:
        grads = torch.empty_like(params)
    if scratch is None:
        scratch = torch.empty(fused_scratch_elems(obs_dim, n_actions, rows, deterministic), dtype=torch.bfloat16, device=dev)
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
                                      _mb_flags(grads_zeroed, accumulate_stats, deterministic), _s()))
    return grads, stats


def a2c_batch(params, wpack, obs, obs_dim, n_actions, actions, advantages, returns, *, index=None, rows=None, global_rows=None,
              adv_sums=None, normalize=False, ent_coef=0.0, vf_coef=0.5, grads=None, scratch=None, stats=None, logits=None,
              values=None, grads_zeroed=False, accumulate_stats=False, deterministic=False):
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
        scratch = torch.empty(fused_scratch_elems(obs_dim, n_actions, rows, deterministic), dtype=torch.bfloat16, device=dev)
    if stats is None:
        stats = torch.empty(8, dtype=torch.float32, device=dev)
    _chk(scratch, torch.bfloat16, "scratch"); _chk(grads, torch.float32, "grads"); _chk(stats, torch.float32, "stats")
    _chk(logits, torch.float32, "logits"); _chk(values, torch.float32, "values")
    if normalize and adv_sums is None:
        adv_sums = adv_stats(advantages, index, rows)
    check(lib.tmla_a2c_batch_bf16(ptr(params), ptr(wpack), obs_dim, HIDDEN, n_actions, ptr(obs), ptr(index), int(rows),
                                  int(global_rows or rows), ptr(actions), ptr(advantages), ptr(returns), ptr(adv_sums),
                                  1 if normalize else 0, float(ent_coef), float(vf_coef), ptr(grads), ptr(scratch), ptr(stats),
                                  ptr(logits), ptr(values), _mb_flags(grads_zeroed, accumulate_stats, deterministic), _s()))
    return grads, stats


def adam_clip(params, grads, m, v, step, *, grad_scale=1.0, max_grad_norm=0.5, lr=3e-4, beta1=0.9, beta2=0.999,
              eps=1e-5, norm_out=None, zero_grads=False, wpack=None, obs_dim=0, n_actions=0, hidden=HIDDEN):
    """clip_grad_norm_ + Adam.step.  zero_grads: clear `grads` once consumed.  wpack (+ obs_dim, n_actions): also refresh the bf16
    operand images of the hidden-layer weights inside `wpack` (what the fused minibatch kernel reads)."""
    if norm_out is None:
        norm_out = torch.zeros(132, dtype=torch.float32, device=params.device)
    _chk(wpack, torch.bfloat16, "wpack")
    check(lib.tmla_adam_clip_fused(ptr(params), ptr(grads), ptr(m), ptr(v), params.numel(), float(grad_scale),
                                   float(max_grad_norm), float(lr), float(beta1), float(beta2), float(eps), int(step),
                                   ptr(norm_out), 1 if zero_grads else 0, ptr(wpack), int(obs_dim), int(hidden), int(n_actions), _s()))
    return norm_out


def adam_clip_allreduce(comm, params, grads, m, v, step, *, grad_scale=1.0, max_grad_norm=0.5, lr=3e-4, beta1=0.9, beta2=0.999,
                        eps=1e-5, norm_out=None, zero_grads=False, wpack=None, obs_dim=0, n_actions=0, hidden=HIDDEN):
    """grads <- sum over ranks (one-shot all-reduce over NVLink peer memory, rank order), then adam_clip — two launches, no NCCL."""
    if norm_out is None:
        norm_out = torch.zeros(132, dtype=torch.float32, device=params.device)
    _chk(wpack, torch.bfloat16, "wpack"); _chk(grads, torch.float32, "grads")
    check(lib.tmla_adam_clip_allreduce(comm.handle, ptr(params), ptr(grads), ptr(m), ptr(v), params.numel(), float(grad_scale),
                                       float(max_grad_norm), float(lr), float(beta1), float(beta2), float(eps), int(step),
                                       ptr(norm_out), 1 if zero_grads else 0, ptr(wpack), int(obs_dim), int(hidden), int(n_actions), _s()))
    return norm_out


def rmsprop_clip(params, grads, sq_avg, *, grad_scale=1.0, max_grad_norm=0.5, lr=7e-4, alpha=0.99, eps=1e-5, norm_out=None,
                 zero_grads=False, wpack=None, obs_dim=0, n_actions=0, hidden=HIDDEN):
    """clip_grad_norm_ + torch.optim.RMSprop.step in one launch (tmla_rmsprop_clip_fused); flags as adam_clip."""
    if norm_out is None:
        norm_out = torch.zeros(132, dtype=torch.float32, device=params.device)
    _chk(wpack, torch.bfloat16, "wpack"); _chk(grads, torch.float32, "grads"); _chk(sq_avg, torch.float32, "sq_avg")
    check(lib.tmla_rmsprop_clip_fused(ptr(params), ptr(grads), ptr(sq_avg), params.numel(), float(grad_scale), float(max_grad_norm),
                                      float(lr), float(alpha), float(eps), ptr(norm_out), 1 if zero_grads else 0, ptr(wpack),
                                      int(obs_dim), int(hidden), int(n_actions), _s()))
    return norm_out


def rmsprop_clip_allreduce(comm, params, grads, sq_avg, step, *, grad_scale=1.0, max_grad_norm=0.5, lr=7e-4, alpha=0.99, eps=1e-5,
                           norm_out=None, zero_grads=False, wpack=None, obs_dim=0, n_actions=0, hidden=HIDDEN):
    """grads <- sum over ranks over NVLink peer memory, then rmsprop_clip, in the same launch; `step` = exchange sequence number."""
    if norm_out is None:
        norm_out = torch.zeros(132, dtype=torch.float32, device=params.device)
    _chk(wpack, torch.bfloat16, "wpack"); _chk(grads, torch.float32, "grads"); _chk(sq_avg, torch.float32, "sq_avg")
    check(lib.tmla_rmsprop_clip_allreduce(comm.handle, ptr(params), ptr(grads), ptr(sq_avg), params.numel(), float(grad_scale),
                                          float(max_grad_norm), float(lr), float(alpha), float(eps), int(step), ptr(norm_out),
                                          1 if zero_grads else 0, ptr(wpack), int(obs_dim), int(hidden), int(n_actions), _s()))
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
