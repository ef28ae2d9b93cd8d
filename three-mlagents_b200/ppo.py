"""CudaPPO — SB3-compatible PPO front-end whose rollout, GAE and update all run in libtmla.so.

Mirrors what the reference builds at backend/mlagents/training.py:150 (`PPO("MlpPolicy", vec_env,
seed=seed, **kwargs)`) and drives at training.py:166-175 (`learn`, `save`), plus `predict`/`load`
(training.py:269,278).  Algorithm = SB3 2.9.0 OnPolicyAlgorithm.collect_rollouts + RolloutBuffer +
PPO.train (SURVEY.md Appendix A), with these documented differences:
  * all N envs advance in one kernel per step, sampling uses per-env Philox streams (not torch's
    global generator), minibatch order is a keyed Feistel permutation (not np.random.permutation);
  * callbacks fire per rollout, not per env step (SURVEY.md §7 "per-step host hooks");
  * with world_size > 1, env shards are per rank, gradients are all-reduced (NCCL) once per
    minibatch and advantage normalisation uses global-minibatch statistics.
"""
from __future__ import annotations

import io
import json
import math
import time
import zipfile
from typing import Any

import numpy as np
import torch
from torch.cuda import nvtx      # NVTX ranges rollout / gae / update / allreduce (SURVEY.md §5; visible in nsys / ncu --nvtx)

from . import native, ops
from .native import ptr
from .distributed import PeerComm, allreduce_sum_, dist_state
from .vec_env import CudaVecEnv

HIDDEN = 256


_dist = dist_state


def _on_device(fn):
    """Run a CudaPPO method with the model's GPU as the current CUDA device: the C entry points enqueue on torch's current
    stream, which is per device — without this a model on cuda:1 called from a thread whose current device is cuda:0 would
    launch on the wrong GPU."""
    import functools

    @functools.wraps(fn)
    def wrapped(self, *args, **kwargs):
        with torch.cuda.device(self.device):
            return fn(self, *args, **kwargs)

    return wrapped


def orthogonal_init(obs_dim: int, n_actions: int, seed: int) -> torch.Tensor:
    """SB3 ActorCriticPolicy init: orthogonal weights with gain sqrt(2) (towers), 0.01 (action_net),
    1.0 (value_net), zero biases; flat vector in policy.parameters() order (include/tmla.h)."""
    g = torch.Generator().manual_seed(int(seed))
    shapes = []
    for _tower in range(2):
        shapes += [((HIDDEN, obs_dim), math.sqrt(2.0)), ((HIDDEN,), None), ((HIDDEN, HIDDEN), math.sqrt(2.0)), ((HIDDEN,), None)]
    shapes += [((n_actions, HIDDEN), 0.01), ((n_actions,), None), ((1, HIDDEN), 1.0), ((1,), None)]
    chunks = []
    for shape, gain in shapes:
        t = torch.zeros(shape, dtype=torch.float32)
        if gain is not None:
            torch.nn.init.orthogonal_(t, gain=gain, generator=g)
        chunks.append(t.reshape(-1))
    return torch.cat(chunks)


class CudaPPO:
    algorithm = "ppo"
    _log_interval = 1                 # learn(): verbose rows every this many iterations
    _row_every_iteration = True       # learn(): a logger / progress.jsonl row after every iteration (A2C: every log_interval)
    _HYPER_KEYS = ("learning_rate", "n_steps", "batch_size", "n_epochs", "gamma", "gae_lambda", "clip_range", "ent_coef", "vf_coef",
                   "max_grad_norm")

    def __init__(self, policy: str, env: CudaVecEnv, *, seed: int = 1, learning_rate: float = 3e-4, n_steps: int = 2048,
                 batch_size: int = 64, n_epochs: int = 10, gamma: float = 0.99, gae_lambda: float = 0.95,
                 clip_range: float = 0.2, ent_coef: float = 0.0, vf_coef: float = 0.5, max_grad_norm: float = 0.5,
                 normalize_advantage: bool = True, policy_kwargs: dict | None = None, tensorboard_log: str | None = None,
                 verbose: int = 0, mlp_impl: str = "auto", fused_update: bool = True, rollout_impl: str = "fused",
                 _params: torch.Tensor | None = None):
        if policy != "MlpPolicy":
            raise ValueError("CudaPPO supports 'MlpPolicy' (vector observations) only")
        arch = (policy_kwargs or {}).get("net_arch", {"pi": [256, 256], "vf": [256, 256]})
        if arch != {"pi": [256, 256], "vf": [256, 256]}:
            raise ValueError("CudaPPO implements net_arch dict(pi=[256,256], vf=[256,256]) (training.py:363-365)")
        self.env = env
        self.seed = int(seed)
        self.lr, self.n_steps, self.batch_size, self.n_epochs = float(learning_rate), int(n_steps), int(batch_size), int(n_epochs)
        self.gamma, self.gae_lambda, self.clip_range = float(gamma), float(gae_lambda), float(clip_range)
        self.ent_coef, self.vf_coef, self.max_grad_norm = float(ent_coef), float(vf_coef), float(max_grad_norm)
        self.normalize_advantage = bool(normalize_advantage)
        self.verbose, self.tensorboard_log = int(verbose), tensorboard_log
        if mlp_impl not in ("auto", "bf16", "fp32"):
            raise ValueError("mlp_impl must be 'auto', 'bf16' (tcgen05 tensor cores) or 'fp32' (CUDA cores)")
        self.mlp_impl = "bf16" if mlp_impl == "auto" else mlp_impl
        self.obs_dim, self.n_actions, self.n_envs = env.obs_dim, env.n_actions, env.num_envs
        # one fused forward+loss+backward kernel per tower and minibatch (csrc/mlp_train.cu) where the shape allows
        self.fused_update = bool(fused_update) and self.mlp_impl == "bf16" and ops.ppo_minibatch_supported(self.obs_dim, self.n_actions)
        self.device = torch.device("cuda", env.device_index)
        self.num_timesteps = 0
        self.n_updates = 0
        self._iterations = 0
        self._adam_step = 0
        self._epoch_counter = 0
        self._dist, self.rank, self.world = _dist()
        with torch.cuda.device(self.device):
            p = orthogonal_init(self.obs_dim, self.n_actions, self.seed) if _params is None else _params.detach().float().cpu()
            assert p.numel() == ops.num_params(self.obs_dim, self.n_actions)
            self.params = p.to(self.device).contiguous()
            self.m = torch.zeros_like(self.params)
            self.v = torch.zeros_like(self.params)
            self.grads = torch.zeros_like(self.params)
            self.wpack = None
            self._repack()
        self._buffers_ready = False
        self._last_obs_valid = False
        self._rollout_args = None
        # the gradient all-reduce: fused into clip + Adam over NVLink peer memory when every rank can map its peers, else NCCL
        self._comm = PeerComm.create(env.device_index, self.params.numel()) if self.world > 1 else None
        self.allreduce_impl = "none" if self.world == 1 else ("peer-memory one-shot, fused with clip+Adam (csrc/comm.cu)" if self._comm else "nccl")
        if rollout_impl not in ("fused", "steps"):
            raise ValueError("rollout_impl must be 'fused' (tmla_rollout: one call per rollout) or 'steps' (one call per step)")
        self.rollout_impl = rollout_impl
        self.logger_rows: list[dict[str, Any]] = []

    def _repack(self):
        """bf16 copies of the hidden-layer weights for the tensor-core path (after every optimizer step)."""
        if self.mlp_impl == "bf16":
            self.wpack = ops.mlp_pack(self.params, self.obs_dim, self.n_actions, self.wpack)

    @property
    def _act_dtype(self):
        return torch.bfloat16 if self.mlp_impl == "bf16" else torch.float32

    # ------------------------------------------------------------------------------------- buffers
    def _alloc(self):
        if self._buffers_ready:
            return
        T, N, D, A, dev = self.n_steps, self.n_envs, self.obs_dim, self.n_actions, self.device
        f32 = dict(dtype=torch.float32, device=dev)
        self.obs = torch.empty((T + 1, N, D), **f32)
        self.act = torch.empty((T, N), dtype=torch.int32, device=dev)
        self.logp = torch.empty((T, N), **f32)
        self.rew = torch.empty((T, N), **f32)
        self.val = torch.empty((T, N), **f32)
        self.step_counter = torch.zeros(1, dtype=torch.int64, device=dev)
        self.adv = torch.empty((T, N), **f32)
        self.ret = torch.empty((T, N), **f32)
        self.done = torch.empty((T, N), dtype=torch.uint8, device=dev)
        self.last_values = torch.empty(N, **f32)
        self.logits_roll = torch.empty((N, A), **f32)
        self.cache_roll = torch.empty((4, N, HIDDEN), dtype=self._act_dtype, device=dev)
        # every env can hit its time limit at most floor(T/limit)+1 times per rollout
        cap = N * (T // self.env.max_episode_steps + 1)
        self.trunc_count = torch.zeros(1, dtype=torch.int32, device=dev)
        self.trunc_index = torch.zeros(cap, dtype=torch.int32, device=dev)
        self.trunc_obs = torch.zeros((cap, D), **f32)
        self.trunc_values = torch.zeros(cap, **f32)
        self.cache_trunc = torch.empty((4, cap, HIDDEN), dtype=self._act_dtype, device=dev) if cap != N else self.cache_roll
        self.ep_stats = torch.zeros(4, **f32)
        total = T * N
        B = min(self.batch_size, total)
        self.mb_rows = B
        self.perm = torch.empty(total, dtype=torch.int32, device=dev)
        if not self.fused_update:
            self.logits_mb = torch.empty((B, A), **f32)
            self.values_mb = torch.empty(B, **f32)
            self.dlogits = torch.empty((B, A), **f32)
            self.dvalues = torch.empty(B, **f32)
            self.cache_mb = torch.empty((4, B, HIDDEN), dtype=self._act_dtype, device=dev)
        n_img = 4 if self.fused_update else 2          # fused: H1 and dZ2 tile images of both towers
        self.scratch_mb = torch.empty(n_img * ((B + 127) // 128 * 128) * HIDDEN, dtype=self._act_dtype, device=dev)
        self.adv_sums = torch.zeros(((total + B - 1) // B, 3), dtype=torch.float64, device=dev)   # one row per minibatch of an epoch
        self.stats = torch.zeros(8, **f32)
        self.stats_acc = torch.zeros(8, **f32)
        self.norm_out = torch.zeros(132, **f32)      # TMLA_ADAM_SCRATCH: norm, 128 partials, grid-barrier words (zeroed once)
        if getattr(self.env, "_monitor", None) is not None and self.env._ep_log is None:
            self.env.attach_episode_log(N * T)          # Monitor rows for the device path (flushed after every rollout)
        self._buffers_ready = True

    # ------------------------------------------------------------------------------------- rollout
    @_on_device
    def collect_rollouts(self):
        """OnPolicyAlgorithm.collect_rollouts + compute_returns_and_advantage, no host round-trip per step."""
        self._alloc()
        nvtx.range_push("rollout")
        T, N, D, A = self.n_steps, self.n_envs, self.obs_dim, self.n_actions
        if not self._last_obs_valid:
            self.obs[0].copy_(self.env.reset_tensor())
            self._last_obs_valid = True
        else:
            self.obs[0].copy_(self.obs[T])
        if self.rollout_impl == "fused":
            # ONE call: T x {tower forward, sample + env step}, last-value and timeout-bootstrap forwards, GAE — a CUDA graph
            # recorded once per buffer set inside libtmla.so and replayed here (include/tmla.h tmla_rollout)
            if self._rollout_args is None:
                keep = self.cache_trunc if self.cache_trunc.numel() >= self.cache_roll.numel() else self.cache_roll
                need_cache = not (self.mlp_impl == "bf16" and D <= 6)
                self._rollout_args = native.RolloutArgs(
                    params=ptr(self.params), wpack=ptr(self.wpack), act_cache=ptr(keep) if need_cache else None,
                    obs=ptr(self.obs), actions=ptr(self.act), log_probs=ptr(self.logp), rewards=ptr(self.rew), values=ptr(self.val),
                    dones=ptr(self.done), last_values=ptr(self.last_values), advantages=ptr(self.adv), returns=ptr(self.ret),
                    logits=ptr(self.logits_roll), trunc_count=ptr(self.trunc_count), trunc_index=ptr(self.trunc_index),
                    trunc_obs=ptr(self.trunc_obs), trunc_values=ptr(self.trunc_values), ep_stats=ptr(self.ep_stats),
                    step_counter=ptr(self.step_counter), gamma=self.gamma, gae_lambda=self.gae_lambda, obs_dim=D, hidden=HIDDEN,
                    n_actions=A, n_steps=T, deterministic=0, trunc_capacity=self.trunc_index.numel())
            native.check(native.lib.tmla_rollout(self.env.handle, self._rollout_args, native.current_stream()))
            nvtx.range_pop()
            self.num_timesteps += T * N * self.world
            return
        self.trunc_count.zero_()
        self.ep_stats.zero_()
        for t in range(T):
            ops.mlp_forward(self.params, self.obs[t], D, A, rows=N, logits=self.logits_roll, values=self.val[t],
                            act_cache=self.cache_roll, wpack=self.wpack, keep_act=False)
            ops.step_policy(self.env, self.logits_roll, t, self.obs[t + 1], self.act[t], self.logp[t], self.rew[t],
                            self.done[t], trunc_count=self.trunc_count, trunc_index=self.trunc_index,
                            trunc_obs=self.trunc_obs, ep_stats=self.ep_stats)
        ops.mlp_forward(self.params, self.obs[T], D, A, rows=N, want_logits=False, values=self.last_values,
                        act_cache=self.cache_roll, wpack=self.wpack, keep_act=False)
        # timeout bootstrap: rewards += gamma * V(terminal_obs) for time-limit truncations
        cap = self.trunc_index.numel()
        ops.mlp_forward(self.params, self.trunc_obs, D, A, rows=cap, rows_dev=self.trunc_count, want_logits=False,
                        values=self.trunc_values, act_cache=self.cache_trunc, wpack=self.wpack, keep_act=False)
        ops.bootstrap_add(self.rew, self.trunc_count, self.trunc_index, self.trunc_values, self.gamma)
        nvtx.range_pop()
        nvtx.range_push("gae")
        ops.gae(self.rew, self.val, self.done, self.last_values, self.gamma, self.gae_lambda, self.adv, self.ret)
        nvtx.range_pop()
        self.num_timesteps += T * N * self.world

    # -------------------------------------------------------------------------------------- update
    @_on_device
    def train(self):
        """PPO.train: n_epochs passes over the rollout in minibatches of batch_size."""
        T, N, D, A = self.n_steps, self.n_envs, self.obs_dim, self.n_actions
        total = T * N
        B = self.mb_rows
        obs_flat = self.obs[:T].reshape(total, D)
        nvtx.range_push("update")
        self.stats_acc.zero_()
        fused = self.fused_update
        if fused:              # no per-minibatch memsets: Adam clears the gradient it consumed, statistics accumulate in place
            self.grads.zero_()
        n_mb = 0
        for _ in range(self.n_epochs):
            ops.permutation(self.seed + 7919 * self.rank, self._epoch_counter, T, N, out=self.perm)
            self._epoch_counter += 1
            if self.normalize_advantage:                  # advantage statistics of all minibatches: one launch, one all-reduce
                ops.adv_stats_batched(self.adv, self.perm, total, B, self.adv_sums)
                allreduce_sum_(self.adv_sums)
            for mb, start in enumerate(range(0, total, B)):
                rows = min(B, total - start)
                idx = self.perm[start:start + rows]
                sums = self.adv_sums[mb] if self.normalize_advantage and rows * self.world > 1 else None
                if self.fused_update:
                    ops.ppo_minibatch(self.params, self.wpack, obs_flat, D, A, self.act, self.adv, self.logp, self.ret,
                                      index=idx, rows=rows, global_rows=rows * self.world, adv_sums=sums,
                                      normalize=sums is not None, clip_range=self.clip_range, ent_coef=self.ent_coef,
                                      vf_coef=self.vf_coef, grads=self.grads, scratch=self.scratch_mb, stats=self.stats_acc,
                                      grads_zeroed=True, accumulate_stats=True)
                else:
                    ops.mlp_forward(self.params, obs_flat, D, A, index=idx, rows=rows, logits=self.logits_mb,
                                    values=self.values_mb, act_cache=self.cache_mb, wpack=self.wpack)
                    ops.ppo_loss(self.logits_mb, self.values_mb, self.act, self.adv, self.logp, self.ret, index=idx,
                                 rows=rows, global_rows=rows * self.world, adv_sums=sums, normalize=sums is not None,
                                 clip_range=self.clip_range, ent_coef=self.ent_coef, vf_coef=self.vf_coef,
                                 dlogits=self.dlogits, dvalues=self.dvalues, stats=self.stats)
                    ops.mlp_backward(self.params, obs_flat, D, A, self.cache_mb, self.dlogits, self.dvalues, index=idx,
                                     rows=rows, grads=self.grads, scratch=self.scratch_mb, wpack=self.wpack)
                self._adam_step += 1
                if self._comm is not None:                # the one collective on the path, inside the optimizer launches
                    nvtx.range_push("allreduce+adam")
                    ops.adam_clip_allreduce(self._comm, self.params, self.grads, self.m, self.v, self._adam_step,
                                            max_grad_norm=self.max_grad_norm, lr=self.lr, eps=1e-5, norm_out=self.norm_out,
                                            zero_grads=fused, wpack=self.wpack if fused else None, obs_dim=D, n_actions=A)
                    nvtx.range_pop()
                else:
                    if self.world > 1:
                        nvtx.range_push("allreduce")
                        self._allreduce_grads(self.grads) # NCCL sum over NVLink
                        nvtx.range_pop()
                    ops.adam_clip(self.params, self.grads, self.m, self.v, self._adam_step, max_grad_norm=self.max_grad_norm,
                                  lr=self.lr, eps=1e-5, norm_out=self.norm_out, zero_grads=fused,
                                  wpack=self.wpack if fused else None, obs_dim=D, n_actions=A)
                if not fused:          # (fused: Adam refreshed the operand images itself; full repack once after the loop)
                    self._repack()
                    self.stats_acc += self.stats
                n_mb += 1
            self.n_updates += 1
        if fused:
            self._repack()
        if self._comm is not None:
            self._comm.check()                            # a rank that never showed up (bounded waits) surfaces here
        nvtx.range_pop()
        return n_mb

    def _allreduce_grads(self, grads: torch.Tensor) -> None:
        allreduce_sum_(grads)

    def close(self) -> None:
        """Release the peer-memory gradient exchange (collective-free; safe to call more than once)."""
        if getattr(self, "_comm", None) is not None:
            self._comm.close()
            self._comm = None

    def __del__(self):  # best effort
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass

    def _log_row(self, n_mb: int, t_roll: float, t_train: float, t0: float) -> dict[str, Any]:
        s = (self.stats_acc / max(n_mb, 1)).cpu().numpy()
        if self.world > 1:
            st = torch.from_numpy(s.copy()).to(self.device)
            self._dist.all_reduce(st)
            s = st.cpu().numpy()
        ep = self.ep_stats.clone()
        if self.world > 1:
            self._dist.all_reduce(ep)
        ep = ep.cpu().numpy()
        var_y = float(self.ret.var())
        ev = float("nan") if var_y == 0 else 1.0 - float((self.ret - self.val).var()) / var_y
        row = {
            "time/total_timesteps": self.num_timesteps, "time/iterations": self._iterations,
            "time/time_elapsed": time.time() - t0,
            "time/fps": self.n_steps * self.n_envs * self.world / max(t_roll + t_train, 1e-9),
            "time/rollout_s": t_roll, "time/train_s": t_train,
            "rollout/ep_rew_mean": float(ep[0] / ep[2]) if ep[2] > 0 else float("nan"),
            "rollout/ep_len_mean": float(ep[1] / ep[2]) if ep[2] > 0 else float("nan"),
            "rollout/episodes": int(ep[2]),
            "train/policy_gradient_loss": float(s[0]), "train/value_loss": float(s[1]), "train/entropy_loss": float(s[2]),
            "train/approx_kl": float(s[3]), "train/clip_fraction": float(s[4]), "train/loss": float(s[5]),
            "train/explained_variance": ev, "train/learning_rate": self.lr, "train/clip_range": self.clip_range,
            "train/n_updates": self.n_updates,
        }
        return row

    @_on_device
    def learn(self, total_timesteps: int, callback=None, progress_bar: bool = False, log_interval: int | None = None):
        log_interval = max(1, int(log_interval or self._log_interval))
        t0 = time.time()
        target = self.num_timesteps + int(total_timesteps)
        it = 0
        while self.num_timesteps < target:
            ts = time.time()
            self.collect_rollouts()
            torch.cuda.synchronize(self.device)
            if getattr(self.env, "_monitor", None) is not None:
                self.env.flush_episode_log()             # Monitor rows of the episodes that ended in this rollout
            tr = time.time()
            n_mb = self.train()
            torch.cuda.synchronize(self.device)
            te = time.time()
            it += 1
            self._iterations += 1
            if self._row_every_iteration or it % log_interval == 0 or self.num_timesteps >= target:
                row = self._log_row(n_mb, tr - ts, te - tr, t0)
                self.logger_rows.append(row)
                if self.verbose and self.rank == 0 and it % log_interval == 0:
                    print(json.dumps({k: (round(v, 5) if isinstance(v, float) else v) for k, v in row.items()}), flush=True)
                if self.tensorboard_log and self.rank == 0:
                    import os

                    os.makedirs(self.tensorboard_log, exist_ok=True)
                    with open(os.path.join(self.tensorboard_log, "progress.jsonl"), "a", encoding="utf-8") as f:
                        f.write(json.dumps(row) + "\n")
            if callback is not None:
                keep = callback(self) if callable(callback) else callback.on_rollout(self)
                if keep is False:
                    break
        return self

    # ------------------------------------------------------------------------- predict / evaluate
    @_on_device
    def policy_logits(self, obs_dev: torch.Tensor) -> torch.Tensor:
        rows = obs_dev.shape[0]
        logits, _, _ = ops.mlp_forward(self.params, obs_dev.contiguous(), self.obs_dim, self.n_actions, rows=rows,
                                       want_values=False, wpack=self.wpack, keep_act=False)
        return logits

    @_on_device
    def predict(self, observation, state=None, episode_start=None, deterministic: bool = False):
        obs = np.asarray(observation, dtype=np.float32)
        single = obs.ndim == 1
        x = torch.from_numpy(obs.reshape(-1, self.obs_dim)).to(self.device)
        logits = self.policy_logits(x)
        if deterministic:
            a = torch.argmax(logits, dim=1)
        else:
            a = torch.distributions.Categorical(logits=logits).sample()
        a = a.cpu().numpy().astype(np.int64)
        return (a[0] if single else a), state

    def evaluate(self, n_episodes: int, seed: int, deterministic: bool = True):
        """evaluate_policy equivalent, batched on the device: `n_episodes` envs run one episode each."""
        env = CudaVecEnv(self.env.task_id, n_episodes, seed=seed, device=self.env.device_index)
        try:
            with torch.cuda.device(self.device):
                obs = env.reset_tensor()
                ret = torch.zeros(n_episodes, device=self.device)
                length = torch.zeros(n_episodes, dtype=torch.int32, device=self.device)
                finished = torch.zeros(n_episodes, dtype=torch.bool, device=self.device)
                for _ in range(env.max_episode_steps):
                    logits = self.policy_logits(obs)
                    if deterministic:
                        a = torch.argmax(logits, dim=1).to(torch.int32)
                    else:
                        a = torch.distributions.Categorical(logits=logits).sample().to(torch.int32)
                    b = env.step_tensor(a.contiguous())
                    new = b["done"].bool() & ~finished
                    ret = torch.where(new, b["ret"], ret)
                    length = torch.where(new, b["len"], length)
                    finished |= new
                    obs = b["obs"]
                    if bool(finished.all()):
                        break
                return ret.cpu().numpy().astype(np.float64), length.cpu().numpy().astype(np.int64)
        finally:
            env.close()

    # ------------------------------------------------------------------------------- persistence
    def save(self, path) -> None:
        """`model.save` (training.py:172-175): a zip in Stable-Baselines3's archive layout (see sb3_zip.py)."""
        from . import sb3_zip

        path = str(path)
        if not path.endswith(".zip"):
            path += ".zip"
        sb3_zip.write_zip(path, self)

    @classmethod
    def load(cls, path, env: CudaVecEnv | None = None, device: int = 0, task_id: str | None = None):
        """`PPO.load` (training.py:269): accepts zips written by this backend and SB3-written zips of the same
        architecture (pass `task_id` for those; it is inferred from the shapes when unambiguous)."""
        from . import sb3_zip

        z = sb3_zip.read_zip(str(path))
        meta = z["meta"] or {}
        data = z["data"]
        task = task_id or meta.get("task_id") or sb3_zip.TASK_BY_SHAPE.get((z["obs_dim"], z["n_actions"]))
        if task is None:
            raise ValueError("cannot infer the task from the policy shapes; pass task_id=")
        seed = int(meta.get("seed", data.get("seed", 0) or 0))
        if env is None:
            env = CudaVecEnv(task, 1, seed=seed, device=device)
        if (env.obs_dim, env.n_actions) != (z["obs_dim"], z["n_actions"]):
            raise ValueError(f"policy is {z['obs_dim']}->{z['n_actions']} but task '{task}' is {env.obs_dim}->{env.n_actions}")
        hyper = dict(meta.get("hyper", {}))
        for k in cls._HYPER_KEYS:
            if k not in hyper and isinstance(data.get(k), (int, float)):
                hyper[k] = data[k]
        model = cls("MlpPolicy", env, seed=seed, _params=z["params"], **hyper)
        model._repack()
        model._load_optimizer_state(z, meta)
        model.num_timesteps = int(meta.get("num_timesteps", data.get("num_timesteps", 0) or 0))
        model.n_updates = int(meta.get("n_updates", data.get("_n_updates", 0) or 0))
        return model

    def _load_optimizer_state(self, z: dict, meta: dict) -> None:
        self.m.copy_(z["adam_m"])
        self.v.copy_(z["adam_v"])
        self._adam_step = int(meta.get("adam_step", z["adam_step"]))


# ---------------------------------------------------------------------------------------- bench / smoke
def params_hash(params: torch.Tensor) -> int:
    """64-bit position-weighted checksum of the parameter BITS (wrap-around int64 arithmetic, deterministic)."""
    w = params.detach().contiguous().view(torch.int32).to(torch.int64)
    k = torch.arange(1, w.numel() + 1, dtype=torch.int64, device=w.device) * 0x9E3779B1
    return int(((w + 0x7F4A7C15) * k).sum().item())


def bench_ppo(local_rank: int, rank: int, world: int, iters: int = 5, warmup: int = 2, n_envs: int = 65536, n_steps: int = 128,
              minibatches: int = 32, task: str = "ball3d", mlp_impl: str = "bf16", fused_update: bool = True,
              sustained_tflops: float | None = None) -> dict[str, Any]:
    """BASELINE configs 3/4/5: PPO end-to-end (rollout + GAE + update), `n_envs` envs per GPU, 128-step rollouts, 2x256 MLP,
    10 epochs x 32 minibatches (SURVEY.md §8(d)): `warmup` untimed iterations, then `iters` timed ones (CUDA events, max over
    ranks).  With world > 1 every rank's parameters are hashed after the timed iterations and compared (`replicas_identical`)."""
    dist, _, _ = _dist()
    env = CudaVecEnv(task, n_envs, seed=1, device=local_rank, env_id_base=rank * n_envs)
    model = CudaPPO("MlpPolicy", env, seed=1, n_steps=n_steps, batch_size=n_envs * n_steps // minibatches, n_epochs=10,
                    ent_coef=0.01, mlp_impl=mlp_impl, fused_update=fused_update)
    dev = model.device

    def sync():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for _ in range(max(1, warmup)):                   # allocations, NCCL setup, graph capture
        model.collect_rollouts(); model.train()
    sync()
    e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    roll_ms = train_ms = 0.0
    for _ in range(iters):
        e[0].record(); model.collect_rollouts(); e[1].record(); model.train(); e[2].record()
        sync()
        roll_ms += e[0].elapsed_time(e[1]); train_ms += e[1].elapsed_time(e[2])
    tot = torch.tensor([roll_ms + train_ms, roll_ms, train_ms], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(tot, op=dist.ReduceOp.MAX)
    tot_ms, roll_ms, train_ms = (float(x) for x in tot)
    # replicas must hold bit-identical parameters (the gradient sum and the norm reduction have a fixed order)
    h = torch.tensor([params_hash(model.params)], dtype=torch.int64, device=dev)
    replicas_identical = True
    if dist is not None:
        hs = [torch.zeros_like(h) for _ in range(world)]
        dist.all_gather(hs, h)
        replicas_identical = all(int(x.item()) == int(hs[0].item()) for x in hs)
    # cost of the one collective on the path, measured alone: the gradient all-reduce of one minibatch
    allreduce_us = 0.0
    if dist is not None:
        g = torch.zeros_like(model.grads)
        if model._comm is None:
            def exchange(k):
                model._allreduce_grads(g)
            base_us = 0.0
        else:                                             # fused path: cost of the exchange = fused launch pair minus the local one
            p2, m2, v2 = model.params.clone(), model.m.clone(), model.v.clone()
            seq = [model._adam_step]

            def exchange(k):
                seq[0] += 1
                ops.adam_clip_allreduce(model._comm, p2, g, m2, v2, seq[0], norm_out=model.norm_out)
            for k in range(5):
                ops.adam_clip(p2, g, m2, v2, 1 + k, norm_out=model.norm_out)
            sync()
            e[0].record()
            for k in range(50):
                ops.adam_clip(p2, g, m2, v2, 6 + k, norm_out=model.norm_out)
            e[1].record()
            sync()
            base_us = e[0].elapsed_time(e[1]) * 1e3 / 50
        for k in range(5):
            exchange(k)
        sync()
        e[0].record()
        for k in range(50):
            exchange(k)
        e[1].record()
        sync()
        t = torch.tensor([e[0].elapsed_time(e[1]) * 1e3 / 50 - base_us], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        allreduce_us = float(t.item())
        if model._comm is not None:
            model._adam_step = seq[0]
            model._comm.check()
    samples = world * n_envs * n_steps * iters
    flop_sample = 807936.0 if env.obs_dim == 6 else 803840.0      # SURVEY.md §8(d): fwd+bwd per sample (ball3d | gridworld, push)
    flop_update = flop_sample * n_envs * n_steps * 10 * iters
    row = model._log_row(10 * minibatches, roll_ms / 1e3 / iters, train_ms / 1e3 / iters, time.time())
    update_tflops = flop_update / (train_ms * 1e-3) / 1e12
    out = {
        "value": samples / (tot_ms * 1e-3), "unit": "samples/s (env-steps consumed per second, rollout+GAE+update)",
        "iters": iters, "warmup": max(1, warmup), "ms_per_iter": tot_ms / iters, "rollout_ms": roll_ms / iters,
        "update_ms": train_ms / iters, "update_us_per_minibatch": train_ms / iters * 1e3 / (10 * minibatches),
        "update_tflops": update_tflops,
        "frac_of_sustained": (update_tflops / sustained_tflops) if sustained_tflops else None,
        "allreduce_us": allreduce_us, "allreduce_impl": model.allreduce_impl, "replicas_identical": replicas_identical,
        "rollout_impl": model.rollout_impl,
        "config": {"task": task, "envs_per_gpu": n_envs, "n_steps": n_steps, "epochs": 10, "minibatches_per_epoch": minibatches,
                   "minibatch_rows_per_gpu": n_envs * n_steps // minibatches,
                   "mlp": f"{env.obs_dim}-256-256-{{{env.n_actions},1}} tanh, separate towers",
                   "mlp_impl": ("bf16 tcgen05/TMEM hidden-layer GEMMs, fp32 accumulate (csrc/mlp_tc.cu)" if mlp_impl == "bf16"
                                else "fp32 CUDA-core SGEMM (csrc/mlp_kernels.cu)"),
                   "update": ("fused forward+loss+backward kernel per tower + MN-major wgrad (csrc/mlp_train.cu)"
                              if model.fused_update else "unfused (forward, loss, backward kernels)")},
        "ep_rew_mean": row["rollout/ep_rew_mean"], "approx_kl": row["train/approx_kl"],
    }
    if dist is not None:
        dist.barrier()                                    # nobody unmaps its exchange memory while a peer may still read it
    model.close()
    env.close()
    del model
    torch.cuda.empty_cache()
    return out


def bench_kernels(device: int = 0, n_envs: int = 65536, n_steps: int = 128) -> dict[str, Any]:
    """Per-kernel roofline evidence for the PPO side at BASELINE config-3 sizes (CUDA events, 20 launches each):
    GAE scan and loss head against the measured HBM peak, the tcgen05 GEMMs in TFLOP/s."""
    from . import native as nat

    dev = torch.device("cuda", device)
    T, N, A = n_steps, n_envs, 5
    g = torch.Generator(device=dev).manual_seed(0)
    rew = torch.randn((T, N), device=dev, generator=g)
    val = torch.randn((T, N), device=dev, generator=g)
    done = (torch.rand((T, N), device=dev, generator=g) < 0.01).to(torch.uint8)
    lastv = torch.randn(N, device=dev, generator=g)
    adv, ret = torch.empty_like(rew), torch.empty_like(rew)
    B = T * N // 32
    logits = torch.randn((B, A), device=dev, generator=g)
    values = torch.randn(B, device=dev, generator=g)
    act = torch.randint(0, A, (T, N), device=dev, dtype=torch.int32)
    logp = -torch.rand((T, N), device=dev, generator=g)
    idx = ops.permutation(1, 0, T, N)[:B].contiguous()
    dl, dv, st = torch.empty_like(logits), torch.empty_like(values), torch.zeros(8, device=dev)
    sums = torch.zeros(3, dtype=torch.float64, device=dev)
    Abf = (torch.randn((B, HIDDEN), device=dev, generator=g) * 0.5).to(torch.bfloat16)
    Hbf = torch.tanh(torch.randn((B, HIDDEN), device=dev, generator=g)).to(torch.bfloat16)
    Wbf = (torch.randn((HIDDEN, HIDDEN), device=dev, generator=g) / 16).to(torch.bfloat16)
    out = torch.empty_like(Abf)
    G = torch.zeros((HIDDEN, HIDDEN), device=dev)
    s = nat.current_stream()

    def timed(fn, reps=20):
        for _ in range(3):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(dev)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize(dev)
        return e0.elapsed_time(e1) * 1e3 / reps            # us per launch

    res = {}
    us = timed(lambda: ops.gae(rew, val, done, lastv, 0.99, 0.95, adv, ret))
    res["gae"] = {"us": us, "GB/s": 17.0 * T * N / us / 1e3, "bytes_per_element": 17,
                  "note": "r,V f32 + done u8 read, A,R f32 written (SURVEY's 20 B counts episode_start as f32)"}
    us = timed(lambda: ops.ppo_loss(logits, values, act, adv, logp, ret, index=idx, adv_sums=ops.adv_stats(adv, idx, B, sums),
                                    dlogits=dl, dvalues=dv, stats=st))
    res["adv_stats+ppo_loss"] = {"us": us, "GB/s": (64.0 + 8.0) * B / us / 1e3, "rows": B}
    flop = 2.0 * B * HIDDEN * HIDDEN
    us = timed(lambda: nat.check(nat.lib.tmla_tc_linear(0, nat.ptr(Abf), nat.ptr(Wbf), nat.ptr(lastv), None, nat.ptr(out), B, None, s)))
    res["tc_linear_fwd"] = {"us": us, "TFLOP/s": flop / us / 1e6, "GB/s": 1024.0 * B / us / 1e3}
    us = timed(lambda: nat.check(nat.lib.tmla_tc_linear(1, nat.ptr(Abf), nat.ptr(Wbf), None, nat.ptr(Hbf), nat.ptr(out), B, None, s)))
    res["tc_linear_dgrad"] = {"us": us, "TFLOP/s": flop / us / 1e6, "GB/s": 1536.0 * B / us / 1e3}
    us = timed(lambda: nat.check(nat.lib.tmla_tc_wgrad(nat.ptr(Abf), nat.ptr(Hbf), nat.ptr(G), B, s)))
    res["tc_wgrad"] = {"us": us, "TFLOP/s": flop / us / 1e6, "GB/s": 1024.0 * B / us / 1e3}
    # fused minibatch path (csrc/mlp_train.cu): the TMA-fed split-K wgrad over tile images, and one whole minibatch
    # (tower kernels for pi and vf + two wgrads) at 807 936 FLOP per sample (SURVEY.md 8(d))
    us = timed(lambda: nat.check(nat.lib.tmla_tc_wgrad_tiled(nat.ptr(Abf), nat.ptr(Hbf), nat.ptr(G), B, s)))
    res["tc_wgrad_tiled"] = {"us": us, "TFLOP/s": flop / us / 1e6, "GB/s": 1024.0 * B / us / 1e3,
                             "note": "bulk-TMA loads of 64 KB tile images, MN-major UMMA operands, 3-stage mbarrier ring"}
    D = 6
    obs = torch.randn((T * N, D), device=dev, generator=g)
    params = orthogonal_init(D, A, 1).to(dev)
    wpack = ops.mlp_pack(params, D, A)
    grads = torch.empty_like(params)
    scratch = torch.empty(nat.lib.tmla_ppo_minibatch_scratch(HIDDEN, B), dtype=torch.bfloat16, device=dev)
    stats = torch.zeros(8, device=dev)
    adv_sums = ops.adv_stats(adv, idx, B, sums)
    us = timed(lambda: ops.ppo_minibatch(params, wpack, obs, D, A, act, adv, logp, ret, index=idx, rows=B, adv_sums=adv_sums,
                                         grads=grads, scratch=scratch, stats=stats))
    res["ppo_minibatch_fused"] = {"us": us, "TFLOP/s": 807936.0 * B / us / 1e6, "rows": B,
                                  "note": "forward + loss + backward of both towers: 2 fused tower kernels + 2 tiled wgrads"}
    return res


def smoke_update() -> None:
    """One tiny rollout + update on cuda:0 (called from __graft_entry__.smoke)."""
    env = CudaVecEnv("ball3d", 256, seed=1)
    model = CudaPPO("MlpPolicy", env, seed=1, n_steps=16, batch_size=1024, n_epochs=2, ent_coef=0.01)
    before = model.params.clone()
    model.learn(256 * 16)
    torch.cuda.synchronize()
    row = model.logger_rows[-1]
    assert torch.isfinite(model.params).all() and not torch.equal(before, model.params)
    assert math.isfinite(row["train/loss"]) and row["train/clip_fraction"] >= 0.0
    env.close()
