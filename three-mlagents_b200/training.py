"""Training / evaluation orchestration — same surface as backend/mlagents/training.py:
`TrainConfig`, `TrainResult`, `make_vector_env`, `make_eval_env`, `train_task`, `evaluate_model`,
`load_model`, `predict_action`, `latest_model_filename`, `ALGORITHMS`, `POLICIES_DIR`, `RUNS_DIR`
(training.py:28-37, 40-68, 71-95, 98-291), with the SB3 objects replaced by the CUDA backend:

    DummyVecEnv[Monitor[env]]  ->  CudaVecEnv           (one kernel launch per vec-step)
    stable_baselines3.PPO      ->  CudaPPO              (rollout, GAE, update in libtmla.so)
    stable_baselines3.A2C      ->  CudaA2C              (the same rollout; one RMSprop step per rollout)
    EvalCallback/evaluate_policy -> CudaPPO.evaluate    (batched deterministic episodes on the device)

PPO and A2C have CUDA backends; asking for dqn/sac/td3 raises the same ValueError the reference raises
for an unsupported algorithm (training.py:110-114).
"""
from __future__ import annotations

import json
import platform
import uuid
import warnings
from dataclasses import asdict, dataclass
from datetime import datetime, timezone
from pathlib import Path
from typing import Any

import numpy as np

from .a2c import CudaA2C
from .ppo import CudaPPO
from .registry import TaskSpec, get_task, make_env
from .vec_env import CudaVecEnv

POLICIES_DIR = Path("policies")
RUNS_DIR = Path("runs")

ALGORITHMS: dict[str, type] = {"ppo": CudaPPO, "a2c": CudaA2C}
_REFERENCE_ALGORITHMS = ("a2c", "dqn", "ppo", "sac", "td3")      # training.py:31-37


@dataclass(frozen=True)
class TrainConfig:                    # field-for-field training.py:40-53
    task_id: str
    total_timesteps: int | None = None
    algorithm: str | None = None
    seed: int = 1
    n_envs: int | None = None
    eval_episodes: int | None = None
    eval_freq: int = 10_000
    deterministic_eval: bool = True
    policy: str | None = None
    run_name: str | None = None
    save_policy: bool = True
    verbose: int = 1


@dataclass(frozen=True)
class TrainResult:                    # field-for-field training.py:56-68
    task_id: str
    algorithm: str
    run_id: str
    model_filename: str
    model_path: str
    run_dir: str
    mean_reward: float
    std_reward: float
    eval_episodes: int
    total_timesteps: int
    metadata_path: str


def make_vector_env(task_id: str, *, n_envs: int, seed: int, monitor_dir: Path | None = None, device: int = 0,
                    env_id_base: int = 0) -> CudaVecEnv:
    """training.py:71-89.  Env i is seeded by (seed, global env id i) through Philox sub-sequences
    instead of `reset(seed=seed+i)` on NumPy's global RNG."""
    task = get_task(task_id)
    if not task.trainable:
        raise ValueError(f"Task '{task_id}' is not a Gymnasium/SB3 trainable task yet.")
    return CudaVecEnv(task.id, n_envs, seed=seed, device=device, env_id_base=env_id_base, monitor_dir=monitor_dir)


def make_eval_env(task_id: str, *, seed: int):
    """training.py:92-95: a single seeded env (Gymnasium 5-tuple API)."""
    env = make_env(task_id)
    env.reset(seed=seed)
    return env


def _default_policy(task: TaskSpec) -> str:          # training.py:326-327
    return "CnnPolicy" if task.observation == "image" else "MlpPolicy"


def _default_model_kwargs(algorithm_name: str, *, train_env, task: TaskSpec, total_timesteps: int, tensorboard_log: str,
                          verbose: int) -> dict[str, Any]:
    """PPO branch of training.py:361-391 (hyper-parameters verbatim).  a2c: SB3 2.9.0 A2C.__init__'s defaults with the PPO
    branch's net_arch (the reference's own a2c branch is not transcribed here; DESIGN.md §8)."""
    if algorithm_name not in ALGORITHMS:
        raise ValueError(f"Algorithm '{algorithm_name}' has no CUDA backend; use one of {sorted(ALGORITHMS)}.")
    if task.observation == "image":
        raise ValueError(f"Task '{task.id}' needs task-specific CNN policy settings.")
    if algorithm_name == "a2c":
        return {
            "tensorboard_log": tensorboard_log, "verbose": verbose,
            "learning_rate": 7e-4, "n_steps": 5, "gamma": 0.99, "gae_lambda": 1.0, "ent_coef": 0.0, "vf_coef": 0.5,
            "max_grad_norm": 0.5, "rms_prop_eps": 1e-5, "use_rms_prop": True, "normalize_advantage": False,
            "policy_kwargs": {"net_arch": {"pi": [256, 256], "vf": [256, 256]}},
        }
    return {
        "tensorboard_log": tensorboard_log, "verbose": verbose,
        "learning_rate": 3e-4,
        "n_steps": 1024 if task.research_tier == "foundation" else 2048,
        "batch_size": 256, "n_epochs": 10, "gamma": 0.99, "gae_lambda": 0.95, "clip_range": 0.2,
        "ent_coef": 0.01, "vf_coef": 0.5, "max_grad_norm": 0.5,
        "policy_kwargs": {"net_arch": {"pi": [256, 256], "vf": [256, 256]}},
    }


def _make_run_id(task_id: str, algorithm_name: str) -> str:
    return f"{task_id}_{algorithm_name}_{datetime.now().strftime('%Y%m%d_%H%M%S')}_{uuid.uuid4().hex[:8]}"


def train_task(config: TrainConfig, *, callback=None, model_kwargs: dict[str, Any] | None = None) -> TrainResult:
    """training.py:98-225."""
    task = get_task(config.task_id)
    if not task.trainable:
        raise ValueError(f"Task '{task.id}' is not trainable through Gymnasium/SB3 yet.")
    algorithm_name = (config.algorithm or task.default_algorithm).lower()
    if config.algorithm is None and algorithm_name not in ALGORITHMS and algorithm_name in _REFERENCE_ALGORITHMS:
        # the registry keeps the reference's per-task default (dqn for basic / gridworld / push / walljump, registry.py:61-112);
        # this backend trains every CUDA task with PPO, so an unspecified algorithm resolves to it
        warnings.warn(f"task '{task.id}' defaults to '{algorithm_name}' in the reference; three-mlagents_b200 has a CUDA backend "
                      f"for PPO only and trains it with 'ppo'", stacklevel=2)
        algorithm_name = "ppo"
    if algorithm_name not in ALGORITHMS:
        if algorithm_name in _REFERENCE_ALGORITHMS:
            raise ValueError(f"Algorithm '{algorithm_name}' has no CUDA backend in three-mlagents_b200 "
                             f"(task default: '{task.default_algorithm}'). Use one of {sorted(ALGORITHMS)} (pass -a ppo).")
        raise ValueError(f"Unsupported algorithm '{algorithm_name}'. Use one of {sorted(ALGORITHMS)}.")

    total_timesteps = config.total_timesteps or task.total_timesteps
    n_envs = config.n_envs or task.n_envs
    eval_episodes = config.eval_episodes or task.eval_episodes
    run_id = config.run_name or _make_run_id(task.id, algorithm_name)
    run_dir = RUNS_DIR / task.id / run_id
    monitor_dir, eval_dir, tb_dir = run_dir / "monitor", run_dir / "eval", run_dir / "tb"
    for path in (POLICIES_DIR, run_dir, monitor_dir, eval_dir, tb_dir):
        path.mkdir(parents=True, exist_ok=True)

    train_env = make_vector_env(task.id, n_envs=n_envs, seed=config.seed, monitor_dir=monitor_dir)
    try:
        policy = config.policy or _default_policy(task)
        kwargs = _default_model_kwargs(algorithm_name, train_env=train_env, task=task, total_timesteps=total_timesteps,
                                       tensorboard_log=str(tb_dir), verbose=config.verbose)
        if model_kwargs:
            kwargs.update(model_kwargs)
        model = ALGORITHMS[algorithm_name](policy, train_env, seed=config.seed, **kwargs)

        # EvalCallback (training.py:152-161) at rollout granularity: evaluate whenever another
        # `eval_freq` timesteps have been consumed; keep the best parameters and evaluations.npz.
        evals: dict[str, list] = {"timesteps": [], "results": [], "ep_lengths": []}
        state = {"next_eval": config.eval_freq, "best": -np.inf}

        def _on_rollout(m: CudaPPO):
            if m.num_timesteps >= state["next_eval"]:
                state["next_eval"] = (m.num_timesteps // max(1, config.eval_freq) + 1) * max(1, config.eval_freq)
                r, l = m.evaluate(eval_episodes, seed=config.seed + 10_000, deterministic=config.deterministic_eval)
                evals["timesteps"].append(m.num_timesteps); evals["results"].append(r); evals["ep_lengths"].append(l)
                np.savez(eval_dir / "evaluations.npz", timesteps=np.array(evals["timesteps"]),
                         results=np.stack(evals["results"]), ep_lengths=np.stack(evals["ep_lengths"]))
                if r.mean() > state["best"]:
                    state["best"] = float(r.mean())
                    (run_dir / "best_model").mkdir(exist_ok=True)
                    m.save(run_dir / "best_model" / "best_model.zip")
                if config.verbose:
                    print(f"Eval num_timesteps={m.num_timesteps}, episode_reward={r.mean():.2f} +/- {r.std():.2f}", flush=True)
            if callback is not None:
                return callback(m) if callable(callback) else callback.on_rollout(m)
            return True

        model.learn(total_timesteps=total_timesteps, callback=_on_rollout, progress_bar=False)

        model_filename = f"{task.policy_prefix}_{run_id}.zip"
        model_path = POLICIES_DIR / model_filename
        if config.save_policy:
            model.save(model_path)

        episode_rewards, episode_lengths = model.evaluate(eval_episodes, seed=config.seed + 10_000,
                                                          deterministic=config.deterministic_eval)
        mean_reward, std_reward = float(np.mean(episode_rewards)), float(np.std(episode_rewards))
        import torch

        from . import native

        metadata = {
            "task": task.card(), "config": asdict(config), "algorithm": algorithm_name, "run_id": run_id,
            "model_filename": model_filename, "model_path": str(model_path),
            "deterministic": bool(model.deterministic),
            "mean_reward": mean_reward, "std_reward": std_reward,
            "episode_rewards": [float(r) for r in episode_rewards],
            "episode_lengths": [int(n) for n in episode_lengths],
            "software": {"python": platform.python_version(), "three_mlagents_b200": "0.1.0",
                         "libtmla": native.lib.tmla_version(), "torch": torch.__version__,
                         "device": torch.cuda.get_device_name(train_env.device_index)},
            "created_at": datetime.now(timezone.utc).isoformat(),
        }
        metadata_path = run_dir / "metadata.json"
        metadata_path.write_text(json.dumps(metadata, indent=2), encoding="utf-8")
        return TrainResult(task_id=task.id, algorithm=algorithm_name, run_id=run_id, model_filename=model_filename,
                           model_path=str(model_path), run_dir=str(run_dir), mean_reward=mean_reward,
                           std_reward=std_reward, eval_episodes=eval_episodes, total_timesteps=total_timesteps,
                           metadata_path=str(metadata_path))
    finally:
        train_env.close()


def evaluate_model(task_id: str, model_filename_or_path: str, *, episodes: int | None = None, deterministic: bool = True,
                   seed: int = 10_001) -> dict[str, Any]:
    """training.py:227-258."""
    task = get_task(task_id)
    model = load_model(task, model_filename_or_path)
    try:
        n_eval_episodes = episodes or task.eval_episodes
        rewards, lengths = model.evaluate(n_eval_episodes, seed=seed, deterministic=deterministic)
        return {
            "task_id": task.id, "model": str(_resolve_model_path(task, model_filename_or_path)),
            "episodes": n_eval_episodes, "mean_reward": float(np.mean(rewards)), "std_reward": float(np.std(rewards)),
            "episode_rewards": [float(r) for r in rewards], "episode_lengths": [int(n) for n in lengths],
        }
    finally:
        model.env.close()


def load_model(task: TaskSpec, model_filename_or_path: str | None = None):
    """training.py:261-269."""
    model_path = _resolve_model_path(task, model_filename_or_path)
    algorithm_name = _infer_algorithm_from_metadata(task, model_path) or _infer_algorithm_from_zip(model_path) or "ppo"
    if algorithm_name not in ALGORITHMS:
        raise ValueError(f"Model '{model_path}' was trained with '{algorithm_name}', which has no CUDA backend.")
    return ALGORITHMS[algorithm_name].load(model_path, task_id=task.id)


def predict_action(task_id: str, obs: np.ndarray, model_filename: str | None = None) -> int | list[float]:
    """training.py:272-283."""
    task = get_task(task_id)
    model = load_model(task, model_filename)
    try:
        action, _ = model.predict(np.asarray(obs, dtype=np.float32), deterministic=True)
    finally:
        model.env.close()
    if isinstance(action, np.ndarray):
        return int(action.item()) if action.ndim == 0 else action.tolist()
    return int(action)


def latest_model_filename(task_id: str) -> str:          # training.py:286-291
    task = get_task(task_id)
    matches = sorted(POLICIES_DIR.glob(f"{task.policy_prefix}_*.zip"), reverse=True)
    if not matches:
        raise FileNotFoundError(f"No SB3 policy zip found for task '{task.id}'.")
    return matches[0].name


def _resolve_model_path(task: TaskSpec, model_filename_or_path: str | None) -> Path:      # training.py:294-305
    if model_filename_or_path is None:
        model_filename_or_path = latest_model_filename(task.id)
    path = Path(model_filename_or_path)
    if path.exists():
        return path
    if not path.is_absolute():
        candidate = POLICIES_DIR / path
        if candidate.exists():
            return candidate
        path = candidate
    raise FileNotFoundError(f"Model not found: {path}")


def _infer_algorithm_from_zip(model_path: Path) -> str | None:
    """The algorithm a policy zip names itself (tmla.json), or, for SB3-written zips, the one its optimizer state implies."""
    from . import sb3_zip

    return sb3_zip.zip_algorithm(str(model_path))


def _infer_algorithm_from_metadata(task: TaskSpec, model_path: Path) -> str | None:       # training.py:308-323
    stem = model_path.name.removesuffix(".zip")
    for meta_file in (RUNS_DIR / task.id).glob("*/metadata.json"):
        try:
            meta = json.loads(meta_file.read_text(encoding="utf-8"))
        except json.JSONDecodeError:
            continue
        if meta.get("model_filename") == model_path.name or (meta.get("run_id") or "\0") in stem:
            return (meta.get("algorithm") or meta.get("config", {}).get("algorithm") or task.default_algorithm).lower()
    return None
