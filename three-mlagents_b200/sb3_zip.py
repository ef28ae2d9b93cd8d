"""Policy artifacts in Stable-Baselines3's zip layout (SURVEY.md §8(f) #1).

The reference saves `policies/<prefix>_<run_id>.zip` with `model.save` (backend/mlagents/training.py:172-175)
and loads it with `algo_cls.load` (training.py:269).  `write_zip` produces the same archive members SB3 2.9.0
writes — `data` (JSON), `policy.pth` (state dict with SB3's parameter names), `policy.optimizer.pth` (torch Adam
state dict), `pytorch_variables.pth`, `_stable_baselines3_version`, `system_info.txt` — plus `tmla.json`, this
backend's own metadata.  A2C models (CudaA2C) write the same members with A2C's `data` attributes and a torch RMSprop state dict.
`read_zip` accepts both this backend's zips and zips written by SB3 itself for the
same architecture (MlpPolicy, net_arch dict(pi=[H,H], vf=[H,H]) with H = 64, 128 or 256; SB3's default is 64), so
SB3-trained policies can be evaluated on the CUDA backend.  The width is read off the state dict's shapes.

What can be checked here IS checked (tests/test_sb3_zip_cpu.py): parameter names/shapes/order, the round trip
flat vector <-> state dict, optimizer state layout, archive members, `data` decodability.  Loading the zip
INTO Stable-Baselines3 cannot be tested in this image (SB3 and gymnasium are not installable, no network): the
pickled class references and space objects inside `data` are written against the attribute layout of
gymnasium 1.3.0 / SB3 2.9.0 (the versions pinned by the reference's uv.lock) on a best-effort basis.
"""
from __future__ import annotations

import base64
import io
import json
import math
import pickle
import sys
import types
import zipfile
from collections import OrderedDict

import numpy as np
import torch

H = 256                    # default hidden width
WIDTHS = (64, 128, 256)
SB3_VERSION = "2.9.0"


def param_layout(obs_dim: int, n_actions: int, hidden: int = H):
    """(SB3 state-dict key, shape) in policy.parameters() order == order of the flat vector (include/tmla.h)."""
    H = int(hidden)
    return [
        ("mlp_extractor.policy_net.0.weight", (H, obs_dim)), ("mlp_extractor.policy_net.0.bias", (H,)),
        ("mlp_extractor.policy_net.2.weight", (H, H)), ("mlp_extractor.policy_net.2.bias", (H,)),
        ("mlp_extractor.value_net.0.weight", (H, obs_dim)), ("mlp_extractor.value_net.0.bias", (H,)),
        ("mlp_extractor.value_net.2.weight", (H, H)), ("mlp_extractor.value_net.2.bias", (H,)),
        ("action_net.weight", (n_actions, H)), ("action_net.bias", (n_actions,)),
        ("value_net.weight", (1, H)), ("value_net.bias", (1,)),
    ]


def flat_to_state_dict(flat: torch.Tensor, obs_dim: int, n_actions: int, hidden: int = H) -> "OrderedDict[str, torch.Tensor]":
    flat = flat.detach().float().cpu().contiguous()
    sd, p = OrderedDict(), 0
    for name, shape in param_layout(obs_dim, n_actions, hidden):
        n = int(np.prod(shape))
        sd[name] = flat[p:p + n].clone().view(shape)
        p += n
    if p != flat.numel():
        raise ValueError(f"flat vector has {flat.numel()} elements, layout needs {p}")
    return sd


def state_dict_to_flat(sd, obs_dim: int, n_actions: int, hidden: int = H) -> torch.Tensor:
    chunks = []
    for name, shape in param_layout(obs_dim, n_actions, hidden):
        if name not in sd:
            raise KeyError(f"state dict has no '{name}' (not an MlpPolicy with net_arch dict(pi=[{hidden},{hidden}], "
                           f"vf=[{hidden},{hidden}])?)")
        t = torch.as_tensor(sd[name]).float()
        if tuple(t.shape) != tuple(shape):
            raise ValueError(f"{name}: shape {tuple(t.shape)} != {shape}")
        chunks.append(t.reshape(-1))
    return torch.cat(chunks)


def hidden_width(sd) -> int:
    """The hidden width of an MlpPolicy state dict: both hidden layers of both towers square and equal, 64, 128 or 256."""
    try:
        shapes = [tuple(sd[f"mlp_extractor.{t}.{i}.weight"].shape) for t in ("policy_net", "value_net") for i in (0, 2)]
    except KeyError as e:
        raise KeyError(f"state dict has no {e} (not an MlpPolicy with a two-layer net_arch?)") from None
    h = shapes[0][0]
    if any(s[0] != h for s in shapes) or shapes[1][1] != h or shapes[3][1] != h or h not in WIDTHS:
        raise ValueError(f"hidden layers {shapes}: supported are net_arch dict(pi=[H,H], vf=[H,H]) with H in {WIDTHS}")
    return int(h)


def adam_state_dict(m, v, step: int, hyper: dict, obs_dim: int, n_actions: int, hidden: int = H) -> dict:
    """torch.optim.Adam.state_dict() layout for the 12 parameter tensors."""
    ms, vs = flat_to_state_dict(m, obs_dim, n_actions, hidden), flat_to_state_dict(v, obs_dim, n_actions, hidden)
    state = {}
    for i, name in enumerate(ms):
        if step > 0:
            state[i] = {"step": torch.tensor(float(step)), "exp_avg": ms[name], "exp_avg_sq": vs[name]}
    group = {"lr": hyper["learning_rate"], "betas": (0.9, 0.999), "eps": 1e-5, "weight_decay": 0, "amsgrad": False,
             "maximize": False, "foreach": None, "capturable": False, "differentiable": False, "fused": None,
             "decoupled_weight_decay": False, "params": list(range(len(ms)))}
    return {"state": state, "param_groups": [group]}


def rmsprop_state_dict(sq_avg, step: int, hyper: dict, obs_dim: int, n_actions: int, hidden: int = H) -> dict:
    """torch.optim.RMSprop(alpha=0.99, eps=rms_prop_eps, weight_decay=0).state_dict() for the 12 parameter tensors, produced by a
    real RMSprop instance so that the layout (state keys, param_group entries) is torch's own."""
    sq = flat_to_state_dict(sq_avg, obs_dim, n_actions, hidden)
    params = [torch.nn.Parameter(torch.zeros(shape)) for _, shape in param_layout(obs_dim, n_actions, hidden)]
    opt = torch.optim.RMSprop(params, lr=hyper["learning_rate"], alpha=0.99, eps=hyper["rms_prop_eps"], weight_decay=0)
    if step > 0:
        for p, name in zip(params, sq):
            opt.state[p] = {"step": torch.tensor(float(step)), "square_avg": sq[name]}
    return opt.state_dict()


# ---- best-effort `data` entries that SB3 stores as base64 cloudpickle -------------------------------------------
_created_stubs: list[str] = []


def _stub_module(name: str) -> types.ModuleType:
    parts = name.split(".")
    for i in range(1, len(parts) + 1):
        sub = ".".join(parts[:i])
        if sub not in sys.modules:
            sys.modules[sub] = types.ModuleType(sub)
            _created_stubs.append(sub)
    return sys.modules[name]


def _drop_stubs() -> None:
    """Remove the placeholder modules again so `import stable_baselines3` keeps failing honestly."""
    while _created_stubs:
        sys.modules.pop(_created_stubs.pop(), None)


def _by_reference(module: str, qualname: str):
    """An object that pickles as a reference to `module.qualname` even when that module is not installed."""
    installed = module in sys.modules and hasattr(sys.modules[module], qualname)
    mod = sys.modules[module] if installed else _stub_module(module)
    if not hasattr(mod, qualname):
        cls = type(qualname, (), {})
        cls.__module__ = module
        setattr(mod, qualname, cls)
    return getattr(mod, qualname)


def _serialized(obj, type_repr: str) -> dict:
    return {":type:": type_repr, ":serialized:": base64.b64encode(pickle.dumps(obj, protocol=4)).decode()}


def _space_entries(obs_space, act_space):
    box_cls = _by_reference("gymnasium.spaces.box", "Box")
    disc_cls = _by_reference("gymnasium.spaces.discrete", "Discrete")
    box = box_cls.__new__(box_cls)
    low = np.asarray(obs_space.low, np.float32)
    high = np.asarray(obs_space.high, np.float32)
    box.__dict__.update(dtype=np.dtype(np.float32), _shape=tuple(low.shape), low=low, high=high,
                        low_repr=str(low.min()), high_repr=str(high.max()), bounded_below=np.isfinite(low),
                        bounded_above=np.isfinite(high), _np_random=None)
    disc = disc_cls.__new__(disc_cls)
    disc.__dict__.update(n=np.int64(act_space.n), start=np.int64(0), _shape=(), dtype=np.dtype(np.int64), _np_random=None)
    obs_e = _serialized(box, "<class 'gymnasium.spaces.box.Box'>")
    obs_e.update(dtype="float32", _shape=list(low.shape), low=repr(low), high=repr(high))
    act_e = _serialized(disc, "<class 'gymnasium.spaces.discrete.Discrete'>")
    act_e.update(n=str(int(act_space.n)), start="0", _shape=[], dtype="int64")
    return obs_e, act_e


def build_data(model) -> dict:
    try:
        return _build_data(model)
    finally:
        _drop_stubs()


def _build_data(model) -> dict:
    obs_e, act_e = _space_entries(model.env.observation_space, model.env.action_space)
    policy_cls = _by_reference("stable_baselines3.common.policies", "ActorCriticPolicy")
    buf_cls = _by_reference("stable_baselines3.common.buffers", "RolloutBuffer")
    pc = _serialized(policy_cls, "<class 'abc.ABCMeta'>")
    pc["__module__"] = "stable_baselines3.common.policies"
    rb = _serialized(buf_cls, "<class 'abc.ABCMeta'>")
    rb["__module__"] = "stable_baselines3.common.buffers"
    hid = getattr(model, "hidden", H)
    net_arch = {"pi": [hid, hid], "vf": [hid, hid]}
    data = {
        "policy_class": pc, "verbose": model.verbose, "policy_kwargs": {"net_arch": net_arch},
        "num_timesteps": model.num_timesteps, "_total_timesteps": model.num_timesteps, "_num_timesteps_at_start": 0,
        "seed": model.seed, "action_noise": None, "start_time": 0, "learning_rate": model.lr,
        "tensorboard_log": model.tensorboard_log, "_last_obs": None, "_last_episode_starts": None,
        "_last_original_obs": None, "_episode_num": 0, "use_sde": False, "sde_sample_freq": -1,
        "_current_progress_remaining": 0.0, "_stats_window_size": 100, "_n_updates": model.n_updates,
        "observation_space": obs_e, "action_space": act_e, "n_envs": model.n_envs, "n_steps": model.n_steps,
        "gamma": model.gamma, "gae_lambda": model.gae_lambda, "ent_coef": model.ent_coef, "vf_coef": model.vf_coef,
        "max_grad_norm": model.max_grad_norm, "rollout_buffer_class": rb, "rollout_buffer_kwargs": {},
    }
    if getattr(model, "algorithm", "ppo") == "a2c":      # A2C.__init__: use_rms_prop puts RMSprop and its kwargs into policy_kwargs
        kwargs = {"net_arch": net_arch, "optimizer_class": torch.optim.RMSprop,
                  "optimizer_kwargs": {"alpha": 0.99, "eps": model.rms_prop_eps, "weight_decay": 0}}
        pk = _serialized(kwargs, "<class 'dict'>")
        pk.update(net_arch=kwargs["net_arch"], optimizer_class=str(torch.optim.RMSprop), optimizer_kwargs=kwargs["optimizer_kwargs"])
        data.update(policy_kwargs=pk, normalize_advantage=model.normalize_advantage, rms_prop_eps=model.rms_prop_eps,
                    use_rms_prop=True)
    else:
        data.update(batch_size=model.batch_size, n_epochs=model.n_epochs, clip_range=model.clip_range, clip_range_vf=None,
                    normalize_advantage=model.normalize_advantage, target_kl=None)
    return data


def _torch_bytes(obj) -> bytes:
    buf = io.BytesIO()
    torch.save(obj, buf)
    return buf.getvalue()


def write_zip(path: str, model) -> None:
    a2c = getattr(model, "algorithm", "ppo") == "a2c"
    hid = getattr(model, "hidden", H)
    if a2c:
        hyper = {"learning_rate": model.lr, "n_steps": model.n_steps, "gamma": model.gamma, "gae_lambda": model.gae_lambda,
                 "ent_coef": model.ent_coef, "vf_coef": model.vf_coef, "max_grad_norm": model.max_grad_norm,
                 "rms_prop_eps": model.rms_prop_eps, "normalize_advantage": model.normalize_advantage}
    else:
        hyper = {"learning_rate": model.lr, "n_steps": model.n_steps, "batch_size": model.batch_size, "n_epochs": model.n_epochs,
                 "gamma": model.gamma, "gae_lambda": model.gae_lambda, "clip_range": model.clip_range, "ent_coef": model.ent_coef,
                 "vf_coef": model.vf_coef, "max_grad_norm": model.max_grad_norm}
    meta = {"format": "three-mlagents_b200/2", "algorithm": "a2c" if a2c else "ppo", "task_id": model.env.task_id, "obs_dim": model.obs_dim,
            "n_actions": model.n_actions, "net_arch": {"pi": [hid, hid], "vf": [hid, hid]}, "seed": model.seed,
            "num_timesteps": model.num_timesteps, "n_updates": model.n_updates,
            **({"opt_step": model._opt_step} if a2c else {"adam_step": model._adam_step}), "mlp_impl": model.mlp_impl, "hyper": hyper}
    if a2c:
        opt_sd = rmsprop_state_dict(model.sq_avg, model._opt_step, hyper, model.obs_dim, model.n_actions, hid)
    else:
        opt_sd = adam_state_dict(model.m, model.v, model._adam_step, hyper, model.obs_dim, model.n_actions, hid)
    with zipfile.ZipFile(path, "w") as z:
        z.writestr("data", json.dumps(build_data(model), indent=4))
        z.writestr("policy.pth", _torch_bytes(flat_to_state_dict(model.params, model.obs_dim, model.n_actions, hid)))
        z.writestr("policy.optimizer.pth", _torch_bytes(opt_sd))
        z.writestr("pytorch_variables.pth", _torch_bytes({}))
        z.writestr("_stable_baselines3_version", SB3_VERSION)
        z.writestr("system_info.txt", f"- three-mlagents_b200 CUDA backend (libtmla), torch {torch.__version__}\n")
        z.writestr("tmla.json", json.dumps(meta, indent=2))


def read_zip(path: str) -> dict:
    """-> {params, adam_m, adam_v, adam_step, sq_avg, opt_step, optimizer, meta (or None), data, obs_dim, n_actions, hidden} for a
    zip written by this backend or by SB3 (hidden: the width read off the policy's hidden layers).  optimizer: "adam" (exp_avg / exp_avg_sq: PPO), "rmsprop" (square_avg: A2C) or None (no optimizer state);
    sq_avg / opt_step are RMSprop's state (None / 0 for Adam)."""
    with zipfile.ZipFile(path) as z:
        names = set(z.namelist())
        if "policy.pth" not in names:
            raise ValueError(f"{path}: no policy.pth member (not an SB3-layout policy zip)")
        sd = torch.load(io.BytesIO(z.read("policy.pth")), map_location="cpu", weights_only=True)
        meta = json.loads(z.read("tmla.json")) if "tmla.json" in names else None
        data = json.loads(z.read("data")) if "data" in names else {}
        obs_dim = int(sd["mlp_extractor.policy_net.0.weight"].shape[1])
        n_actions = int(sd["action_net.weight"].shape[0])
        hidden = hidden_width(sd)
        flat = state_dict_to_flat(sd, obs_dim, n_actions, hidden)
        m, v, step = torch.zeros_like(flat), torch.zeros_like(flat), 0
        sq, opt_step, kind = None, 0, None
        if "policy.optimizer.pth" in names:
            opt = torch.load(io.BytesIO(z.read("policy.optimizer.pth")), map_location="cpu", weights_only=True)
            st = opt.get("state", {})
            kind = _optimizer_kind(opt)
            if len(st) == 12:
                layout = param_layout(obs_dim, n_actions, hidden)
                cat = lambda key: torch.cat([torch.as_tensor(st[i][key]).float().reshape(-1) for i in range(12)])
                if kind == "rmsprop":
                    sq, opt_step = cat("square_avg"), int(float(st[0]["step"]))
                    assert sq.numel() == flat.numel()
                else:
                    m, v = cat("exp_avg"), cat("exp_avg_sq")
                    step = int(float(st[0]["step"]))
                    assert m.numel() == sum(int(np.prod(s)) for _, s in layout)
    return {"params": flat, "adam_m": m, "adam_v": v, "adam_step": step, "sq_avg": sq, "opt_step": opt_step, "optimizer": kind,
            "meta": meta, "data": data, "obs_dim": obs_dim, "n_actions": n_actions, "hidden": hidden}


def _optimizer_kind(opt_state_dict: dict) -> str | None:
    st = opt_state_dict.get("state", {})
    keys = set(next(iter(st.values()))) if st else set()
    if "square_avg" in keys:
        return "rmsprop"
    if "exp_avg" in keys:
        return "adam"
    group = (opt_state_dict.get("param_groups") or [{}])[0]          # no state yet (never stepped): RMSprop groups carry alpha
    return "rmsprop" if "alpha" in group else ("adam" if "betas" in group else None)


def zip_algorithm(path: str) -> str | None:
    """The algorithm a policy zip was trained with: tmla.json's `algorithm`, else (SB3-written zips) the optimizer state's kind
    (square_avg: A2C's RMSprop, exp_avg: PPO's Adam), else None."""
    with zipfile.ZipFile(path) as z:
        names = set(z.namelist())
        if "tmla.json" in names:
            algo = json.loads(z.read("tmla.json")).get("algorithm")
            if algo:
                return str(algo).lower()
        if "policy.optimizer.pth" in names:
            opt = torch.load(io.BytesIO(z.read("policy.optimizer.pth")), map_location="cpu", weights_only=True)
            return {"rmsprop": "a2c", "adam": "ppo"}.get(_optimizer_kind(opt))
    return None


TASK_BY_SHAPE = {(21, 3): "basic", (6, 5): "ball3d", (4, 4): "walljump", (45, 3): "brickbreak", (7, 3): "bicycle", (16, 5): "glider"}      # (4,5) is ambiguous (gridworld / push): needs the task id
