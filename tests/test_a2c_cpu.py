"""A2C without a GPU: the oracle's invariants (A2C gradient = PPO gradient at ratio 1; RMSprop step = its written-out rule),
the A2C policy archive (data, RMSprop state layout, algorithm detection), the training-layer registration and defaults."""
import base64
import json
import pickle
import types
import zipfile

import numpy as np
import pytest
import torch

from oracle import a2c_oracle as ao, ppo_oracle as po
from three_mlagents_b200 import sb3_zip
from three_mlagents_b200.spaces import spaces_for


def _batch(d, a, rows, seed):
    g = torch.Generator().manual_seed(seed)
    flat = torch.from_numpy(po.init_params(d, a, seed)) + 0.05 * torch.randn(po.init_params(d, a, seed).size, generator=g)
    obs = torch.randn(rows, d, generator=g)
    act = torch.randint(0, a, (rows,), generator=g)
    adv = torch.randn(rows, generator=g) * 2.0 + 0.3
    ret = torch.randn(rows, generator=g) * 3.0
    return flat, obs, act, adv, ret


@pytest.mark.parametrize("normalize", [False, True])
def test_a2c_gradient_is_the_ppo_gradient_at_ratio_one(normalize):
    """With old_logp = log_prob the PPO ratio is 1 and its clip inactive: d/dθ of -min(A r, A clip(r)) is -A dlogp/dθ, the A2C
    policy gradient; the value and entropy terms are the same expressions."""
    d, a, rows = 6, 5, 512
    flat, obs, act, adv, ret = _batch(d, a, rows, 3)
    grads = []
    for algo in ("a2c", "ppo"):
        p = flat.clone().requires_grad_(True)
        logits, values = po.forward(p, obs, d, a)
        if algo == "a2c":
            loss, _ = ao.a2c_loss(logits, values, act, adv, ret, ent_coef=0.01, vf_coef=0.5, normalize=normalize)
        else:
            logp, _ = po.categorical(logits, act)
            loss, st = po.ppo_loss(logits, values, act, adv, logp.detach(), ret, clip=0.2, ent_coef=0.01, vf_coef=0.5,
                                   normalize=normalize)
            assert st["clip_fraction"] == 0.0
        loss.backward()
        grads.append(p.grad.clone())
    assert torch.allclose(grads[0], grads[1], rtol=1e-5, atol=1e-7)


def test_oracle_rmsprop_step_is_the_written_rule():
    d, a, rows = 4, 5, 300
    flat, obs, act, adv, ret = _batch(d, a, rows, 5)
    learner = ao.OracleA2C(d, a, params=flat.numpy(), lr=7e-4, max_grad_norm=0.5)
    p = flat.numpy().copy()
    sq = np.zeros_like(p)
    for _ in range(3):
        stats, g = learner.step(obs.numpy(), act.numpy(), adv.numpy(), ret.numpy())
        coef = min(0.5 / (stats["grad_norm"] + 1e-6), 1.0)
        p, sq = ao.rmsprop_reference(p, (g * np.float32(coef)).astype(np.float32), sq, lr=7e-4)
        np.testing.assert_allclose(learner.flat.detach().numpy(), p, rtol=1e-6, atol=1e-8)     # a few ulp of a 7e-4 step
        p = learner.flat.detach().numpy().copy()        # continue from torch's rounding


class _FakeEnv:
    def __init__(self, task):
        self.task_id = task
        self.observation_space, self.action_space = spaces_for(task)


def _fake_a2c(task="gridworld", d=4, a=5):
    m = types.SimpleNamespace(algorithm="a2c")
    m.env, m.obs_dim, m.n_actions, m.n_envs = _FakeEnv(task), d, a, 16
    m.params = torch.from_numpy(po.init_params(d, a, 4))
    m.sq_avg = torch.rand_like(m.params)
    m._opt_step, m.num_timesteps, m.n_updates, m.seed = 9, 720, 9, 4
    m.lr, m.n_steps, m.gamma, m.gae_lambda, m.ent_coef, m.vf_coef, m.max_grad_norm = 7e-4, 5, 0.99, 1.0, 0.0, 0.5, 0.5
    m.rms_prop_eps, m.normalize_advantage, m.verbose, m.tensorboard_log, m.mlp_impl = 1e-5, False, 0, None, "bf16"
    return m


def test_a2c_zip_round_trip_and_rmsprop_layout(tmp_path):
    m = _fake_a2c()
    path = str(tmp_path / "gridworld_policy_a.zip")
    sb3_zip.write_zip(path, m)
    with zipfile.ZipFile(path) as z:
        data = json.loads(z.read("data"))
        meta = json.loads(z.read("tmla.json"))
        opt = torch.load(__import__("io").BytesIO(z.read("policy.optimizer.pth")), weights_only=True)
    assert meta["algorithm"] == "a2c" and meta["opt_step"] == 9 and meta["hyper"]["rms_prop_eps"] == 1e-5
    # data: A2C's attributes, not PPO's
    for k in ("batch_size", "n_epochs", "clip_range", "clip_range_vf", "target_kl"):
        assert k not in data
    assert data["normalize_advantage"] is False and data["rms_prop_eps"] == 1e-5 and data["use_rms_prop"] is True
    assert data["n_steps"] == 5 and data["gae_lambda"] == 1.0 and data["learning_rate"] == 7e-4
    pk = data["policy_kwargs"]
    assert pk["net_arch"] == {"pi": [256, 256], "vf": [256, 256]} and pk["optimizer_kwargs"] == {"alpha": 0.99, "eps": 1e-5, "weight_decay": 0}
    unpickled = pickle.loads(base64.b64decode(pk[":serialized:"]))
    assert unpickled["optimizer_class"] is torch.optim.RMSprop
    # optimizer state: the layout of a real torch.optim.RMSprop over the 12 tensors after a step
    params = [torch.nn.Parameter(torch.randn(s)) for _, s in sb3_zip.param_layout(4, 5)]
    ref = torch.optim.RMSprop(params, lr=7e-4, alpha=0.99, eps=1e-5, weight_decay=0)
    sum(p.sum() for p in params).backward()
    ref.step()
    want = ref.state_dict()
    assert opt["param_groups"][0].keys() == want["param_groups"][0].keys()
    assert {k: v for k, v in opt["param_groups"][0].items() if k != "lr"} == {k: v for k, v in want["param_groups"][0].items() if k != "lr"}
    assert sorted(opt["state"]) == sorted(want["state"]) == list(range(12))
    for i, (name, shape) in enumerate(sb3_zip.param_layout(4, 5)):
        assert opt["state"][i].keys() == want["state"][i].keys()
        assert tuple(opt["state"][i]["square_avg"].shape) == tuple(shape)
        assert float(opt["state"][i]["step"]) == 9.0
    # read back
    r = sb3_zip.read_zip(path)
    assert r["optimizer"] == "rmsprop" and r["opt_step"] == 9
    assert torch.equal(r["params"], m.params) and torch.equal(r["sq_avg"], m.sq_avg)
    assert sb3_zip.zip_algorithm(path) == "a2c"


def test_algorithm_of_sb3_written_zips_comes_from_the_optimizer_state(tmp_path):
    """A zip without tmla.json (what SB3 writes): square_avg -> a2c, exp_avg -> ppo."""
    m = _fake_a2c()
    src = str(tmp_path / "a.zip")
    sb3_zip.write_zip(src, m)
    for name, want in (("sb3_a2c.zip", "a2c"),):
        dst = str(tmp_path / name)
        with zipfile.ZipFile(src) as zi, zipfile.ZipFile(dst, "w") as zo:
            for n in zi.namelist():
                if n != "tmla.json":
                    zo.writestr(n, zi.read(n))
        assert sb3_zip.zip_algorithm(dst) == want
        assert sb3_zip.read_zip(dst)["optimizer"] == "rmsprop"
    # an Adam state dict (PPO) written the same way
    ppo = types.SimpleNamespace(**{k: v for k, v in vars(m).items() if k not in ("algorithm", "sq_avg", "_opt_step")})
    ppo.m, ppo.v, ppo._adam_step, ppo.batch_size, ppo.n_epochs, ppo.clip_range = torch.rand_like(m.params), torch.rand_like(m.params), 3, 64, 10, 0.2
    dst = str(tmp_path / "p.zip")
    sb3_zip.write_zip(dst, ppo)
    stripped = str(tmp_path / "sb3_ppo.zip")
    with zipfile.ZipFile(dst) as zi, zipfile.ZipFile(stripped, "w") as zo:
        for n in zi.namelist():
            if n != "tmla.json":
                zo.writestr(n, zi.read(n))
    assert sb3_zip.zip_algorithm(stripped) == "ppo" and sb3_zip.zip_algorithm(dst) == "ppo"


def test_training_registers_a2c_with_sb3_defaults():
    from three_mlagents_b200.a2c import CudaA2C
    from three_mlagents_b200.registry import get_task
    from three_mlagents_b200.training import ALGORITHMS, _default_model_kwargs

    assert ALGORITHMS["a2c"] is CudaA2C and "dqn" not in ALGORITHMS
    kw = _default_model_kwargs("a2c", train_env=None, task=get_task("gridworld"), total_timesteps=1000, tensorboard_log="tb", verbose=0)
    assert kw == {"tensorboard_log": "tb", "verbose": 0, "learning_rate": 7e-4, "n_steps": 5, "gamma": 0.99, "gae_lambda": 1.0,
                  "ent_coef": 0.0, "vf_coef": 0.5, "max_grad_norm": 0.5, "rms_prop_eps": 1e-5, "use_rms_prop": True,
                  "normalize_advantage": False, "policy_kwargs": {"net_arch": {"pi": [256, 256], "vf": [256, 256]}}}


def test_dqn_still_has_no_backend(tmp_path, monkeypatch):
    from three_mlagents_b200.training import TrainConfig, train_task

    monkeypatch.chdir(tmp_path)
    with pytest.raises(ValueError, match="no CUDA backend"):
        train_task(TrainConfig("gridworld", algorithm="dqn"))
