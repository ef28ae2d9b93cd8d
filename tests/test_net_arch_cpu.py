"""Policy widths 64 and 128 (net_arch [H, H]) without a GPU: net_arch parsing, parameter counts of the C ABI, the SB3 state-dict
layout at every width, and a zip laid out the way stock Stable-Baselines3 writes one with its default arguments (64 wide)."""
import io
import json
import zipfile

import numpy as np
import pytest
import torch

from oracle import ppo_oracle as po
from three_mlagents_b200 import sb3_zip
from three_mlagents_b200.ppo import orthogonal_init, parse_net_arch

TASK_SHAPES = {"basic": (21, 3), "ball3d": (6, 5), "gridworld": (4, 5), "push": (4, 5), "walljump": (4, 4), "brickbreak": (45, 3),
               "bicycle": (7, 3), "glider": (16, 5)}


@pytest.mark.parametrize("pk,width", [
    (None, 256), ({}, 256), ({"net_arch": [64, 64]}, 64), ({"net_arch": (128, 128)}, 128), ({"net_arch": [256, 256]}, 256),
    ({"net_arch": {"pi": [64, 64], "vf": [64, 64]}}, 64), ({"net_arch": {"pi": [128, 128], "vf": [128, 128]}}, 128),
    ({"net_arch": {"pi": [256, 256], "vf": [256, 256]}}, 256),
    ({"net_arch": [64, 64], "activation_fn": torch.nn.Tanh, "ortho_init": True}, 64)])
def test_accepted_net_arch_forms(pk, width):
    assert parse_net_arch(pk) == width


@pytest.mark.parametrize("pk", [
    {"net_arch": [64, 128]}, {"net_arch": [64]}, {"net_arch": [64, 64, 64]}, {"net_arch": [96, 96]}, {"net_arch": [512, 512]},
    {"net_arch": {"pi": [64, 64], "vf": [128, 128]}}, {"net_arch": {"pi": [64, 64]}}, {"net_arch": 64},
    {"net_arch": [64, 64], "activation_fn": torch.nn.ReLU}, {"net_arch": [64, 64], "ortho_init": False},
    {"net_arch": [64, 64], "share_features_extractor": False}, {"log_std_init": 0.0}])
def test_rejected_net_arch_forms(pk):
    with pytest.raises(ValueError, match="supported"):
        parse_net_arch(pk)


@pytest.mark.parametrize("hidden", [64, 128])
def test_num_params_matches_the_state_dict_layout(hidden):
    from three_mlagents_b200 import native, ops

    for task, (d, a) in TASK_SHAPES.items():
        want = sum(int(np.prod(s)) for _, s in sb3_zip.param_layout(d, a, hidden))
        assert native.lib.tmla_mlp_num_params(d, hidden, a) == want == ops.num_params(d, a, hidden=hidden), task
        assert native.lib.tmla_ppo_minibatch_supported(d, hidden, a) == 0          # the fused bf16 update is 256-only
    assert native.lib.tmla_mlp_num_params(6, 64, 5) == 9606      # 2*(6*64+64+64*64+64) + 5*64+5 + 64+1
    for bad in (96, 512, 0):
        assert native.lib.tmla_mlp_num_params(6, bad, 5) == native.TMLA_EINVAL
        assert b"64, 128 or 256" in native.lib.tmla_last_error()
    with pytest.raises(ValueError):
        ops.num_params(6, 5, hidden=96)


@pytest.mark.parametrize("hidden", [64, 128])
def test_state_dict_round_trip(hidden):
    for d, a in ((6, 5), (4, 5), (21, 3), (45, 3)):
        flat = orthogonal_init(d, a, 2, hidden=hidden)
        sd = sb3_zip.flat_to_state_dict(flat, d, a, hidden)
        assert sd["mlp_extractor.policy_net.2.weight"].shape == (hidden, hidden) and sd["action_net.weight"].shape == (a, hidden)
        assert sb3_zip.hidden_width(sd) == hidden
        assert torch.equal(sb3_zip.state_dict_to_flat(sd, d, a, hidden), flat)
        with pytest.raises(ValueError):
            sb3_zip.state_dict_to_flat(sd, d, a)                                    # a 256-wide layout does not fit


def test_oracle_init_matches_at_width_64(monkeypatch):
    """The SB3 restatement at H = 64 (its module width pinned for this test) draws the same orthogonal init."""
    monkeypatch.setattr(po, "H", 64)
    for d, a in ((6, 5), (21, 3)):
        assert np.array_equal(po.init_params(d, a, 5), orthogonal_init(d, a, 5, hidden=64).numpy())
        assert sb3_zip.param_layout(d, a, 64) == po.param_shapes(d, a)


def write_stock_sb3_zip(path, d=4, a=5, seed=9):
    """A zip with only the members stock SB3 writes, 64 wide, with the empty policy_kwargs of PPO("MlpPolicy", env)."""
    flat = orthogonal_init(d, a, seed, hidden=64)
    with zipfile.ZipFile(path, "w") as z:
        z.writestr("data", json.dumps({"policy_kwargs": {}, "learning_rate": 3e-4, "n_steps": 2048, "gamma": 0.99,
                                       "num_timesteps": 4096, "seed": 3}))
        buf = io.BytesIO(); torch.save(sb3_zip.flat_to_state_dict(flat, d, a, 64), buf); z.writestr("policy.pth", buf.getvalue())
        z.writestr("_stable_baselines3_version", "2.9.0")
    return flat


def test_reads_a_stock_sb3_default_zip(tmp_path):
    path = str(tmp_path / "sb3_default.zip")
    flat = write_stock_sb3_zip(path)
    z = sb3_zip.read_zip(path)
    assert z["hidden"] == 64 and (z["obs_dim"], z["n_actions"]) == (4, 5) and z["meta"] is None
    assert torch.equal(z["params"], flat) and z["data"]["policy_kwargs"] == {}


@pytest.mark.parametrize("algo", ["ppo", "a2c"])
def test_written_zip_records_the_width(tmp_path, algo):
    import types

    from three_mlagents_b200.spaces import spaces_for

    d, a, hidden = 6, 5, 128
    m = types.SimpleNamespace(algorithm=algo, hidden=hidden, obs_dim=d, n_actions=a, n_envs=4, seed=1, verbose=0,
                              tensorboard_log=None, mlp_impl="fp32", num_timesteps=10, n_updates=1, lr=3e-4, n_steps=8,
                              batch_size=16, n_epochs=2, gamma=0.99, gae_lambda=0.95, clip_range=0.2, ent_coef=0.0,
                              vf_coef=0.5, max_grad_norm=0.5, normalize_advantage=True, rms_prop_eps=1e-5,
                              _adam_step=3, _opt_step=3)
    m.env = types.SimpleNamespace(task_id="ball3d")
    m.env.observation_space, m.env.action_space = spaces_for("ball3d")
    m.params = orthogonal_init(d, a, 1, hidden=hidden)
    m.m, m.v, m.sq_avg = torch.rand_like(m.params), torch.rand_like(m.params), torch.rand_like(m.params)
    path = str(tmp_path / "w.zip")
    sb3_zip.write_zip(path, m)
    with zipfile.ZipFile(path) as zf:
        data = json.loads(zf.read("data"))
        meta = json.loads(zf.read("tmla.json"))
    assert data["policy_kwargs"]["net_arch"] == {"pi": [hidden, hidden], "vf": [hidden, hidden]}
    assert meta["net_arch"] == {"pi": [hidden, hidden], "vf": [hidden, hidden]}
    z = sb3_zip.read_zip(path)
    assert z["hidden"] == hidden and torch.equal(z["params"], m.params)
    if algo == "a2c":
        assert z["optimizer"] == "rmsprop" and torch.equal(z["sq_avg"], m.sq_avg)
    else:
        assert z["optimizer"] == "adam" and torch.equal(z["adam_m"], m.m) and torch.equal(z["adam_v"], m.v)


@pytest.mark.parametrize("hidden", [64, 128])
def test_backward_scratch_never_shrinks_with_more_rows(hidden):
    """Scratch sized for a minibatch of B rows must also hold the backward of every shorter batch (an epoch's last minibatch),
    so the required size may not decrease as rows grow."""
    from three_mlagents_b200 import native

    f = native.lib.tmla_mlp_backward_scratch
    P = native.lib.tmla_mlp_num_params(6, hidden, 5)
    prev = 0
    for rows in range(1, 300_001):
        n = f(6, hidden, 5, rows)
        assert n >= prev and n % P == 0 and n // P <= 148, rows
        prev = n
    assert f(6, hidden, 5, 10_000) >= f(6, hidden, 5, 8_000)      # 1000 envs x 128 steps, batch 10 000: last minibatch 8000


@pytest.mark.parametrize("hidden", [64, 128])
def test_backward_scratch_rejects_empty_batches(hidden):
    from three_mlagents_b200 import native, ops

    for rows in (0, -5):
        assert native.lib.tmla_mlp_backward_scratch(6, hidden, 5, rows) == native.TMLA_EINVAL
        assert b"rows" in native.lib.tmla_last_error()
    with pytest.raises(ValueError, match="rows"):
        ops.mlp_backward(torch.zeros(ops.num_params(6, 5, hidden=hidden)), torch.zeros((0, 6)), 6, 5, None, None, None, rows=0,
                         hidden=hidden)
