"""Deterministic mode without a GPU: the CLI switch, the metadata field, the rejections and the scratch-size queries."""
import json
import types

import pytest
import torch


@pytest.fixture
def restore_flag():
    before = torch.are_deterministic_algorithms_enabled()
    yield
    torch.use_deterministic_algorithms(before)


def test_cli_deterministic_sets_the_torch_flag(monkeypatch, restore_flag, capsys):
    from three_mlagents_b200 import cli, training

    assert cli.build_parser().parse_args(["train", "basic", "--deterministic"]).deterministic is True
    assert cli.build_parser().parse_args(["train", "basic"]).deterministic is False
    seen = []

    def fake_train(config):
        seen.append(torch.are_deterministic_algorithms_enabled())
        return training.TrainResult("basic", "ppo", "r", "m.zip", "m.zip", "d", 0.0, 0.0, 1, 1, "meta.json")

    monkeypatch.setattr(training, "train_task", fake_train)
    torch.use_deterministic_algorithms(False)
    cli.main(["train", "basic", "-t", "10"])
    cli.main(["train", "basic", "-t", "10", "--deterministic"])
    assert seen == [False, True]


class _FakeModel:
    def __init__(self, policy, env, seed=1, **kw):
        self.deterministic = torch.are_deterministic_algorithms_enabled()
        self.num_timesteps = 0

    def learn(self, total_timesteps, callback=None, progress_bar=False):
        return self

    def save(self, path):
        open(str(path), "wb").close()

    def evaluate(self, n, seed, deterministic=True):
        import numpy as np

        return np.zeros(n), np.ones(n, dtype=np.int64)


@pytest.mark.parametrize("flag", [False, True])
def test_metadata_records_the_flag(tmp_path, monkeypatch, restore_flag, flag):
    from three_mlagents_b200 import training

    monkeypatch.chdir(tmp_path)
    env = types.SimpleNamespace(device_index=0, close=lambda: None)
    monkeypatch.setattr(training, "make_vector_env", lambda *a, **k: env)
    monkeypatch.setitem(training.ALGORITHMS, "ppo", _FakeModel)
    monkeypatch.setattr(torch.cuda, "get_device_name", lambda *a: "test device")
    torch.use_deterministic_algorithms(flag)
    res = training.train_task(training.TrainConfig("basic", algorithm="ppo", total_timesteps=10, verbose=0))
    assert json.loads((tmp_path / res.metadata_path).read_text())["deterministic"] is flag


def _env():
    return types.SimpleNamespace(obs_dim=6, n_actions=5, num_envs=4, device_index=0)


def test_deterministic_rejects_fp32_256(restore_flag):
    from three_mlagents_b200.ppo import CudaPPO

    torch.use_deterministic_algorithms(True)
    with pytest.raises(ValueError, match="mlp_impl='fp32'"):
        CudaPPO("MlpPolicy", _env(), mlp_impl="fp32")


def test_deterministic_rejects_data_parallel(restore_flag, monkeypatch):
    from three_mlagents_b200 import ppo
    from three_mlagents_b200.a2c import CudaA2C

    monkeypatch.setattr(ppo, "_dist", lambda: (None, 0, 2))
    torch.use_deterministic_algorithms(True)
    with pytest.raises(ValueError, match="world_size > 1"):
        ppo.CudaPPO("MlpPolicy", _env())
    with pytest.raises(ValueError, match="world_size > 1"):
        CudaA2C("MlpPolicy", _env())


def test_scratch_queries_never_shrink_as_rows_grow():
    from three_mlagents_b200 import native

    lib = native.lib
    for d, a in ((6, 5), (4, 4), (7, 3), (21, 3), (45, 3), (16, 5)):
        last = 0
        for rows in (1, 63, 64, 127, 128, 1000, 4737, 40000, 262144, 1 << 21):
            n = lib.tmla_det_scratch_bytes(d, 256, a, rows)
            assert n >= last and n % 4 == 0, (d, a, rows, n, last)
            last = n
        assert lib.tmla_det_scratch_bytes(d, 64, a, 1000) == 4 * 8 * 4        # small widths: loss statistics rows only
    assert lib.tmla_det_scratch_bytes(6, 256, 5, 0) == native.TMLA_EINVAL
    assert lib.tmla_adv_stats_det_scratch_bytes(1 << 20, 1 << 15) == 16 * 32 * 16
    assert lib.tmla_adv_stats_det_scratch_bytes(0, 1) == native.TMLA_EINVAL
