"""Deterministic mode (torch.use_deterministic_algorithms(True)): the update's sums run in a fixed order, so a run repeats
bit for bit.

Kernel level: every deterministic entry point is called twice on the same inputs with other work queued between the calls,
and the two results must be bit-identical.  Against the default atomic path they differ only by the order of fp32 sums:
  * gradient, per parameter tensor t ..... ||det_t - atomic_t|| <= 1e-5 ||atomic_t|| + 1e-6 ||atomic||
    (every value is the same set of fp32 partials added in another order: a relative error of a few fp32 ulps, 6e-8 each,
    times the depth of the sum, far below 1e-5; the absolute term covers tensors whose gradient nearly cancels)
  * loss statistics ....................... |det - atomic| <= 1e-5 max(1, |atomic|)
  * advantage sums (float64) .............. |det - atomic| <= 1e-12 max(1, |atomic|)
Against the float64 reference (oracle/ppo_oracle.py), the tolerances of tests/test_default_path_oracle_gpu.py.

End to end: each run twice with the flag on must give equal parameters (params_hash of the saved zip), equal optimizer state,
a byte-equal evaluations.npz and equal progress.jsonl rows apart from the time/* keys and rollout/ep_rew_mean (a logging value
summed with float atomics in the rollout kernel, DESIGN.md §8).  A second seed must give other parameters.
"""
import json
import os

import numpy as np
import pytest
import torch

from three_mlagents_b200 import ops, sb3_zip
from three_mlagents_b200.ppo import CudaPPO, orthogonal_init, params_hash
from three_mlagents_b200.training import TrainConfig, train_task
from three_mlagents_b200.vec_env import CudaVecEnv
from test_default_path_oracle_gpu import _check_grad, _check_stats, _oracle_grad, _tensor_slices

pytestmark = pytest.mark.gpu


@pytest.fixture
def det_flag():
    before = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True)
    yield
    torch.use_deterministic_algorithms(before)


def _inputs(d, a, total, rows, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    obs = torch.randn((total, d), device="cuda", generator=g)
    act = torch.randint(0, a, (total,), device="cuda", dtype=torch.int32, generator=g)
    adv = torch.randn(total, device="cuda", generator=g)
    logp = -torch.rand(total, device="cuda", generator=g) - 0.5
    ret = torch.randn(total, device="cuda", generator=g)
    idx = ops.permutation(seed + 3, 0, total // 64, 64)[:rows].contiguous()
    sums = ops.adv_stats(adv, idx, rows)
    return obs, act, adv, logp, ret, idx, sums


def _close_to_atomic(det, atomic, d, a, label):
    g, w = det.double().cpu(), atomic.double().cpu()
    wn = float(w.norm())
    for name, lo, hi in _tensor_slices(d, a):
        err, tn = float((g[lo:hi] - w[lo:hi]).norm()), float(w[lo:hi].norm())
        assert err <= 1e-5 * tn + 1e-6 * wn, (label, name, err, tn)


def _close_stats(det, atomic, label):
    d, w = det.double().cpu(), atomic.double().cpu()
    assert ((d - w).abs() <= 1e-5 * w.abs().clamp(min=1.0)).all(), (label, d, w)


FUSED_SHAPES = [("ball3d", 6, 5), ("gridworld", 4, 5), ("walljump", 4, 4), ("bicycle", 7, 3)]


@pytest.mark.parametrize("loss", ["ppo", "a2c"])
@pytest.mark.parametrize("task,d,a", FUSED_SHAPES)
def test_fused_batch_repeats_bit_for_bit(task, d, a, loss):
    total, rows = 64 * 1024, 40000                 # 313 tiles over 148 CTAs, a partial last tile
    obs, act, adv, logp, ret, idx, sums = _inputs(d, a, total, rows)
    params = orthogonal_init(d, a, 1).cuda()
    wpack = ops.mlp_pack(params, d, a)
    scratch = torch.empty(ops.fused_scratch_elems(d, a, rows, True), dtype=torch.bfloat16, device="cuda")

    def run(det, p=params, wp=wpack):
        if loss == "ppo":
            return ops.ppo_minibatch(p, wp, obs, d, a, act, adv, logp, ret, index=idx, rows=rows, adv_sums=sums, scratch=scratch,
                                     grads=torch.empty_like(p), stats=torch.zeros(8, device="cuda"), deterministic=det)
        return ops.a2c_batch(p, wp, obs, d, a, act, adv, ret, index=idx, rows=rows, adv_sums=sums, normalize=True, ent_coef=0.01,
                             scratch=scratch, grads=torch.empty_like(p), stats=torch.zeros(8, device="cuda"), deterministic=det)

    g1, s1 = run(True)
    other = orthogonal_init(d, a, 2).cuda()
    for _ in range(3):                             # other work between the two calls: the atomic path and other inputs
        run(False)
        run(True, other, ops.mlp_pack(other, d, a))
    g2, s2 = run(True)
    torch.cuda.synchronize()
    assert torch.equal(g1.view(torch.int32), g2.view(torch.int32)), f"{task} {loss}: gradients differ between two calls"
    assert torch.equal(s1.view(torch.int32), s2.view(torch.int32)), f"{task} {loss}: statistics differ between two calls"
    ga, sa = run(False)
    _close_to_atomic(g1, ga, d, a, f"{task} {loss}")
    _close_stats(s1, sa, f"{task} {loss}")
    if loss == "ppo" and task in ("ball3d", "bicycle"):
        sel = idx.long()
        want, tot, _, _ = _oracle_grad(params.cpu().numpy(), obs[sel].cpu().numpy(), act[sel].cpu().numpy(), adv[sel].cpu().numpy(),
                                       logp[sel].cpu().numpy(), ret[sel].cpu().numpy(), d, a, dtype=torch.float64)
        _check_grad(g1.cpu().numpy(), want, d, a, f"{task} deterministic")
        _check_stats(s1.cpu(), tot, f"{task} deterministic")


@pytest.mark.parametrize("task,d,a", [("basic", 21, 3), ("glider", 16, 5), ("brickbreak", 45, 3)])
def test_three_call_backward_repeats_bit_for_bit(task, d, a):
    total, rows = 32 * 1024, 20000
    obs, act, adv, logp, ret, idx, sums = _inputs(d, a, total, rows, seed=1)
    params = orthogonal_init(d, a, 1).cuda()
    wpack = ops.mlp_pack(params, d, a)
    logits, values, cache = ops.mlp_forward(params, obs, d, a, index=idx, rows=rows, wpack=wpack)
    part = torch.empty(ops.det_scratch_bytes(d, a, rows), dtype=torch.uint8, device="cuda")
    scratch = torch.empty(2 * rows * 256, dtype=torch.bfloat16, device="cuda")

    def run(det):
        dl, dv, st = ops.ppo_loss(logits, values, act, adv, logp, ret, index=idx, rows=rows, adv_sums=sums,
                                  partials=part if det else None)
        g = ops.mlp_backward(params, obs, d, a, cache, dl, dv, index=idx, rows=rows, scratch=scratch, wpack=wpack,
                             partials=part if det else None)
        return g, st

    g1, s1 = run(True)
    for _ in range(3):
        run(False)
    g2, s2 = run(True)
    torch.cuda.synchronize()
    assert torch.equal(g1.view(torch.int32), g2.view(torch.int32)), f"{task}: gradients differ between two calls"
    assert torch.equal(s1.view(torch.int32), s2.view(torch.int32)), f"{task}: statistics differ between two calls"
    ga, sa = run(False)
    _close_to_atomic(g1, ga, d, a, task)
    _close_stats(s1, sa, task)
    st_a = ops.a2c_loss(logits, values, act, adv, ret, index=idx, rows=rows, partials=part)[2]
    st_b = ops.a2c_loss(logits, values, act, adv, ret, index=idx, rows=rows, partials=part)[2]
    assert torch.equal(st_a, st_b)
    if task == "basic":
        sel = idx.long()
        want, tot, _, _ = _oracle_grad(params.cpu().numpy(), obs[sel].cpu().numpy(), act[sel].cpu().numpy(), adv[sel].cpu().numpy(),
                                       logp[sel].cpu().numpy(), ret[sel].cpu().numpy(), d, a, dtype=torch.float64)
        _check_grad(g1.cpu().numpy(), want, d, a, "basic deterministic three-call")
        _check_stats(s1.cpu(), tot, "basic deterministic three-call")


def test_adv_stats_batched_repeats_bit_for_bit():
    T, N, B = 128, 8192, 8192 * 4
    total = T * N
    g = torch.Generator(device="cuda").manual_seed(5)
    adv = torch.randn(total, device="cuda", generator=g) * 3 + 0.5
    perm = ops.permutation(7, 0, T, N)
    part = torch.empty(ops.adv_det_scratch_bytes(total, B), dtype=torch.uint8, device="cuda")
    s1 = ops.adv_stats_batched(adv, perm, total, B, partials=part).clone()
    ops.adv_stats_batched(adv, None, total, B)
    ops.adv_stats_batched(adv, None, total, B, partials=part)
    s2 = ops.adv_stats_batched(adv, perm, total, B, partials=part)
    assert torch.equal(s1, s2)
    sa = ops.adv_stats_batched(adv, perm, total, B)
    assert ((s1 - sa).abs() <= 1e-12 * sa.abs().clamp(min=1.0)).all()
    x = adv[perm.long()].double().cpu().numpy().reshape(-1, B)
    want = np.stack([x.sum(1), (x * x).sum(1), np.full(len(x), B)], 1)
    np.testing.assert_allclose(s1.cpu().numpy(), want, rtol=1e-12, atol=1e-9)
    one = ops.adv_stats_batched(adv, None, total, total, partials=part)     # A2C's single batch
    np.testing.assert_allclose(one[0, :2].cpu().numpy(), [x.sum(), (x * x).sum()], rtol=1e-12)
    assert float(one[0, 2]) == total


# ---------------------------------------------------------------------------------------------------------------- end to end
_DROP = ("rollout/ep_rew_mean",)


def _run(tmp_path, name, cfg: dict, model_kwargs=None):
    """train_task in its own working directory; -> (params hash, optimizer state, evaluations.npz bytes, progress rows)"""
    cwd = os.getcwd()
    d = tmp_path / name
    d.mkdir()
    os.chdir(d)
    try:
        res = train_task(TrainConfig(run_name="run", verbose=0, **cfg), model_kwargs=model_kwargs)
        z = sb3_zip.read_zip(res.model_path)
        state = {k: z[k].clone() for k in ("adam_m", "adam_v", "sq_avg") if isinstance(z.get(k), torch.Tensor)}
        state["step"] = (z["adam_step"], z["opt_step"])
        ev = (d / res.run_dir / "eval" / "evaluations.npz").read_bytes()
        rows = [json.loads(ln) for ln in (d / res.run_dir / "tb" / "progress.jsonl").read_text().splitlines()]
        rows = [{k: v for k, v in r.items() if not k.startswith("time/") and k not in _DROP} for r in rows]
        meta = json.loads((d / res.metadata_path).read_text())
        assert meta["deterministic"] is True
        return params_hash(z["params"]), state, ev, rows
    finally:
        os.chdir(cwd)


def _same(a, b, label):
    assert a[0] == b[0], f"{label}: parameters differ"
    assert a[1].keys() == b[1].keys()
    for k in a[1]:
        if isinstance(a[1][k], torch.Tensor):
            assert torch.equal(a[1][k].view(torch.int32), b[1][k].view(torch.int32)), f"{label}: optimizer state {k} differs"
        else:
            assert a[1][k] == b[1][k]
    assert a[2] == b[2], f"{label}: evaluations.npz differs"
    assert len(a[3]) == len(b[3]) > 0
    for ra, rb in zip(a[3], b[3]):
        assert json.dumps(ra, sort_keys=True) == json.dumps(rb, sort_keys=True), (label, ra, rb)


def test_basic_ppo_baseline_config_repeats(tmp_path, det_flag):
    cfg = dict(task_id="basic", algorithm="ppo", total_timesteps=25000, seed=1)
    a, b = _run(tmp_path, "a", cfg), _run(tmp_path, "b", cfg)
    _same(a, b, "basic ppo")
    c = _run(tmp_path, "c", dict(cfg, seed=2))
    assert c[0] != a[0], "a second seed gave the same parameters"


def test_ball3d_fused_ppo_repeats(tmp_path, det_flag):
    n, T = 4096, 64
    cfg = dict(task_id="ball3d", algorithm="ppo", total_timesteps=3 * n * T, n_envs=n, eval_freq=n * T, eval_episodes=32)
    kw = {"n_steps": T, "batch_size": n * T // 8, "n_epochs": 4}
    a, b = _run(tmp_path, "a", cfg, kw), _run(tmp_path, "b", cfg, kw)
    _same(a, b, "ball3d ppo")
    assert _run(tmp_path, "c", dict(cfg, seed=2), kw)[0] != a[0]


def test_gridworld_a2c_repeats(tmp_path, det_flag):
    n = 1024
    cfg = dict(task_id="gridworld", algorithm="a2c", total_timesteps=120 * n * 5, n_envs=n, eval_freq=40 * n * 5, eval_episodes=32)
    a, b = _run(tmp_path, "a", cfg), _run(tmp_path, "b", cfg)
    _same(a, b, "gridworld a2c")


def test_ball3d_net_arch_64_repeats(tmp_path, det_flag):
    n, T = 1024, 32
    cfg = dict(task_id="ball3d", algorithm="ppo", total_timesteps=4 * n * T, n_envs=n, eval_freq=2 * n * T, eval_episodes=32)
    kw = {"n_steps": T, "batch_size": n * T // 4, "n_epochs": 3, "policy_kwargs": {"net_arch": [64, 64]}}
    a, b = _run(tmp_path, "a", cfg, kw), _run(tmp_path, "b", cfg, kw)
    _same(a, b, "ball3d net_arch [64, 64]")


def test_rejections(det_flag, monkeypatch):
    env = CudaVecEnv("ball3d", 64, seed=1)
    try:
        with pytest.raises(ValueError, match="fp32"):
            CudaPPO("MlpPolicy", env, mlp_impl="fp32")
        CudaPPO("MlpPolicy", env, mlp_impl="fp32", policy_kwargs={"net_arch": [64, 64]})     # the small widths are deterministic
        from three_mlagents_b200 import ppo

        monkeypatch.setattr(ppo, "_dist", lambda: (None, 0, 2))
        with pytest.raises(ValueError, match="world_size"):
            CudaPPO("MlpPolicy", env)
    finally:
        env.close()
