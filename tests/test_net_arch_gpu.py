"""Policy widths 64 and 128 on the device (csrc/mlp_small.cu): the float32 kernels against float64 autograd, one PPO and one A2C
iteration against the SB3 restatement at those widths, the fused rollout graph against per-step calls, artifacts, learning.

Stated tolerances (those of the 256-wide float32 path, tests/test_ppo_gpu.py and DESIGN.md section 5):
  forward   logits / values within 2e-5 abs of float64 autograd on the same parameters
  backward  every parameter block within 2e-3 x its largest |gradient| (+1e-7) of float64 autograd; two calls bit-identical
  PPO       rollout values / log-probs 2e-5 abs, rewards after the timeout bootstrap 1e-4, GAE bit-exact on the device's own
            buffers, parameters after 2 epochs 2e-5 abs (as tests/test_trainer_gpu.py)
  A2C       values / log-probs 2e-5 abs, GAE bit-exact, batch gradient relative L2 error < 1e-4, RMSprop update cosine > 0.9999
The SB3 restatement (oracle/ppo_oracle.py) is written for width 256; these tests pin its module width H with monkeypatch.
"""
import numpy as np
import pytest
import torch

from oracle import a2c_oracle as ao, envs_oracle as eo, ppo_oracle as po

pytestmark = pytest.mark.gpu

SHAPES = [(21, 3), (6, 5), (4, 5), (4, 4), (45, 3), (7, 3), (16, 5)]


@pytest.fixture
def oracle_width(monkeypatch):
    def pin(h):
        monkeypatch.setattr(po, "H", h)
        # the restatement reads H at call time; were it ever captured elsewhere, these layouts would not match and every
        # comparison below would fail on shapes instead of passing at the wrong width
        assert po.param_shapes(6, 5)[2][1] == (h, h) and po.init_params(6, 5, 0).size == 2 * (6 * h + h + h * h + h) + 6 * h + 6
    return pin


@pytest.mark.parametrize("hidden", [64, 128])
@pytest.mark.parametrize("d,a", SHAPES)
def test_kernels_match_float64_autograd(hidden, d, a, oracle_width):
    from three_mlagents_b200 import ops

    oracle_width(hidden)
    rng = np.random.default_rng(hidden * 1000 + d * 10 + a)
    params = po.init_params(d, a, 3) + rng.normal(scale=0.02, size=po.init_params(d, a, 3).shape).astype(np.float32)
    for rows in (1, 1000, 5000):                           # 1000, 5000: not multiples of the 32-row tile
        buf_rows = rows * 2 + 7
        xbuf = rng.normal(size=(buf_rows, d)).astype(np.float32)
        index = rng.permutation(buf_rows)[:rows].astype(np.int32)
        P, X, I = torch.from_numpy(params).cuda(), torch.from_numpy(xbuf).cuda(), torch.from_numpy(index).cuda()
        logits, values, cache = ops.mlp_forward(P, X, d, a, index=I, hidden=hidden)
        flat = torch.from_numpy(params).double().requires_grad_(True)
        wl, wv = po.forward(flat, torch.from_numpy(xbuf[index]).double(), d, a)
        np.testing.assert_allclose(logits.cpu().numpy(), wl.detach().numpy(), rtol=0, atol=2e-5)
        np.testing.assert_allclose(values.cpu().numpy(), wv.detach().numpy(), rtol=0, atol=2e-5)
        # act_cache = NULL (inference): same outputs bit for bit
        l2, v2, c2 = ops.mlp_forward(P, X, d, a, index=I, hidden=hidden, keep_act=False)
        assert c2 is None and torch.equal(l2, logits) and torch.equal(v2, values)
        dl = rng.normal(size=(rows, a)).astype(np.float32) / rows
        dv = rng.normal(size=rows).astype(np.float32) / rows
        DL, DV = torch.from_numpy(dl).cuda(), torch.from_numpy(dv).cuda()
        grads = ops.mlp_backward(P, X, d, a, cache, DL, DV, index=I, hidden=hidden)
        again = ops.mlp_backward(P, X, d, a, cache, DL, DV, index=I, hidden=hidden)
        assert torch.equal(grads.view(torch.int32), again.view(torch.int32))          # fixed-order reduction
        ((wl * torch.from_numpy(dl).double()).sum() + (wv * torch.from_numpy(dv).double()).sum()).backward()
        want, got, p = flat.grad.numpy(), grads.cpu().numpy().astype(np.float64), 0
        for name, shape in po.param_shapes(d, a):
            k = int(np.prod(shape))
            scale = np.abs(want[p:p + k]).max() + 1e-12
            assert np.abs(got[p:p + k] - want[p:p + k]).max() <= 2e-3 * scale + 1e-7, (rows, name)
            p += k
        # value-only pass with a device-side row count below `rows` (the timeout-bootstrap forward)
        cnt = torch.tensor([max(1, rows // 3)], dtype=torch.int32, device="cuda")
        _, v3, _ = ops.mlp_forward(P, X, d, a, index=I, rows_dev=cnt, want_logits=False, hidden=hidden, keep_act=False,
                                   values=torch.full((rows,), 7.0, device="cuda"))
        k = int(cnt.item())
        assert torch.equal(v3[:k], values[:k]) and bool((v3[k:] == 7.0).all())


@pytest.mark.parametrize("hidden", [64, 128])
@pytest.mark.parametrize("task,n,T,B", [("ball3d", 64, 32, 256), ("gridworld", 96, 120, 1000), ("basic", 50, 60, 512)])
def test_one_ppo_iteration_matches_sb3_restatement(hidden, task, n, T, B, oracle_width):
    from three_mlagents_b200.ppo import CudaPPO
    from three_mlagents_b200.vec_env import CudaVecEnv

    oracle_width(hidden)
    env = CudaVecEnv(task, n, seed=3)
    model = CudaPPO("MlpPolicy", env, seed=3, n_steps=T, batch_size=B, n_epochs=2, ent_coef=0.01,
                    policy_kwargs={"net_arch": [hidden, hidden]})
    assert model.hidden == hidden and model.mlp_impl == "fp32" and not model.fused_update
    d, a = env.obs_dim, env.n_actions
    p0 = model.params.cpu().numpy().copy()
    np.testing.assert_array_equal(p0, po.init_params(d, a, 3))
    ora_env = eo.OracleVecEnv(task, n, seed=3)
    model.collect_rollouts()
    torch.cuda.synchronize()
    obs, act = model.obs.cpu().numpy(), model.act.cpu().numpy()
    rew, done = model.rew.cpu().numpy(), model.done.cpu().numpy().astype(bool)
    val, logp = model.val.cpu().numpy(), model.logp.cpu().numpy()
    learner = po.OraclePPO(d, a, params=p0)
    tol = 1e-5 if task == "ball3d" else 0.0
    cur = eo.observe(task, ora_env.state)
    want_rew = np.zeros((T, n), np.float32)
    n_boot = 0
    for t in range(T):
        assert np.abs(obs[t] - cur).max() <= tol, t
        logits, values = learner.evaluate(obs[t])
        np.testing.assert_allclose(val[t], values.numpy(), rtol=0, atol=2e-5)
        lp, _ = po.categorical(logits, torch.from_numpy(act[t]))
        np.testing.assert_allclose(logp[t], lp.numpy(), rtol=0, atol=2e-5)
        cur, r, dn, tl, info = ora_env.step(act[t])
        assert np.array_equal(done[t], dn)
        if tl.any():
            _, tv = learner.evaluate(info["terminal_obs"][tl])
            r = r.copy()
            r[tl] = r[tl] + np.float32(0.99) * tv.numpy()
            n_boot += int(tl.sum())
        want_rew[t] = r
    np.testing.assert_allclose(rew, want_rew, rtol=0, atol=1e-4)
    assert int(model.trunc_count.item()) == n_boot
    if task != "ball3d":
        assert n_boot > 0
    _, last_v = learner.evaluate(obs[T])
    np.testing.assert_allclose(model.last_values.cpu().numpy(), last_v.numpy(), rtol=0, atol=2e-5)
    adv_dev, ret_dev = model.adv.cpu().numpy(), model.ret.cpu().numpy()
    w_adv, _ = po.gae(rew, val, done, model.last_values.cpu().numpy(), 0.99, 0.95)
    assert np.array_equal(adv_dev.view(np.uint32), w_adv.view(np.uint32))
    n_mb = model.train()
    torch.cuda.synchronize()
    total = T * n
    fo, fl = obs[:T].reshape(total, d), (lambda x: x.reshape(total))
    steps = 0
    for epoch in range(2):
        perm = po.permutation(3, epoch, T, n)
        for s in range(0, total, B):
            idx = perm[s:s + B]
            stats, _ = learner.minibatch_step(fo[idx], fl(act)[idx], fl(adv_dev)[idx], fl(logp)[idx], fl(ret_dev)[idx])
            steps += 1
    assert steps == n_mb
    got, want = model.params.cpu().numpy(), learner.flat.detach().numpy()
    assert np.abs(want - p0).max() > 1e-4
    np.testing.assert_allclose(got, want, rtol=0, atol=2e-5)
    last = model.stats.cpu().numpy()
    assert abs(last[5] - stats["loss"]) <= 1e-4 * max(1.0, abs(stats["loss"]))
    env.close()


@pytest.mark.parametrize("task,n,T", [("ball3d", 256, 5), ("gridworld", 300, 8)])
def test_one_a2c_iteration_matches_oracle(task, n, T, oracle_width):
    from three_mlagents_b200 import ops
    from three_mlagents_b200.a2c import CudaA2C
    from three_mlagents_b200.vec_env import CudaVecEnv

    oracle_width(64)
    env = CudaVecEnv(task, n, seed=4)
    model = CudaA2C("MlpPolicy", env, seed=4, n_steps=T, ent_coef=0.01, policy_kwargs={"net_arch": dict(pi=[64, 64], vf=[64, 64])})
    d, a = env.obs_dim, env.n_actions
    assert model.hidden == 64 and model.mlp_impl == "fp32" and not model.fused_update      # the three-call branch
    p0 = model.params.cpu().numpy().copy()
    np.testing.assert_array_equal(p0, po.init_params(d, a, 4))
    ora_env = eo.OracleVecEnv(task, n, seed=4)
    model.collect_rollouts()
    torch.cuda.synchronize()
    obs, act = model.obs.cpu().numpy(), model.act.cpu().numpy()
    rew, done = model.rew.cpu().numpy(), model.done.cpu().numpy().astype(bool)
    val, logp = model.val.cpu().numpy(), model.logp.cpu().numpy()
    learner = ao.OracleA2C(d, a, params=p0, ent_coef=0.01)
    cur = eo.observe(task, ora_env.state)
    for t in range(T):
        assert np.abs(obs[t] - cur).max() <= (1e-5 if task == "ball3d" else 0.0), t
        logits, values = learner.evaluate(obs[t])
        np.testing.assert_allclose(val[t], values.numpy(), rtol=0, atol=2e-5)
        lp, _ = po.categorical(logits, torch.from_numpy(act[t]))
        np.testing.assert_allclose(logp[t], lp.numpy(), rtol=0, atol=2e-5)
        cur, _, dn, _, _ = ora_env.step(act[t])
        assert np.array_equal(done[t], dn)
    adv_dev, ret_dev = model.adv.cpu().numpy(), model.ret.cpu().numpy()
    w_adv, w_ret = po.gae(rew, val, done, model.last_values.cpu().numpy(), 0.99, 1.0)
    assert np.array_equal(adv_dev.view(np.uint32), w_adv.view(np.uint32))
    assert np.array_equal(ret_dev.view(np.uint32), w_ret.view(np.uint32))
    total = T * n
    fo, fl = obs[:T].reshape(total, d), (lambda x: x.reshape(total))
    g_want, _ = learner.gradient(fo, fl(act), fl(adv_dev), fl(ret_dev))
    flat_obs = model.obs[:T].reshape(total, d)
    lg, vl, cache = ops.mlp_forward(model.params, flat_obs, d, a, rows=total, hidden=64)
    dl, dv, _ = ops.a2c_loss(lg, vl, model.act, model.adv, model.ret, ent_coef=0.01)
    g_dev = ops.mlp_backward(model.params, flat_obs, d, a, cache, dl, dv, rows=total, hidden=64)
    torch.cuda.synchronize()
    gd, gw = torch.from_numpy(g_dev.cpu().numpy()).double(), torch.from_numpy(g_want).double()
    rel = float((gd - gw).norm() / gw.norm())
    print(f"{task}: A2C gradient at width 64 vs oracle: relative L2 error {rel:.2e}")
    assert rel < 1e-4
    assert model.train() == 1
    torch.cuda.synchronize()
    learner.step(fo, fl(act), fl(adv_dev), fl(ret_dev))
    got, want = model.params.cpu().numpy(), learner.flat.detach().numpy()
    du_dev, du_ora = torch.from_numpy(got - p0).double(), torch.from_numpy(want - p0).double()
    cos_u = float(torch.nn.functional.cosine_similarity(du_dev, du_ora, dim=0))
    print(f"{task}: parameters after one RMSprop step: update cosine {cos_u:.7f}, max |dp| {np.abs(got - want).max():.2e}")
    # RMSprop's first step moves a coordinate by up to lr / sqrt(1 - alpha) = 7e-3 whatever its gradient's size: a coordinate
    # whose gradient is at rounding level may move the other way, so the per-coordinate bound is 2 x that step
    assert cos_u > 0.9999 and np.abs(got - want).max() <= 2 * 7e-4 / np.sqrt(0.01) + 1e-6
    env.close()


@pytest.mark.parametrize("task,n,T", [("ball3d", 512, 32), ("gridworld", 300, 120)])
def test_fused_rollout_equals_per_step_rollout_at_width_64(task, n, T):
    from three_mlagents_b200.ppo import CudaPPO
    from three_mlagents_b200.vec_env import CudaVecEnv

    models = [CudaPPO("MlpPolicy", CudaVecEnv(task, n, seed=7), seed=7, n_steps=T, batch_size=n * T // 2, n_epochs=1,
                      ent_coef=0.01, rollout_impl=impl, policy_kwargs={"net_arch": [64, 64]}) for impl in ("fused", "steps")]
    fused, steps = models
    for it in range(3):
        for m in models:
            m.collect_rollouts()
        torch.cuda.synchronize()
        # (the timeout records trunc_index / trunc_values are appended in atomic order; their effect is in `rew`)
        for name in ("obs", "act", "logp", "rew", "val", "done", "last_values", "adv", "ret"):
            x, y = getattr(fused, name), getattr(steps, name)
            assert torch.equal(x.view(torch.uint8), y.view(torch.uint8)), (task, it, name)
        assert int(fused.trunc_count.item()) == int(steps.trunc_count.item())
        if it == 1:                              # deterministic update: both models stay bit-identical through it
            for m in models:
                m.train()
            torch.cuda.synchronize()
            assert torch.equal(fused.params.view(torch.int32), steps.params.view(torch.int32))
    if task == "gridworld":
        assert int(fused.trunc_count.item()) > 0
    for m in models:
        m.env.close()


def test_train_save_load_evaluate_at_width_64(tmp_path):
    from three_mlagents_b200.ppo import CudaPPO
    from three_mlagents_b200.vec_env import CudaVecEnv

    env = CudaVecEnv("basic", 256, seed=1)
    model = CudaPPO("MlpPolicy", env, seed=1, n_steps=64, batch_size=2048, n_epochs=4, ent_coef=0.01,
                    policy_kwargs={"net_arch": [64, 64]})
    model.learn(256 * 64 * 4)
    path = tmp_path / "basic_policy_w64.zip"
    model.save(path)
    loaded = CudaPPO.load(path)
    assert loaded.hidden == 64 and torch.equal(loaded.params, model.params) and torch.equal(loaded.m, model.m)
    obs = np.random.default_rng(0).normal(size=(64, 21)).astype(np.float32)
    a0, _ = model.predict(obs, deterministic=True)
    a1, _ = loaded.predict(obs, deterministic=True)
    assert np.array_equal(a0, a1)
    r0, _ = model.evaluate(32, seed=11)
    r1, _ = loaded.evaluate(32, seed=11)
    assert np.array_equal(r0, r1)
    env.close(); loaded.env.close()


def test_stock_sb3_default_zip_evaluates_and_predicts(tmp_path, monkeypatch):
    from test_net_arch_cpu import write_stock_sb3_zip
    from three_mlagents_b200 import cli
    from three_mlagents_b200.training import evaluate_model, predict_action

    monkeypatch.chdir(tmp_path)
    path = str(tmp_path / "sb3_default.zip")
    write_stock_sb3_zip(path, 4, 5)
    res = evaluate_model("gridworld", path, episodes=16)
    assert res["episodes"] == 16 and np.isfinite(res["mean_reward"])
    act = predict_action("gridworld", np.zeros(4, np.float32), path)
    assert isinstance(act, int) and 0 <= act < 5
    assert cli.main(["evaluate", "gridworld", path, "--episodes", "8"]) in (0, None)


def test_train_task_a2c_records_width_128(tmp_path, monkeypatch):
    import json
    import zipfile

    from three_mlagents_b200.training import TrainConfig, train_task

    monkeypatch.chdir(tmp_path)
    res = train_task(TrainConfig("gridworld", algorithm="a2c", total_timesteps=64 * 5 * 20, n_envs=64, eval_episodes=8,
                                 eval_freq=10**12, verbose=0, run_name="w128"),
                     model_kwargs={"policy_kwargs": {"net_arch": [128, 128]}})
    with zipfile.ZipFile(res.model_path) as z:
        data = json.loads(z.read("data"))
    assert data["policy_kwargs"]["net_arch"] == {"pi": [128, 128], "vf": [128, 128]}
    assert np.isfinite(res.mean_reward)


@pytest.mark.parametrize("task,steps,episodes", [("ball3d", 40_000_000, 256), ("gridworld", 80_000_000, 8192)])
def test_ppo_at_width_64_reaches_registry_reward_threshold(task, steps, episodes, tmp_path, monkeypatch):
    """As tests/test_training_gpu.py's threshold test (same seeds, budget and rollout geometry), with net_arch [64, 64]."""
    from three_mlagents_b200.registry import get_task
    from three_mlagents_b200.training import TrainConfig, train_task

    monkeypatch.chdir(tmp_path)
    thr = get_task(task).reward_threshold
    seen = []
    for seed in (1, 2, 3):
        res = train_task(TrainConfig(task, total_timesteps=steps, algorithm="ppo", n_envs=4096, eval_episodes=episodes,
                                     eval_freq=10**12, verbose=0, seed=seed, run_name=f"w64_{seed}"),
                         model_kwargs={"n_steps": 128, "batch_size": 32768, "policy_kwargs": {"net_arch": [64, 64]}})
        seen.append(res.mean_reward)
        print(f"{task} net_arch [64, 64], seed {seed}, {steps} steps: eval mean reward {res.mean_reward:.4f} (threshold {thr})")
        if res.mean_reward >= thr:
            return
    raise AssertionError(f"no run reached {thr}; eval mean rewards per seed: {seen}")


def test_partial_last_minibatch_stays_inside_its_scratch():
    """1000 envs x 128 steps in minibatches of 10 000 rows: the epoch's last minibatch has 8000 rows.  Its backward, run on the
    scratch sized for 10 000 rows, must not write past that size (canary), and a whole update must leave the per-minibatch
    advantage statistics (allocated right after the scratch) as computed."""
    from three_mlagents_b200 import native, ops
    from three_mlagents_b200.ppo import CudaPPO, orthogonal_init
    from three_mlagents_b200.vec_env import CudaVecEnv

    d, a, hidden, B, rows = 6, 5, 64, 10_000, 8_000
    size = native.lib.tmla_mlp_backward_scratch(d, hidden, a, B)
    assert native.lib.tmla_mlp_backward_scratch(d, hidden, a, rows) <= size
    g = torch.Generator(device="cuda").manual_seed(1)
    params = orthogonal_init(d, a, 1, hidden=hidden).cuda()
    x = torch.randn((rows, d), device="cuda", generator=g)
    _, _, cache = ops.mlp_forward(params, x, d, a, hidden=hidden)
    dl, dv = torch.randn((rows, a), device="cuda", generator=g) / rows, torch.randn(rows, device="cuda", generator=g) / rows
    buf = torch.full((size + 4096,), 12345.0, device="cuda")
    grads = ops.mlp_backward(params, x, d, a, cache, dl, dv, scratch=buf[:size], hidden=hidden)
    ref = ops.mlp_backward(params, x, d, a, cache, dl, dv, hidden=hidden)
    torch.cuda.synchronize()
    assert bool((buf[size:] == 12345.0).all()) and torch.equal(grads, ref)

    env = CudaVecEnv("ball3d", 1000, seed=2)
    model = CudaPPO("MlpPolicy", env, seed=2, n_steps=128, batch_size=B, n_epochs=2, ent_coef=0.01,
                    policy_kwargs={"net_arch": [hidden, hidden]})
    model.collect_rollouts()
    model.train()
    torch.cuda.synchronize()
    assert model.scratch_mb.numel() == size and torch.isfinite(model.params).all()
    fresh = ops.adv_stats_batched(model.adv, model.perm, 128 * 1000, B)
    assert torch.allclose(model.adv_sums, fresh, rtol=1e-12, atol=0)
    env.close()
