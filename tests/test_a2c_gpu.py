"""A2C on the device: the fused A2C batch against the three-call bf16 path and fp32, the one-launch clip + RMSprop step
against torch.optim.RMSprop, one whole A2C iteration against the CPU restatement (oracle/a2c_oracle.py), and the training /
CLI / websocket surface for every CUDA task.

Stated tolerances (as test_train_fused_gpu.py / test_default_path_oracle_gpu.py for the PPO kernels):
  * head outputs fused vs unfused bf16: 5e-3 abs; loss statistics 1e-4 abs/rel
  * gradients fused vs unfused bf16: cosine > 0.9999, relative L2 error < 1e-2; vs fp32: cosine > 0.999, rel < 5e-2
  * RMSprop step vs torch.optim.RMSprop on the same clipped gradient: square_avg within 4 ulp; new parameters within 4 ulp of
    the update + 2 ulp of the parameter (observed maximum printed)
  * rollout values / log-probs vs the oracle 3e-2; GAE (lambda = 1) bit-exact; batch gradient cosine > 0.999, rel < 5e-2
"""
import json
import os

import numpy as np
import pytest
import torch

from oracle import a2c_oracle as ao, envs_oracle as eo, ppo_oracle as po

pytestmark = pytest.mark.gpu

TASKS = ["basic", "ball3d", "gridworld", "push", "walljump", "brickbreak", "bicycle", "glider"]


def _model(task, n, T, seed=5, **kw):
    from three_mlagents_b200.a2c import CudaA2C
    from three_mlagents_b200.vec_env import CudaVecEnv

    env = CudaVecEnv(task, n, seed=seed)
    m = CudaA2C("MlpPolicy", env, seed=seed, n_steps=T, ent_coef=0.01, **kw)
    return env, m


@pytest.mark.parametrize("task,n,T,normalize", [("ball3d", 512, 5, False), ("gridworld", 300, 8, True), ("walljump", 400, 5, False),
                                                ("bicycle", 4096, 5, True), ("push", 65536, 5, False)])
def test_fused_a2c_batch_matches_three_call_paths(task, n, T, normalize):
    from three_mlagents_b200 import ops

    env, m = _model(task, n, T)
    with torch.no_grad():
        g = torch.Generator(device=m.params.device).manual_seed(77)
        m.params += 0.05 * torch.randn(m.params.shape, device=m.params.device, generator=g)
    m._repack()
    m.collect_rollouts()
    d, a, rows = env.obs_dim, env.n_actions, n * T
    obs = m.obs[:T].reshape(rows, d)
    sums = ops.adv_stats(m.adv, None, rows) if normalize else None
    l16, v16, c16 = ops.mlp_forward(m.params, obs, d, a, rows=rows, wpack=m.wpack)
    dl, dv, st_ref = ops.a2c_loss(l16, v16, m.act, m.adv, m.ret, adv_sums=sums, normalize=normalize, ent_coef=0.01)
    g_ref = ops.mlp_backward(m.params, obs, d, a, c16, dl, dv, rows=rows, wpack=m.wpack).clone()
    l32, v32, c32 = ops.mlp_forward(m.params, obs, d, a, rows=rows)
    dl32, dv32, _ = ops.a2c_loss(l32, v32, m.act, m.adv, m.ret, adv_sums=sums, normalize=normalize, ent_coef=0.01)
    g32 = ops.mlp_backward(m.params, obs, d, a, c32, dl32, dv32, rows=rows)
    logits = torch.full((rows, a), float("nan"), device="cuda")
    values = torch.full((rows,), float("nan"), device="cuda")
    g_f, st_f = ops.a2c_batch(m.params, m.wpack, obs, d, a, m.act, m.adv, m.ret, rows=rows, adv_sums=sums, normalize=normalize,
                              ent_coef=0.01, logits=logits, values=values)
    torch.cuda.synchronize()
    assert float((logits - l16).abs().max()) < 5e-3 and float((values - v16).abs().max()) < 5e-3
    assert torch.allclose(st_f[:6], st_ref[:6], rtol=1e-4, atol=1e-4), (st_f, st_ref)
    assert float(st_f[3]) == 0.0 and float(st_f[4]) == 0.0           # approx_kl / clip_fraction: not A2C quantities
    # the three-call loss against the fp32 path's own statistics and the oracle's loss on the same head outputs
    _, want = ao.a2c_loss(l32.cpu(), v32.cpu(), m.act.reshape(-1).long().cpu(), m.adv.reshape(-1).cpu(), m.ret.reshape(-1).cpu(),
                          ent_coef=0.01, normalize=normalize)
    assert abs(float(st_f[0]) - want["policy_loss"]) <= 2e-2 * max(1.0, abs(want["policy_loss"]))
    cos = float(torch.nn.functional.cosine_similarity(g_f, g_ref, dim=0))
    rel = float((g_f - g_ref).norm() / g_ref.norm())
    cos32 = float(torch.nn.functional.cosine_similarity(g_f, g32, dim=0))
    rel32 = float((g_f - g32).norm() / g32.norm())
    print(f"{task} rows={rows}: fused A2C vs bf16 cos {cos:.7f} rel {rel:.5f}; vs fp32 cos {cos32:.6f} rel {rel32:.4f}")
    assert cos > 0.9999 and rel < 1e-2
    assert cos32 > 0.999 and rel32 < 5e-2
    env.close()


@pytest.mark.parametrize("with_wpack", [False, True])
def test_rmsprop_kernel_matches_torch_rmsprop(with_wpack):
    from three_mlagents_b200 import ops
    from three_mlagents_b200.ppo import orthogonal_init

    d, a = 6, 5
    p = orthogonal_init(d, a, 3).cuda()
    sq = torch.zeros_like(p)
    ref = torch.nn.Parameter(p.clone())
    opt = torch.optim.RMSprop([ref], lr=7e-4, alpha=0.99, eps=1e-5, weight_decay=0)
    wpack = ops.mlp_pack(p, d, a) if with_wpack else None
    norm_out = torch.zeros(132, device="cuda")
    g = torch.Generator(device="cuda").manual_seed(1)
    worst = 0.0
    eps32 = torch.finfo(torch.float32).eps
    for step in range(5):
        grad = torch.randn(p.shape, device="cuda", generator=g) * (0.02 if step % 2 else 1.0)    # clipped and unclipped steps
        grads = grad.clone()
        p_old = p.clone()
        ops.rmsprop_clip(p, grads, sq, max_grad_norm=0.5, lr=7e-4, norm_out=norm_out, zero_grads=True, wpack=wpack, obs_dim=d, n_actions=a)
        torch.cuda.synchronize()
        norm = float(norm_out[0])
        assert abs(norm - float(grad.norm())) <= 1e-5 * float(grad.norm())
        assert bool((grads == 0).all())                                  # zero_grads honoured
        coef = min(0.5 / (norm + 1e-6), 1.0)
        ref.grad = grad * coef
        opt.step()
        torch.testing.assert_close(sq, opt.state[ref]["square_avg"], rtol=4 * eps32, atol=1e-30)     # values are 1e-9 .. 1e-7
        # new parameters: 4 ulp of the update plus 2 ulp of the parameter (the kernel adds its update with one rounding, torch's
        # foreach kernels may round the product and the sum separately; a CPU emulation of both orders differs by up to 2 ulp)
        du_ref = ref.detach() - p_old
        err = (p - ref.detach()).abs()
        mag = torch.maximum(p_old.abs(), ref.detach().abs())
        assert bool((err <= 4 * eps32 * du_ref.abs() + 2 * eps32 * mag + 1e-12).all()), float(err.max())
        worst = max(worst, float((err / (eps32 * mag.clamp(min=1e-30))).max()))
        if with_wpack:       # the hidden-layer operand images equal a fresh pack of the updated parameters
            fresh = ops.mlp_pack(p, d, a)
            assert torch.equal(wpack[4:], fresh[4:])
        p.copy_(ref.detach())                                            # continue from torch's rounding
    print(f"RMSprop kernel vs torch.optim.RMSprop over 5 steps: max parameter error {worst:.2f} ulp of the parameter")


def test_rmsprop_rejects_a_shape_it_does_not_cover():
    from three_mlagents_b200 import ops

    p = torch.zeros(300_000, device="cuda")
    with pytest.raises(ValueError, match="one launch"):
        ops.rmsprop_clip(p, torch.zeros_like(p), torch.zeros_like(p))


@pytest.mark.parametrize("task,n,T", [("ball3d", 256, 5), ("gridworld", 300, 8)])
def test_a2c_iteration_matches_oracle(task, n, T):
    env, model = _model(task, n, T, seed=4)
    d, a = env.obs_dim, env.n_actions
    assert model.fused_update and model.gae_lambda == 1.0
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
    tol_env = 1e-5 if task == "ball3d" else 0.0
    for t in range(T):
        assert np.abs(obs[t] - cur).max() <= tol_env, t
        logits, values = learner.evaluate(obs[t])
        np.testing.assert_allclose(val[t], values.numpy(), rtol=0, atol=3e-2)
        lp, _ = po.categorical(logits, torch.from_numpy(act[t]))
        np.testing.assert_allclose(logp[t], lp.numpy(), rtol=0, atol=3e-2)
        cur, _, dn, _, _ = ora_env.step(act[t])
        assert np.array_equal(done[t], dn)
    adv_dev, ret_dev = model.adv.cpu().numpy(), model.ret.cpu().numpy()
    w_adv, w_ret = po.gae(rew, val, done, model.last_values.cpu().numpy(), 0.99, 1.0)
    assert np.array_equal(adv_dev.view(np.uint32), w_adv.view(np.uint32))
    assert np.array_equal(ret_dev.view(np.uint32), w_ret.view(np.uint32))
    total = T * n
    fo, fl = obs[:T].reshape(total, d), (lambda x: x.reshape(total))
    g_want, _ = learner.gradient(fo, fl(act), fl(adv_dev), fl(ret_dev))
    from three_mlagents_b200 import ops

    g_dev, _ = ops.a2c_batch(model.params, model.wpack, model.obs[:T].reshape(total, d), d, a, model.act, model.adv, model.ret,
                             rows=total, ent_coef=0.01)
    torch.cuda.synchronize()
    gd, gw = torch.from_numpy(g_dev.cpu().numpy()).double(), torch.from_numpy(g_want).double()
    cos, rel = float(torch.nn.functional.cosine_similarity(gd, gw, dim=0)), float((gd - gw).norm() / gw.norm())
    print(f"{task}: A2C batch gradient vs oracle: cosine {cos:.7f}, relative L2 error {rel:.5f}")
    assert cos > 0.999 and rel < 5e-2
    assert model.train() == 1
    torch.cuda.synchronize()
    learner.step(fo, fl(act), fl(adv_dev), fl(ret_dev))
    got, want = model.params.cpu().numpy(), learner.flat.detach().numpy()
    du_dev, du_ora = torch.from_numpy(got - p0).double(), torch.from_numpy(want - p0).double()
    cos_u = float(torch.nn.functional.cosine_similarity(du_dev, du_ora, dim=0))
    print(f"{task}: parameters after one RMSprop step: update cosine {cos_u:.5f}, max |dp| {np.abs(got - want).max():.2e}")
    # RMSprop's first step moves every coordinate by about lr / sqrt(1 - alpha) = 7e-3 whatever its gradient's size, so a
    # coordinate whose gradient is within the bf16 noise may move the other way: bound as for Adam, 2 x that step
    assert cos_u > 0.98 and np.abs(got - want).max() <= 2 * 7e-4 / np.sqrt(0.01) + 1e-6
    env.close()


@pytest.mark.parametrize("task", TASKS)
def test_train_task_a2c_every_cuda_task(task, tmp_path, monkeypatch):
    from three_mlagents_b200 import training
    from three_mlagents_b200.training import TrainConfig, train_task

    monkeypatch.chdir(tmp_path)
    res = train_task(TrainConfig(task, total_timesteps=64 * 5 * 250, algorithm="a2c", n_envs=64, eval_episodes=4, eval_freq=10**12,
                                 verbose=0, run_name="a2c"))
    assert res.algorithm == "a2c" and np.isfinite(res.mean_reward) and res.total_timesteps == 80_000
    meta = json.loads(open(res.metadata_path).read())
    assert meta["algorithm"] == "a2c" and meta["config"]["algorithm"] == "a2c"
    rows = open(os.path.join(res.run_dir, "monitor", "0.monitor.csv")).read().splitlines()
    assert rows[0].startswith("#") and rows[1] == "r,l,t"
    prog = [json.loads(l) for l in open(os.path.join(res.run_dir, "tb", "progress.jsonl"))]
    assert len(prog) == 3 and [r["time/iterations"] for r in prog] == [100, 200, 250]        # every log_interval (100) + the last
    for k in ("train/policy_loss", "train/value_loss", "train/entropy_loss", "train/explained_variance", "train/n_updates",
              "train/learning_rate", "rollout/ep_rew_mean", "time/fps", "time/total_timesteps"):
        assert k in prog[-1], k
    assert "train/approx_kl" not in prog[-1] and prog[-1]["train/n_updates"] == 250 and prog[-1]["train/learning_rate"] == 7e-4
    ev = training.evaluate_model(task, res.model_filename, episodes=4)
    assert ev["episodes"] == 4 and np.all(np.isfinite(ev["episode_rewards"]))
    d, n_act = eo.TASKS[task][0], eo.TASKS[task][1]
    assert training.predict_action(task, np.zeros(d, np.float32), res.model_filename) in range(n_act)
    # load_model by file name and by path, with and without the run metadata: CudaA2C, square_avg and counters restored
    from three_mlagents_b200.a2c import CudaA2C

    for ref in (res.model_filename, os.path.abspath(res.model_path)):
        m = training.load_model(training.get_task(task), ref)
        assert isinstance(m, CudaA2C) and m._opt_step == 250 and m.n_updates == 250 and float(m.sq_avg.abs().sum()) > 0
        m.env.close()
    os.remove(res.metadata_path)
    m = training.load_model(training.get_task(task), os.path.abspath(res.model_path))
    assert isinstance(m, CudaA2C)
    m.env.close()


def test_cli_train_gridworld_a2c_then_evaluate(tmp_path, monkeypatch, capsys):
    from three_mlagents_b200 import cli

    monkeypatch.chdir(tmp_path)
    cli.main(["train", "gridworld", "-a", "a2c", "-t", "100000", "--run-name", "cli", "--quiet"])
    result = json.loads(capsys.readouterr().out)
    assert result["algorithm"] == "a2c" and result["total_timesteps"] == 100000 and os.path.exists(result["model_path"])
    cli.main(["evaluate", "gridworld", result["model_path"], "--episodes", "8"])
    ev = json.loads(capsys.readouterr().out)
    assert ev["episodes"] == 8 and ev["task_id"] == "gridworld"


def test_websocket_training_sends_a2c(tmp_path, monkeypatch):
    import asyncio

    from three_mlagents_b200 import websocket_training as wst

    class _Socket:
        application_state = "CONNECTED"

        def __init__(self):
            self.frames = []

        async def send_json(self, payload):
            self.frames.append(payload)

    monkeypatch.chdir(tmp_path)
    sock = _Socket()
    result = asyncio.run(wst.train_task_for_websocket(sock, "gridworld", total_timesteps=16 * 5 * 400, algorithm="a2c", n_envs=16,
                                                      eval_episodes=8, progress_freq=16 * 5 * 100))
    assert sock.frames[-1]["type"] == "trained" and sock.frames[-1]["algorithm"] == "a2c"
    assert wst.predict_policy_action("gridworld", np.array([0.25, -0.5, 1.0, 0.0], np.float32), result["model_filename"]) in range(5)


@pytest.mark.parametrize("task,steps,episodes", [("ball3d", 50_000_000, 256), ("gridworld", 50_000_000, 8192)])
def test_a2c_reaches_registry_reward_threshold(task, steps, episodes, tmp_path, monkeypatch):
    """A2C with SB3's defaults (n_steps 5, RMSprop 7e-4) at 4096 envs learns: evaluation return at or above the registry's
    reward_threshold (ball3d 150.0, gridworld 0.75).  Measured on one B200 (profiles/a2c_time_1gpu.json, 50 M steps, two seeds,
    256 evaluation episodes): ball3d 184.4 / 184.3, gridworld 0.798 / 0.783; gridworld is evaluated on 8192 episodes (standard
    error 0.006) as in the PPO threshold test.  Up to three seeds (test_training_gpu._train_until's rule)."""
    from three_mlagents_b200.registry import get_task
    from three_mlagents_b200.training import TrainConfig, train_task

    monkeypatch.chdir(tmp_path)
    thr = get_task(task).reward_threshold
    seen = []
    for seed in (1, 2, 3):
        res = train_task(TrainConfig(task, total_timesteps=steps, algorithm="a2c", n_envs=4096, eval_episodes=episodes, eval_freq=10**12,
                                     verbose=0, seed=seed, run_name=f"a2c_thr{seed}"))
        seen.append(res.mean_reward)
        if res.mean_reward >= thr:
            return
    raise AssertionError(f"no run met the threshold {thr}; eval mean rewards per seed: {seen}")
