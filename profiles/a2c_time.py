"""A2C on the CUDA backend, measured: end-to-end samples/s at 65 536 envs x 5 steps (ball3d / gridworld / push), the fused A2C
batch at 327 680 rows, the one-launch clip + RMSprop step against the clip + Adam step, and learning runs of the default A2C
hyper-parameters at 4096 envs (the budget and criterion of tests/test_a2c_gpu.py's learning-outcome test).

    python profiles/a2c_time.py [--out a2c_time.json] [--skip-learn]

CUDA events, warmed up; every timed window is at least 1 s of work.  The card name and power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    name, power, clk = ([x.strip() for x in q.stdout.strip().splitlines()[0].split(",")] + ["?"] * 3)[:3]
    return {"name": name, "power_limit": power, "max_sm_clock": clk, "torch_device": torch.cuda.get_device_name(0)}


def timed(fn, min_s=1.0):
    """us per call over a window of at least min_s seconds (after 3 warm-up calls)."""
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 1
    while True:
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if ms >= min_s * 1e3:
            return ms * 1e3 / reps, reps
        reps = max(reps * 2, int(reps * 1.2 * min_s * 1e3 / max(ms, 1e-3)))


def end_to_end(task: str, n_envs=65536, n_steps=5) -> dict:
    from three_mlagents_b200.a2c import CudaA2C
    from three_mlagents_b200.vec_env import CudaVecEnv

    env = CudaVecEnv(task, n_envs, seed=1)
    m = CudaA2C("MlpPolicy", env, seed=1, n_steps=n_steps)
    e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    for _ in range(5):
        m.collect_rollouts(); m.train()
    torch.cuda.synchronize()
    iters, roll, train = 0, 0.0, 0.0
    while roll + train < 2000.0:                            # >= 2 s of iterations
        e[0].record(); m.collect_rollouts(); e[1].record(); m.train(); e[2].record()
        torch.cuda.synchronize()
        roll += e[0].elapsed_time(e[1]); train += e[1].elapsed_time(e[2]); iters += 1
    out = {"task": task, "envs": n_envs, "n_steps": n_steps, "fused_update": m.fused_update, "iters": iters,
           "samples_per_s": n_envs * n_steps * iters / ((roll + train) * 1e-3), "rollout_ms": roll / iters, "update_ms": train / iters}
    env.close()
    return out


def kernels(rows=327680) -> dict:
    from three_mlagents_b200 import native, ops
    from three_mlagents_b200.ppo import orthogonal_init

    g = torch.Generator(device="cuda").manual_seed(0)
    D, A, T = 6, 5, 5
    N = rows // T
    params = orthogonal_init(D, A, 1).cuda()
    wpack = ops.mlp_pack(params, D, A)
    obs = torch.randn((rows, D), device="cuda", generator=g)
    act = torch.randint(0, A, (T, N), device="cuda", dtype=torch.int32, generator=g)
    adv, ret = torch.randn((T, N), device="cuda", generator=g), torch.randn((T, N), device="cuda", generator=g)
    logp = -torch.rand((T, N), device="cuda", generator=g)
    grads = torch.zeros_like(params)
    scratch = torch.empty(native.lib.tmla_ppo_minibatch_scratch(256, rows), dtype=torch.bfloat16, device="cuda")
    stats = torch.zeros(8, device="cuda")
    res = {}
    us, reps = timed(lambda: ops.a2c_batch(params, wpack, obs, D, A, act, adv, ret, rows=rows, grads=grads, scratch=scratch, stats=stats))
    res["a2c_batch_fused"] = {"rows": rows, "us": us, "reps": reps, "TFLOP/s": 807936.0 * rows / us / 1e6,
                              "note": "ball3d shape; forward + loss + backward of both towers (807 936 FLOP per row)"}
    us, reps = timed(lambda: ops.ppo_minibatch(params, wpack, obs, D, A, act, adv, logp, ret, rows=rows, normalize=False, grads=grads,
                                               scratch=scratch, stats=stats))
    res["ppo_minibatch_fused_same_rows"] = {"rows": rows, "us": us, "reps": reps, "TFLOP/s": 807936.0 * rows / us / 1e6}
    p = params.clone()
    gr = torch.randn(p.shape, device="cuda", generator=g) * 1e-3
    sq, m, v = torch.zeros_like(p), torch.zeros_like(p), torch.zeros_like(p)
    norm_out = torch.zeros(132, device="cuda")
    step = [0]

    def adam():
        step[0] += 1
        ops.adam_clip(p, gr, m, v, step[0], norm_out=norm_out)
    us_r, reps_r = timed(lambda: ops.rmsprop_clip(p, gr, sq, norm_out=norm_out))
    us_a, reps_a = timed(adam)
    res["rmsprop_step"] = {"us": us_r, "reps": reps_r, "num_params": p.numel()}
    res["adam_step"] = {"us": us_a, "reps": reps_a, "num_params": p.numel()}
    return res


def learn(task: str, steps: int, seed: int, n_envs=4096) -> dict:
    from three_mlagents_b200.training import TrainConfig, train_task

    t0 = time.time()
    r = train_task(TrainConfig(task, total_timesteps=steps, algorithm="a2c", n_envs=n_envs, eval_episodes=256, eval_freq=10**12, verbose=0,
                               seed=seed, run_name=f"a2c_learn_{task}_{seed}"))
    return {"task": task, "steps": steps, "seed": seed, "n_envs": n_envs, "mean_reward": r.mean_reward, "std_reward": r.std_reward,
            "wall_s": time.time() - t0}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="a2c_time.json")
    ap.add_argument("--skip-learn", action="store_true")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "a2c_time.py measures on a GPU; there is no CPU fallback"
    rec = {"card": card()}
    print(json.dumps(rec), flush=True)
    rec["kernels"] = kernels()
    print(json.dumps(rec["kernels"]), flush=True)
    rec["end_to_end"] = []
    for task in ("ball3d", "gridworld", "push"):
        rec["end_to_end"].append(end_to_end(task))
        print(json.dumps(rec["end_to_end"][-1]), flush=True)
    if not args.skip_learn:
        import tempfile

        cwd = os.getcwd()
        rec["learn"] = []
        with tempfile.TemporaryDirectory() as tmp:
            os.chdir(tmp)
            try:
                for task, steps in (("ball3d", 50_000_000), ("gridworld", 50_000_000)):
                    for seed in (1, 2):
                        rec["learn"].append(learn(task, steps, seed))
                        print(json.dumps(rec["learn"][-1]), flush=True)
            finally:
                os.chdir(cwd)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=2)


if __name__ == "__main__":
    main()
