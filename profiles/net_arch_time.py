"""Timing of the 64- and 128-wide policies (csrc/mlp_small.cu) at the bench geometry: 65 536 envs x 128 steps, 32 minibatches.

    python profiles/net_arch_time.py [--out profiles/net_arch_time_1gpu.json] [--iters 3]

Per width in {64, 128} and task in {ball3d, gridworld, push}:
  * the rollout forward (both towers, no activation cache) over 65 536 rows and the backward over one 262 144-row minibatch, in us
    (CUDA events, mean of 20 launches after 3 warm-up launches), with their FLOP rate as a fraction of the float32 FMA peak
    SMs x 128 FMA/clk x 2 FLOP x SM clock, the clock read with nvidia-smi right after the kernel timings;
  * PPO end to end (rollout + GAE + 10 epochs x 32 minibatches) in samples/s;
  * A2C end to end at n_steps 5 (one update per 5-step rollout) in samples/s.
This is separate from bench.py, which times the default 256-wide bf16 network only.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from three_mlagents_b200 import native, ops  # noqa: E402
from three_mlagents_b200.a2c import CudaA2C  # noqa: E402
from three_mlagents_b200.ppo import CudaPPO, orthogonal_init  # noqa: E402
from three_mlagents_b200.vec_env import CudaVecEnv  # noqa: E402

N, T, MB = 65536, 128, 32


def timed_us(fn, reps=20):
    for _ in range(3):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / reps


def flops(d, a, h):
    """(forward, backward) FLOP per row, both towers: forward 2(DH + H^2 + H n), backward 2(2Hn + 2H^2 + DH) per tower."""
    fwd = sum(2 * (d * h + h * h + h * n) for n in (a, 1))
    bwd = sum(2 * (2 * h * n + 2 * h * h + d * h) for n in (a, 1))
    return fwd, bwd


def sm_clock_mhz():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=clocks.sm,clocks.max.sm,power.limit", "--format=csv,noheader,nounits",
                              "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout
        sm, smax, plim = (x.strip() for x in out.strip().split(","))
        return float(sm), float(smax), plim
    except Exception:  # noqa: BLE001
        return None, None, None


def kernel_times(task, h):
    env = CudaVecEnv(task, 1, seed=1)
    d, a = env.obs_dim, env.n_actions
    env.close()
    dev = torch.device("cuda")
    g = torch.Generator(device=dev).manual_seed(0)
    params = orthogonal_init(d, a, 1, hidden=h).to(dev)
    x = torch.randn((N * T, d), device=dev, generator=g)
    B = N * T // MB
    idx = ops.permutation(1, 0, T, N)[:B].contiguous()
    logits = torch.empty((N, a), device=dev)
    values = torch.empty(N, device=dev)
    fwd_us = timed_us(lambda: ops.mlp_forward(params, x, d, a, rows=N, logits=logits, values=values, keep_act=False, hidden=h))
    lg, vl, cache = ops.mlp_forward(params, x, d, a, index=idx, hidden=h)
    dl, dv = torch.randn_like(lg) / B, torch.randn_like(vl) / B
    grads = torch.empty_like(params)
    scratch = torch.empty(native.lib.tmla_mlp_backward_scratch(d, h, a, B), device=dev)
    bwd_us = timed_us(lambda: ops.mlp_backward(params, x, d, a, cache, dl, dv, index=idx, grads=grads, scratch=scratch, hidden=h))
    fwd_cache_us = timed_us(lambda: ops.mlp_forward(params, x, d, a, index=idx, act_cache=cache, logits=lg, values=vl, hidden=h))
    ff, fb = flops(d, a, h)
    return {"rollout_forward_us_65536_rows": fwd_us, "backward_us_262144_rows": bwd_us,
            "train_forward_us_262144_rows_with_cache": fwd_cache_us,
            "flop_per_row_fwd": ff, "flop_per_row_bwd": fb,
            "forward_tflops": ff * N / fwd_us / 1e6, "backward_tflops": fb * B / bwd_us / 1e6}


def e2e(cls, task, h, iters, **kw):
    env = CudaVecEnv(task, N, seed=1)
    model = cls("MlpPolicy", env, seed=1, ent_coef=0.01, policy_kwargs={"net_arch": [h, h]}, **kw)
    for _ in range(2):
        model.collect_rollouts(); model.train()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        model.collect_rollouts(); model.train()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / iters
    out = {"ms_per_iter": ms, "samples_per_s": model.n_steps * N / (ms * 1e-3)}
    env.close()
    del model
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.abspath(__file__)), "net_arch_time_1gpu.json"))
    ap.add_argument("--iters", type=int, default=3)
    args = ap.parse_args()
    props = torch.cuda.get_device_properties(0)
    res = {"device": props.name, "sms": props.multi_processor_count,
           "geometry": {"envs": N, "n_steps": T, "minibatches": MB, "minibatch_rows": N * T // MB, "epochs": 10}, "results": {}}
    for h in (64, 128):
        for task in ("ball3d", "gridworld", "push"):
            k = kernel_times(task, h)
            sm, smax, plim = sm_clock_mhz()
            clk = sm or smax
            if clk:
                peak = props.multi_processor_count * 128 * 2 * clk * 1e6 / 1e12
                k.update(sm_clock_mhz=sm, max_sm_clock_mhz=smax, power_limit_w=plim, fp32_fma_peak_tflops=peak,
                         forward_frac_of_fp32_peak=k["forward_tflops"] / peak, backward_frac_of_fp32_peak=k["backward_tflops"] / peak)
            k["ppo"] = e2e(CudaPPO, task, h, args.iters, n_steps=T, batch_size=N * T // MB, n_epochs=10)
            k["a2c_n_steps_5"] = e2e(CudaA2C, task, h, args.iters * 10, n_steps=5)
            res["results"][f"{task}_h{h}"] = k
            print(json.dumps({f"{task}_h{h}": k}), flush=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
