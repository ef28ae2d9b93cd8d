"""Cost of deterministic mode on one GPU (DESIGN.md §6), flag off and on alternated in one session:
  * one minibatch update (forward + loss + backward + clip/Adam), CUDA events over 20 launches after 3 warm-up launches:
    ball3d, 262 144 rows, fused path (tmla_ppo_minibatch_bf16 with / without TMLA_MB_DETERMINISTIC);
    glider, 262 144 rows, three-call path (tmla_mlp_forward_bf16 + tmla_ppo_loss(_det) + tmla_mlp_backward_bf16(_det));
  * PPO end to end at 65 536 envs x 128 steps, 32 minibatches x 10 epochs (ppo.bench_ppo), samples/s;
  * the card's name, power limit and SM clocks, read in the same call.

    python profiles/deterministic_time.py [out.json]      (default: profiles/deterministic_time_1gpu.json)
"""
from __future__ import annotations

import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from three_mlagents_b200 import ops  # noqa: E402
from three_mlagents_b200.ppo import bench_ppo, orthogonal_init  # noqa: E402


def gpu_info() -> dict:
    q = "name,power.limit,clocks.max.sm,clocks.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True).stdout
    return dict(zip(q.split(","), [x.strip() for x in out.splitlines()[0].split(",")])) if out else {"name": torch.cuda.get_device_name(0)}


def timed(fn, reps=20) -> float:
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


def minibatch_case(task: str, d: int, a: int, rows: int):
    """-> fn(det) running one minibatch update of `rows` rows out of a 128 x 65 536 rollout"""
    T, N = 128, 65536
    g = torch.Generator(device="cuda").manual_seed(0)
    obs = torch.randn((T * N, d), device="cuda", generator=g)
    act = torch.randint(0, a, (T * N,), device="cuda", dtype=torch.int32, generator=g)
    adv, ret = torch.randn(T * N, device="cuda", generator=g), torch.randn(T * N, device="cuda", generator=g)
    logp = -torch.rand(T * N, device="cuda", generator=g) - 0.5
    idx = ops.permutation(1, 0, T, N)[:rows].contiguous()
    sums = ops.adv_stats(adv, idx, rows)
    params = orthogonal_init(d, a, 1).cuda()
    wpack = ops.mlp_pack(params, d, a)
    m, v, grads = torch.zeros_like(params), torch.zeros_like(params), torch.zeros_like(params)
    stats, norm = torch.zeros(8, device="cuda"), torch.zeros(132, device="cuda")
    fused = ops.ppo_minibatch_supported(d, a)
    if fused:
        scratch = torch.empty(ops.fused_scratch_elems(d, a, rows, True), dtype=torch.bfloat16, device="cuda")
    else:
        part = torch.empty(ops.det_scratch_bytes(d, a, rows), dtype=torch.uint8, device="cuda")
        scratch = torch.empty(2 * rows * 256, dtype=torch.bfloat16, device="cuda")
        logits, values = torch.empty((rows, a), device="cuda"), torch.empty(rows, device="cuda")
        cache = torch.empty((4, rows, 256), dtype=torch.bfloat16, device="cuda")
        dl, dv = torch.empty((rows, a), device="cuda"), torch.empty(rows, device="cuda")

    def step(det: bool):
        if fused:
            ops.ppo_minibatch(params, wpack, obs, d, a, act, adv, logp, ret, index=idx, rows=rows, adv_sums=sums, grads=grads,
                              scratch=scratch, stats=stats, grads_zeroed=True, accumulate_stats=True, deterministic=det)
        else:
            ops.mlp_forward(params, obs, d, a, index=idx, rows=rows, logits=logits, values=values, act_cache=cache, wpack=wpack)
            ops.ppo_loss(logits, values, act, adv, logp, ret, index=idx, rows=rows, adv_sums=sums, dlogits=dl, dvalues=dv, stats=stats,
                         partials=part if det else None)
            ops.mlp_backward(params, obs, d, a, cache, dl, dv, index=idx, rows=rows, grads=grads, scratch=scratch, wpack=wpack,
                             partials=part if det else None)
        ops.adam_clip(params, grads, m, v, 1, norm_out=norm, zero_grads=fused, wpack=wpack if fused else None, obs_dim=d, n_actions=a)

    return step, "fused (tmla_ppo_minibatch_bf16)" if fused else "three-call (forward, loss, backward)"


def main() -> None:
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "deterministic_time_1gpu.json")
    torch.cuda.set_device(0)
    res = {"gpu": gpu_info(), "minibatch_us": {}, "ppo_samples_per_s": {}}
    for task, d, a in (("ball3d", 6, 5), ("glider", 16, 5)):
        step, path = minibatch_case(task, d, a, 262144)
        off, on = [], []
        for _ in range(4):                                   # alternated: off, on, off, on, ...
            off.append(timed(lambda: step(False)))
            on.append(timed(lambda: step(True)))
        res["minibatch_us"][task] = {"path": path, "rows": 262144, "off": off, "on": on, "off_min": min(off), "on_min": min(on),
                                     "on_over_off": min(on) / min(off)}
        print(task, res["minibatch_us"][task], flush=True)
        del step
        torch.cuda.empty_cache()
    for task in ("ball3d", "gridworld"):
        runs = {"off": [], "on": []}
        for _ in range(2):
            for flag in ("off", "on"):
                torch.use_deterministic_algorithms(flag == "on")
                r = bench_ppo(0, 0, 1, iters=3, warmup=1, task=task)
                runs[flag].append({"samples_per_s": r["value"], "update_us_per_minibatch": r["update_us_per_minibatch"],
                                   "rollout_ms": r["rollout_ms"]})
        torch.use_deterministic_algorithms(False)
        best = {k: max(x["samples_per_s"] for x in v) for k, v in runs.items()}
        res["ppo_samples_per_s"][task] = {"config": "65536 envs x 128 steps, 32 minibatches x 10 epochs", "runs": runs, "best": best,
                                          "on_over_off": best["on"] / best["off"]}
        print(task, res["ppo_samples_per_s"][task]["best"], flush=True)
    res["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as f:
        json.dump(res, f, indent=2)
    print(json.dumps({"minibatch_us": {k: (v["off_min"], v["on_min"]) for k, v in res["minibatch_us"].items()},
                      "ppo": {k: v["best"] for k, v in res["ppo_samples_per_s"].items()}, "gpu": res["gpu"]}))


if __name__ == "__main__":
    main()
