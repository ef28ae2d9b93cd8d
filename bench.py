#!/usr/bin/env python
"""bench.py — headline benchmark of the three-mlagents hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Metric (BASELINE.json): env-steps/sec for ball3d at 65 536 envs per GPU, random policy.
A "step" of this bench is ONE pass of the hot path over the whole batch: one fused 128-step
rollout of all 65 536 environments (`tmla_rollout_random`, 8 388 608 env-steps, 277 MB written).
  value      whole-job env-steps/s with state and buffers resident in HBM, timed with CUDA events,
             max over ranks
  e2e        the same metric through the reference-facing API `CudaVecEnv.step(numpy actions)`
             (C ABI `tmla_step_host`): host buffers, H2D + kernel + D2H inside the timed region
  roofline   rollout kernel: algorithmic bytes / measured launch duration vs the measured HBM peak
  cpu_baseline   the scalar reference port (oracle/ref_port.py) timed on this box's host cores
  ppo        end-to-end PPO samples/s on BASELINE configs 3/4/5 (ball3d 64K envs/GPU, gridworld and push 32K envs/GPU; T=128,
             2x256 MLP), each with update TFLOP/s against the measured sustained bf16 peak, the all-reduce cost and a
             replicas-identical check; `cpu_baseline.ppo` is the CPU restatement of SB3 PPO at the reference defaults
Multi-GPU: one process per GPU under torchrun; environments shard by global env id, no data-path
collective for the env-step metric (weak scaling); PPO adds one gradient all-reduce per minibatch.

--dump-outputs DIR writes what the last timed rollout launch returned on rank 0, for a fixed sample of DUMP_ENVS
environments (seeded choice, sorted env ids) over all T_ROLLOUT steps, as float32 arrays: obs.npy [T, DUMP_ENVS, 6],
actions.npy, rewards.npy and dones.npy [T, DUMP_ENVS] (37.7 MB in all).  Every launch before the last timed one has a
fixed count for given --steps / --warmup, so two builds run with the same arguments can be compared array for array.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

TASK = "ball3d"
N_ENVS = 65536
T_ROLLOUT = 128
OBS_DIM = 6
# SURVEY.md §8(d): fused-rollout path writes obs 24 + reward 4 + done 1 + action 4 per env-step,
# plus the 56 B/env state read+write amortised over the T steps of one launch.
BYTES_PER_ENV_STEP = 33.0 + 56.0 / T_ROLLOUT
DUMP_ENVS, DUMP_SEED = 8192, 0
# untimed launches that load the GPU before the timed ones while nvidia-smi samples clocks: 130 x 50 launches, ~0.4 s on a
# B200.  A count rather than a time budget, so that the timed launches start from the same environment state in every run.
PRELOAD_BATCHES = 130


NCU_TRAFFIC_CSV = "profiles/r2_rollout_fast_ncu_raw.csv"


def _ncu_traffic():
    """dram bytes (read+write) per rollout launch from the committed `ncu --set full` capture of the same kernel, or None.
    (ncu cannot run inside a timed bench; the line names the file the figure comes from as `traffic_source`.)"""
    path = os.path.join(ROOT, NCU_TRAFFIC_CSV)
    try:
        vals = {}
        with open(path) as f:
            for line in f:
                parts = line.strip().split(",")
                if len(parts) < 3:
                    continue
                k, unit, v = parts[:3]
                if k.startswith("dram__bytes_"):
                    vals[k] = float(v) * {"Mbyte": 1e6, "Gbyte": 1e9, "Kbyte": 1e3, "byte": 1.0}[unit]
        return vals["dram__bytes_read.sum"] + vals["dram__bytes_write.sum"]
    except Exception:  # noqa: BLE001
        return None


def _peaks():
    """(HBM GB/s, sustained bf16 TFLOP/s, source): the driver-measured peaks of this pool, else the recipe's fallback."""
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), float(d.get("bf16_tflops_sustained") or 1400.0), "measured (MEASURED_PEAKS.json)"
    except Exception:  # noqa: BLE001
        return 6650.0, 1400.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """Samples nvidia-smi clocks/throttle reasons while the timed region runs."""

    QUERY = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self._stop, self._thr = index, [], threading.Event(), None

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                                      "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:  # noqa: BLE001
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._thr = threading.Thread(target=self._run, daemon=True)
        self._thr.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        self._thr.join(timeout=6)

    def summary(self):
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            for name, val in zip(names, r[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.rows)}


def _cpu_baseline(seconds_target: float = 12.0):
    """Reference CPU path: serial DummyVecEnv-style loop over 8 scalar Python envs (1 core)."""
    from oracle import ref_port

    n_envs = 8                                   # ball3d's registry default (registry.py:79)
    t_probe = ref_port.time_random_policy(TASK, n_envs, 500)
    vec_steps = max(1000, int(500 * seconds_target / max(t_probe, 1e-3)))
    dt = ref_port.time_random_policy(TASK, n_envs, vec_steps)
    out = {"value": n_envs * vec_steps / dt, "unit": "env-steps/s", "cores": 1, "kind": "port",
           "sample": f"ball3d, {n_envs} envs x {vec_steps} serial vec-steps, uniform random actions, "
                     f"scalar Python port of the reference env + adapter + DummyVecEnv loop ({dt:.1f} s)"}
    # For scale, the same semantics restated as vectorised NumPy over all 65 536 envs (oracle/envs_oracle.py, the parity
    # checker): what one host core reaches once the per-env Python objects of the reference are gone.
    try:
        import numpy as np
        from oracle import envs_oracle as eo

        ora = eo.OracleVecEnv(TASK, N_ENVS, seed=1)
        acts = np.random.default_rng(0).integers(0, 5, size=(8, N_ENVS))
        ora.step(acts[0])
        t0 = time.perf_counter()
        k = 0
        while time.perf_counter() - t0 < 3.0:
            ora.step(acts[k % 8])
            k += 1
        out["numpy_vectorised"] = {"value": N_ENVS * k / (time.perf_counter() - t0), "unit": "env-steps/s", "cores": 1,
                                   "sample": f"{k} vec-steps of {N_ENVS} envs (NumPy restatement with Philox auto-reset, 3 s)"}
    except Exception as e:  # noqa: BLE001
        out["numpy_vectorised"] = {"error": f"{type(e).__name__}: {e}"}
    # PPO end to end on the CPU at the reference defaults (registry.py:77-80 n_envs=8; training.py:379-389 n_steps=1024,
    # batch 256, 10 epochs): the CPU figure that stands beside `ppo.*.value`
    try:
        from oracle import ppo_cpu_baseline

        out["ppo"] = ppo_cpu_baseline.time_ppo("ball3d", n_envs=8, n_steps=1024, batch_size=256, n_epochs=10, iterations=3)
    except Exception as e:  # noqa: BLE001
        out["ppo"] = {"error": f"{type(e).__name__}: {e}"}
    return out


def _config1_pair():
    """BASELINE configs[0] — `three-mlagents train basic -a ppo -t 25000 --seed 1` — as a (wall-clock, eval reward) pair on the
    CPU restatement and through this backend's own `train_task` (same registry defaults: n_envs=1, 50 eval episodes)."""
    import tempfile

    pair = {}
    try:
        from oracle import ppo_cpu_baseline

        pair["cpu"] = ppo_cpu_baseline.train_config1(25_000, seed=1)
    except Exception as e:  # noqa: BLE001
        pair["cpu"] = {"error": f"{type(e).__name__}: {e}"}
    try:
        from three_mlagents_b200.training import TrainConfig, train_task

        cwd = os.getcwd()
        with tempfile.TemporaryDirectory() as tmp:
            os.chdir(tmp)
            try:
                t0 = time.perf_counter()
                res = train_task(TrainConfig(task_id="basic", total_timesteps=25_000, algorithm="ppo", seed=1, verbose=0))
                pair["cuda"] = {"wall_s": time.perf_counter() - t0, "timesteps": res.total_timesteps, "eval_mean_reward": res.mean_reward,
                                "eval_std_reward": res.std_reward, "eval_episodes": res.eval_episodes,
                                "note": "n_envs=1: launch-latency bound (one env per kernel launch), the reference's own configuration"}
            finally:
                os.chdir(cwd)
    except Exception as e:  # noqa: BLE001
        pair["cuda"] = {"error": f"{type(e).__name__}: {e}"}
    return pair


def run_reference(args):
    """--impl reference: the reference's CPU implementation (port; the Python reference cannot travel)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import ref_port

    n_envs, vec_steps = 8, 4000                  # one bench step = 32 000 env-steps (~1 s)
    for _ in range(max(0, args.warmup)):
        ref_port.time_random_policy(TASK, n_envs, 200)
    times = [ref_port.time_random_policy(TASK, n_envs, vec_steps, seed=1 + i) for i in range(args.steps)]
    total = sum(times)
    value = n_envs * vec_steps * args.steps / total
    sample = (f"each step = {n_envs} envs x {vec_steps} serial vec-steps of ball3d with uniform random actions "
              f"(scalar Python port of the reference; DummyVecEnv is single-threaded by construction)")
    try:      # the other half of BASELINE's metric on the CPU: PPO end to end at the reference defaults (bounded: 2 iterations)
        from oracle import ppo_cpu_baseline

        ppo = ppo_cpu_baseline.time_ppo("ball3d", n_envs=8, n_steps=1024, batch_size=256, n_epochs=10, iterations=2)
    except Exception as e:  # noqa: BLE001
        ppo = {"error": f"{type(e).__name__}: {e}"}
    print(json.dumps({
        "impl": "reference", "metric": "env_steps_per_sec", "value": value, "unit": "env-steps/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32+f64", "data": "synthetic",
        "config": {"workload": "ball3d random-policy step throughput (reference CPU path, bounded sample)",
                   "envs": n_envs, "vec_steps_per_step": vec_steps},
        "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": 1, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "ppo": {"ball3d": ppo},
    }))


def run_cuda(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: three-mlagents_b200 has no CPU fallback "
                         "(use --impl reference for the CPU baseline)")
    from three_mlagents_b200.distributed import bind_to_gpu_numa_node

    numa_cpus = bind_to_gpu_numa_node(local_rank)      # pinned host buffers on the GPU's own NUMA node (host-step e2e)
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    from three_mlagents_b200.vec_env import CudaVecEnv

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    K, W = args.steps, max(3, args.warmup)
    env = CudaVecEnv(TASK, N_ENVS, seed=1, device=local_rank, env_id_base=rank * N_ENVS)
    dev = torch.device("cuda", local_rank)
    obs = torch.empty((T_ROLLOUT, N_ENVS, OBS_DIM), dtype=torch.float32, device=dev)
    act = torch.empty((T_ROLLOUT, N_ENVS), dtype=torch.int32, device=dev)
    rew = torch.empty((T_ROLLOUT, N_ENVS), dtype=torch.float32, device=dev)
    done = torch.empty((T_ROLLOUT, N_ENVS), dtype=torch.uint8, device=dev)

    # ---- device-resident fused rollout (value + roofline) ------------------------------------------
    for _ in range(W):
        env.rollout_random(T_ROLLOUT, obs, act, rew, done)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    # The timed region is only K x ~70 us long; nvidia-smi needs ~100 ms per sample.  The sampler therefore
    # brackets the timed region with the same kernel running back to back (load before, during and after):
    # untimed launches first, then the K timed launches, then untimed launches until >= 5 samples exist.
    dumped = None
    with ClockSampler(local_rank) as clocks:
        for _ in range(PRELOAD_BATCHES):
            for _ in range(50):
                env.rollout_random(T_ROLLOUT, obs, act, rew, done)
            torch.cuda.synchronize()
        barrier()
        e0.record()
        for _ in range(K):
            env.rollout_random(T_ROLLOUT, obs, act, rew, done)
        e1.record()
        barrier()
        if args.dump_outputs and rank == 0:      # before the launches below overwrite the buffers
            idx = torch.from_numpy(np.sort(np.random.default_rng(DUMP_SEED).choice(N_ENVS, DUMP_ENVS, replace=False))).to(dev)
            dumped = {name: t.index_select(1, idx).float().cpu().numpy()
                      for name, t in (("obs", obs), ("actions", act), ("rewards", rew), ("dones", done))}
        t_load = time.perf_counter()
        while len(clocks.rows) < 5 and time.perf_counter() - t_load < 3.0:
            for _ in range(50):
                env.rollout_random(T_ROLLOUT, obs, act, rew, done)
            torch.cuda.synchronize()
    if dumped is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dumped.items():
            np.save(os.path.join(args.dump_outputs, f"{name}.npy"), a)
    ms = max_over_ranks(e0.elapsed_time(e1))
    steps_per_launch = N_ENVS * T_ROLLOUT
    value = world * steps_per_launch * K / (ms * 1e-3)
    launch_ms = ms / K
    peak, tensor_sustained, peak_src = _peaks()
    achieved = BYTES_PER_ENV_STEP * steps_per_launch / (launch_ms * 1e-3) / 1e9
    done_rate = float(done.float().mean().item())

    if args.quick:      # profiling runs (ncu): only the fused rollout
        if rank == 0:
            print(json.dumps({"metric": "env_steps_per_sec", "value": value, "ms_per_step": launch_ms, "quick": True}))
        env.close()
        return
    # ---- per-launch VecEnv.step on device tensors (launch-bound; reported, not the headline) -------
    a_dev = torch.randint(0, 5, (N_ENVS,), dtype=torch.int32, device=dev)
    for _ in range(20):
        env.step_tensor(a_dev)
    barrier()
    n_api = 2000
    e0.record()
    for _ in range(n_api):
        env.step_tensor(a_dev)
    e1.record()
    barrier()
    api_ms = max_over_ranks(e0.elapsed_time(e1))
    step_api = world * N_ENVS * n_api / (api_ms * 1e-3)

    # ---- e2e: SB3 VecEnv.step contract, NumPy in / NumPy out through tmla_step_host ----------------
    rng = np.random.default_rng(rank)
    host_actions = rng.integers(0, 5, size=(64, N_ENVS)).astype(np.int32)
    env.reset()
    for i in range(10):
        env.step(host_actions[i % 64])
    barrier()
    n_e2e = 300
    t0 = time.perf_counter()
    for i in range(n_e2e):
        o, r, d, infos = env.step(host_actions[i % 64])
    barrier()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    e2e = world * N_ENVS * n_e2e / e2e_s

    out = {
        "metric": "env_steps_per_sec", "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": launch_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32+f64", "data": "synthetic",
        "config": {"workload": "ball3d random-policy step throughput, 65536 envs/GPU (BASELINE configs[1]); "
                               "one bench step = one fused 128-step rollout launch",
                   "envs_per_gpu": N_ENVS, "rollout_steps": T_ROLLOUT, "actions": "in-kernel Philox4x32-10",
                   "l2": "each step writes 277 MB of rollout rows (> 126 MB L2); no flush needed",
                   "done_rate": done_rate},
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": _ncu_traffic(), "traffic_source": NCU_TRAFFIC_CSV + " (ncu --set full capture of this kernel, per launch)",
                     "algorithmic_bytes": BYTES_PER_ENV_STEP * steps_per_launch,
                     "kernel": "rollout_fast_kernel<Ball3DTask>",
                     "bytes_per_env_step": BYTES_PER_ENV_STEP, "peak_source": peak_src},
        "e2e": {"value": e2e, "unit": "env-steps/s", "h2d_bytes_per_step": 4 * N_ENVS,
                "d2h_bytes_per_step": N_ENVS * (4 * OBS_DIM + 4 + 1 + 1),
                "api": "CudaVecEnv.step(np.ndarray int32) -> tmla_step_block_begin / _end (range check + narrowing of the actions into pinned "
                       "memory, ONE kernel that reads them and writes obs/reward/done/truncated/records over PCIe into a pooled pinned "
                       "result block, host polls the sequence word); the returned NumPy arrays are slices of that block, reused only "
                       "when dropped", "steps": n_e2e,
                "numa_cpus": None if numa_cpus is None else len(numa_cpus)},
        "step_api": {"value": step_api, "unit": "env-steps/s", "us_per_launch": 1e3 * api_ms / n_api,
                     "frac_hbm": (89.0 * N_ENVS / (api_ms / n_api * 1e-3) / 1e9) / peak,
                     "note": "one tmla_step launch per env step on device tensors; 5.8 MB working set, launch-bound"},
        "gpu_launches": K,
        "clocks": clocks.summary(),
    }
    if not args.no_ppo:
        # BASELINE configs[2..4]: ball3d 64K envs/GPU, gridworld 32K envs/GPU (256K over 8), push 32K envs/GPU — every one at the
        # N this run uses, `--ppo-warmup` untimed + `--ppo-iters` timed iterations each
        from three_mlagents_b200.ppo import bench_ppo

        out["ppo"] = {}
        for task in [t for t in args.ppo_tasks.split(",") if t]:
            try:
                ppo_envs = args.ppo_envs or (N_ENVS if task == "ball3d" else 32768)
                out["ppo"][task] = bench_ppo(local_rank, rank, world, iters=args.ppo_iters, warmup=args.ppo_warmup, task=task,
                                             n_envs=ppo_envs, sustained_tflops=tensor_sustained)
            except Exception as e:  # noqa: BLE001 - the env-step headline must still print
                out["ppo"][task] = {"error": f"{type(e).__name__}: {e}"}
        if world == 1 and "ball3d" in out["ppo"] and "error" not in out["ppo"]["ball3d"] and not args.no_kernels:
            try:
                from three_mlagents_b200.ppo import bench_kernels

                out["ppo"]["ball3d"]["kernels"] = bench_kernels(local_rank)
            except Exception as e:  # noqa: BLE001
                out["ppo"]["ball3d"]["kernels"] = {"error": f"{type(e).__name__}: {e}"}
        # the second half of BASELINE's metric, where the driver's parser keeps it (it retains `config` whole)
        out["config"]["ppo_samples_per_sec"] = {
            t: ({k: r.get(k) for k in ("value", "update_tflops", "frac_of_sustained", "allreduce_us", "replicas_identical", "rollout_ms", "update_ms")}
                if "error" not in r else r) for t, r in out["ppo"].items()}
        out["config"]["ppo_workload"] = "PPO end-to-end samples/s: ball3d 65536 envs/GPU | gridworld 32768 | push 32768; T=128, 2x256 MLP, 10 epochs x 32 minibatches"
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        out["cpu_baseline"] = _cpu_baseline()
        if not args.no_config1:
            out["config1_basic_ppo_25k"] = _config1_pair()
    elif rank == 0:
        out["cpu_baseline"] = None
    env.close()
    if rank == 0:
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--no-ppo", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--ppo-iters", type=int, default=5)
    ap.add_argument("--ppo-warmup", type=int, default=2)
    ap.add_argument("--ppo-tasks", default="ball3d,gridworld,push", help="comma-separated subset of ball3d,gridworld,push")
    ap.add_argument("--no-kernels", action="store_true", help="skip the per-kernel PPO micro-benchmarks")
    ap.add_argument("--no-config1", action="store_true", help="skip the BASELINE configs[0] wall-clock/eval-reward pair")
    ap.add_argument("--ppo-envs", type=int, default=0, help="envs per GPU for the PPO section (default: 65536 ball3d, 32768 otherwise)")
    ap.add_argument("--quick", action="store_true", help="fused rollout only (for ncu runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write a fixed sample of the last timed rollout's obs / actions / rewards / dones to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "cuda":
        ap.error("--dump-outputs writes the outputs of the CUDA rollout (--impl cuda)")
    # Exactly ONE line on stdout: libraries that print there on their own (NCCL's version banner under NCCL_DEBUG, a
    # stray warning) are sent to stderr at the file-descriptor level; the JSON line goes to the real stdout.
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(real_stdout, "w", buffering=1)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_cuda(args)
    sys.stdout.flush()


if __name__ == "__main__":
    main()
