"""A/B of ball3d's fused random-policy rollout (what bench.py times): the parent commit's tree against this tree, in one
session on one GPU.

    python profiles/rollout_ab.py --parent DIR [--rounds 4] [--steps 200] [--tasks gridworld,push] [--out FILE]

DIR is an untracked export of the parent commit (`git archive <parent> | tar -x -C DIR`).  The script reads the card's name,
power limit and max SM clock, builds both trees, checks that `bench.py --quick --steps 50 --dump-outputs` gives equal arrays
for both, then alternates `bench.py --quick --steps K` between them `rounds` times and reports the median µs per launch
(one 65 536 x 128 rollout), the per-run spread and the gain over the parent.  In the same rounds it times each of
`--tasks` (default gridworld and push) through `env.rollout_random` at 65 536 x 128 with CUDA events, `--steps` launches
after a warm-up, the same way for both trees.
"""
from __future__ import annotations

import argparse
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(cmd, cwd):
    r = subprocess.run(cmd, cwd=cwd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"{' '.join(cmd)} in {cwd} failed ({r.returncode}):\n{r.stdout[-2000:]}\n{r.stderr[-4000:]}")
    return r.stdout


def _bench(tree, steps, dump=None):
    cmd = [sys.executable, "bench.py", "--quick", "--steps", str(steps)] + (["--dump-outputs", dump] if dump else [])
    return json.loads(_run(cmd, tree).strip().splitlines()[-1])


_TASK_TIMER = """
import sys, torch
sys.path.insert(0, '.')
from three_mlagents_b200.vec_env import CudaVecEnv
task, n, T, K = sys.argv[1], 65536, 128, int(sys.argv[2])
env = CudaVecEnv(task, n, seed=1)
obs = torch.empty((T, n, env.obs_dim), device='cuda')
act = torch.empty((T, n), dtype=torch.int32, device='cuda')
rew = torch.empty((T, n), device='cuda')
done = torch.empty((T, n), dtype=torch.uint8, device='cuda')
for _ in range(50):
    env.rollout_random(T, obs, act, rew, done)
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(K):
    env.rollout_random(T, obs, act, rew, done)
e1.record()
torch.cuda.synchronize()
print(e0.elapsed_time(e1) / K * 1e3)
"""


def _time_task(tree, task, steps):
    return float(_run([sys.executable, "-c", _TASK_TIMER, task, str(steps)], tree).strip().splitlines()[-1])


def _summary(runs, base_name="parent"):
    base = statistics.median(runs[base_name])
    return {name: {"us_per_launch": us, "median_us": statistics.median(us), "spread": (max(us) - min(us)) / statistics.median(us),
                   "gain_vs_parent": 1.0 - statistics.median(us) / base} for name, us in runs.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent", required=True, help="untracked export of the parent commit")
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--tasks", default="gridworld,push", help="tasks also timed through env.rollout_random ('' for none)")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "rollout_blocks_ab_1gpu.json"))
    args = ap.parse_args()
    trees = {"parent": os.path.abspath(args.parent), "new": ROOT}
    q = "name,power.limit,clocks.max.sm"
    card = _run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], ROOT).strip()
    result = {"card": dict(zip(q.split(","), [c.strip() for c in card.split(",")])),
              "bench": f"bench.py --quick --steps {args.steps}", "rounds": args.rounds}
    for tree in trees.values():
        _run([sys.executable, os.path.join(tree, "three-mlagents_b200", "build.py")], tree)
    tmp = tempfile.mkdtemp(prefix="rollout_ab_")
    try:
        for name, tree in trees.items():
            _bench(tree, 50, dump=os.path.join(tmp, name))
        result["dump_equal"] = {f: bool(np.array_equal(np.load(os.path.join(tmp, "parent", f)), np.load(os.path.join(tmp, "new", f))))
                                for f in ("obs.npy", "actions.npy", "rewards.npy", "dones.npy")}
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    tasks = [t for t in args.tasks.split(",") if t]
    runs = {name: [] for name in trees}
    task_runs = {task: {name: [] for name in trees} for task in tasks}
    for _ in range(args.rounds):
        for name, tree in trees.items():
            runs[name].append(_bench(tree, args.steps)["ms_per_step"] * 1e3)
            print(name, f"{runs[name][-1]:.2f} us", file=sys.stderr, flush=True)
            for task in tasks:
                task_runs[task][name].append(_time_task(tree, task, args.steps))
                print(name, task, f"{task_runs[task][name][-1]:.2f} us", file=sys.stderr, flush=True)
    result["runs"] = _summary(runs)
    if tasks:
        result["rollout_random_65536x128"] = {task: _summary(r) for task, r in task_runs.items()}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
