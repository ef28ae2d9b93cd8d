"""SASS accounting of the fused random-policy rollout (`rollout_fast_kernel`), no GPU needed.

    python profiles/rollout_sass.py [--tree DIR] [--tasks Ball3D,GridWorld,Push]

Compiles DIR's csrc/env_kernels.cu (default: this tree) with the library's nvcc flags and prints, per task:
registers, stack frame and spill bytes (ptxas), and for every innermost loop of the kernel its span in bytes and the
instructions and branches on its shortest path.  That path skips every conditional block: the episode reset, the spare
refill, the first-step-after-reset rounding and the sqrt slow path, so it is the common path of a step.  Steps per loop
iteration are counted as the one-byte `done` stores on the path (one per step), and the per-step figures divide by it.
"""
from __future__ import annotations

import argparse
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "--expt-relaxed-constexpr"]
INS = re.compile(r"^\s+/\*([0-9a-f]{4,})\*/\s+(.*?)\s*;")


def _compile(tree, tmp):
    csrc = os.path.join(tree, "three-mlagents_b200", "csrc")
    cubin = os.path.join(tmp, "env_kernels.cubin")
    nvcc = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "nvcc")
    r = subprocess.run([nvcc, *FLAGS, "-I", os.path.join(tree, "include"), "-Xptxas", "-v", "-cubin", "-o", cubin,
                        os.path.join(csrc, "env_kernels.cu")], capture_output=True, text=True)
    if r.returncode != 0:
        raise SystemExit(r.stdout + r.stderr)
    return cubin, r.stdout + r.stderr


def _ptxas(log, mangled):
    lines = log.splitlines()
    for n, line in enumerate(lines):
        if f"'{mangled}'" in line and "Compiling entry" in line:
            text = " ".join(lines[n + 1:n + 4])
            num = lambda pat: int(re.search(pat, text).group(1))
            return {"registers": num(r"Used (\d+) registers"), "stack_bytes": num(r"(\d+) bytes stack frame"),
                    "spill_store_bytes": num(r"(\d+) bytes spill stores"), "spill_load_bytes": num(r"(\d+) bytes spill loads")}
    raise SystemExit(f"{mangled}: no ptxas report")


def _sass(cubin, mangled):
    out = subprocess.run(["cuobjdump", "-sass", "-fun", mangled, cubin], capture_output=True, text=True, check=True).stdout
    return [(int(m.group(1), 16), m.group(2)) for m in map(INS.match, out.splitlines()) if m]


def _branch(ins):
    """(target, conditional) of a branch instruction, else None."""
    m = re.match(r"(@!?U?P\w+\s+)?BRA(\.U)?\s+(!?U?P\w+,\s*)?(0x[0-9a-f]+)", ins)
    if not m:
        return None
    return int(m.group(4), 16), bool(m.group(1) or m.group(3))


def _loops(code):
    loops = []
    for addr, ins in code:
        b = _branch(ins)
        if b and b[0] <= addr:
            loops.append((b[0], addr))
    return [(h, e) for h, e in loops if not any(h <= h2 and e2 <= e and (h2, e2) != (h, e) for h2, e2 in loops)]


def _shortest(code, head, end):
    """Fewest instructions from `head` through the back edge at `end`, and the branches and done stores on that path."""
    body = [(a, ins) for a, ins in code if head <= a <= end]
    index = {a: n for n, (a, _) in enumerate(body)}
    inf = (1 << 30, 0, 0)
    best = [inf] * (len(body) + 1)
    best[0] = (0, 0, 0)
    for n, (a, ins) in enumerate(body):
        if best[n] == inf:
            continue
        c, br, st = best[n]
        here = (c + 1, br + (_branch(ins) is not None), st + ("STG" in ins and ".U8" in ins))
        if a == end:
            best[len(body)] = min(best[len(body)], here)
            continue
        b = _branch(ins)
        nxt = []
        if b is None or b[1]:
            if not re.match(r"(EXIT|RET)", ins):
                nxt.append(n + 1)
        if b and head < b[0] <= end and b[0] in index:
            nxt.append(index[b[0]])
        for m in nxt:
            best[m] = min(best[m], here)
    return best[len(body)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tree", default=ROOT, help="repository tree whose env_kernels.cu is compiled")
    ap.add_argument("--tasks", default="Ball3D,GridWorld,Push")
    args = ap.parse_args()
    with tempfile.TemporaryDirectory(prefix="rollout_sass_") as tmp:
        cubin, log = _compile(os.path.abspath(args.tree), tmp)
        for task in args.tasks.split(","):
            name = f"{task}Task"
            mangled = f"_Z19rollout_fast_kernelI{len(name)}{name}Ev7EnvPtrsjmmmiP6float4PiPfPh"
            res = _ptxas(log, mangled)
            code = _sass(cubin, mangled)
            print(f"rollout_fast_kernel<{name}>: {res['registers']} registers, stack {res['stack_bytes']} B, "
                  f"spills {res['spill_store_bytes']} B stored / {res['spill_load_bytes']} B loaded, {len(code) * 16} B of code")
            for head, end in _loops(code):
                ins, br, steps = _shortest(code, head, end)
                if not steps:                                    # a wait loop, not a step loop
                    continue
                per = f", per step {ins / steps:.1f} instructions and {br / steps:.1f} branches"
                print(f"    loop 0x{head:x}-0x{end:x}: {end + 16 - head} B, shortest path {ins} instructions, "
                      f"{br} branches, {steps} steps{per}")


if __name__ == "__main__":
    sys.exit(main())
