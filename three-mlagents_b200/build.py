"""Builds libtmla.so (the C-ABI CUDA library) in-tree for sm_100a with nvcc.

    python three-mlagents_b200/build.py [--force]

nvcc cross-compiles without a GPU; the resulting `lib/libtmla.so` is git-ignored but travels to the
GPU box with the repository snapshot.
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_DIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIB_DIR, "libtmla.so")
SOURCES = ["error.cu", "env_kernels.cu", "rollout.cu", "comm.cu", "ppo_kernels.cu", "mlp_kernels.cu", "mlp_small.cu", "mlp_tc.cu", "mlp_fwd_pipe.cu", "mlp_train.cu", "det_reduce.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr",
] + os.environ.get("TMLA_EXTRA_NVCC_FLAGS", "").split()      # e.g. -DTMLA_PHASE_CLOCKS for profiles/phase_clocks.py


def _nvcc() -> str:
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found: libtmla.so cannot be built (there is no CPU fallback)")
    return exe


def _digest(paths) -> str:
    h = hashlib.sha256()
    for p in sorted(paths):
        with open(p, "rb") as f:
            h.update(p.encode())
            h.update(f.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(LIB_DIR, exist_ok=True)
    srcs = [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    deps = srcs + [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    deps.append(os.path.join(os.path.dirname(HERE), "include", "tmla.h"))
    stamp = os.path.join(LIB_DIR, "libtmla.sha256")
    digest = _digest(deps)
    if not force and os.path.exists(LIB) and os.path.exists(stamp) and open(stamp).read().strip() == digest:
        return LIB
    nvcc = _nvcc()
    objs = []
    procs = []
    for s in srcs:
        o = os.path.join(LIB_DIR, os.path.basename(s)[:-3] + ".o")
        objs.append(o)
        cmd = [nvcc, *NVCC_FLAGS, "-c", s, "-o", o]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for cmd, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            raise RuntimeError("nvcc failed: " + " ".join(cmd) + "\n" + out)
        if verbose and out:
            print(out)
    link = [nvcc, "-shared", "-o", LIB, *objs, "-gencode", "arch=compute_100a,code=sm_100a"]
    r = subprocess.run(link, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed: " + " ".join(link) + "\n" + r.stdout)
    with open(stamp, "w") as f:
        f.write(digest)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
