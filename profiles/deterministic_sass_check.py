"""Check that the default (atomic) kernels of this build compile to the same SASS as another build's (e.g. the parent commit's).

    python profiles/deterministic_sass_check.py <other build's lib dir> [<this build's lib dir>]

Deterministic mode adds a `bool DET = false` template parameter to the reducing kernels, which renames their default
instantiations (`tc_wgrad_tiled_kernel` -> `tc_wgrad_tiled_kernel<false>`, `ppo_loss_kernel<5, 0>` -> `ppo_loss_kernel<5, 0,
false>`).  Kernels are matched by their demangled name with that trailing `false` removed; the DET=true instantiations and
other kernels new in this build are listed separately.  Runs on the CPU (cuobjdump + c++filt), no GPU needed.
"""
from __future__ import annotations

import os
import re
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CUOBJDUMP = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "cuobjdump")


def kernels(obj: str) -> dict[str, str]:
    """demangled kernel name -> SASS body (header lines dropped)"""
    out = subprocess.run([CUOBJDUMP, "-sass", obj], capture_output=True, text=True, check=True).stdout
    parts = re.split(r"^\s*Function : (\S+)\s*$", out, flags=re.M)
    names = parts[1::2]
    dem = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True, check=True).stdout.splitlines()
    res = {}
    for name, body in zip(dem, parts[2::2]):
        lines = [ln.strip() for ln in body.splitlines() if ln.strip() and not ln.strip().startswith(("..", "Fatbin", "code for", "arch =", "host ="))]
        res[name] = "\n".join(lines)
    return res


def default_name(name: str) -> str:
    """the parent's name of a DET=false instantiation: `void f<false>(...)` -> `f(...)`, `void f<6, 5, 0, false>(...)` ->
    `void f<6, 5, 0>(...)` (only the template argument list right before the parameter list is touched)"""
    m = re.match(r"^void (\w+)<false>\(", name)
    if m:
        return name[len("void "):].replace("<false>(", "(", 1)
    return re.sub(r", false>\(", ">(", name, count=1)


def strip_registers(body: str) -> str:
    """instructions with register numbers and encodings removed (register allocation only)"""
    out = []
    for ln in body.splitlines():
        if ln.startswith("/* 0x"):
            continue
        out.append(re.sub(r"\bU?R\d+\b", "R", ln.split(";")[0]))
    return "\n".join(out)


def main() -> None:
    other = sys.argv[1]
    mine = sys.argv[2] if len(sys.argv) > 2 else os.path.join(HERE, "..", "three-mlagents_b200", "lib")
    print("SASS of every kernel of the parent build vs this build (cuobjdump -sass per object, sm_100a; header lines dropped;")
    print("default instantiations matched by name with the new trailing DET=false template argument removed):")
    ok = True
    for obj in sorted(f for f in os.listdir(mine) if f.endswith(".o")):
        if not os.path.exists(os.path.join(other, obj)):
            print(f"{obj} is new: " + ", ".join(k.split("(")[0] for k in kernels(os.path.join(mine, obj))))
            continue
        a, b = kernels(os.path.join(other, obj)), kernels(os.path.join(mine, obj))
        match, renamed = {}, 0
        for k in a:                                    # the same name, else a DET=false instantiation that carried it
            if k in b:
                match[k] = k
            else:
                cand = [x for x in b if default_name(x) == k]
                if cand:
                    match[k] = cand[0]
                    renamed += 1
        same = [k for k in match if b[match[k]] == a[k]]
        regs = [k for k in match if b[match[k]] != a[k] and strip_registers(b[match[k]]) == strip_registers(a[k])]
        diff = [k for k in match if k not in same and k not in regs]
        gone = [k for k in a if k not in match]
        new = [k for k in b if k not in match.values()]
        line = f"{obj}: {len(same)} of {len(a)} kernels SASS-identical"
        if renamed:
            line += f" ({renamed} of them renamed by the DET=false template argument)"
        if new:
            line += f"; {len(new)} new kernels"
        print(line)
        for k in new:
            print(f"  new: {k.split('(')[0]}")
        for k in regs:
            print(f"  same instructions, different register numbers: {k.split('(')[0]}")
        for k in diff:
            print(f"  DIFFERENT: {k}")
        for k in gone:
            print(f"  MISSING: {k}")
        ok = ok and not diff and not gone
    print("no existing kernel differs beyond register numbering" if ok else "DIFFERENCES FOUND")
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
