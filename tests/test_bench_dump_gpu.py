"""bench.py --dump-outputs: the sample of the last timed rollout is the same from run to run with the same arguments, changes
with --steps, and stays within 64 MB of float32 arrays."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = ("obs", "actions", "rewards", "dones")


def _bench_dump(out_dir, steps):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--quick", "--steps", str(steps), "--warmup", "1",
                        "--dump-outputs", str(out_dir)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    assert json.loads(p.stdout.strip())["value"] > 0
    return {n: np.load(os.path.join(out_dir, f"{n}.npy")) for n in NAMES}


@pytest.mark.gpu
def test_dump_outputs_are_reproducible_and_follow_steps(tmp_path):
    a = _bench_dump(tmp_path / "a", 2)
    b = _bench_dump(tmp_path / "b", 2)
    c = _bench_dump(tmp_path / "c", 3)
    T, n = a["actions"].shape
    assert a["obs"].shape == (T, n, 6) and a["rewards"].shape == a["dones"].shape == (T, n)
    assert all(x.dtype == np.float32 for x in a.values()) and sum(x.nbytes for x in a.values()) <= 64 << 20
    assert set(np.unique(a["actions"]).tolist()) == {0, 1, 2, 3, 4} and set(np.unique(a["dones"]).tolist()) == {0, 1}
    assert np.isfinite(a["obs"]).all() and np.isfinite(a["rewards"]).all()
    for name in NAMES:
        assert np.array_equal(a[name], b[name]), name
    assert not np.array_equal(a["actions"], c["actions"]) and not np.array_equal(a["obs"], c["obs"])
