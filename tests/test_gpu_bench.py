"""GPU: bench.py times exactly --steps steps, and --dump-outputs writes the results of the last timed step, identical
from run to run with the same arguments."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(steps, dump=None):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "C1", "--steps", str(steps), "--warmup", "0",
           "--no-cpu-baseline", "--no-extras"] + (["--dump-outputs", str(dump)] if dump else [])
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-3000:]
    return json.loads([ln for ln in out.stdout.splitlines() if ln.startswith("{")][-1])


def test_steps_and_dump_outputs(tmp_path):
    one, two = _bench(1), _bench(2, tmp_path / "a")
    assert one["steps"] == 1 and two["steps"] == 2
    assert two["gpu_launches"] == 2 * one["gpu_launches"] > 0
    _bench(2, tmp_path / "b")
    a = {n: np.load(tmp_path / "a" / (n + ".npy")) for n in ("x", "atom_class", "bond_orders", "sample_id")}
    b = {n: np.load(tmp_path / "b" / (n + ".npy")) for n in a}
    B, N = 20, 19  # C1: 20 molecules of 15..19 atoms
    assert a["x"].shape == (B, N, 3) and a["atom_class"].shape == (B, N) and a["bond_orders"].shape == (B, 42, 42)
    assert np.array_equal(a["sample_id"], np.arange(B)) and all(v.dtype == np.float32 for k, v in a.items() if k != "sample_id")
    assert np.isfinite(a["x"]).all() and a["atom_class"].max() >= 0
    for n in a:
        assert np.array_equal(a[n], b[n]), n
