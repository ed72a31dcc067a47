"""CPU: the reference arm of bench.py (the reference's own formulation on host cores) runs without a GPU and prints one JSON
line with the keys the bench contract asks for."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--ref-mols", "2"],
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "mols/s" and d["higher_is_better"] is True
    assert d["metric"].startswith("generated mols/sec") and d["n_gpus"] == 1 and d["steps"] == 1
    assert d["value"] > 0 and d["ms_per_step"] > 0
    # "reference" = the reference's own modules (staged copy oracle/_ref or /root/reference), "port" = oracle fallback
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "mols/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and d["config"]["workload"].startswith("C3")


def test_committed_bench_lines_follow_contract():
    """The bench lines kept under profiles/ (what DESIGN.md section 8 quotes) carry every key the contract asks for, and their
    derived numbers are consistent: roofline.frac = achieved / peak, achieved = algorithmic FLOPs per launch / launch time,
    value = molecules per step / step time, e2e below the device-timed value, clocks sampled and not thermally throttled."""
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r2_bench_default*.json")) +
                   glob.glob(os.path.join(ROOT, "profiles", "r2_bench_bf16.json")) +
                   glob.glob(os.path.join(ROOT, "profiles", "r2_bench_2gpu.json")))
    assert files
    for f in files:
        d = json.loads([ln for ln in open(f).read().splitlines() if ln.startswith("{")][-1])
        for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                  "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "clocks", "roofline"):
            assert k in d, (f, k)
        assert d["unit"] == "mols/s" and d["higher_is_better"] is True and d["vs_baseline"] is None and d["warmup"] >= 3
        assert d["dtype"] in ("fp16", "bf16") and d["data"] == "synthetic" and "workload" in d["config"] and "model" not in d["config"]
        per_gpu = int(d["config"]["per_gpu_batch"])
        assert abs(d["value"] - d["n_gpus"] * per_gpu / (d["ms_per_step"] * 1e-3)) / d["value"] < 1e-6
        e = d["e2e"]
        assert e["unit"] == "mols/s" and e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0
        assert 0.9 * d["value"] < e["value"] < 1.02 * d["value"]   # host buffers in the timed region: a little below
        assert d["gpu_launches"] > 10000                           # 101 forwards x 117 launches + step kernels + GCN
        r = d["roofline"]
        assert r["bound"] == "tensor" and r["unit"] == "TFLOP/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
        assert abs(r["achieved"] - r["alg_flops_per_launch"] / (r["launch_ms"] * 1e-3) / 1e12) / r["achieved"] < 1e-6
        assert 0.3 < r["frac"] < 1.0
        c = d["clocks"]
        assert c["sm_mhz"] > 0.8 * c["sm_max_mhz"] and not set(c["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
        if d["n_gpus"] == 1 and "cpu_baseline" in d:
            b = d["cpu_baseline"]
            assert b["kind"] in ("reference", "port") and b["cores"] >= 1 and b["unit"] == "mols/s" and b["value"] > 0


def test_dump_outputs_writes_float_arrays_within_budget(tmp_path):
    """--dump-outputs: every array is float32 / float64, all of them together fit DUMP_BYTES, and a job larger than that is
    written as the same seeded sample of molecules on every run."""
    import numpy as np
    import torch
    import bench
    g = torch.Generator().manual_seed(0)
    for B, whole in ((20, True), (9000, False)):
        x = torch.randn(B, 39, 3, generator=g)
        cls = torch.randint(-1, 7, (B, 39), generator=g, dtype=torch.int32)
        bonds = torch.randint(0, 5, (B, 42, 42), generator=g).to(torch.int8)
        runs = []
        for k in range(2):
            d = tmp_path / ("%d_%d" % (B, k))
            bench.dump_outputs(str(d), x, cls, bonds)
            out = {p.stem: np.load(p) for p in d.glob("*.npy")}
            assert sorted(out) == ["atom_class", "bond_orders", "sample_id", "x"]
            assert all(a.dtype in (np.float32, np.float64) for a in out.values())
            assert sum(p.stat().st_size for p in d.glob("*.npy")) <= bench.DUMP_BYTES
            ids = out["sample_id"].astype(np.int64)
            assert np.array_equal(out["sample_id"], ids) and np.all(np.diff(ids) > 0)
            assert (len(ids) == B) == whole and np.array_equal(ids, np.arange(B)) == whole
            assert np.array_equal(out["x"], x.numpy()[ids]) and np.array_equal(out["atom_class"], cls.numpy()[ids])
            assert np.array_equal(out["bond_orders"], bonds.numpy()[ids])
            runs.append(ids)
        assert np.array_equal(runs[0], runs[1])


def test_bench_rejects_arguments_it_cannot_honour():
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True, text=True,
                             timeout=300, cwd=ROOT)
        assert out.returncode == 2 and "error" in out.stderr, (extra, out.stderr[-500:])
