"""GPU: scoring many jobs against their own reference conformers in one pass (ShapeScorer.evaluate_jobs ->
mlcg_shape_tanimoto_jobs) and the scored path of generate_jobs / generate_jobs_sharded.  The acceptance rule is bit
equality with the single-reference scorer (ShapeScorer.evaluate, itself pinned to the reference's outputs by
test_gpu_properties) on every job: float bit patterns of scores, aligned coordinates and moments, and the orientation."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import golden
from ml_conformer_generator_b200 import jobs as J
from ml_conformer_generator_b200.shape_similarity import MAX_JOB_REFERENCES, ShapeScorer

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
T, L = 8, 4


def _bits(t):
    t = torch.as_tensor(t).detach().cpu()
    return t.view(torch.int32) if t.dtype == torch.float32 else t


def _same(a, b, what=""):
    a, b = _bits(a), _bits(b)
    assert a.dtype == b.dtype and a.shape == b.shape and torch.equal(a, b), what


def _molecule(rng, n):
    """A compact random heavy-atom skeleton: a random walk of 1.5 A steps, rotated and shifted."""
    steps = rng.normal(size=(n, 3))
    steps *= 1.5 / np.linalg.norm(steps, axis=1, keepdims=True)
    x = np.cumsum(steps, axis=0) * 0.6
    q, _ = np.linalg.qr(rng.normal(size=(3, 3)))
    return torch.from_numpy((x @ q + rng.normal(scale=3.0, size=3)).astype(np.float32))


def test_golden(engines):
    g = golden("shape")
    sc = ShapeScorer(engines("bf16"))
    B = g["coords"].shape[0]
    out = sc.evaluate_jobs([torch.from_numpy(g["ref_xyz"])], torch.from_numpy(g["coords"]), torch.from_numpy(g["n_nodes"]),
                           torch.zeros(B, dtype=torch.long))
    assert out["scores"].is_cuda and out["shape_tanimoto"].is_cuda
    assert float(np.abs(out["scores"].cpu().numpy() - g["scores"]).max()) < 2e-4
    assert np.array_equal(out["best_orientation"].cpu().numpy(), g["best_idx"])
    assert np.allclose(out["aligned_coords"].cpu().numpy(), g["best_coord"], atol=5e-4)
    assert np.allclose(out["reference_coords"][0].cpu().numpy(), g["ref_pts"], atol=5e-4)


def test_many_references_equal_evaluate_per_job_bit_for_bit(engines):
    """~300 jobs, each with its own reference of 3-64 atoms (its own grid), samples in shuffled job order padded to one
    N while each job alone pads to its own, across the 256-reference boundary between calls."""
    sc = ShapeScorer(engines("bf16"))
    rng = np.random.default_rng(11)
    n_jobs = 300
    assert n_jobs > MAX_JOB_REFERENCES
    refs = [_molecule(rng, int(n)) for n in np.concatenate([[3, 64], rng.integers(3, 65, n_jobs - 2)])]
    per_job = rng.integers(1, 4, n_jobs)
    job = rng.permutation(np.repeat(np.arange(n_jobs), per_job))
    n_nodes = rng.integers(5, 49, job.size)
    N = 52
    coords = torch.zeros(job.size, N, 3)
    for b in range(job.size):  # a perturbed copy of (part of) the reference, or an unrelated skeleton
        r = refs[job[b]]
        if b % 3 and r.size(0) >= n_nodes[b]:
            coords[b, :n_nodes[b]] = r[:n_nodes[b]] + torch.from_numpy(rng.normal(scale=0.3, size=(n_nodes[b], 3))).float()
        else:
            coords[b, :n_nodes[b]] = _molecule(rng, int(n_nodes[b]))
    got = sc.evaluate_jobs(refs, coords.cuda(), torch.from_numpy(n_nodes), torch.from_numpy(job))
    assert got["shape_tanimoto"].is_cuda and got["aligned_coords"].shape == (job.size, N, 3)
    assert float(got["shape_tanimoto"].max()) > 0.5  # the scores are not all trivial
    for j in range(n_jobs):
        rows = np.nonzero(job == j)[0]
        nj = int(n_nodes[rows].max())
        want = sc.evaluate(refs[j], coords[rows, :nj], torch.from_numpy(n_nodes[rows]))
        r = torch.from_numpy(rows)
        for k in ("shape_tanimoto", "best_orientation", "scores", "moments"):
            _same(got[k].cpu()[r], want[k], "%s of job %d" % (k, j))
        _same(got["aligned_coords"].cpu()[r, :nj], want["aligned_coords"], "aligned_coords of job %d" % j)
        assert not bool(got["aligned_coords"].cpu()[r, nj:].any())
        _same(got["reference_coords"][j], want["reference_coords"], "reference_coords %d" % j)
        _same(got["reference_moments"][j], want["reference_moments"], "reference_moments %d" % j)
    # a sample's score does not depend on the others in the call
    sub = np.sort(rng.choice(job.size, 40, replace=False))
    part = sc.evaluate_jobs(refs, coords[sub], torch.from_numpy(n_nodes[sub]), torch.from_numpy(job[sub]))
    _same(part["scores"], got["scores"].cpu()[torch.from_numpy(sub)])


def test_input_errors(engines):
    sc = ShapeScorer(engines("bf16"))
    ref, x, nn = torch.randn(5, 3), torch.randn(2, 10, 3), torch.tensor([10, 8])
    with pytest.raises(ValueError, match="3 <= n_ref <= 64"):
        sc.evaluate_jobs([torch.randn(2, 3)], x, nn, [0, 0])
    with pytest.raises(ValueError, match="3 <= n_ref <= 64"):
        sc.evaluate_jobs([ref, torch.randn(65, 3)], x, nn, [0, 0])
    with pytest.raises(ValueError, match=r"job indices must lie in \[0, 2\)"):
        sc.evaluate_jobs([ref, ref], x, nn, [0, 2])
    with pytest.raises(ValueError, match=r"job indices must lie in \[0, 1\)"):
        sc.evaluate_jobs([ref], x, nn, [-1, 0])
    with pytest.raises(ValueError, match="same length"):
        sc.evaluate_jobs([ref], x, nn, [0])
    with pytest.raises(ValueError, match="same length"):
        sc.evaluate_jobs([ref], x, torch.tensor([10]), [0, 0])
    empty = sc.evaluate_jobs([ref], x[:0], nn[:0], [])
    assert empty["shape_tanimoto"].shape == (0,) and len(empty["reference_coords"]) == 1


def _raw(e, J_=2, B=3, N=10, G=8, n_orient=4, null=None):
    """mlcg_shape_tanimoto_jobs through ctypes with valid device buffers unless named in `null`."""
    d = torch.device("cuda:0")
    buf = {"ref_pts": torch.zeros(max(J_, 1), 64, 3, device=d), "n_ref": torch.full((max(J_, 1),), 4, dtype=torch.int32, device=d),
           "axes": torch.zeros(max(J_, 1), 3, max(G, 1), device=d), "coords": torch.zeros(max(B, 1), max(N, 1), 3, device=d),
           "n_nodes": torch.ones(max(B, 1), dtype=torch.int32, device=d), "job": torch.zeros(max(B, 1), dtype=torch.int32, device=d),
           "frames": torch.zeros(max(B, 1), 12, device=d), "orient": torch.eye(3, device=d).reshape(1, 9).repeat(4, 1),
           "workspace": torch.zeros(max(J_, 1) * (max(G, 1) ** 3 + 1), device=d),
           "scores": torch.zeros(max(B, 1), 4, device=d), "aligned": torch.zeros(max(B, 1), 4, max(N, 1), 3, device=d)}
    p = {k: C.c_void_p(v.data_ptr()) for k, v in buf.items()}
    for k in null or ():
        p[k] = None
    rc = e.lib.mlcg_shape_tanimoto_jobs(e.h, p["ref_pts"], p["n_ref"], p["axes"], J_, p["coords"], p["n_nodes"], p["job"], B,
                                        N, p["frames"], p["orient"], n_orient, G, 2.7, 1.6, p["workspace"], p["scores"],
                                        p["aligned"], e._stream())
    e._check(rc, "shape_tanimoto_jobs")
    torch.cuda.synchronize()
    return buf


def test_c_abi_argument_errors(engines):
    e = engines("bf16")
    for k in ("ref_pts", "n_ref", "axes", "coords", "n_nodes", "job", "frames", "orient", "workspace", "scores"):
        with pytest.raises(ValueError, match="shape_tanimoto_jobs"):
            _raw(e, null=[k])
    for kw in (dict(J_=0), dict(B=0), dict(N=0), dict(N=65), dict(n_orient=0), dict(n_orient=65536), dict(G=1), dict(G=49)):
        with pytest.raises(ValueError, match="shape_tanimoto_jobs"):
            _raw(e, **kw)
    _raw(e, null=["aligned"])  # aligned is optional
    _raw(e, N=64, G=48)
    test_golden(engines)  # a failed call leaves the handle usable


@pytest.fixture(scope="module")
def generators(state_dicts):
    from ml_conformer_generator_b200 import MLConformerGenerator
    gen = MLConformerGenerator(diffusion_steps=T, device=torch.device("cuda:0"), precision="bf16",
                               edm_state_dict=state_dicts[0], adj_mat_seer_state_dict=state_dicts[1])
    yield gen
    gen.engine.close()


def _conformer(k):
    """The golden reference conformer, rotated and stretched per job."""
    x = torch.from_numpy(golden("shape")["ref_xyz"])
    a = 0.4 * k
    rot = torch.tensor([[np.cos(a), -np.sin(a), 0.0], [np.sin(a), np.cos(a), 0.0], [0.0, 0.0, 1.0]], dtype=torch.float32)
    return (x - x.mean(0)) @ rot * (1.0 + 0.05 * k)


def _jobs(kind, scored=(0, 1, 2, 3, 4, 5)):
    import test_gpu_jobs as G
    return [dict(j, reference_conformer=_conformer(k)) if k in scored else j for k, j in enumerate(G._jobs(kind))]


@pytest.mark.parametrize("kind", ["plain", "ifm"])
def test_generate_jobs_scores_equal_evaluate_and_keep_best_keeps_the_top(generators, kind):
    gen = generators
    sc = ShapeScorer(gen.engine)
    plain = gen.generate_jobs(_jobs(kind, scored=()), ifm_diffusion_level=L, seed=5)
    mixed = gen.generate_jobs(_jobs(kind, scored=(0, 2, 3)), ifm_diffusion_level=L, seed=5)
    full = gen.generate_jobs(_jobs(kind), ifm_diffusion_level=L, seed=5)
    for j in range(len(plain)):
        for res in (mixed, full):
            for k in plain[j]:
                _same(res[j][k], plain[j][k], k)  # the molecules are those generated without references
        if j not in (0, 2, 3):
            assert mixed[j].keys() == plain[j].keys()
        r = full[j]
        assert bool(torch.isfinite(r["x"]).all())
        want = sc.evaluate(_conformer(j), r["x"], r["n_nodes"])
        for k in ("shape_tanimoto", "best_orientation", "aligned_coords", "reference_coords"):
            _same(r[k], want[k], "%s of job %d" % (k, j))
            if j in (0, 2, 3):
                _same(mixed[j][k], want[k], k)
    for k_best in (3, 100):
        best = gen.generate_jobs(_jobs(kind), ifm_diffusion_level=L, seed=5, keep_best=k_best)
        for j, r in enumerate(best):
            f = full[j]
            n = f["x"].shape[0]
            order = sorted(range(n), key=lambda i: (-float(f["shape_tanimoto"][i]), i))[:k_best]
            assert r["sample_index"].tolist() == order
            idx = torch.tensor(order)
            for k in ("x", "atom_class", "n_nodes", "bonds", "shape_tanimoto", "best_orientation", "aligned_coords"):
                _same(r[k], f[k][idx], k)
            _same(r["reference_coords"], f["reference_coords"])
    with pytest.raises(ValueError, match="every job needs a reference_conformer"):
        gen.generate_jobs(_jobs(kind, scored=(1,)), keep_best=2)


_TWO_RANK = r"""
import os, sys, numpy as np, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
sys.path.insert(0, os.path.join(sys.argv[1], "tests"))
from ml_conformer_generator_b200.engine import Engine
from ml_conformer_generator_b200.shape_similarity import ShapeScorer
from ml_conformer_generator_b200.weights import random_state_dicts
from ml_conformer_generator_b200 import parallel as P, jobs as J
import test_gpu_jobs as G
import test_gpu_shape_jobs as S
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(rank)
dev = torch.device("cuda", rank)
dist.init_process_group("nccl", device_id=dev)
sd, ssd = random_state_dicts(0)
e = Engine(dev, "bf16"); e.load_edm_state_dict(sd); e.load_seer_state_dict(ssd)
ok = True
for kind, scored, keep in (("plain", (0, 2, 5), None), ("ifm", (0, 1, 2, 3, 4, 5), 3)):
    jobs = S._jobs(kind, scored)
    got = P.generate_jobs_sharded(e, jobs, T=G.T, ifm_diffusion_level=G.L, seed=5, keep_best=keep)
    if rank == 0:
        packed = J.flatten_jobs(jobs, seed=5)
        idx = np.arange(packed.ids.size)
        x, cls, bonds = G._packed(e, packed, device_out=True)
        want = J.attach_scores(packed, J.split_jobs(packed, x, cls, bonds),
                               *J.score_packed(ShapeScorer(e), packed, idx, x), keep)
        for a, b in zip(got, want):
            ok = ok and a.keys() == b.keys()
            for k in a:
                u, v = S._bits(a[k]), S._bits(b[k])
                ok = ok and u.shape == v.shape and torch.equal(u, v)
if rank == 0:
    print("SHARDED_SCORED_JOBS_EQUAL_SINGLE", ok)
dist.barrier()
dist.destroy_process_group()
"""


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_rank_sharded_scored_jobs_equal_single_gpu(tmp_path):
    script = tmp_path / "two_rank_scored_jobs.py"
    script.write_text(_TWO_RANK)
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
                          "127.0.0.1", "--master-port", "29557", str(script), ROOT], capture_output=True, text=True,
                         timeout=900)
    assert out.returncode == 0, out.stderr[-3000:]
    assert "SHARDED_SCORED_JOBS_EQUAL_SINGLE" in out.stdout and "SHARDED_SCORED_JOBS_EQUAL_SINGLE True" in out.stdout
