"""GPU: analogue jobs -- a parent molecule forward-diffused to a diffusion level and denoised from there, optionally with
some atoms fixed (mlcg_analogue_inputs, mlcg_sample modes 2 and 3, mlcg_generate_analogue_jobs, jobs.run_packed,
MLConformerGenerator.generate_jobs).  The loop is checked against the CPU reference edm_analogue with injected noise in fp32;
the graphed call against the eager composition, and every packed job against the job alone, bit for bit: float bit
patterns, so NaN positions count (random-init 16-bit trajectories may leave the finite range, DESIGN section 3)."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from analogue_oracle import edm_analogue
from conftest import GOLDEN, rel_l2
from ml_conformer_generator_b200 import _lib
from ml_conformer_generator_b200 import jobs as J
from ml_conformer_generator_b200.config import CONTEXT_NORMS
from ml_conformer_generator_b200.mol_utils import (get_context_shape, normalise_context, read_mol_heavy_atoms,
                                                   symbols_to_one_hot)

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
T, L = 10, 4


def _mol(name):
    """Heavy atoms of a stored molfile: (coordinates (n,3), one-hot (n,8))."""
    symbols, x = read_mol_heavy_atoms(os.path.join(GOLDEN, name + ".mol"))
    return x.float(), symbols_to_one_hot(symbols).float()


def _parent(n, seed):
    """A compact random skeleton of n atoms (1.5 A random walk) away from the origin, classes 0..6."""
    g = torch.Generator().manual_seed(seed)
    steps = torch.randn(n, 3, generator=g)
    steps = 1.5 * steps / steps.norm(dim=1, keepdim=True)
    x = torch.cumsum(steps, 0) * 0.6 + torch.tensor([2.0, -1.0, 4.0]) * (seed % 4)
    return x, torch.eye(8)[torch.randint(0, 7, (n,), generator=g)]


def _bits(t):
    t = torch.as_tensor(t).detach().cpu()
    return t.view(torch.int32) if t.dtype == torch.float32 else t


def _same(a, b, what=""):
    if isinstance(a, dict):
        assert a.keys() == b.keys()
        for k in a:
            _same(a[k], b[k], k)
        return
    u, v = _bits(a), _bits(b)
    assert u.dtype == v.dtype and u.shape == v.shape, what
    assert torch.equal(u, v), what


def _flags(n, idx):
    f = np.zeros(n, np.int32)
    f[list(idx)] = 1
    return f


@pytest.mark.parametrize("fixed", [False, True])
def test_parent_inputs_and_loop_match_the_oracle_fp32(engines, state_dicts, fixed):
    from oracle import edm_oracle as O
    e = engines("fp32")
    parents = [_mol("yibfeu"), _mol("ceyyag")]
    job = np.array([0, 1, 0], np.int32)
    n_of = [p[0].shape[0] for p in parents]
    n_nodes = torch.tensor([n_of[j] for j in job])
    B, N = len(job), max(n_of) + 1  # one padded slot even for the larger parent
    centred = [(x - x.mean(0), h) for x, h in parents]
    flags = [_flags(n, [0, 2, 5]) for n in n_of] if fixed else None
    zk, fm = e.analogue_inputs(job, centred, flags, N)
    want_zk, want_fm = torch.zeros(B, N, 11), torch.zeros(B, N)
    for b, j in enumerate(job):
        n = n_of[j]
        want_zk[b, :n, :3], want_zk[b, :n, 3:] = centred[j]
        if fixed:
            want_fm[b, :n] = torch.from_numpy(flags[j]).float()
    _same(zk, want_zk, "z_known")
    _same(fm, want_fm, "fixed_mask")
    ctx = torch.stack([normalise_context(get_context_shape(centred[j][0])[0], CONTEXT_NORMS) for j in job])
    nm, em = O.prepare_masks(n_nodes, N)
    r, bp = 1, 3
    n_draw = 1 + (L + 1) * (2 if fixed else 1) * r + 1
    tape = O.NoiseTape.draw(n_draw, B, N, 7)
    with torch.no_grad():
        x_ref, h_ref = edm_analogue(state_dicts[0], O.gamma_table(T), nm, em, want_fm.unsqueeze(-1),
                                    ctx.view(B, 1, 3) * nm, want_zk, tape, L, r, bp)
    e.set_batch(n_nodes.numpy(), N)
    x, cls = e.sample(ctx, T, "merge" if fixed else "analogue", r, z_known=zk, fixed_mask=fm, diffusion_level=L,
                      blend_power=bp, noise_tape=tape.stacked())
    err = rel_l2(x.cpu(), x_ref)
    print("analogue fixed=%s free-running x rel-L2 %.3e" % (fixed, err))
    assert err < 5e-3  # the merge golden test's tolerance
    real = nm.squeeze(-1) > 0
    assert bool((cls.cpu().long()[real] == h_ref.argmax(-1)[real]).all())
    assert bool((cls.cpu()[~real] == -1).all())


def _eager(e, nn, N, ctx, job, parents, flags, seed, ids):
    """mlcg_generate_analogue_jobs composed of its eager steps: parent inputs -> mlcg_sample -> GCN."""
    e.set_batch(nn, N)
    zk, fm = e.analogue_inputs(job, parents, flags, N)
    fixed = flags is not None and any(np.asarray(f).any() for f in flags)
    x, cls = e.sample(torch.from_numpy(ctx), T, "merge" if fixed else "analogue", 0, z_known=zk, fixed_mask=fm,
                      diffusion_level=L, blend_power=3, seed=seed, sample_ids=ids)
    el, dist, adj = e.seer_inputs(x, cls)
    _, bonds = e.seer_forward(el, dist, adj, want_logits=False)
    return x.cpu(), cls.cpu(), bonds.cpu()


def _call_inputs(seed, fixed, sizes=(14, 22, 9)):
    parents = [_parent(n, seed + k) for k, n in enumerate(sizes)]
    parents = [(x - x.mean(0), h) for x, h in parents]
    flags = [_flags(x.shape[0], [1, 4]) for x, _ in parents] if fixed else None
    job = np.array([2, 0, 1, 0, 2, 2, 1, 0], np.int32)
    nn = np.array([sizes[j] for j in job], np.int32)
    ctx = np.stack([normalise_context(get_context_shape(parents[j][0])[0], CONTEXT_NORMS).numpy() for j in job])
    ids = ((300 + job.astype(np.int64)) << 32) + np.arange(job.size)
    return nn, max(sizes), ctx.astype(np.float32), job, parents, flags, ids


@pytest.mark.parametrize("precision", ["fp16", "bf16"])
@pytest.mark.parametrize("fixed", [False, True])
def test_graphed_call_equals_the_eager_composition(engines, precision, fixed):
    e = engines(precision)
    nn, N, ctx, job, parents, flags, ids = _call_inputs(0, fixed)
    want = _eager(e, nn, N, ctx, job, parents, flags, 5, ids)
    captures = []
    for _ in range(3):  # 1st call eager, 2nd captured into a CUDA graph, 3rd a replay
        c0 = e.graph_captures()
        got = e.generate_analogue_jobs_host(nn, N, ctx, job, parents, flags, T, 0, 3, L, seed=5, sample_ids=ids)
        captures.append(e.graph_captures() - c0)
        for a, b, k in zip(got, want, ("x", "atom_class", "bonds")):
            _same(a, b, k)
    assert captures == [0, 1, 0]
    # other parents (and flags) of the same sizes replay the graph with the new inputs
    nn2, _, ctx2, _, parents2, flags2, _ = _call_inputs(10, fixed)
    if fixed:
        flags2 = [_flags(x.shape[0], [0, 3, 5]) for x, _ in parents2]
    c0 = e.graph_captures()
    got = e.generate_analogue_jobs_host(nn2, N, ctx2, job, parents2, flags2, T, 0, 3, L, seed=5, sample_ids=ids)
    assert e.graph_captures() == c0
    want2 = _eager(e, nn2, N, ctx2, job, parents2, flags2, 5, ids)
    for a, b, k in zip(got, want2, ("x", "atom_class", "bonds")):
        _same(a, b, k)
    assert not torch.equal(_bits(got[0]), _bits(want[0]))


@pytest.fixture(scope="module")
def generators(state_dicts):
    from ml_conformer_generator_b200 import MLConformerGenerator
    made = {}

    def get(precision, steps=T):
        if (precision, steps) not in made:
            made[precision, steps] = MLConformerGenerator(diffusion_steps=steps, device=torch.device("cuda:0"),
                                                          precision=precision, edm_state_dict=state_dicts[0],
                                                          adj_mat_seer_state_dict=state_dicts[1])
        return made[precision, steps]

    yield get
    for g in made.values():
        g.engine.close()


def _analogue_jobs():
    """Analogue jobs with and without fixed atoms at two levels, one of them a stored molecule."""
    return [
        dict(parent_molecule=_parent(17, 1), n_samples=5, job_id=500),
        dict(parent_molecule=_parent(24, 2), n_samples=4, fixed_atoms=[0, 5, 9], job_id=501),
        dict(parent_molecule=_parent(11, 3), n_samples=3, diffusion_level=2, job_id=502),
        dict(parent_molecule=_mol("yibfeu"), n_samples=6, fixed_atoms=[2], diffusion_level=2, job_id=503),
        dict(parent_molecule=_parent(30, 4), n_samples=2, reference_context=[60.0, 120.0, 170.0], job_id=504),
    ]


def test_packed_analogue_jobs_equal_each_job_alone(generators):
    import test_gpu_jobs as G
    gen = generators("bf16")
    jobs = _analogue_jobs()
    whole = gen.generate_jobs(jobs, ifm_diffusion_level=L, seed=5)
    for j, job in enumerate(jobs):
        _same(whole[j], gen.generate_jobs([job], ifm_diffusion_level=L, seed=5)[0])
        assert whole[j]["x"].shape == (job["n_samples"], job["parent_molecule"][0].shape[0], 3)
    perm = [3, 0, 4, 2, 1]
    shuffled = gen.generate_jobs([jobs[p] for p in perm], ifm_diffusion_level=L, seed=5)
    for k, p in enumerate(perm):
        _same(shuffled[k], whole[p])
    straddled = gen.generate_jobs(jobs, ifm_diffusion_level=L, seed=5, max_batch=4)  # jobs straddle calls
    for a, b in zip(whole, straddled):
        _same(a, b)
    # next to plain, inpainting and IFM jobs in one call: every output as without the others
    others = [dict(j, job_id=600 + k) for k, j in enumerate(G._jobs("plain")[:2] + G._jobs("inpaint")[2:4] +
                                                             G._jobs("ifm")[4:])]
    mixed = gen.generate_jobs(others[:3] + jobs + others[3:], ifm_diffusion_level=L, seed=5)
    alone = gen.generate_jobs(others, ifm_diffusion_level=L, seed=5)
    for a, b in zip(mixed[:3] + mixed[-3:], alone):
        _same(a, b)
    for a, b in zip(mixed[3:-3], whole):
        _same(a, b)


def test_level_one_returns_the_parent_and_fixed_atoms_keep_their_classes(generators):
    # fp32 keeps the random-init trajectories finite; L = 1 of T = 100 noises the parent by sigma ~ 0.014
    gen = generators("fp32", 100)
    parents = [_parent(18, 7), _mol("ceyyag")]
    res = gen.generate_jobs([dict(parent_molecule=p, n_samples=8, diffusion_level=1) for p in parents], seed=2)
    for (x, h), r in zip(parents, res):
        ok = h[:, :7].sum(1) > 0  # class 7 (Br) cannot be decoded
        assert bool((r["atom_class"][:, ok].long() == h.argmax(-1)[ok].view(1, -1)).all())
        rms = float(((r["x"] - x.view(1, -1, 3)) ** 2).sum(-1).mean().sqrt())
        print("L = 1: RMS distance to the parent %.4f A" % rms)
        assert rms < 0.1  # measured 0.03 A on a B200; in the parent's input frame
    gen = generators("fp32")
    x, h = _parent(20, 8)
    fix = [0, 3, 4, 11, 19]
    for level in (1, L, T):
        r = gen.generate_jobs([dict(parent_molecule=(x, h), n_samples=6, fixed_atoms=fix, diffusion_level=level)], seed=3)[0]
        assert bool((r["atom_class"][:, fix].long() == h.argmax(-1)[fix].view(1, -1)).all()), level


def test_scores_and_keep_best_on_analogue_jobs_equal_evaluate(generators):
    from ml_conformer_generator_b200.shape_similarity import ShapeScorer
    gen = generators("bf16")
    sc = ShapeScorer(gen.engine)
    jobs = [dict(j, reference_conformer=j["parent_molecule"][0], diffusion_level=2) for j in _analogue_jobs()]
    plain = gen.generate_jobs([{k: v for k, v in j.items() if k != "reference_conformer"} for j in jobs], seed=5)
    full = gen.generate_jobs(jobs, seed=5)
    for j, r in enumerate(full):
        for k in plain[j]:
            _same(r[k], plain[j][k], k)
        assert bool(torch.isfinite(r["x"]).all())
        want = sc.evaluate(jobs[j]["reference_conformer"], r["x"], r["n_nodes"])
        for k in ("shape_tanimoto", "best_orientation", "aligned_coords", "reference_coords"):
            _same(r[k], want[k], "%s of job %d" % (k, j))
    best = gen.generate_jobs(jobs, seed=5, keep_best=2)
    for j, r in enumerate(best):
        f = full[j]
        order = sorted(range(f["x"].shape[0]), key=lambda i: (-float(f["shape_tanimoto"][i]), i))[:2]
        assert r["sample_index"].tolist() == order
        for k in ("x", "atom_class", "n_nodes", "bonds", "shape_tanimoto", "best_orientation", "aligned_coords"):
            _same(r[k], f[k][torch.tensor(order)], k)
    # the kept rows go back in as parents
    again = [dict(parent_molecule=(r["x"][0], torch.nn.functional.one_hot(r["atom_class"][0].long(), 8)), n_samples=3,
                  fixed_atoms=[0]) for r in best]
    for r, job in zip(gen.generate_jobs(again, ifm_diffusion_level=L, seed=6), again):
        assert r["x"].shape == (3, job["parent_molecule"][0].shape[0], 3)
        assert bool((r["atom_class"][:, 0] == job["parent_molecule"][1][0].argmax()).all())


def _raw(e, job, n_atoms, fixed, n_nodes, level=L, N=25, null=None, T_=T):
    """mlcg_generate_analogue_jobs through ctypes with every pointer valid unless named in `null`."""
    B, J_ = len(n_nodes), len(n_atoms)
    job = np.ascontiguousarray(job, dtype=np.int32)
    na = np.ascontiguousarray(n_atoms, dtype=np.int32)
    tot = max(int(na.clip(min=0).sum()), 1)
    px, ph = np.zeros((tot, 3), np.float32), np.tile(np.eye(8, dtype=np.float32)[:1], (tot, 1))
    fx = np.zeros(tot, np.int32)
    fx[:len(fixed)] = fixed
    ptr = {"job": job.ctypes.data, "n_atoms": na.ctypes.data, "coords": px.ctypes.data, "one_hot": ph.ctypes.data,
           "fixed": fx.ctypes.data}
    for k in null or ():
        ptr[k] = None
    aj = _lib.AnalogueJobs(J_, ptr["job"], ptr["n_atoms"], ptr["coords"], ptr["one_hot"], ptr["fixed"], level, 0.5, 0.5)
    nn = np.ascontiguousarray(n_nodes, dtype=np.int32)
    ctx = np.zeros((B, 3), np.float32)
    steps = e._steps_cached(T_, 3)[1]
    out = [torch.empty(B, N, 3), torch.empty(B, N, dtype=torch.int32), torch.empty(B, 42, 42, dtype=torch.int8)]
    rc = e.lib.mlcg_generate_analogue_jobs(e.h, C.byref(aj), nn.ctypes.data_as(C.c_void_p), B, N, ctx.ctypes.data, T_,
                                           steps, 0, 1.0, 1.0, 1.0, 0, 0, None, out[0].data_ptr(), out[1].data_ptr(),
                                           out[2].data_ptr(), e._stream())
    e._check(rc, "generate_analogue")


def test_c_abi_argument_errors(engines):
    e = engines("fp16")
    nn = [10, 12, 10, 12]
    _raw(e, [0, 1, 0, 1], [10, 12], [], nn)  # valid
    with pytest.raises(ValueError, match="job index out of range"):
        _raw(e, [0, 2, 0, 1], [10, 12], [], nn)
    with pytest.raises(ValueError, match="job index out of range"):
        _raw(e, [0, -1, 0, 1], [10, 12], [], nn)
    with pytest.raises(ValueError, match="n_nodes must equal the parent's atom count"):
        _raw(e, [0, 1, 0, 1], [10, 12], [], [10, 12, 11, 12])
    with pytest.raises(ValueError, match="all have fixed atoms or all have none"):
        _raw(e, [0, 1, 0, 1], [10, 12], [1], nn)  # job 0 has a fixed atom, job 1 none
    with pytest.raises(ValueError, match="every atom of the parent is fixed"):
        _raw(e, [0, 0, 0, 0], [3], [1, 1, 1], [3] * 4)
    for level in (0, T + 1):
        with pytest.raises(ValueError, match=r"diffusion_level must lie in \[1, T\]"):
            _raw(e, [0, 1, 0, 1], [10, 12], [], nn, level=level)
    with pytest.raises(ValueError, match="1 <= n_atoms <= N"):
        _raw(e, [0, 1, 0, 1], [10, 26], [], [10, 26, 10, 26])
    with pytest.raises(ValueError, match="n_jobs >= 1"):
        _raw(e, [0, 0, 0, 0], [], [], nn)
    with pytest.raises(ValueError, match="1 <= N <= 39"):
        _raw(e, [0, 1, 0, 1], [10, 12], [], nn, N=40)
    for k in ("job", "n_atoms", "coords", "one_hot", "fixed"):
        with pytest.raises(ValueError, match="null pointer"):
            _raw(e, [0, 1, 0, 1], [10, 12], [], nn, null=[k])
    with pytest.raises(ValueError, match="analogue needs z_known"):
        e.set_batch([10, 12], 12)
        e.sample(torch.zeros(2, 3), T, "analogue", 0, diffusion_level=L)
    from ml_conformer_generator_b200.engine import Engine
    bare = Engine(torch.device("cuda:0"), "fp16")  # no weights
    try:
        with pytest.raises(ValueError, match="load both weight sets first"):
            _raw(bare, [0, 1, 0, 1], [10, 12], [], nn)
    finally:
        bare.close()
    # a failed call leaves the handle usable
    nn_, N, ctx, job, parents, flags, ids = _call_inputs(0, True)
    got = e.generate_analogue_jobs_host(nn_, N, ctx, job, parents, flags, T, 0, 3, L, seed=5, sample_ids=ids)
    for a, b, k in zip(got, _eager(e, nn_, N, ctx, job, parents, flags, 5, ids), ("x", "atom_class", "bonds")):
        _same(a, b, k)


_TWO_RANK = r"""
import os, sys, numpy as np, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
sys.path.insert(0, os.path.join(sys.argv[1], "tests"))
from ml_conformer_generator_b200.engine import Engine
from ml_conformer_generator_b200.shape_similarity import ShapeScorer
from ml_conformer_generator_b200.weights import random_state_dicts
from ml_conformer_generator_b200 import parallel as P, jobs as J
import test_gpu_analogue_jobs as A
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(rank)
dev = torch.device("cuda", rank)
dist.init_process_group("nccl", device_id=dev)
sd, ssd = random_state_dicts(0)
e = Engine(dev, "bf16"); e.load_edm_state_dict(sd); e.load_seer_state_dict(ssd)
ok = True
scored = [dict(j, reference_conformer=j["parent_molecule"][0], diffusion_level=2) for j in A._analogue_jobs()]
for jobs, keep in ((A._analogue_jobs(), None), (scored, 2)):
    got = P.generate_jobs_sharded(e, jobs, T=A.T, ifm_diffusion_level=A.L, seed=5, keep_best=keep)
    if rank == 0:
        packed = J.flatten_jobs(jobs, seed=5)
        idx = np.arange(packed.ids.size)
        x, cls, bonds = J.run_packed(e, packed, idx, A.T, 0, 3, A.L, 5, 8192, True)
        want = J.split_jobs(packed, x, cls, bonds)
        if keep:
            want = J.attach_scores(packed, want, *J.score_packed(ShapeScorer(e), packed, idx, x), keep)
        for a, b in zip(got, want):
            ok = ok and a.keys() == b.keys()
            for k in a:
                u, v = A._bits(a[k]), A._bits(b[k])
                ok = ok and u.shape == v.shape and torch.equal(u, v)
if rank == 0:
    print("SHARDED_ANALOGUE_JOBS_EQUAL_SINGLE", ok)
dist.barrier()
dist.destroy_process_group()
"""


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_rank_sharded_analogue_jobs_equal_single_gpu(tmp_path):
    script = tmp_path / "two_rank_analogue.py"
    script.write_text(_TWO_RANK)
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
                          "127.0.0.1", "--master-port", "29549", str(script), ROOT], capture_output=True, text=True,
                         timeout=900)
    assert out.returncode == 0, out.stderr[-3000:]
    assert "SHARDED_ANALOGUE_JOBS_EQUAL_SINGLE" in out.stdout and "SHARDED_ANALOGUE_JOBS_EQUAL_SINGLE True" in out.stdout
