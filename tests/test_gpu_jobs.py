"""GPU: many generation jobs packed into few device calls (MLConformerGenerator.generate_jobs, jobs.run_packed,
Engine.generate_fragment_jobs_host -> mlcg_generate_fragment_jobs).  The acceptance rule is that every job's output
equals that job run alone (generate_host / generate_fragment_host with its own atom counts, its own max_n_nodes and the
same sample ids), bit for bit: float bit patterns, so NaN positions count (fp16 random-init inpainting diverges).  The
job alone pads to its own N (and N - n_ff in the first IFM loop); the packed call pads to the largest N of its jobs and to
N - min n_ff, so these tests also cover the sampler's padding and batch invariance."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import golden
from ml_conformer_generator_b200 import _lib
from ml_conformer_generator_b200 import jobs as J
from ml_conformer_generator_b200.config import CONTEXT_NORMS

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
T, L = 8, 4  # small T: random-init inpainting trajectories diverge at large T
KIND_ARGS = {"plain": None, "inpaint": False, "ifm": True}


def _ref(k):
    base = torch.from_numpy(golden("host_utils")["yibfeu_context"]).float()
    return base * (1.0 + 0.07 * k)


def _frag(n, seed):
    """A fragment of n atoms: coordinates around the origin, classes among C N O F S Cl."""
    g = torch.Generator().manual_seed(seed)
    x = 1.4 * torch.randn(n, 3, generator=g)
    return x, torch.eye(8)[torch.randint(0, 6, (n,), generator=g)]


# (n_atoms, variance, n_samples, fragment atoms): different references, atom ranges, sample counts and fragments of
# 2-8 atoms, including a one-sample job
SPECS = [(23, 2, 9, 3), (21, 2, 1, 8), (30, 3, 6, 2), (18, 2, 5, 5), (35, 4, 12, 7), (26, 1, 4, 4)]


def _jobs(kind, frag_seed=0, ref_shift=0):
    out = []
    for k, (n_atoms, var, n, n_ff) in enumerate(SPECS):
        job = dict(reference_context=_ref(k + ref_shift), n_atoms=n_atoms, variance=var, n_samples=n, job_id=100 + k)
        if KIND_ARGS[kind] is not None:
            job["fixed_fragment"] = _frag(n_ff, 10 * frag_seed + k)
            job["inertial_fragment_matching"] = KIND_ARGS[kind]
        out.append(job)
    return out


def _packed(e, packed, idx=None, seed=5, max_batch=8192, device_out=False):
    idx = np.arange(packed.ids.size) if idx is None else idx
    return J.run_packed(e, packed, idx, T, 0, 3, L, seed, max_batch, device_out)


def _alone(e, packed, j, seed=5):
    """Job j of `packed` run alone, as a user calls it today."""
    a, b = int(packed.starts[j]), int(packed.starts[j + 1])
    nn, N, ctx, ids = packed.n_nodes[a:b], int(packed.max_n_nodes[j]), packed.ctx[a:b], packed.ids[a:b]
    if packed.kind[j] == 0:
        out = e.generate_host(nn, N, ctx, T, 0, seed=seed, sample_ids=ids)
    else:
        fx, fh = packed.fragments[j]
        out = e.generate_fragment_host(nn, N, ctx, fx, fh, packed.kind[j] == 2, packed.references[j], None, T, 0, 3, L,
                                       seed=seed, sample_ids=ids)
    return {"x": out[0].clone(), "atom_class": out[1].clone(), "n_nodes": torch.from_numpy(nn.astype(np.int64)),
            "bonds": out[2].clone()}


def _same(a, b):
    assert a.keys() == b.keys()
    for k in a:
        u, v = a[k].cpu(), b[k].cpu()
        assert u.dtype == v.dtype and u.shape == v.shape, k
        if u.dtype == torch.float32:
            u, v = u.view(torch.int32), v.view(torch.int32)
        assert torch.equal(u, v), k


@pytest.fixture(scope="module")
def generators(state_dicts):
    from ml_conformer_generator_b200 import MLConformerGenerator
    made = {}

    def get(precision):
        if precision not in made:
            made[precision] = MLConformerGenerator(diffusion_steps=T, device=torch.device("cuda:0"), precision=precision,
                                                   edm_state_dict=state_dicts[0], adj_mat_seer_state_dict=state_dicts[1])
        return made[precision]

    yield get
    for g in made.values():
        g.engine.close()


@pytest.mark.parametrize("precision", ["fp16", "bf16"])
@pytest.mark.parametrize("kind", ["plain", "inpaint", "ifm"])
def test_packed_jobs_equal_each_job_alone_on_eager_capture_and_replay_calls(engines, precision, kind):
    e = engines(precision)
    packed = J.flatten_jobs(_jobs(kind), seed=5)
    calls, captures = [], []
    for _ in range(3):  # 1st call eager, 2nd captured into a CUDA graph, 3rd a replay
        c0, l0 = e.graph_captures(), e.kernel_launches()
        calls.append(J.split_jobs(packed, *_packed(e, packed)))
        assert e.kernel_launches() > l0
        captures.append(e.graph_captures() - c0)
    assert captures == [0, 1, 0]
    for j in range(len(SPECS)):
        want = _alone(e, packed, j)
        for got in calls:
            _same(got[j], want)
    if kind == "ifm":  # the merge loop ends with a re-injection: the fixed atoms keep the fragment's classes
        for j, r in enumerate(calls[0]):
            fh = packed.fragments[j][1]
            assert bool((r["atom_class"][:, :fh.shape[0]].long() == fh.argmax(-1).view(1, -1)).all())


@pytest.mark.parametrize("kind", ["inpaint", "ifm"])
def test_replay_with_other_fragments_and_references_uses_the_new_inputs(engines, kind):
    e = engines("bf16")
    packed = J.flatten_jobs(_jobs(kind), seed=5)
    for _ in range(2):
        first = J.split_jobs(packed, *_packed(e, packed))
    other = J.flatten_jobs(_jobs(kind, frag_seed=1, ref_shift=3), seed=5)  # same sizes, other fragments and references
    assert np.array_equal(other.n_nodes, packed.n_nodes)
    c0 = e.graph_captures()
    got = J.split_jobs(other, *_packed(e, other))
    assert e.graph_captures() == c0  # a replay, not a re-capture
    for j in range(len(SPECS)):
        _same(got[j], _alone(e, other, j))
        assert not torch.equal(got[j]["x"], first[j]["x"])


@pytest.mark.parametrize("kind", ["plain", "inpaint", "ifm"])
def test_generate_jobs_is_independent_of_job_order_and_call_boundaries(generators, kind):
    gen = generators("bf16")
    jobs = _jobs(kind)
    whole = gen.generate_jobs(jobs, ifm_diffusion_level=L, seed=5)
    perm = [3, 5, 0, 4, 1, 2]
    shuffled = gen.generate_jobs([jobs[p] for p in perm], ifm_diffusion_level=L, seed=5)
    for k, p in enumerate(perm):
        _same(shuffled[k], whole[p])
    straddled = gen.generate_jobs(jobs, ifm_diffusion_level=L, seed=5, max_batch=7)  # jobs straddle calls
    for a, b in zip(whole, straddled):
        _same(a, b)
    packed = J.flatten_jobs(jobs, seed=5)
    for j in range(len(SPECS)):
        _same(whole[j], _alone(gen.engine, packed, j))


def test_mixed_kinds_are_grouped_and_equal_each_job_alone(generators):
    gen = generators("bf16")
    jobs = [dict(j, job_id=200 + k) for k, j in enumerate(_jobs("ifm")[:2] + _jobs("plain")[2:4] + _jobs("inpaint")[4:])]
    res = gen.generate_jobs(jobs, ifm_diffusion_level=L, seed=5)
    packed = J.flatten_jobs(jobs, seed=5)
    assert packed.kind.tolist() == [2, 2, 0, 0, 1, 1]
    for j in range(len(jobs)):
        _same(res[j], _alone(gen.engine, packed, j))


@pytest.mark.parametrize("kind", ["plain", "inpaint", "ifm"])
def test_sharding_by_arbitrary_id_subsets_is_bit_exact(engines, kind):
    e = engines("bf16")
    packed = J.flatten_jobs(_jobs(kind), seed=5)
    full = _packed(e, packed)
    S = packed.ids.size
    perm = np.random.RandomState(1).permutation(S)
    outs = [torch.empty_like(t) for t in full]
    for ids in (np.sort(perm[:11]), np.sort(perm[11:12]), np.sort(perm[12:])):
        res = _packed(e, packed, ids, device_out=True)
        for o, r in zip(outs, res):
            o[torch.as_tensor(ids)] = r.cpu()
    for a, b in zip(outs, full):
        if a.dtype == torch.float32:
            a, b = a.view(torch.int32), b.view(torch.int32)
        assert torch.equal(a, b)


def _raw_call(e, mode, job_of_sample, n_ff, n_nodes, n=25, null=None):
    """mlcg_generate_fragment_jobs through ctypes with every pointer valid unless named in `null`."""
    B, J_ = len(n_nodes), len(n_ff)
    job = np.ascontiguousarray(job_of_sample, dtype=np.int32)
    nff = np.ascontiguousarray(n_ff, dtype=np.int32)
    tot = max(int(nff.clip(min=0).sum()), 1)
    fx, fh = np.zeros((tot, 3), np.float32), np.zeros((tot, 8), np.float32)
    moi, com = np.tile(np.eye(3, dtype=np.float32).reshape(1, 9) * 100, (J_, 1)), np.ones((J_, 3), np.float32)
    mean, mad = (np.asarray(CONTEXT_NORMS[k], np.float32) for k in ("mean", "mad"))
    ptr = {"job": job.ctypes.data, "n_ff": nff.ctypes.data, "ff_x": fx.ctypes.data, "ff_h": fh.ctypes.data}
    for k in null or ():
        ptr[k] = None
    fj = _lib.FragmentJobs(mode, J_, ptr["job"], ptr["n_ff"], ptr["ff_x"], ptr["ff_h"], L, 0.5, 0.5, moi.ctypes.data,
                           com.ctypes.data, mean.ctypes.data, mad.ctypes.data)
    nn = np.ascontiguousarray(n_nodes, dtype=np.int32)
    ctx = np.zeros((B, 3), np.float32)
    steps = e._steps_cached(T, 3)[1]
    out = [torch.empty(B, n, 3), torch.empty(B, n, dtype=torch.int32), torch.empty(B, 42, 42, dtype=torch.int8)]
    rc = e.lib.mlcg_generate_fragment_jobs(e.h, C.byref(fj), nn.ctypes.data_as(C.c_void_p), B, n, ctx.ctypes.data, T,
                                           steps, 0, 1.0, 1.0, 1.0, 0, 0, None, out[0].data_ptr(), out[1].data_ptr(),
                                           out[2].data_ptr(), e._stream())
    e._check(rc, "generate_fragment")


def test_argument_errors(engines, generators):
    e = engines("fp16")
    nn = [21, 22, 23, 24]
    with pytest.raises(ValueError, match="mode must be 1"):
        _raw_call(e, 0, [0, 1, 0, 1], [3, 4], nn)
    with pytest.raises(ValueError, match="job index out of range"):
        _raw_call(e, 2, [0, 2, 0, 1], [3, 4], nn)
    with pytest.raises(ValueError, match="job index out of range"):
        _raw_call(e, 1, [0, -1, 0, 1], [3, 4], nn)
    with pytest.raises(ValueError, match="at least one atom"):
        _raw_call(e, 1, [0, 1, 0, 1], [3, 0], nn)
    with pytest.raises(ValueError, match="fewer atoms than every sample"):
        _raw_call(e, 2, [0, 1, 0, 1], [3, 22], nn)
    with pytest.raises(ValueError, match="fewer atoms than N"):
        _raw_call(e, 1, [0, 0, 0, 0], [3, 25], nn)
    with pytest.raises(ValueError, match="n_jobs >= 1"):
        _raw_call(e, 1, [0, 0, 0, 0], [], nn)
    for k in ("job", "n_ff", "ff_x", "ff_h"):
        with pytest.raises(ValueError, match="null pointer"):
            _raw_call(e, 1, [0, 1, 0, 1], [3, 4], nn, null=[k])
    ffx, ffh = _frag(3, 0)
    with pytest.raises(ValueError, match="reference_context of every job"):
        e.generate_fragment_jobs_host(np.array(nn), 25, np.zeros((4, 3), np.float32), [0, 1, 0, 1], [(ffx, ffh)] * 2,
                                      True, [_ref(0)], T=T)
    with pytest.raises(ValueError, match="one job per sample"):
        e.generate_fragment_jobs_host(np.array(nn), 25, np.zeros((4, 3), np.float32), [0, 1], [(ffx, ffh)] * 2, False, T=T)
    with pytest.raises(ValueError, match="fewer atoms than minimum generation size"):
        generators("bf16").generate_jobs([dict(reference_context=_ref(0), n_atoms=20, n_samples=2,
                                               fixed_fragment=_frag(18, 0))])
    # a failed call leaves the handle usable
    packed = J.flatten_jobs(_jobs("inpaint")[:2], seed=5)
    got = J.split_jobs(packed, *_packed(e, packed))
    for j in range(2):
        _same(got[j], _alone(e, packed, j))


_TWO_RANK = r"""
import os, sys, numpy as np, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
sys.path.insert(0, os.path.join(sys.argv[1], "tests"))
from ml_conformer_generator_b200.engine import Engine
from ml_conformer_generator_b200.weights import random_state_dicts
from ml_conformer_generator_b200 import parallel as P, jobs as J
import test_gpu_jobs as G
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(rank)
dev = torch.device("cuda", rank)
dist.init_process_group("nccl", device_id=dev)
sd, ssd = random_state_dicts(0)
e = Engine(dev, "bf16"); e.load_edm_state_dict(sd); e.load_seer_state_dict(ssd)
ok = True
for kind in ("plain", "inpaint", "ifm"):
    jobs = G._jobs(kind)
    got = P.generate_jobs_sharded(e, jobs, T=G.T, ifm_diffusion_level=G.L, seed=5)
    if rank == 0:
        packed = J.flatten_jobs(jobs, seed=5)
        want = J.split_jobs(packed, *G._packed(e, packed))
        for a, b in zip(got, want):
            for k in a:
                u, v = a[k].cpu(), b[k].cpu()
                if u.dtype == torch.float32:
                    u, v = u.view(torch.int32), v.view(torch.int32)
                ok = ok and u.shape == v.shape and torch.equal(u, v)
if rank == 0:
    print("SHARDED_JOBS_EQUAL_SINGLE", ok)
dist.barrier()
dist.destroy_process_group()
"""


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_rank_sharded_jobs_equal_single_gpu(tmp_path):
    script = tmp_path / "two_rank_jobs.py"
    script.write_text(_TWO_RANK)
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
                          "127.0.0.1", "--master-port", "29547", str(script), ROOT], capture_output=True, text=True,
                         timeout=900)
    assert out.returncode == 0, out.stderr[-3000:]
    assert "SHARDED_JOBS_EQUAL_SINGLE True" in out.stdout
