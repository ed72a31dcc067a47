"""CPU: the host logic of packed generation jobs (jobs.py, parallel.generate_jobs_sharded) -- flattening and the split
back per job, the id mapping, per-job atom-count determinism, grouping by kind and chunking with straddling jobs,
validation, and sharding on gloo (world size 2) -- with a stand-in engine whose every output row is a pure function of
the sample's own inputs, like the keyed device RNG and the per-molecule kernels."""
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from ml_conformer_generator_b200 import jobs as J
from ml_conformer_generator_b200 import parallel as P
from ml_conformer_generator_b200.config import CONTEXT_NORMS
from ml_conformer_generator_b200.mol_utils import normalise_context

REFS = [[89.87, 210.78, 217.78], [53.64, 108.30, 151.44], [60.0, 120.0, 170.0], [70.0, 150.0, 190.0]]


def _frag(n, shift=0.0):
    return torch.arange(3 * n, dtype=torch.float32).view(n, 3) + shift, torch.eye(8)[[k % 7 for k in range(n)]]


def _jobs():
    return [
        dict(reference_context=REFS[0], n_atoms=20, n_samples=5),
        dict(reference_context=REFS[1], n_atoms=24, variance=1, n_samples=4, fixed_fragment=_frag(3)),
        dict(reference_context=REFS[2], n_nodes=[30, 31, 29], fixed_fragment=_frag(5, 1.0),
             inertial_fragment_matching=False),
        dict(reference_context=REFS[3], n_atoms=37, n_samples=1, job_id=11),
        dict(reference_context=REFS[0], n_atoms=22, n_samples=6, fixed_fragment=_frag(8, 2.0)),
        dict(reference_context=REFS[1], n_atoms=17, n_samples=2, fixed_fragment=_frag(2), inertial_fragment_matching=False),
    ]


class FakeEngine:
    """Stand-in for Engine: row b of every output depends only on sample b's id, atom count and context, its job's
    fragment and reference, and the shared settings; x / atom_class rows beyond the atom count are 0 / -1 as the kernels
    write them.  Records every call."""
    device = torch.device("cpu")

    def __init__(self):
        self.calls = []

    def _out(self, n_nodes, N, ctx, ids, tag):
        B = len(ids)
        ids = torch.as_tensor(np.asarray(ids))
        val = (ids % 1000 + (ids >> 32) * 1000).double().view(B, 1, 1) + torch.as_tensor(tag).double().view(B, 1, 1) \
            + torch.as_tensor(ctx, dtype=torch.float64)[:, :1].view(B, 1, 1)
        real = torch.arange(N).view(1, N) < torch.as_tensor(np.asarray(n_nodes)).view(B, 1)
        x = (val + torch.arange(N).double().view(1, N, 1) / 64 + torch.zeros(1, 1, 3, dtype=torch.float64)).float()
        x = x * real.unsqueeze(-1)
        cls = torch.where(real, torch.as_tensor(np.asarray(n_nodes)).view(B, 1).to(torch.int32) % 7, -1).to(torch.int32)
        bonds = (ids % 5).view(B, 1, 1).repeat(1, 42, 42).to(torch.int8)
        return x, cls, bonds

    def generate_host(self, n_nodes, max_n_nodes, ctx, T=100, resample_steps=0, seed=0, sample_offset=0, out=None,
                      sample_ids=None, device_out=False):
        self.calls.append(dict(kind=0, ids=np.asarray(sample_ids).copy(), N=max_n_nodes, T=T, r=resample_steps, seed=seed,
                               device_out=device_out))
        assert np.asarray(n_nodes).max() <= max_n_nodes
        return self._out(n_nodes, max_n_nodes, ctx, sample_ids, np.full(len(sample_ids), 7.0 * seed))

    def generate_fragment_jobs_host(self, n_nodes, max_n_nodes, ctx, job_of_sample, fragments,
                                    inertial_fragment_matching=True, reference_contexts=None, context_norms=None, T=100,
                                    resample_steps=0, blend_power=3, diffusion_level=50, seed=0, sample_offset=0,
                                    sample_ids=None, out=None, device_out=False):
        job = np.asarray(job_of_sample)
        assert job.min() >= 0 and job.max() < len(fragments) and len(reference_contexts) == len(fragments)
        n_ff = np.array([f[0].shape[0] for f in fragments])
        assert (n_ff[job] < np.asarray(n_nodes)).all() and np.asarray(n_nodes).max() <= max_n_nodes
        self.calls.append(dict(kind=2 if inertial_fragment_matching else 1, ids=np.asarray(sample_ids).copy(),
                               N=max_n_nodes, n_jobs=len(fragments), T=T, r=resample_steps, bp=blend_power,
                               L=diffusion_level, seed=seed, device_out=device_out))
        tag = np.array([float(fragments[j][0].sum()) + 0.25 * float(torch.as_tensor(reference_contexts[j]).sum())
                        + 100.0 * inertial_fragment_matching + 10.0 * diffusion_level + 7.0 * seed for j in job])
        return self._out(n_nodes, max_n_nodes, ctx, sample_ids, tag)


def _run(jobs, max_batch=8192, seed=3, engine=None):
    e = engine or FakeEngine()
    packed = J.flatten_jobs(jobs, seed)
    res = J.split_jobs(packed, *J.run_packed(e, packed, np.arange(packed.ids.size), T=7, resample_steps=1, blend_power=2,
                                             ifm_diffusion_level=4, seed=seed, max_batch=max_batch))
    return res, e.calls, packed


def _flat(packed, ids):
    """Flat sample positions of global sample ids."""
    pos = {int(g): k for k, g in enumerate(packed.ids)}
    return np.array([pos[int(g)] for g in ids], dtype=np.int64)


def _same(a, b):
    assert a.keys() == b.keys()
    for k in a:
        assert a[k].dtype == b[k].dtype and a[k].shape == b[k].shape, k
        assert torch.equal(a[k], b[k]), k


def test_flatten_maps_ids_context_and_kinds_and_split_restores_each_job():
    jobs = _jobs()
    packed = J.flatten_jobs(jobs, seed=5)
    sizes = [5, 4, 3, 1, 6, 2]
    assert packed.starts.tolist() == np.concatenate([[0], np.cumsum(sizes)]).tolist()
    assert packed.kind.tolist() == [0, 2, 1, 0, 2, 1]
    assert packed.job_ids.tolist() == [0, 1, 2, 11, 4, 5]
    assert packed.max_n_nodes.tolist() == [22, 25, 31, 39, 24, 19]
    assert packed.N == 39
    for j, job in enumerate(jobs):
        a, b = packed.starts[j], packed.starts[j + 1]
        assert packed.ids[a:b].tolist() == [(int(packed.job_ids[j]) << 32) + k for k in range(b - a)]
        assert (packed.job[a:b] == j).all()
        want = normalise_context(torch.tensor(job["reference_context"]), CONTEXT_NORMS).numpy()
        assert np.array_equal(packed.ctx[a:b], np.tile(want, (b - a, 1)))
    assert packed.n_nodes[packed.starts[2]:packed.starts[3]].tolist() == [30, 31, 29]
    # the split slices every job to its own max atom count, in input order
    S = packed.ids.size
    x = torch.arange(S * 39 * 3, dtype=torch.float32).view(S, 39, 3)
    cls = torch.arange(S * 39, dtype=torch.int32).view(S, 39)
    bonds = (torch.arange(S, dtype=torch.int8).view(S, 1, 1)).repeat(1, 42, 42)
    res = J.split_jobs(packed, x, cls, bonds)
    assert len(res) == len(jobs)
    for j, r in enumerate(res):
        a, b, nj = packed.starts[j], packed.starts[j + 1], packed.max_n_nodes[j]
        assert torch.equal(r["x"], x[a:b, :nj]) and torch.equal(r["atom_class"], cls[a:b, :nj])
        assert torch.equal(r["bonds"], bonds[a:b]) and r["n_nodes"].tolist() == packed.n_nodes[a:b].tolist()


def test_atom_counts_depend_only_on_the_seed_and_the_job_id():
    job = dict(reference_context=REFS[0], n_atoms=30, variance=9, n_samples=200, job_id=42)
    alone = J.flatten_jobs([job], seed=8).n_nodes
    others = J.flatten_jobs(_jobs() + [job], seed=8)
    assert np.array_equal(others.n_nodes[others.starts[-2]:], alone)
    assert np.array_equal(alone, J.job_atom_counts(8, 42, 21, 39, 200))
    assert alone.min() == 21 and alone.max() == 39  # clipped to [n_atoms - variance, max_n_nodes]
    assert not np.array_equal(J.flatten_jobs([job], seed=9).n_nodes, alone)
    assert not np.array_equal(J.flatten_jobs([dict(job, job_id=43)], seed=8).n_nodes, alone)
    # a job's position sets its default id, and so its atom counts
    a = J.flatten_jobs([{k: v for k, v in job.items() if k != "job_id"}], seed=8)
    assert a.job_ids.tolist() == [0] and np.array_equal(a.n_nodes, J.job_atom_counts(8, 0, 21, 39, 200))


def test_grouping_by_kind_and_chunking_with_straddling_jobs():
    jobs = _jobs()
    whole, calls, packed = _run(jobs)
    assert [c["kind"] for c in calls] == [0, 1, 2]  # one call per kind
    straddled, calls7, _ = _run(jobs, max_batch=7)
    kinds = [c["kind"] for c in calls7]
    assert kinds == sorted(kinds) and all(len(c["ids"]) <= 7 for c in calls7)
    # plain: 6 samples -> 1 call; inpaint: 5 -> 1; IFM: 10 -> 2 calls, the 8-atom job straddles them
    assert kinds == [0, 1, 2, 2]
    ifm_calls = [set(packed.job[_flat(packed, c["ids"])].tolist()) for c in calls7[2:]]
    assert ifm_calls == [{1, 4}, {4}]
    for c in calls7:
        here = np.unique(packed.job[_flat(packed, c["ids"])])
        assert c["N"] == packed.max_n_nodes[here].max()  # padded to the largest job in the call
        assert (c["T"], c["r"], c["seed"]) == (7, 1, 3)
        if c["kind"]:
            assert c["n_jobs"] == here.size and (c["bp"], c["L"]) == (2, 4)
    for a, b in zip(whole, straddled):
        _same(a, b)
    # every job equals the job run alone
    for j, job in enumerate(jobs):
        alone, _, _ = _run([dict(job, job_id=int(packed.job_ids[j]))])
        _same(alone[0], whole[j])


def test_permuting_the_jobs_leaves_every_job_unchanged():
    jobs = [dict(j, job_id=k) for k, j in enumerate(_jobs())]
    whole, _, _ = _run(jobs)
    perm = [4, 0, 5, 2, 3, 1]
    shuffled, _, _ = _run([jobs[p] for p in perm])
    for k, p in enumerate(perm):
        _same(shuffled[k], whole[p])


def test_validation_messages():
    ref = REFS[0]
    with pytest.raises(ValueError, match="fewer atoms than minimum generation size"):
        J.flatten_jobs([dict(reference_context=ref, n_atoms=20, n_samples=2, fixed_fragment=_frag(18))])
    with pytest.raises(ValueError, match="fewer atoms than minimum generation size"):
        J.flatten_jobs([dict(reference_context=ref, n_nodes=[25, 9, 30], fixed_fragment=_frag(9))])
    with pytest.raises(ValueError, match="one-hot"):
        J.flatten_jobs([dict(reference_context=ref, n_atoms=20, n_samples=2, fixed_fragment=(torch.zeros(3, 3),
                                                                                           torch.zeros(3, 7)))])
    with pytest.raises(ValueError, match="unique"):
        J.flatten_jobs([dict(reference_context=ref, n_atoms=20, n_samples=2, job_id=3),
                        dict(reference_context=ref, n_atoms=21, n_samples=2, job_id=3)])
    with pytest.raises(ValueError, match="unknown field"):
        J.flatten_jobs([dict(reference_context=ref, n_atoms=20, n_sample=2)])
    with pytest.raises(ValueError, match="3 principal moments"):
        J.flatten_jobs([dict(reference_context=[1.0, 2.0], n_atoms=20, n_samples=2)])
    with pytest.raises(ValueError, match="does not match"):
        J.flatten_jobs([dict(reference_context=ref, n_nodes=[20, 21], n_samples=3)])
    with pytest.raises(ValueError, match="n_nodes must lie"):
        J.flatten_jobs([dict(reference_context=ref, n_nodes=[20, 40])])
    with pytest.raises(ValueError, match="at least 1"):
        J.flatten_jobs([dict(reference_context=ref, n_atoms=20, n_samples=0)])
    with pytest.raises(ValueError, match="job_id"):
        J.flatten_jobs([dict(reference_context=ref, n_atoms=20, n_samples=1, job_id=-1)])
    with pytest.raises(ValueError, match="no atom count"):
        J.flatten_jobs([dict(reference_context=ref, n_atoms=60, variance=2, n_samples=1)])
    with pytest.raises(ValueError, match="no jobs"):
        J.flatten_jobs([])


def _sharded(max_batch):
    e = FakeEngine()
    res = P.generate_jobs_sharded(e, _jobs(), T=7, resample_steps=1, blend_power=2, ifm_diffusion_level=4, seed=3,
                                  max_batch=max_batch)
    return res, e.calls


def _worker(rank, world, port, tmp, max_batch):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.save(_sharded(max_batch), tmp + ".%d" % rank)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("max_batch,port", [(8192, 29541), (4, 29542)])
def test_sharded_jobs_match_the_single_process_result(tmp_path, max_batch, port):
    want, _, packed = _run(_jobs())
    single, _ = _sharded(max_batch)
    for a, b in zip(want, single):
        _same(a, b)
    out_file = str(tmp_path / "jobs.pt")
    mp.spawn(_worker, args=(2, port, out_file, max_batch), nprocs=2, join=True)
    shards = P.shard_indices(packed.n_nodes, 2)
    for r in range(2):
        got, calls = torch.load(out_file + ".%d" % r, weights_only=False)
        for a, b in zip(want, got):  # every rank holds every job
            _same(a, b)
        # each rank ran exactly its own samples, one kind per call, at most max_batch per call, on the device
        ran = np.sort(np.concatenate([_flat(packed, c["ids"]) for c in calls]))
        assert np.array_equal(ran, shards[r])
        assert all(len(c["ids"]) <= max_batch and c["device_out"] for c in calls)
        for c in calls:
            assert (packed.kind[packed.job[_flat(packed, c["ids"])]] == c["kind"]).all()
