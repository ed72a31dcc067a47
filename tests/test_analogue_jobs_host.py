"""CPU: the host logic of analogue jobs (a parent molecule forward-diffused to a diffusion level and denoised from there)
-- validation, the default context, grouping by (has fixed atoms, diffusion level) and cutting at max_batch, the parent's
input frame restored, independence of packing and order, and sharding on gloo (world size 2, with scoring, and with an
empty shard) -- with the stand-in engine of test_jobs_host extended by a stand-in analogue call whose every output row is
a pure function of the sample's own inputs.  Also the CPU reference edm_analogue against edm_merge_fragments."""
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from analogue_oracle import edm_analogue
from ml_conformer_generator_b200 import jobs as J
from ml_conformer_generator_b200 import parallel as P
from ml_conformer_generator_b200.config import CONTEXT_NORMS
from ml_conformer_generator_b200.mol_utils import get_context_shape, normalise_context
from test_jobs_host import REFS, FakeEngine, _flat, _frag, _same
from test_shape_jobs_host import FakeScorer, _conf

T_, L_DEFAULT = 7, 4


def _parent(n, seed):
    """A parent of n atoms away from the origin (so centring matters), classes among C N O F P S Cl."""
    g = torch.Generator().manual_seed(seed)
    x = 1.5 * torch.randn(n, 3, generator=g) + torch.tensor([3.0, -2.0, 5.0]) * (1 + seed % 3)
    return x, torch.eye(8)[torch.randint(0, 7, (n,), generator=g)]


class FakeAnalogueEngine(FakeEngine):
    """FakeEngine with a stand-in Engine.generate_analogue_jobs_host: sample b's real atoms are its parent's (centred)
    coordinates plus an offset that depends only on its id, context, fixed flags, the level and the seed."""

    def generate_analogue_jobs_host(self, n_nodes, max_n_nodes, ctx, job_of_sample, parents, fixed=None, T=100,
                                    resample_steps=0, blend_power=3, diffusion_level=50, seed=0, sample_offset=0,
                                    sample_ids=None, out=None, device_out=False):
        job = np.asarray(job_of_sample)
        n_at = np.array([p[0].shape[0] for p in parents])
        assert job.min() >= 0 and job.max() < len(parents) and len(fixed) == len(parents)
        assert (n_at[job] == np.asarray(n_nodes)).all() and n_at.max() <= max_n_nodes
        any_fixed = {bool(np.asarray(f).any()) for f in fixed}
        assert len(any_fixed) == 1  # one call never mixes jobs with and without fixed atoms
        for (px, _), f in zip(parents, fixed):  # the engine gets the centred parent and one flag per atom
            assert torch.allclose(px.mean(0), torch.zeros(3), atol=1e-5) and np.asarray(f).size == px.shape[0]
        self.calls.append(dict(kind=3, ids=np.asarray(sample_ids).copy(), N=max_n_nodes, n_jobs=len(parents), T=T,
                               r=resample_steps, bp=blend_power, L=diffusion_level, fixed=any_fixed.pop(), seed=seed,
                               device_out=device_out))
        ids = np.asarray(sample_ids)
        B = ids.size
        x = torch.zeros(B, max_n_nodes, 3)
        cls = torch.full((B, max_n_nodes), -1, dtype=torch.int32)
        for b in range(B):
            px, ph = parents[job[b]]
            n = px.shape[0]
            off = 1e-3 * float(ids[b] % 1000 + (ids[b] >> 32) * 1000) + 0.01 * diffusion_level + 7.0 * seed \
                + 0.1 * float(np.asarray(fixed[job[b]]).sum()) + float(ctx[b][0])
            x[b, :n] = px + off
            cls[b, :n] = ph.argmax(-1).to(torch.int32)
        bonds = torch.as_tensor(ids % 5).view(B, 1, 1).repeat(1, 42, 42).to(torch.int8)
        return x, cls, bonds


def _jobs():
    """Analogue jobs with and without fixed atoms at two levels, next to plain and fragment jobs."""
    return [
        dict(parent_molecule=_parent(12, 0), n_samples=4),
        dict(reference_context=REFS[0], n_atoms=20, n_samples=3),
        dict(parent_molecule=_parent(20, 1), n_samples=5, fixed_atoms=[0, 3, 7]),
        dict(parent_molecule=_parent(9, 2), n_samples=3, diffusion_level=2, reference_context=REFS[1]),
        dict(reference_context=REFS[1], n_atoms=24, n_samples=2, fixed_fragment=_frag(3)),
        dict(parent_molecule=_parent(15, 3), n_samples=6, fixed_atoms=np.array([14]), diffusion_level=2),
        dict(parent_molecule=_parent(30, 4), n_samples=2, job_id=40),
        dict(parent_molecule=_parent(3, 5), n_samples=1, fixed_atoms=[1, 2]),
    ]


def _run(jobs, max_batch=8192, seed=3, level=L_DEFAULT):
    e = FakeAnalogueEngine()
    packed = J.flatten_jobs(jobs, seed)
    x, cls, bonds = J.run_packed(e, packed, np.arange(packed.ids.size), T=T_, resample_steps=1, blend_power=2,
                                 ifm_diffusion_level=level, seed=seed, max_batch=max_batch)
    return J.split_jobs(packed, x, cls, bonds), e.calls, packed, x


def test_validation_messages():
    base = dict(parent_molecule=_parent(10, 0), n_samples=2)
    for k, v in (("n_atoms", 10), ("variance", 1), ("n_nodes", [10, 10]), ("fixed_fragment", _frag(2)),
                 ("inertial_fragment_matching", False)):
        with pytest.raises(ValueError, match="cannot go with it"):
            J.flatten_jobs([dict(base, **{k: v})])
    with pytest.raises(ValueError, match="needs n_samples"):
        J.flatten_jobs([dict(parent_molecule=_parent(10, 0))])
    with pytest.raises(ValueError, match=r"parent_molecule must be \(coordinates"):
        J.flatten_jobs([dict(base, parent_molecule=torch.zeros(10, 3))])
    with pytest.raises(ValueError, match=r"parent_molecule must be \(coordinates"):
        J.flatten_jobs([dict(base, parent_molecule=(torch.zeros(10, 2), torch.zeros(10, 8)))])
    with pytest.raises(ValueError, match=r"parent_molecule must be \(coordinates"):
        J.flatten_jobs([dict(base, parent_molecule=(torch.zeros(10, 3), torch.zeros(9, 8)))])
    for n in (2, 40):
        with pytest.raises(ValueError, match="3 <= n <= 39"):
            J.flatten_jobs([dict(base, parent_molecule=_parent(n, 0))])
    with pytest.raises(ValueError, match="3 <= n <= 30"):
        J.flatten_jobs([dict(base, parent_molecule=_parent(31, 0))], max_n_nodes=30)
    x, h = _parent(10, 0)
    for bad in (h * 2, h * 0, h + torch.eye(8)[[7] * 10]):
        with pytest.raises(ValueError, match="one 1 per atom"):
            J.flatten_jobs([dict(base, parent_molecule=(x, bad))])
    with pytest.raises(ValueError, match="must be finite"):
        J.flatten_jobs([dict(base, parent_molecule=(x * float("nan"), h))])
    with pytest.raises(ValueError, match="must be atom indices"):
        J.flatten_jobs([dict(base, fixed_atoms=[0.5, 1.0])])
    for bad in ([-1, 2], [3, 10]):
        with pytest.raises(ValueError, match="must index the parent's 10 atoms"):
            J.flatten_jobs([dict(base, fixed_atoms=bad)])
    with pytest.raises(ValueError, match="must be distinct"):
        J.flatten_jobs([dict(base, fixed_atoms=[1, 4, 1])])
    with pytest.raises(ValueError, match="at most n - 1 = 9"):
        J.flatten_jobs([dict(base, fixed_atoms=list(range(10)))])
    for k in ("fixed_atoms", "diffusion_level"):
        with pytest.raises(ValueError, match="%s needs a parent_molecule" % k):
            J.flatten_jobs([dict(reference_context=REFS[0], n_atoms=20, n_samples=2, **{k: 1})])
    for bad in (0, -5):
        with pytest.raises(ValueError, match="diffusion_level must be at least 1"):
            J.flatten_jobs([dict(base, diffusion_level=bad)])
    with pytest.raises(ValueError, match="3 principal moments"):
        J.flatten_jobs([dict(base, reference_context=[1.0, 2.0])])
    # the level's upper bound is T, known when the jobs run
    with pytest.raises(ValueError, match=r"diffusion_level must lie in \[1, T=7\], got 8"):
        _run([dict(base, diffusion_level=8)])
    with pytest.raises(ValueError, match=r"diffusion_level must lie in \[1, T=7\], got 50"):
        _run([base], level=50)
    with pytest.raises(ValueError, match=r"diffusion_level must lie in \[1, T=7\]"):
        P.generate_jobs_sharded(FakeAnalogueEngine(), [base], T=7, ifm_diffusion_level=9)
    # accepted edge cases: an empty fixed set, n - 1 fixed atoms, L = 1 and L = T
    for ok in (dict(base, fixed_atoms=[]), dict(base, fixed_atoms=list(range(9)), diffusion_level=T_),
               dict(base, diffusion_level=1), dict(base, parent_molecule=_parent(3, 0)), dict(base, job_id=5)):
        _run([ok])
    # the other kinds still need a reference_context
    with pytest.raises(KeyError):
        J.flatten_jobs([dict(n_atoms=20, n_samples=2)])


def test_default_context_is_the_centred_parents_principal_moments():
    jobs = _jobs()
    packed = J.flatten_jobs(jobs, seed=3)
    assert packed.kind.tolist() == [3, 0, 3, 3, 2, 3, 3, 3]
    for j, job in enumerate(jobs):
        if "parent_molecule" not in job:
            assert packed.parents[j] is None and packed.levels[j] == 0
            continue
        coords, oh = job["parent_molecule"]
        a, b = packed.starts[j], packed.starts[j + 1]
        assert packed.n_nodes[a:b].tolist() == [coords.shape[0]] * job["n_samples"]
        assert packed.max_n_nodes[j] == coords.shape[0]
        if job.get("reference_context") is None:
            want = get_context_shape(coords - coords.mean(dim=0))[0]  # as generate_conformers computes it
        else:
            want = torch.as_tensor(job["reference_context"], dtype=torch.float32)
        assert torch.equal(packed.references[j], want)
        assert np.array_equal(packed.ctx[a:b], np.tile(normalise_context(want, CONTEXT_NORMS).numpy(), (b - a, 1)))
        cx, ph, fixed, mean = packed.parents[j]
        assert torch.equal(mean, coords.mean(dim=0)) and torch.equal(cx, coords - mean) and torch.equal(ph, oh)
        assert fixed.dtype == np.int32 and np.nonzero(fixed)[0].tolist() == sorted(np.asarray(job.get("fixed_atoms", [])).tolist())
        assert packed.levels[j] == job.get("diffusion_level", 0)


def test_grouping_by_fixed_atoms_and_level_and_cutting_at_max_batch():
    jobs = _jobs()
    whole, calls, packed, _ = _run(jobs)
    # plain, IFM, then the analogue groups (has fixed atoms, level) in order: (no, 2) (no, 4) (yes, 2) (yes, 4)
    assert [c["kind"] for c in calls] == [0, 2, 3, 3, 3, 3]
    groups = [(c["fixed"], c["L"]) for c in calls[2:]]
    assert groups == [(False, 2), (False, 4), (True, 2), (True, 4)]
    members = [sorted(set(packed.job[_flat(packed, c["ids"])].tolist())) for c in calls[2:]]
    assert members == [[3], [0, 6], [5], [2, 7]]
    for c in calls[2:]:
        here = np.unique(packed.job[_flat(packed, c["ids"])])
        assert c["N"] == packed.max_n_nodes[here].max() and c["n_jobs"] == here.size
        assert (c["T"], c["r"], c["bp"], c["seed"]) == (T_, 1, 2, 3)
    small, calls3, _, _ = _run(jobs, max_batch=3)
    assert all(len(c["ids"]) <= 3 for c in calls3)
    analogue = [c for c in calls3 if c["kind"] == 3]
    # (no, 2): 3 samples -> 1 call; (no, 4): 4 + 2 -> 2; (yes, 2): 6 -> 2; (yes, 4): 5 + 1 -> 2, job 2 straddles them
    assert [(c["fixed"], c["L"], len(c["ids"])) for c in analogue] == [
        (False, 2, 3), (False, 4, 3), (False, 4, 3), (True, 2, 3), (True, 2, 3), (True, 4, 3), (True, 4, 3)]
    for a, b in zip(whole, small):
        _same(a, b)
    for j, job in enumerate(jobs):  # every job equals the job run alone
        alone, _, _, _ = _run([dict(job, job_id=int(packed.job_ids[j]))])
        _same(alone[0], whole[j])


def test_results_are_in_the_parents_input_frame():
    jobs = _jobs()
    res, _, packed, x = _run(jobs)
    e = FakeAnalogueEngine()
    for j, job in enumerate(jobs):
        if "parent_molecule" not in job:
            continue
        coords, oh = job["parent_molecule"]
        n = coords.shape[0]
        cx, _, fixed, mean = packed.parents[j]
        a, b = int(packed.starts[j]), int(packed.starts[j + 1])
        raw = e.generate_analogue_jobs_host(packed.n_nodes[a:b], n, packed.ctx[a:b], np.zeros(b - a, np.int32), [(cx, oh)],
                                            [fixed], T_, 1, 2, job.get("diffusion_level", L_DEFAULT), seed=3,
                                            sample_ids=packed.ids[a:b])[0]
        assert torch.equal(res[j]["x"], raw + mean)  # the engine's output with the parent's mean added back
        off = (raw - cx)[:, :1]
        assert torch.allclose(res[j]["x"], coords + off, atol=1e-4)
        assert res[j]["x"].shape == (b - a, n, 3) and torch.equal(res[j]["atom_class"], oh.argmax(-1).repeat(b - a, 1).int())
        # in the packed output, rows beyond the parent stay padding
        assert bool((x[a:b, n:] == 0).all())


def test_permuting_the_jobs_leaves_every_job_unchanged():
    jobs = [dict(j, job_id=k) for k, j in enumerate(_jobs())]
    whole, _, _, _ = _run(jobs)
    perm = [5, 0, 7, 2, 6, 3, 1, 4]
    shuffled, _, _, _ = _run([jobs[p] for p in perm])
    for k, p in enumerate(perm):
        _same(shuffled[k], whole[p])
    # other jobs' outputs are the same with or without the analogue jobs next to them
    others = [j for j in jobs if "parent_molecule" not in j]
    without, _, _, _ = _run(others)
    for a, j in zip(without, others):
        _same(a, whole[jobs.index(j)])


def test_edm_analogue_is_merge_fragments_with_fixed_atoms_and_skips_reinjection_without():
    from ml_conformer_generator_b200.weights import random_state_dicts
    from oracle import edm_oracle as O
    sd = random_state_dicts(0)[0]
    T, L, r, bp = 5, 3, 1, 3
    n_nodes = torch.tensor([7, 9])
    N, B = 9, 2
    nm, em = O.prepare_masks(n_nodes, N)
    zk = torch.zeros(B, N, 11)
    for b, seed in enumerate((0, 1)):
        x, h = _parent(int(n_nodes[b]), seed)
        zk[b, : n_nodes[b], :3] = x - x.mean(0)
        zk[b, : n_nodes[b], 3:] = h
    ctx = O.batch_context(normalise_context(torch.tensor(REFS[0]), CONTEXT_NORMS), nm)
    gamma = O.gamma_table(T)
    n_active = L + 1
    fm = torch.zeros(B, N, 1)
    fm[0, [1, 4]] = 1.0
    fm[1, [0]] = 1.0
    with torch.no_grad():
        n_draw = 1 + n_active * 2 * r + 1
        a = edm_analogue(sd, gamma, nm, em, fm, ctx, zk, O.NoiseTape.draw(n_draw, B, N, 4), L, r, bp)
        m = O.edm_merge_fragments(sd, gamma, nm, em, fm, ctx, zk, O.NoiseTape.draw(n_draw, B, N, 4), L, r, bp)
        for u, v in zip(a, m):
            assert torch.equal(u.view(torch.int32) if u.dtype == torch.float32 else u,
                               v.view(torch.int32) if v.dtype == torch.float32 else v)
        # nothing fixed: merge_fragments' loop without re-injection, which draws no re-injection noise
        tape = O.NoiseTape.draw(1 + n_active * r + 1, B, N, 4)
        x, h = edm_analogue(sd, gamma, nm, em, torch.zeros(B, N, 1), ctx, zk, tape, L, r, bp)
        assert tape.pos == len(tape.pairs) and bool(torch.isfinite(x).all())
        with pytest.raises(ValueError, match="every sample has fixed atoms or none"):
            edm_analogue(sd, gamma, nm, em, fm * torch.tensor([1.0, 0.0]).view(B, 1, 1), ctx, zk,
                           O.NoiseTape.draw(n_draw, B, N, 4), L, r, bp)


def _case(name):
    if name == "mixed":
        return _jobs(), None
    if name == "scored":
        return [dict(j, reference_conformer=_conf(3 + k, k)) for k, j in enumerate(_jobs())], 2
    # one molecule in all: the second rank's shard is empty
    return [dict(parent_molecule=_parent(11, 0), n_samples=1, fixed_atoms=[2], reference_conformer=_conf(11))], 1


def _single(jobs, keep_best):
    e, sc = FakeAnalogueEngine(), FakeScorer()
    packed = J.flatten_jobs(jobs, 3)
    J.check_keep_best(packed, keep_best)
    idx = np.arange(packed.ids.size)
    x, cls, bonds = J.run_packed(e, packed, idx, T=T_, resample_steps=1, blend_power=2, ifm_diffusion_level=L_DEFAULT,
                                 seed=3)
    res = J.split_jobs(packed, x, cls, bonds)
    if packed.scored:
        res = J.attach_scores(packed, res, *J.score_packed(sc, packed, idx, x), keep_best)
    return res, packed


def _sharded(jobs, keep_best, max_batch):
    e = FakeAnalogueEngine()
    res = P.generate_jobs_sharded(e, jobs, T=T_, resample_steps=1, blend_power=2, ifm_diffusion_level=L_DEFAULT, seed=3,
                                  max_batch=max_batch, keep_best=keep_best, scorer=FakeScorer())
    return res, e.calls


def _worker(rank, world, port, tmp, name, max_batch):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    jobs, k = _case(name)
    torch.save(_sharded(jobs, k, max_batch), tmp + ".%d" % rank)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("name,max_batch,port", [("mixed", 8192, 29571), ("scored", 3, 29572), ("empty_shard", 8192, 29573)])
def test_sharded_analogue_jobs_match_the_single_process_result(tmp_path, name, max_batch, port):
    jobs, k = _case(name)
    want, packed = _single(jobs, k)
    single, _ = _sharded(jobs, k, max_batch)
    for a, b in zip(want, single):
        _same(a, b)
    out_file = str(tmp_path / "analogue.pt")
    mp.spawn(_worker, args=(2, port, out_file, name, max_batch), nprocs=2, join=True)
    shards = P.shard_indices(packed.n_nodes, 2)
    if name == "empty_shard":
        assert [len(s) for s in shards] == [1, 0]
    for r in range(2):
        got, calls = torch.load(out_file + ".%d" % r, weights_only=False)
        assert len(got) == len(want)
        for a, b in zip(want, got):  # every rank holds every job
            _same(a, b)
        ran = np.sort(np.concatenate([_flat(packed, c["ids"]) for c in calls])) if calls else np.zeros(0, np.int64)
        assert np.array_equal(ran, shards[r])
        assert all(len(c["ids"]) <= max_batch and c["device_out"] for c in calls)
