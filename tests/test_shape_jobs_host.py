"""CPU: the host logic of scoring generation jobs against their reference conformers (jobs.score_packed,
jobs.attach_scores, the scored path of parallel.generate_jobs_sharded) -- validation, the top-k selection, jobs without a
conformer left as they are, and sharding on gloo (world size 2) -- with the stand-in engine of test_jobs_host and a
stand-in scorer whose every output row is a pure function of the sample and its own reference, like the shape kernels."""
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from ml_conformer_generator_b200 import jobs as J
from ml_conformer_generator_b200 import parallel as P
from test_jobs_host import REFS, FakeEngine, _frag, _jobs, _run, _same


def _conf(n, shift=0.0):
    return torch.linspace(-2.0, 2.0, 3 * n).view(n, 3) + shift


class FakeScorer:
    """Stand-in for ShapeScorer.evaluate_jobs.  A score takes few values, so a job has ties; it depends on the sample's
    coordinates and atom count and on its reference only.  Records every call."""

    def __init__(self):
        self.calls = []

    def evaluate_jobs(self, references, coords, n_nodes, job):
        job = torch.as_tensor(job).long()
        n_nodes = torch.as_tensor(n_nodes).long()
        self.calls.append(dict(n_refs=len(references), B=coords.shape[0], job=job.clone()))
        assert coords.shape[0] == n_nodes.numel() == job.numel()
        assert job.numel() == 0 or 0 <= int(job.min()) <= int(job.max()) < len(references)
        refsum = torch.tensor([float(r.sum()) for r in references] + [0.0])
        first = coords[:, 0, 0].double().round()
        score = ((first % 4) / 4 + (n_nodes % 2) / 8 + 1e-3 * refsum[job]).float()
        orient = (first.long() + n_nodes) % 4
        aligned = coords * (1 + orient).view(-1, 1, 1).float()
        return {"shape_tanimoto": score, "best_orientation": orient, "aligned_coords": aligned,
                "reference_coords": [r - r.mean(0) for r in references]}


def _scored_jobs():
    """Jobs of every kind; four with a reference conformer, two without."""
    jobs = _jobs()
    for j, n in ((0, 12), (1, 5), (3, 64), (4, 3)):
        jobs[j] = dict(jobs[j], reference_conformer=_conf(n, j))
    return jobs


def _single(jobs, keep_best=None, seed=3):
    """The single-process scored path, as MLConformerGenerator.generate_jobs runs it."""
    e, sc = FakeEngine(), FakeScorer()
    packed = J.flatten_jobs(jobs, seed)
    J.check_keep_best(packed, keep_best)
    idx = np.arange(packed.ids.size)
    x, cls, bonds = J.run_packed(e, packed, idx, T=7, resample_steps=1, blend_power=2, ifm_diffusion_level=4, seed=seed)
    res = J.attach_scores(packed, J.split_jobs(packed, x, cls, bonds), *J.score_packed(sc, packed, idx, x), keep_best)
    return res, sc.calls, packed


def test_reference_conformer_validation():
    ref = REFS[0]
    base = dict(reference_context=ref, n_atoms=20, n_samples=2)
    with pytest.raises(ValueError, match=r"reference_conformer must be heavy-atom coordinates \(n, 3\)"):
        J.flatten_jobs([dict(base, reference_conformer=torch.zeros(5, 2))])
    with pytest.raises(ValueError, match=r"reference_conformer must be heavy-atom coordinates \(n, 3\)"):
        J.flatten_jobs([dict(base, reference_conformer=torch.zeros(15))])
    with pytest.raises(ValueError, match="3 <= n <= 64"):
        J.flatten_jobs([dict(base, reference_conformer=_conf(2))])
    with pytest.raises(ValueError, match="3 <= n <= 64"):
        J.flatten_jobs([dict(base, reference_conformer=_conf(65))])
    for n in (3, 64):
        packed = J.flatten_jobs([dict(base, reference_conformer=_conf(n).numpy())])
        assert packed.scored and packed.conformers[0].dtype == torch.float32 and packed.conformers[0].shape == (n, 3)
    packed = J.flatten_jobs([base])
    assert packed.conformers == [None] and not packed.scored
    # PackedJobs built without the new field keeps working
    old = J.PackedJobs(*[getattr(packed, f) for f in ("kind", "job_ids", "max_n_nodes", "starts", "fragments",
                                                       "references", "n_nodes", "ctx", "job", "ids")])
    assert old.conformers is None and not old.scored


def test_keep_best_validation():
    scored = J.flatten_jobs([dict(reference_context=REFS[0], n_atoms=20, n_samples=2, reference_conformer=_conf(4))])
    for k in (0, -3):
        with pytest.raises(ValueError, match="keep_best must be at least 1"):
            J.check_keep_best(scored, k)
    J.check_keep_best(scored, 1)
    J.check_keep_best(scored, None)
    mixed = J.flatten_jobs(_scored_jobs())
    J.check_keep_best(mixed, None)
    with pytest.raises(ValueError, match="every job needs a reference_conformer"):
        J.check_keep_best(mixed, 2)
    with pytest.raises(ValueError, match="every job needs a reference_conformer"):
        P.generate_jobs_sharded(FakeEngine(), _scored_jobs(), keep_best=2, scorer=FakeScorer())
    with pytest.raises(ValueError, match="keep_best must be at least 1"):
        P.generate_jobs_sharded(FakeEngine(), [dict(reference_context=REFS[0], n_atoms=20, n_samples=2,
                                                    reference_conformer=_conf(4))], keep_best=0, scorer=FakeScorer())


def _toy(scores):
    """One scored job whose samples carry the given scores; rows of x / aligned tell the samples apart."""
    n = len(scores)
    packed = J.flatten_jobs([dict(reference_context=REFS[0], n_nodes=[20] * n, reference_conformer=_conf(4))])
    x = torch.arange(n, dtype=torch.float32).view(n, 1, 1).expand(n, 20, 3).contiguous()
    cls = torch.arange(n, dtype=torch.int32).view(n, 1).expand(n, 20).contiguous()
    bonds = torch.arange(n, dtype=torch.int8).view(n, 1, 1).expand(n, 42, 42).contiguous()
    res = J.split_jobs(packed, x, cls, bonds)
    return packed, res, torch.tensor(scores, dtype=torch.float32), torch.arange(n) % 4, x * 2


def test_keep_best_orders_by_score_with_ties_to_the_lower_index():
    scores = [0.5, 0.9, float("nan"), 0.5, 0.9, 0.1, 0.5]
    packed, res, s, o, al = _toy(scores)
    ref = [_conf(4)]
    full = J.attach_scores(packed, J.split_jobs(packed, *[res[0][k] for k in ("x", "atom_class", "bonds")]), s, o, al,
                           ref)[0]
    for k, want in ((3, [1, 4, 0]), (5, [1, 4, 0, 3, 6]), (1, [1]), (7, [1, 4, 0, 3, 6, 5, 2]), (50, [1, 4, 0, 3, 6, 5, 2])):
        packed, res, s, o, al = _toy(scores)
        got = J.attach_scores(packed, res, s, o, al, ref, keep_best=k)[0]
        assert got["sample_index"].dtype == torch.int64 and got["sample_index"].tolist() == want  # NaN ranks last
        keep = torch.tensor(want)
        for key in ("x", "atom_class", "bonds", "n_nodes", "shape_tanimoto", "best_orientation", "aligned_coords"):
            a, b = got[key], full[key][keep]
            if a.dtype == torch.float32:  # bit patterns: NaN rows count
                a, b = a.view(torch.int32), b.view(torch.int32)
            assert torch.equal(a, b), key
        assert torch.equal(got["reference_coords"], ref[0])
        assert set(got) == set(full) | {"sample_index"}


def test_scores_of_the_scored_jobs_and_unscored_jobs_unchanged():
    jobs = _scored_jobs()
    res, calls, packed = _single(jobs)
    plain, _, _ = _run(_jobs())
    # one scorer call over the samples of the scored jobs only, their jobs renumbered 0..3
    assert len(calls) == 1 and calls[0]["n_refs"] == 4
    scored = [0, 1, 3, 4]
    assert calls[0]["B"] == sum(int(packed.starts[j + 1] - packed.starts[j]) for j in scored)
    assert calls[0]["job"].tolist() == sorted(calls[0]["job"].tolist())
    for j in range(len(jobs)):
        if j not in scored:
            _same(res[j], plain[j])  # the same keys, dtypes and values as without scoring
            continue
        r, p = res[j], plain[j]
        assert set(r) == set(p) | {"shape_tanimoto", "best_orientation", "aligned_coords", "reference_coords"}
        for k in p:
            assert torch.equal(r[k], p[k])
        # each job's scores equal the scorer run on that job alone
        alone = FakeScorer().evaluate_jobs([packed.conformers[j]], p["x"], p["n_nodes"], torch.zeros(len(p["x"])))
        assert torch.equal(r["shape_tanimoto"], alone["shape_tanimoto"])
        assert torch.equal(r["best_orientation"], alone["best_orientation"])
        assert torch.equal(r["aligned_coords"], alone["aligned_coords"])
        assert torch.equal(r["reference_coords"], alone["reference_coords"][0])
        assert r["shape_tanimoto"].shape == (len(p["x"]),) and r["aligned_coords"].shape == p["x"].shape


def _sharded(jobs, keep_best, max_batch):
    e, sc = FakeEngine(), FakeScorer()
    res = P.generate_jobs_sharded(e, jobs, T=7, resample_steps=1, blend_power=2, ifm_diffusion_level=4, seed=3,
                                  max_batch=max_batch, keep_best=keep_best, scorer=sc)
    return res, e.calls, sc.calls


def _case(name):
    if name == "mixed":
        return _scored_jobs(), None
    if name == "keep_best":
        return [dict(j, reference_conformer=_conf(3 + k, k)) for k, j in enumerate(_jobs())], 3
    # one molecule in all: the second rank's shard is empty
    return [dict(reference_context=REFS[1], n_atoms=24, n_samples=1, fixed_fragment=_frag(3),
                 reference_conformer=_conf(7))], 1


def _worker(rank, world, port, tmp, name, max_batch):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    jobs, k = _case(name)
    torch.save(_sharded(jobs, k, max_batch), tmp + ".%d" % rank)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("name,max_batch,port", [("mixed", 8192, 29561), ("keep_best", 4, 29562), ("empty_shard", 8192, 29563)])
def test_sharded_scored_jobs_match_the_single_process_result(tmp_path, name, max_batch, port):
    jobs, k = _case(name)
    want, _, packed = _single(jobs, k)
    single, _, _ = _sharded(jobs, k, max_batch)
    for a, b in zip(want, single):
        _same(a, b)
    out_file = str(tmp_path / "scored.pt")
    mp.spawn(_worker, args=(2, port, out_file, name, max_batch), nprocs=2, join=True)
    shards = P.shard_indices(packed.n_nodes, 2)
    if name == "empty_shard":
        assert [len(s) for s in shards] == [1, 0]
    for r in range(2):
        got, calls, score_calls = torch.load(out_file + ".%d" % r, weights_only=False)
        assert len(got) == len(want)
        for a, b in zip(want, got):  # every rank holds every job, scores and selection included
            _same(a, b)
        # each rank scored its own samples only
        assert sum(c["B"] for c in score_calls) == sum(packed.conformers[packed.job[i]] is not None for i in shards[r])
        assert sum(len(c["ids"]) for c in calls) == len(shards[r])
