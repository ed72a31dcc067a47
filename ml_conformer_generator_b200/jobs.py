"""Many small generation jobs packed into few device calls.

A job is one reference (and optionally one fixed fragment) with its own atom counts and sample count -- what one call of
the reference's `generate_conformers` asks for -- or, for an analogue job, one parent molecule whose analogues are wanted:
the parent forward-diffused to a diffusion level and denoised from there (the reference's merge_fragments loop run on a
whole molecule), optionally with some of its atoms kept fixed.  Jobs are flattened into per-sample arrays (atom counts,
normalised context, job index, global sample id), grouped by kind (plain, inpainting, inertial fragment matching,
analogue -- the analogue jobs further by (has fixed atoms, diffusion level): one group per device call) and cut into calls
of at most `max_batch` samples; a job may straddle two calls.

Determinism: sample k of a job has the global id `job_id * 2**32 + k`, which keys its device noise, and the job's atom
counts are drawn from a generator seeded by `(seed, job_id)`.  Every kernel works on each sample alone, so a job's
molecules depend only on `seed`, its `job_id`, its own fields and the shared loop settings -- never on the other jobs,
their order or how the samples are cut into calls or shards.

A job with a `reference_conformer` also has its molecules scored by Gaussian shape Tanimoto against that conformer
(`score_packed`, one `ShapeScorer.evaluate_jobs` pass over the samples of all scored jobs) and may keep only its best ones
(`attach_scores`).  Scoring works on each sample alone too, so the same independence holds for the scores."""
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from .config import CONTEXT_NORMS, MAX_N_NODES, MIN_N_NODES
from .mol_utils import _check_fragment_size, get_context_shape, normalise_context

KINDS = ("plain", "inpaint", "ifm", "analogue")
JOB_ID_SHIFT = 32
_JOB_KEYS = {"reference_context", "n_atoms", "variance", "n_nodes", "n_samples", "fixed_fragment",
             "inertial_fragment_matching", "job_id", "reference_conformer", "parent_molecule", "fixed_atoms",
             "diffusion_level"}
_NOT_WITH_PARENT = ("n_atoms", "variance", "n_nodes", "fixed_fragment", "inertial_fragment_matching")
SHAPE_MAX_ATOMS = 64  # atoms of a reference conformer (the shape kernels' limit)


@dataclass
class PackedJobs:
    """Jobs flattened into per-sample arrays (S samples, J jobs, samples of job j at starts[j]:starts[j+1])."""
    kind: np.ndarray         # (J,) index into KINDS
    job_ids: np.ndarray      # (J,) int64
    max_n_nodes: np.ndarray  # (J,) padded atom count of each job's results
    starts: np.ndarray       # (J+1,) int64
    fragments: List[Optional[tuple]]  # (J) (coordinates (n,3) f32, one-hot (n,8) f32) or None
    references: List[torch.Tensor]    # (J) raw reference context (3,) f32
    n_nodes: np.ndarray      # (S,) int32
    ctx: np.ndarray          # (S,3) f32 normalised context
    job: np.ndarray          # (S,) int32 job index
    ids: np.ndarray          # (S,) int64 global sample id (the noise key)
    conformers: Optional[List[Optional[torch.Tensor]]] = None  # (J) heavy-atom reference conformer (n_ref,3) f32 or None
    # (J) analogue jobs: (coordinates centred on their mean (n,3) f32, one-hot (n,8) f32, fixed flags (n,) i32, the mean
    # (3,) f32), else None
    parents: Optional[List[Optional[tuple]]] = None
    levels: Optional[np.ndarray] = None  # (J,) i32 the analogue job's own diffusion_level, 0 = the call's default

    @property
    def scored(self) -> bool:
        """Whether any job has a reference conformer to score its molecules against."""
        return self.conformers is not None and any(c is not None for c in self.conformers)

    @property
    def N(self) -> int:
        return int(self.max_n_nodes.max())


def job_atom_counts(seed: int, job_id: int, lo: int, hi: int, n_samples: int) -> np.ndarray:
    """Atom counts of a job, uniform in [lo, hi], from a generator seeded by (seed, job_id) alone."""
    return np.random.default_rng([seed, job_id]).integers(lo, hi + 1, n_samples).astype(np.int32)


def flatten_jobs(jobs: Sequence[Dict], seed: int = 0, context_norms: Dict = CONTEXT_NORMS,
                 min_n_nodes: int = MIN_N_NODES, max_n_nodes: int = MAX_N_NODES) -> PackedJobs:
    """Validates the jobs and flattens them (see MLConformerGenerator.generate_jobs for the job fields)."""
    if seed < 0:
        raise ValueError("seed must be non-negative")
    if len(jobs) == 0:
        raise ValueError("generate_jobs: no jobs")
    kind, job_ids, tops, fragments, refs, confs, parents, levels = [], [], [], [], [], [], [], []
    n_nodes, ctx = [], []
    for p, job in enumerate(jobs):
        unknown = set(job) - _JOB_KEYS
        if unknown:
            raise ValueError("job %d: unknown field(s) %s" % (p, sorted(unknown)))
        job_id = int(job.get("job_id", p))
        if not 0 <= job_id < 2 ** 31:
            raise ValueError("job %d: job_id must be in [0, 2**31)" % p)
        parent, level = _parent(p, job, max_n_nodes), 0
        if parent is None:
            for k in ("fixed_atoms", "diffusion_level"):
                if job.get(k) is not None:
                    raise ValueError("job %d: %s needs a parent_molecule" % (p, k))
        elif job.get("diffusion_level") is not None:
            level = int(job["diffusion_level"])
            if level < 1:
                raise ValueError("job %d: diffusion_level must be at least 1" % p)
        if parent is not None and job.get("reference_context") is None:
            # the parent's own principal moments, as generate_conformers takes them from a reference conformer
            ref = get_context_shape(parent[0])[0]
        else:
            ref = torch.as_tensor(job["reference_context"], dtype=torch.float32).detach().cpu().reshape(-1)
        if ref.numel() != 3:
            raise ValueError("job %d: reference_context must hold 3 principal moments" % p)
        if parent is not None:
            if job.get("n_samples") is None:
                raise ValueError("job %d: an analogue job needs n_samples" % p)
            lo = hi = int(parent[0].shape[0])
            nn = np.full(int(job["n_samples"]), lo, dtype=np.int32)
        elif job.get("n_nodes") is not None:
            nn = np.asarray(job["n_nodes"]).reshape(-1).astype(np.int32)
            if "n_samples" in job and int(job["n_samples"]) != nn.size:
                raise ValueError("job %d: n_samples does not match len(n_nodes)" % p)
            if nn.size and (nn.min() < 1 or nn.max() > max_n_nodes):
                raise ValueError("job %d: n_nodes must lie in [1, %d]" % (p, max_n_nodes))
            lo, hi = (int(nn.min()), int(nn.max())) if nn.size else (0, 0)
        else:
            n_atoms, variance = int(job["n_atoms"]), int(job.get("variance", 2))
            lo, hi = max(n_atoms - variance, min_n_nodes), min(n_atoms + variance, max_n_nodes)
            if lo > hi:
                raise ValueError("job %d: n_atoms +- variance leaves no atom count in [%d, %d]" % (p, min_n_nodes,
                                                                                                  max_n_nodes))
            nn = job_atom_counts(seed, job_id, lo, hi, int(job["n_samples"]))
        if not 1 <= nn.size < 2 ** JOB_ID_SHIFT:
            raise ValueError("job %d: n_samples must be at least 1" % p)
        frag = job.get("fixed_fragment")
        if parent is not None:
            kind.append(3)
            fragments.append(None)
        elif frag is None:
            kind.append(0)
            fragments.append(None)
        else:
            fx = torch.as_tensor(frag[0]).detach().cpu().to(torch.float32)
            fh = torch.as_tensor(frag[1]).detach().cpu().to(torch.float32)
            if fx.dim() != 2 or fx.shape[1] != 3 or tuple(fh.shape) != (fx.shape[0], 8):
                raise ValueError("job %d: the fragment must be coordinates (n,3) and a one-hot (n,8)" % p)
            _check_fragment_size(int(fx.shape[0]), lo, hi)
            kind.append(2 if job.get("inertial_fragment_matching", True) else 1)
            fragments.append((fx, fh))
        conf = job.get("reference_conformer")
        if conf is not None:
            conf = torch.as_tensor(conf).detach().cpu().to(torch.float32)
            if conf.dim() != 2 or conf.shape[1] != 3:
                raise ValueError("job %d: reference_conformer must be heavy-atom coordinates (n, 3)" % p)
            if not 3 <= conf.shape[0] <= SHAPE_MAX_ATOMS:
                raise ValueError("job %d: reference_conformer must have 3 <= n <= %d atoms" % (p, SHAPE_MAX_ATOMS))
        confs.append(conf)
        parents.append(parent)
        levels.append(level)
        job_ids.append(job_id)
        tops.append(hi)
        refs.append(ref)
        n_nodes.append(nn)
        ctx.append(np.tile(normalise_context(ref, context_norms).numpy().reshape(1, 3), (nn.size, 1)))
    job_ids = np.asarray(job_ids, dtype=np.int64)
    if np.unique(job_ids).size != job_ids.size:
        raise ValueError("job ids must be unique: two jobs with one id would draw the same noise")
    sizes = np.array([a.size for a in n_nodes], dtype=np.int64)
    starts = np.concatenate([[0], np.cumsum(sizes)])
    job = np.repeat(np.arange(len(jobs), dtype=np.int32), sizes)
    ids = (job_ids[job] << JOB_ID_SHIFT) + (np.arange(starts[-1], dtype=np.int64) - starts[job])
    return PackedJobs(np.asarray(kind, dtype=np.int32), job_ids, np.asarray(tops, dtype=np.int32), starts, fragments, refs,
                      np.concatenate(n_nodes).astype(np.int32), np.concatenate(ctx).astype(np.float32), job, ids, confs,
                      parents, np.asarray(levels, dtype=np.int32))


def _parent(p: int, job: Dict, max_n_nodes: int) -> Optional[tuple]:
    """The validated parent of an analogue job (see PackedJobs.parents), or None for the other kinds."""
    mol = job.get("parent_molecule")
    if mol is None:
        return None
    clash = [k for k in _NOT_WITH_PARENT if k in job]
    if clash:
        raise ValueError("job %d: parent_molecule fixes the atoms of every sample; %s cannot go with it" % (p, clash))
    try:
        px, ph = mol
    except (TypeError, ValueError):
        raise ValueError("job %d: parent_molecule must be (coordinates (n,3), one-hot (n,8))" % p) from None
    px = torch.as_tensor(px).detach().cpu().to(torch.float32)
    ph = torch.as_tensor(ph).detach().cpu().to(torch.float32)
    if px.dim() != 2 or px.shape[1] != 3 or tuple(ph.shape) != (px.shape[0], 8):
        raise ValueError("job %d: parent_molecule must be (coordinates (n,3), one-hot (n,8))" % p)
    n = int(px.shape[0])
    if not 3 <= n <= max_n_nodes:
        raise ValueError("job %d: parent_molecule must have 3 <= n <= %d atoms" % (p, max_n_nodes))
    if not bool(((ph == 0) | (ph == 1)).all()) or not bool((ph.sum(1) == 1).all()):
        raise ValueError("job %d: the parent's one-hot must hold one 1 per atom, zeros elsewhere" % p)
    if not bool(torch.isfinite(px).all()):
        raise ValueError("job %d: the parent's coordinates must be finite" % p)
    fixed = np.zeros(n, dtype=np.int32)
    fa = job.get("fixed_atoms")
    if fa is not None:
        fa = np.asarray(fa).reshape(-1)
        if fa.size and not np.issubdtype(fa.dtype, np.integer):
            raise ValueError("job %d: fixed_atoms must be atom indices" % p)
        fa = fa.astype(np.int64)
        if fa.size and (fa.min() < 0 or fa.max() >= n):
            raise ValueError("job %d: fixed_atoms must index the parent's %d atoms" % (p, n))
        if np.unique(fa).size != fa.size:
            raise ValueError("job %d: fixed_atoms must be distinct" % p)
        if fa.size > n - 1:
            raise ValueError("job %d: at most n - 1 = %d atoms can be fixed" % (p, n - 1))
        fixed[fa] = 1
    mean = px.mean(dim=0)
    # the loop is free of the centre of mass: the parent enters centred, and its mean is added back to the results
    return px - mean, ph, fixed, mean


def analogue_levels(packed: PackedJobs, default_level: int, T: int) -> np.ndarray:
    """(J,) diffusion level of every analogue job -- its own, else `default_level` -- and 0 for the other kinds.  Raises
    unless every level lies in [1, T]."""
    out = np.zeros(len(packed.job_ids), dtype=np.int64)
    for j in np.nonzero(packed.kind == 3)[0]:
        out[j] = packed.levels[j] if packed.levels[j] > 0 else int(default_level)
        if not 1 <= out[j] <= T:
            raise ValueError("job %d: diffusion_level must lie in [1, T=%d], got %d" % (j, T, out[j]))
    return out


def run_packed(engine, packed: PackedJobs, idx: np.ndarray, T: int = 100, resample_steps: int = 0, blend_power: int = 3,
               ifm_diffusion_level: int = 50, seed: int = 0, max_batch: int = 8192, device_out: bool = False,
               context_norms: Optional[Dict] = None):
    """Generates the flat samples `idx`: per kind, calls of at most `max_batch` of them -- Engine.generate_host for plain
    jobs, Engine.generate_fragment_jobs_host for fragment jobs, Engine.generate_analogue_jobs_host for analogue jobs (one
    group per (has fixed atoms, diffusion level), the level defaulting to `ifm_diffusion_level`; coordinates returned in
    the parent's input frame) -- padded to the largest max_n_nodes of the jobs in the call.  Returns (x (n,N,3) f32, atom_class (n,N) i32, bonds (n,42,42) i8) in the order of `idx`, N = packed.N; rows
    beyond a call's padding are x = 0, atom_class = -1.  On the engine's device with `device_out`, else on the host."""
    idx = np.asarray(idx, dtype=np.int64).reshape(-1)
    dev = engine.device if device_out else torch.device("cpu")
    n, N = idx.size, packed.N
    x = torch.zeros(n, N, 3, device=dev)
    cls = torch.full((n, N), -1, dtype=torch.int32, device=dev)
    bonds = torch.zeros(n, 42, 42, dtype=torch.int8, device=dev)
    # one group per device call kind; analogue jobs further by (has fixed atoms, diffusion level)
    levels = analogue_levels(packed, ifm_diffusion_level, T)
    has_fixed = np.array([p is not None and bool(p[2].any()) for p in (packed.parents or [None] * len(packed.kind))])
    group = np.stack([packed.kind, has_fixed, levels], axis=1)[packed.job[idx]]
    for g in np.unique(group, axis=0):
        k = int(g[0])
        rows = np.nonzero((group == g).all(axis=1))[0]
        for s in range(0, rows.size, max_batch):
            r = rows[s:s + max_batch]
            sel = idx[r]
            here = np.unique(packed.job[sel])
            nc = int(packed.max_n_nodes[here].max())
            if k == 0:
                out = engine.generate_host(packed.n_nodes[sel], nc, packed.ctx[sel], T, resample_steps, seed=seed,
                                           sample_ids=packed.ids[sel], device_out=device_out)
            elif k == 3:
                out = engine.generate_analogue_jobs_host(
                    packed.n_nodes[sel], nc, packed.ctx[sel], np.searchsorted(here, packed.job[sel]),
                    [packed.parents[j][:2] for j in here], [packed.parents[j][2] for j in here], T, resample_steps,
                    blend_power, int(g[2]), seed=seed, sample_ids=packed.ids[sel], device_out=device_out)
                # back to the parent's input frame: its mean added to the real atoms
                xo = out[0]
                mean = torch.stack([packed.parents[j][3] for j in packed.job[sel]]).to(xo.device).view(-1, 1, 3)
                real = (torch.arange(nc).view(1, nc) < torch.from_numpy(packed.n_nodes[sel]).view(-1, 1)).to(xo.device)
                out = (torch.where(real.unsqueeze(-1), xo + mean, xo),) + tuple(out[1:])
            else:
                out = engine.generate_fragment_jobs_host(
                    packed.n_nodes[sel], nc, packed.ctx[sel], np.searchsorted(here, packed.job[sel]),
                    [packed.fragments[j] for j in here], k == 2, [packed.references[j] for j in here], context_norms, T,
                    resample_steps, blend_power, ifm_diffusion_level, seed=seed, sample_ids=packed.ids[sel],
                    device_out=device_out)
            rr = torch.as_tensor(r, device=dev)
            x[rr, :nc] = out[0].to(dev)
            cls[rr, :nc] = out[1].to(dev)
            bonds[rr] = out[2].to(dev)
    return x, cls, bonds


def split_jobs(packed: PackedJobs, x: torch.Tensor, cls: torch.Tensor, bonds: torch.Tensor) -> List[Dict[str, torch.Tensor]]:
    """All samples in flat order -> one dict per job, in input order, sliced to the job's own max atom count."""
    res = []
    for j in range(len(packed.job_ids)):
        a, b, nj = int(packed.starts[j]), int(packed.starts[j + 1]), int(packed.max_n_nodes[j])
        res.append({"x": x[a:b, :nj].clone(), "atom_class": cls[a:b, :nj].clone(),
                    "n_nodes": torch.from_numpy(packed.n_nodes[a:b].astype(np.int64)), "bonds": bonds[a:b].clone()})
    return res


def check_keep_best(packed: PackedJobs, keep_best: Optional[int]) -> None:
    if keep_best is None:
        return
    if int(keep_best) < 1:
        raise ValueError("keep_best must be at least 1")
    if packed.conformers is None or any(c is None for c in packed.conformers):
        raise ValueError("keep_best ranks by shape: every job needs a reference_conformer")


def score_row_spec(N: int) -> Tuple[Tuple[torch.dtype, tuple], ...]:
    """dtype and per-sample shape of score_packed's per-sample outputs, for packing them next to the molecules."""
    return ((torch.float32, ()), (torch.int64, ()), (torch.float32, (N, 3)))


def score_packed(scorer, packed: PackedJobs, idx: np.ndarray, x: torch.Tensor):
    """Scores the flat samples `idx` (x (n,N,3) in the order of `idx`, N = packed.N) of the jobs with a reference conformer
    in one `scorer.evaluate_jobs` pass.  Returns (shape_tanimoto (n,) f32, best_orientation (n,) i64, aligned_coords
    (n,N,3) f32) on x's device -- rows of jobs without a conformer are 0 -- and the list over the jobs of each reference in
    its principal frame (None for jobs without one)."""
    idx = np.asarray(idx, dtype=np.int64).reshape(-1)
    has = np.array([c is not None for c in packed.conformers])
    scored_jobs = np.nonzero(has)[0]
    rows = np.nonzero(has[packed.job[idx]])[0]
    dev, n = x.device, idx.size
    rr = torch.as_tensor(rows, device=dev)
    out = scorer.evaluate_jobs([packed.conformers[j] for j in scored_jobs], x[rr],
                               torch.from_numpy(packed.n_nodes[idx[rows]]),
                               torch.from_numpy(np.searchsorted(scored_jobs, packed.job[idx[rows]]).astype(np.int64)))
    score = torch.zeros(n, device=dev)
    orient = torch.zeros(n, dtype=torch.int64, device=dev)
    aligned = torch.zeros(n, x.shape[1], 3, device=dev)
    score[rr], orient[rr], aligned[rr] = (out[k].to(dev) for k in ("shape_tanimoto", "best_orientation", "aligned_coords"))
    ref_coords = [None] * len(packed.conformers)
    for k, j in enumerate(scored_jobs):
        ref_coords[j] = out["reference_coords"][k]
    return score, orient, aligned, ref_coords


def attach_scores(packed: PackedJobs, res: List[Dict[str, torch.Tensor]], score: torch.Tensor, orient: torch.Tensor,
                  aligned: torch.Tensor, ref_coords: List[Optional[torch.Tensor]],
                  keep_best: Optional[int] = None) -> List[Dict[str, torch.Tensor]]:
    """Adds shape_tanimoto, best_orientation, aligned_coords and reference_coords to the dict (split_jobs) of every job
    with a reference conformer; `score` etc. hold all samples in flat order.  With `keep_best` = k each such job keeps its
    min(k, n) best molecules, by shape_tanimoto descending (NaN last), ties to the lower sample index, with
    `sample_index` the row of each in the unfiltered job.  Jobs without a conformer are left as they are."""
    for j, r in enumerate(res):
        if packed.conformers[j] is None:
            continue
        a, b, nj = int(packed.starts[j]), int(packed.starts[j + 1]), int(packed.max_n_nodes[j])
        r.update(shape_tanimoto=score[a:b].clone(), best_orientation=orient[a:b].clone(),
                 aligned_coords=aligned[a:b, :nj].clone())
        if keep_best is not None:
            s = r["shape_tanimoto"]
            key = torch.where(torch.isnan(s), torch.full_like(s, -float("inf")), s)
            keep = torch.sort(key, descending=True, stable=True).indices[:int(keep_best)]
            for k in list(r):
                r[k] = r[k][keep.to(r[k].device)]
            r["sample_index"] = keep
        r["reference_coords"] = ref_coords[j]
    return res
