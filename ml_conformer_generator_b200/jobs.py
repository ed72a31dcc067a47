"""Many small generation jobs packed into few device calls.

A job is one reference (and optionally one fixed fragment) with its own atom counts and sample count -- what one call of
the reference's `generate_conformers` asks for.  Jobs are flattened into per-sample arrays (atom counts, normalised
context, job index, global sample id), grouped by kind (plain, inpainting, inertial fragment matching: one kind per device
call) and cut into calls of at most `max_batch` samples; a job may straddle two calls.

Determinism: sample k of a job has the global id `job_id * 2**32 + k`, which keys its device noise, and the job's atom
counts are drawn from a generator seeded by `(seed, job_id)`.  Every kernel works on each sample alone, so a job's
molecules depend only on `seed`, its `job_id`, its own fields and the shared loop settings -- never on the other jobs,
their order or how the samples are cut into calls or shards."""
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence

import numpy as np
import torch

from .config import CONTEXT_NORMS, MAX_N_NODES, MIN_N_NODES
from .mol_utils import _check_fragment_size, normalise_context

KINDS = ("plain", "inpaint", "ifm")
JOB_ID_SHIFT = 32
_JOB_KEYS = {"reference_context", "n_atoms", "variance", "n_nodes", "n_samples", "fixed_fragment",
             "inertial_fragment_matching", "job_id"}


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
    kind, job_ids, tops, fragments, refs = [], [], [], [], []
    n_nodes, ctx = [], []
    for p, job in enumerate(jobs):
        unknown = set(job) - _JOB_KEYS
        if unknown:
            raise ValueError("job %d: unknown field(s) %s" % (p, sorted(unknown)))
        job_id = int(job.get("job_id", p))
        if not 0 <= job_id < 2 ** 31:
            raise ValueError("job %d: job_id must be in [0, 2**31)" % p)
        ref = torch.as_tensor(job["reference_context"], dtype=torch.float32).detach().cpu().reshape(-1)
        if ref.numel() != 3:
            raise ValueError("job %d: reference_context must hold 3 principal moments" % p)
        if job.get("n_nodes") is not None:
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
        if frag is None:
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
                      np.concatenate(n_nodes).astype(np.int32), np.concatenate(ctx).astype(np.float32), job, ids)


def run_packed(engine, packed: PackedJobs, idx: np.ndarray, T: int = 100, resample_steps: int = 0, blend_power: int = 3,
               ifm_diffusion_level: int = 50, seed: int = 0, max_batch: int = 8192, device_out: bool = False,
               context_norms: Optional[Dict] = None):
    """Generates the flat samples `idx`: per kind, calls of at most `max_batch` of them -- Engine.generate_host for plain
    jobs, Engine.generate_fragment_jobs_host for fragment jobs -- padded to the largest max_n_nodes of the jobs in the
    call.  Returns (x (n,N,3) f32, atom_class (n,N) i32, bonds (n,42,42) i8) in the order of `idx`, N = packed.N; rows
    beyond a call's padding are x = 0, atom_class = -1.  On the engine's device with `device_out`, else on the host."""
    idx = np.asarray(idx, dtype=np.int64).reshape(-1)
    dev = engine.device if device_out else torch.device("cpu")
    n, N = idx.size, packed.N
    x = torch.zeros(n, N, 3, device=dev)
    cls = torch.full((n, N), -1, dtype=torch.int32, device=dev)
    bonds = torch.zeros(n, 42, 42, dtype=torch.int8, device=dev)
    kinds = packed.kind[packed.job[idx]]
    for k in range(len(KINDS)):
        rows = np.nonzero(kinds == k)[0]
        for s in range(0, rows.size, max_batch):
            r = rows[s:s + max_batch]
            sel = idx[r]
            here = np.unique(packed.job[sel])
            nc = int(packed.max_n_nodes[here].max())
            if k == 0:
                out = engine.generate_host(packed.n_nodes[sel], nc, packed.ctx[sel], T, resample_steps, seed=seed,
                                           sample_ids=packed.ids[sel], device_out=device_out)
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
