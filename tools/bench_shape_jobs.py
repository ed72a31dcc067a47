"""Shape scoring of many jobs on one GPU, each job against its own reference conformer.

  (a) scoring: 8192 samples of 15-39 atoms spread over 64 jobs with 64 different references (15-39 atoms each).  One
      ShapeScorer.evaluate call per job (the loop a user writes today: slice the job's samples, score, repeat) against
      one ShapeScorer.evaluate_jobs call.  The outputs are asserted equal bit for bit.
  (b) scoring inside generation: MLConformerGenerator.generate_jobs on 64 jobs x 128 samples at C3 sizes (atom counts
      15-39, T = 100), without and with a reference_conformer on every job; the difference is the cost of scoring, as a
      share of generation.  The molecules of the two arms are asserted identical bit for bit.

  python tools/bench_shape_jobs.py --out profiles/shape_jobs_bench.jsonl [--T 100] [--reps 3] [--precision fp16]

Both arms of each part are warmed up, then alternate `--reps` times; every timed call ends in a device synchronise.  One
JSON line per (part, arm) with the card's name and power limit read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from ml_conformer_generator_b200 import MLConformerGenerator  # noqa: E402
from ml_conformer_generator_b200.shape_similarity import ShapeScorer  # noqa: E402
from ml_conformer_generator_b200.weights import random_state_dicts  # noqa: E402

N_JOBS, PER_JOB = 64, 128
BASE_CONTEXT = np.array([53.6424, 108.3042, 151.4399], np.float32)  # raw context of configs C2-C5


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    return q or torch.cuda.get_device_name(0)


def skeleton(rng, n):
    """A compact random heavy-atom skeleton: a random walk of 1.5 A steps, rotated and shifted."""
    steps = rng.normal(size=(n, 3))
    steps *= 1.5 / np.linalg.norm(steps, axis=1, keepdims=True)
    q, _ = np.linalg.qr(rng.normal(size=(3, 3)))
    return torch.from_numpy(((np.cumsum(steps, axis=0) * 0.6) @ q + rng.normal(scale=3.0, size=3)).astype(np.float32))


def scoring_inputs():
    """64 references of 15-39 atoms; 128 samples per job of 15-39 atoms (perturbed copies of part of the reference or
    unrelated skeletons), in shuffled job order, padded to 39."""
    rng = np.random.default_rng(7)
    refs = [skeleton(rng, int(n)) for n in rng.integers(15, 40, N_JOBS)]
    job = rng.permutation(np.repeat(np.arange(N_JOBS), PER_JOB))
    n_nodes = rng.integers(15, 40, job.size)
    coords = torch.zeros(job.size, 39, 3)
    for b in range(job.size):
        r, n = refs[job[b]], int(n_nodes[b])
        if b % 2 and r.size(0) >= n:
            coords[b, :n] = r[:n] + torch.from_numpy(rng.normal(scale=0.4, size=(n, 3))).float()
        else:
            coords[b, :n] = skeleton(rng, n)
    return refs, coords, torch.from_numpy(n_nodes), torch.from_numpy(job)


def bits(t):
    t = torch.as_tensor(t).detach().cpu()
    return t.view(torch.int32) if t.dtype == torch.float32 else t


def timed(f):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = f()
    torch.cuda.synchronize()
    return out, time.perf_counter() - t0


def part_a(sc, reps):
    refs, coords, n_nodes, job = scoring_inputs()
    coords_d = coords.to(sc.device)
    rows = [torch.nonzero(job == j).view(-1) for j in range(N_JOBS)]

    def per_job():  # the samples of a job sliced out of the device batch, scored, and the next job
        return [sc.evaluate(refs[j], coords_d[r.to(sc.device)], n_nodes[r]) for j, r in enumerate(rows)]

    def packed():
        return sc.evaluate_jobs(refs, coords_d, n_nodes, job)

    arms = {"evaluate_per_job": per_job, "evaluate_jobs": packed}
    ref = {k: f() for k, f in arms.items()}
    for j, r in enumerate(rows):
        w, g = ref["evaluate_per_job"][j], ref["evaluate_jobs"]
        for k in ("shape_tanimoto", "best_orientation", "aligned_coords", "scores", "moments"):
            assert torch.equal(bits(g[k].cpu()[r]), bits(w[k])), "part a: %s of job %d differs" % (k, j)
        assert torch.equal(bits(g["reference_coords"][j]), bits(w["reference_coords"]))
    times = {k: [] for k in arms}
    for _ in range(reps):
        for k, f in arms.items():
            times[k].append(timed(f)[1])
    return times, int(job.numel())


def make_jobs(with_refs):
    rng = np.random.RandomState(7)
    out = []
    for k in range(N_JOBS):
        job = dict(reference_context=torch.from_numpy(BASE_CONTEXT * rng.uniform(0.8, 1.25, 3).astype(np.float32)),
                   n_atoms=27, variance=12, n_samples=PER_JOB)
        conf = skeleton(np.random.default_rng([7, k]), 15 + k % 25)
        if with_refs:
            job["reference_conformer"] = conf
        out.append(job)
    return out


def part_b(gen, reps, seed=3):
    jobs = {"generate_jobs": make_jobs(False), "generate_jobs_scored": make_jobs(True)}
    arms = {k: (lambda j=j: gen.generate_jobs(j, seed=seed)) for k, j in jobs.items()}
    ref = {k: f() for k, f in arms.items()}
    for a, b in zip(ref["generate_jobs"], ref["generate_jobs_scored"]):
        for k in a:
            assert torch.equal(bits(a[k]), bits(b[k])), "part b: the molecules differ with references (%s)" % k
    finite = all(bool(torch.isfinite(r["shape_tanimoto"]).all()) for r in ref["generate_jobs_scored"])
    times = {k: [] for k in arms}
    for _ in range(reps):
        for k, f in arms.items():
            times[k].append(timed(f)[1])
    return times, sum(j["n_samples"] for j in jobs["generate_jobs"]), finite


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--T", type=int, default=100)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--precision", default="fp16")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_shape_jobs.py measures the GPU; no CUDA device is visible")
    sd, ssd = random_state_dicts(0)
    gen = MLConformerGenerator(diffusion_steps=args.T, device=torch.device("cuda:0"), precision=args.precision,
                               edm_state_dict=sd, adj_mat_seer_state_dict=ssd)
    info = card()
    recs = []
    times, S = part_a(ShapeScorer(gen.engine), args.reps)
    for arm, ts in times.items():
        recs.append({"part": "a: scoring", "arm": arm, "jobs": N_JOBS, "references": N_JOBS, "samples": S, "atoms": "15-39",
                     "grid_points": 40, "seconds": ts, "seconds_median": float(np.median(ts)),
                     "outputs_bit_identical": True})
    times, S, finite = part_b(gen, args.reps)
    med = {k: float(np.median(v)) for k, v in times.items()}
    for arm, ts in times.items():
        recs.append({"part": "b: scoring inside generate_jobs", "arm": arm, "jobs": N_JOBS, "samples": S, "atoms": "15-39",
                     "T": args.T, "precision": args.precision, "seconds": ts, "seconds_median": med[arm],
                     "molecules_bit_identical": True, "scores_finite": finite})
    recs[-1]["scoring_share_of_generation"] = (med["generate_jobs_scored"] - med["generate_jobs"]) / med["generate_jobs"]
    with open(args.out, "a") as fh:
        for rec in recs:
            rec["card(name, power.limit, clocks.sm, clocks.max.sm)"] = info
            line = json.dumps(rec)
            print(line, flush=True)
            fh.write(line + "\n")
    gen.engine.close()


if __name__ == "__main__":
    main()
