"""Many small jobs: MLConformerGenerator.generate_jobs (jobs packed into one call per kind) against one call per job
(Engine.generate_host / generate_fragment_host, as a user calls the library for one reference at a time), on one GPU.

Workloads, 64 jobs x 128 samples each (8192 molecules), every job with its own reference context:
  plain    atom counts 15-39 (n_atoms 27 +- 12), no fragment
  ifm      C4-like: 21-25 atoms (23 +- 2), a fixed fragment of 3-8 atoms per job, inertial fragment matching (L = 50)
  inpaint  the same sizes and fragments as ifm, inpainted

  python tools/bench_jobs.py --out profiles/jobs_bench.jsonl [--T 100] [--reps 2] [--precision fp16]

Both arms are warmed up, then alternate `--reps` times.  The outputs of the two arms are asserted identical bit for bit in
the same run.  One JSON line per (workload, arm) with the card's name, power limit and clocks read in the same run."""
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
from ml_conformer_generator_b200 import jobs as J  # noqa: E402
from ml_conformer_generator_b200.weights import random_state_dicts  # noqa: E402

N_JOBS, PER_JOB, IFM_LEVEL = 64, 128, 50
BASE_CONTEXT = np.array([53.6424, 108.3042, 151.4399], np.float32)  # raw context of configs C2-C5


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    return q or torch.cuda.get_device_name(0)


def make_jobs(kind):
    rng = np.random.RandomState(7)
    out = []
    for k in range(N_JOBS):
        ref = torch.from_numpy(BASE_CONTEXT * rng.uniform(0.8, 1.25, 3).astype(np.float32))
        if kind == "plain":
            out.append(dict(reference_context=ref, n_atoms=27, variance=12, n_samples=PER_JOB))
            continue
        n_ff = 3 + k % 6
        frag = (torch.from_numpy(rng.normal(0, 1.4, (n_ff, 3)).astype(np.float32)),
                torch.eye(8)[torch.from_numpy(rng.randint(0, 6, n_ff))])
        out.append(dict(reference_context=ref, n_atoms=23, variance=2, n_samples=PER_JOB, fixed_fragment=frag,
                        inertial_fragment_matching=kind == "ifm"))
    return out


def per_job(gen, packed, T, seed):
    """One host call per job; results in flat sample order, padded to packed.N like run_packed's."""
    e = gen.engine
    S, N = packed.ids.size, packed.N
    x, cls, bonds = torch.zeros(S, N, 3), torch.full((S, N), -1, dtype=torch.int32), torch.zeros(S, 42, 42, dtype=torch.int8)
    for j in range(len(packed.job_ids)):
        a, b, nj = int(packed.starts[j]), int(packed.starts[j + 1]), int(packed.max_n_nodes[j])
        args = (packed.n_nodes[a:b], nj, packed.ctx[a:b])
        if packed.kind[j] == 0:
            o = e.generate_host(*args, T, 0, seed=seed, sample_ids=packed.ids[a:b])
        else:
            fx, fh = packed.fragments[j]
            o = e.generate_fragment_host(*args, fx, fh, packed.kind[j] == 2, packed.references[j], gen.context_norms, T, 0,
                                         3, IFM_LEVEL, seed=seed, sample_ids=packed.ids[a:b])
        x[a:b, :nj], cls[a:b, :nj], bonds[a:b] = o
    return J.split_jobs(packed, x, cls, bonds)


def same(r1, r2):
    for a, b in zip(r1, r2):
        for k in a:
            u, v = a[k], b[k]
            if u.dtype == torch.float32:
                u, v = u.view(torch.int32), v.view(torch.int32)
            if u.shape != v.shape or not torch.equal(u, v):
                return False
    return True


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--T", type=int, default=100)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--precision", default="fp16")
    ap.add_argument("--workloads", default="plain,ifm,inpaint")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_jobs.py measures the GPU; no CUDA device is visible")
    sd, ssd = random_state_dicts(0)
    gen = MLConformerGenerator(diffusion_steps=args.T, device=torch.device("cuda:0"), precision=args.precision,
                               edm_state_dict=sd, adj_mat_seer_state_dict=ssd)
    info = card()
    seed = 3
    with open(args.out, "a") as fh:
        for kind in args.workloads.split(","):
            jobs = make_jobs(kind)
            packed = J.flatten_jobs(jobs, seed, gen.context_norms, gen.min_n_nodes, gen.max_n_nodes)
            arms = {"packed": lambda: gen.generate_jobs(jobs, ifm_diffusion_level=IFM_LEVEL, seed=seed),
                    "per_job": lambda: per_job(gen, packed, args.T, seed)}
            ref = {name: f() for name, f in arms.items()}  # warm-up of both arms
            assert same(ref["packed"], ref["per_job"]), "%s: packed and per-job outputs differ" % kind
            times = {name: [] for name in arms}
            for _ in range(args.reps):
                for name, f in arms.items():
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    res = f()  # ends in a stream synchronise (host outputs)
                    times[name].append(time.perf_counter() - t0)
                    assert same(res, ref["packed"]), "%s/%s: outputs changed between repetitions" % (kind, name)
            S = int(packed.ids.size)
            for name, ts in times.items():
                rec = {"workload": kind, "arm": name, "jobs": N_JOBS, "samples_per_job": PER_JOB, "molecules": S,
                       "T": args.T, "precision": args.precision, "ifm_diffusion_level": IFM_LEVEL if kind == "ifm" else None,
                       "seconds": ts, "mols_per_s_median": S / float(np.median(ts)), "outputs_bit_identical": True,
                       "card(name, power.limit, clocks.sm, clocks.max.sm)": info}
                line = json.dumps(rec)
                print(line, flush=True)
                fh.write(line + "\n")
    gen.engine.close()


if __name__ == "__main__":
    main()
