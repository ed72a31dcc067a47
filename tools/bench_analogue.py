"""Analogue jobs on one GPU: 8192 samples from 64 parent molecules of 15-39 atoms (128 analogues each), fp16, T = 100.

  (a) For each diffusion level L in --levels: MLConformerGenerator.generate_jobs on the 64 analogue jobs (one packed call)
      against plain generation of the same atom counts and contexts (64 plain jobs with n_nodes = the parent's atom count,
      one packed call).  The analogue loop runs (L + 1) * r + 1 denoiser forwards per molecule (r = max(resample_steps,
      1) = 1), plain generation T + 1; both rates are reported, in molecules/s and in forwards/s.
  (b) At L = --per-job-level: the packed call against one generate_jobs call per job (the loop a user writes without
      packing).  The outputs of the two are asserted equal bit for bit.

  python tools/bench_analogue.py --out profiles/analogue_bench.jsonl [--reps 3] [--levels 10 25 50 100]

Each packed arm is warmed up with two calls (the first runs eagerly, the second captures the CUDA graph), then timed over
`--reps` replays; every timed call ends in a device synchronise.  One JSON line per arm with the card's name and power
limit read in the same run."""
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
from ml_conformer_generator_b200.mol_utils import get_context_shape  # noqa: E402
from ml_conformer_generator_b200.weights import random_state_dicts  # noqa: E402

N_JOBS, PER_JOB, T = 64, 128, 100


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    return q or torch.cuda.get_device_name(0)


def parent(rng, n):
    """A compact random heavy-atom skeleton (1.5 A random walk), classes among C N O F P S Cl."""
    steps = rng.normal(size=(n, 3))
    steps *= 1.5 / np.linalg.norm(steps, axis=1, keepdims=True)
    x = torch.from_numpy((np.cumsum(steps, axis=0) * 0.6 + rng.normal(scale=3.0, size=3)).astype(np.float32))
    return x, torch.eye(8)[torch.from_numpy(rng.integers(0, 7, n))]


def make_jobs():
    rng = np.random.default_rng(11)
    parents = [parent(rng, int(n)) for n in rng.integers(15, 40, N_JOBS)]
    analogue = [dict(parent_molecule=p, n_samples=PER_JOB) for p in parents]
    plain = [dict(reference_context=get_context_shape(p[0] - p[0].mean(0))[0], n_nodes=[p[0].shape[0]] * PER_JOB)
             for p in parents]
    return analogue, plain


def bits(t):
    t = torch.as_tensor(t).detach().cpu()
    return t.view(torch.int32) if t.dtype == torch.float32 else t


def timed(f):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = f()
    torch.cuda.synchronize()
    return out, time.perf_counter() - t0


def run_arm(f, reps, warm=2):
    for _ in range(warm):
        out = f()
    return out, [timed(f)[1] for _ in range(reps)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--levels", type=int, nargs="+", default=[10, 25, 50, 100])
    ap.add_argument("--per-job-level", type=int, default=50)
    ap.add_argument("--precision", default="fp16")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_analogue.py measures the GPU; no CUDA device is visible")
    sd, ssd = random_state_dicts(0)
    gen = MLConformerGenerator(diffusion_steps=T, device=torch.device("cuda:0"), precision=args.precision,
                               edm_state_dict=sd, adj_mat_seer_state_dict=ssd)
    info = card()
    analogue, plain = make_jobs()
    S = N_JOBS * PER_JOB
    base = dict(jobs=N_JOBS, samples=S, atoms="15-39", T=T, resample_steps=1, precision=args.precision)
    recs = []
    _, ts = run_arm(lambda: gen.generate_jobs(plain, seed=3), args.reps)
    med_plain = float(np.median(ts))
    recs.append(dict(base, arm="plain generation, same atom counts", seconds=ts, seconds_median=med_plain,
                     mols_per_s=S / med_plain, forwards_per_molecule=T + 1, forwards_per_s=S * (T + 1) / med_plain))
    for L in args.levels:
        _, ts = run_arm(lambda: gen.generate_jobs(analogue, resample_steps=1, ifm_diffusion_level=L, seed=3), args.reps)
        med = float(np.median(ts))
        fw = (L + 1) * 1 + 1
        recs.append(dict(base, arm="analogue packed", diffusion_level=L, seconds=ts, seconds_median=med, mols_per_s=S / med,
                         forwards_per_molecule=fw, forwards_per_s=S * fw / med, speedup_vs_plain=med_plain / med,
                         cost_model_speedup=(T + 1) / fw))
    L = args.per_job_level
    packed, ts_p = run_arm(lambda: gen.generate_jobs(analogue, resample_steps=1, ifm_diffusion_level=L, seed=3), args.reps)
    per_job = lambda: [gen.generate_jobs([j], resample_steps=1, ifm_diffusion_level=L, seed=3)[0]  # noqa: E731
                       for j in [dict(a, job_id=k) for k, a in enumerate(analogue)]]
    each, ts_j = run_arm(per_job, args.reps, warm=1)
    for a, b in zip(packed, each):
        for k in a:
            assert torch.equal(bits(a[k]), bits(b[k])), "per-job arm differs from the packed call (%s)" % k
    for arm, ts in (("analogue packed (one call)", ts_p), ("analogue, one generate_jobs call per job", ts_j)):
        med = float(np.median(ts))
        recs.append(dict(base, arm=arm, diffusion_level=L, seconds=ts, seconds_median=med, mols_per_s=S / med,
                         outputs_bit_identical=True))
    recs[-1]["packed_speedup"] = float(np.median(ts_j)) / float(np.median(ts_p))
    with open(args.out, "a") as fh:
        for rec in recs:
            rec["card(name, power.limit, clocks.sm, clocks.max.sm)"] = info
            line = json.dumps(rec)
            print(line, flush=True)
            fh.write(line + "\n")
    gen.engine.close()


if __name__ == "__main__":
    main()
