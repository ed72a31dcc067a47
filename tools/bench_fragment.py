"""Fragment-conditioned generation: the eager composition (MLConformerGenerator.edm_sample_tensors: set_batch + one
Engine.sample per loop, then the GCN entry points) against Engine.generate_fragment_host (mlcg_generate_fragment: one
call, replayed as a CUDA graph), on BASELINE.json configs[3] (C4: 4096 samples of 21-25 atoms around 8 fixed atoms, T=100,
resample_steps=1) reproduced from bench.py's workload("C4").

  python tools/bench_fragment.py --out profiles/fragment_bench.jsonl            # one GPU: C4 inpaint, C4 IFM, B=64
  torchrun --nproc-per-node W tools/bench_fragment.py --out ... --scaling       # weak scaling, 4096 samples per GPU

One JSON line per measurement, each with the card's name and power limit read in the same run.  Single GPU: the arms --
eager, new path with device outputs, new path end to end with pinned host buffers -- alternate in one process, each
repeated, and their outputs are checked identical (bit patterns)."""
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

from bench import T_STEPS, normed_ctx, workload  # noqa: E402
from ml_conformer_generator_b200.config import CONTEXT_NORMS  # noqa: E402
from ml_conformer_generator_b200.engine import Engine  # noqa: E402
from ml_conformer_generator_b200.weights import random_state_dicts  # noqa: E402

IFM_LEVEL = 50


def card(index):
    q = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    return {"gpu": q or torch.cuda.get_device_name(index)}


def c4():
    wl = workload("C4")
    zk = wl["z_known"]
    n_ff = int(wl["fixed_mask"][0].sum())
    return wl, torch.from_numpy(zk[0, :n_ff, :3].copy()), torch.from_numpy(zk[0, :n_ff, 3:].copy())


def eager(e, ifm, nn, N, ctx_dev, ffx, ffh, ref, seed, ids):
    """edm_sample_tensors' launch sequence for one batch + seer_inputs + seer_forward (device outputs)."""
    n_ff = ffx.shape[0]
    if ifm:
        f_ctx, shift, rot, _ = e.ifm_context(ffx, ref, CONTEXT_NORMS, torch.from_numpy(nn))
        e.set_batch(nn - n_ff, N - n_ff)
        xg, cg = e.sample(f_ctx, T_STEPS, "forward", 1, seed=seed, sample_ids=ids)
        zk, fm = e.ifm_merge_inputs(xg, cg, shift, rot, ffx, ffh, N)
        e.set_batch(nn, N)
        x, cls = e.sample(ctx_dev, T_STEPS, "merge", 1, z_known=zk, fixed_mask=fm, diffusion_level=IFM_LEVEL, seed=seed,
                          sample_ids=ids)
    else:
        zk = torch.zeros(len(nn), N, 11)
        zk[:, :n_ff, :3], zk[:, :n_ff, 3:] = ffx, ffh
        fm = torch.zeros(len(nn), N)
        fm[:, :n_ff] = 1.0
        e.set_batch(nn, N)
        x, cls = e.sample(ctx_dev, T_STEPS, "inpaint", 1, z_known=zk.to(e.device), fixed_mask=fm.to(e.device), seed=seed,
                          sample_ids=ids)
    el, dist, adj = e.seer_inputs(x, cls)
    _, bonds = e.seer_forward(el, dist, adj, want_logits=False)
    return x, cls, bonds


def fast(e, ifm, nn, N, ctx, ffx, ffh, ref, seed, ids, out=None, device_out=True):
    return e.generate_fragment_host(nn, N, ctx, ffx, ffh, ifm, ref, None, T_STEPS, 1, 3, IFM_LEVEL, seed=seed,
                                    sample_ids=ids, out=out, device_out=device_out)


def same(a, b):
    return all(torch.equal(u.cpu().view(torch.int32) if u.dtype == torch.float32 else u.cpu(),
                           v.cpu().view(torch.int32) if v.dtype == torch.float32 else v.cpu()) for u, v in zip(a, b))


def timed(fn, dev):
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    r = fn()
    torch.cuda.synchronize(dev)
    return time.perf_counter() - t0, r


def single_gpu(args, emit):
    dev = torch.device("cuda", 0)
    e = Engine(dev, args.precision)
    sd, ssd = random_state_dicts(0)
    e.load_edm_state_dict(sd)
    e.load_seer_state_dict(ssd)
    wl, ffx, ffh = c4()
    ref = torch.tensor(wl["ctx"], dtype=torch.float32)
    gn_all = wl["global_n_nodes"]
    for label, B, ifm in (("C4 inpaint", 4096, False), ("C4 IFM", 4096, True), ("B=64 inpaint", 64, False),
                          ("B=64 IFM", 64, True)):
        nn, N = gn_all[:B], wl["N"]
        ids = np.arange(B)
        ctx = normed_ctx(wl["ctx"], B)
        ctx_dev = torch.from_numpy(ctx).to(dev)
        host = [torch.empty(B, N, 3).pin_memory(), torch.empty(B, N, dtype=torch.int32).pin_memory(),
                torch.empty(B, 42, 42, dtype=torch.int8).pin_memory()]
        arms = {
            "eager": lambda s: eager(e, ifm, nn, N, ctx_dev, ffx, ffh, ref, s, ids),
            "graph_device_out": lambda s: fast(e, ifm, nn, N, ctx, ffx, ffh, ref, s, ids),
            "graph_host_e2e": lambda s: fast(e, ifm, nn, N, ctx, ffx, ffh, ref, s, ids, out=host, device_out=False),
        }
        outs = {k: [t.cpu().clone() for t in f(7)] for k, f in arms.items()}  # same seed: outputs must agree
        identical = same(outs["eager"], outs["graph_device_out"]) and same(outs["eager"], outs["graph_host_e2e"])
        finite = bool(torch.isfinite(outs["eager"][0]).all())
        times = {k: [] for k in arms}
        for rep in range(args.repeats):
            for k, f in arms.items():
                for w in range(2):  # the eager arm's set_batch drops the graph: eager call, then capture, before timing
                    f(100 + w)
                launches0 = e.kernel_launches()
                dt, _ = timed(lambda: f(200 + rep), dev)
                times[k].append(dt)
                launches = e.kernel_launches() - launches0
        rec = dict(card(0), config=label, B=B, N=N, n_ff=int(ffx.shape[0]), T=T_STEPS, resample_steps=1,
                   ifm_diffusion_level=IFM_LEVEL if ifm else None, precision=args.precision, outputs_identical=identical,
                   outputs_finite=finite, launches_per_call=launches,
                   seconds={k: [round(v, 4) for v in t] for k, t in times.items()},
                   mols_per_s={k: round(B / min(t), 1) for k, t in times.items()})
        emit(rec)


def scaling(args, emit):
    import torch.distributed as dist
    from ml_conformer_generator_b200 import parallel as P
    world, rank, local = int(os.environ["WORLD_SIZE"]), int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    e = Engine(dev, args.precision)
    sd, ssd = random_state_dicts(0)
    e.load_edm_state_dict(sd)
    e.load_seer_state_dict(ssd)
    wl, ffx, ffh = c4()
    gn = np.random.RandomState(1234).randint(21, 26, 4096 * world).astype(np.int32)  # 4096 samples per GPU
    ctx = normed_ctx(wl["ctx"], len(gn))
    ref = torch.tensor(wl["ctx"], dtype=torch.float32)

    def job(seed, ifm):
        return P.generate_sharded_engine(e, gn, wl["N"], ctx, T_STEPS, 1, seed=seed, fixed_fragment=(ffx, ffh),
                                         inertial_fragment_matching=ifm, reference_context=ref,
                                         ifm_diffusion_level=IFM_LEVEL)

    for ifm in (False, True):
        for s in range(2):
            job(s, ifm)
        best = float("inf")
        for rep in range(args.repeats):
            if world > 1:
                dist.barrier()
            dt, _ = timed(lambda: job(10 + rep, ifm), dev)
            best = min(best, dt)
        if rank == 0:
            emit(dict(card(local), config="C4 %s weak scaling" % ("IFM" if ifm else "inpaint"), gpus=world,
                      samples=len(gn), precision=args.precision, seconds=round(best, 4),
                      mols_per_s=round(len(gn) / best, 1)))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="JSON lines are appended here")
    ap.add_argument("--precision", default="fp16", choices=["fp16", "bf16", "tf32"])
    ap.add_argument("--repeats", type=int, default=2)
    ap.add_argument("--scaling", action="store_true", help="weak scaling through parallel.generate_sharded_engine")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_fragment.py needs a B200")

    def emit(rec):
        line = json.dumps(rec)
        print(line, flush=True)
        with open(args.out, "a") as fh:
            fh.write(line + "\n")

    (scaling if args.scaling else single_gpu)(args, emit)


if __name__ == "__main__":
    main()
