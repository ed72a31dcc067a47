#!/usr/bin/env python
"""Headline benchmark: generated molecules / second through the hot path (T=100 reverse steps = 101 EGNN forwards,
then GCN-input build + AdjMatSeer + bond argmax), one process per GPU.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--precision fp16|bf16|tf32] [--workload C3|C2|C1|C4|C5]
                  [--dump-outputs DIR]
  python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...      (N > 1)
  python bench.py --impl reference ...        (the reference's own torch CPU path on the host cores)

A "step" is one pass of the hot path over one batch of synthetic molecules (random-init weights of the named
architecture; the HuggingFace checkpoints are not available offline).  Default workload: BASELINE.json configs[2]
(8192 molecules of 15-39 atoms + AdjMatSeer) per GPU, weak scaling -- at 8 GPUs that is configs[4]'s 65 536 samples,
sharded by the product path (parallel.generate_sharded_engine: size-balanced shards keyed by global sample ids, one
packed NCCL all-gather).  `value` is timed with inputs resident in HBM; `e2e` goes through the host-buffer API (pinned
host -> device -> pinned host inside the timed region).  Inputs, weights and noise seeds depend only on the arguments, so
`--dump-outputs DIR` lets two builds of the project be compared output for output."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ONNX_CONTEXT = [53.6424, 108.3042, 151.4399]  # raw context of configs C2-C5 (SURVEY.md 8d)
CEYYAG_CONTEXT = [50.5897, 105.3132, 133.5223]
T_STEPS = 100
MAC_PER_EDGE = 420 * 420 + 420 + 2 * 420  # second edge layer + gate/coord head + rank-2 distance terms (SURVEY 8d)
MAC_PER_NODE = 19_061_280                 # per node per forward (SURVEY 8d)
METRIC = "generated mols/sec (100 EGNN steps + GCN, <=39 atoms)"


def workload(name, world=1, rank=0):
    """Per-GPU batch of the named BASELINE.json config.  `global_n_nodes` lists the atom counts of ALL samples of the job
    (world * per-GPU batch for the weak-scaling workloads), from which every rank derives its shard."""
    if name == "C3":
        B = 8192
        sizes = np.random.RandomState(5).randint(15, 40, 65536).astype(np.int32)[: world * B]
        return dict(B=B, N=39, global_n_nodes=sizes, ctx=ONNX_CONTEXT,
                    desc="C3 per GPU (configs[2]): %d samples of 15-39 atoms on %d GPU(s)%s, T=100 (101 EGNN forwards) + "
                         "AdjMatSeer GCN + bond argmax" % (world * B, world, " = configs[4]'s 65 536-sample sweep" if world == 8 else ""))
    if name == "C5":
        sizes = np.random.RandomState(5).randint(15, 40, 65536).astype(np.int32)
        return dict(B=65536 // world, N=39, global_n_nodes=sizes, ctx=ONNX_CONTEXT, strong=True,
                    desc="C5 (configs[4]): 65536 samples of 15-39 atoms in total over %d GPU(s) (strong scaling), T=100 + "
                         "AdjMatSeer GCN" % world)
    if name == "C2":
        return dict(B=1024, N=39, global_n_nodes=np.full(1024 * world, 39, np.int32), ctx=ONNX_CONTEXT,
                    desc="C2 per GPU (configs[1]): %d samples x 39 atoms, T=100 (101 EGNN forwards) + AdjMatSeer GCN" % (1024 * world))
    rng = np.random.RandomState(1234)
    if name == "C4":
        # SURVEY 8d C4: simple inpainting around the 8 heavy atoms of frag_yibfeu (Cl, Cl, C x 6), resample_steps = 1
        # => 201 EGNN forwards per sample.  Fragment coordinates are synthetic (seeded), one-hot raw 0/1.
        B, N = 4096, 25
        frag = rng.randn(8, 3).astype(np.float32) * 1.5
        zk = np.zeros((B, N, 11), np.float32)
        zk[:, :8, :3] = frag
        for k, c in enumerate([6, 6, 0, 0, 0, 0, 0, 0]):
            zk[:, k, 3 + c] = 1.0
        fm = np.zeros((B, N), np.float32)
        fm[:, :8] = 1.0
        return dict(B=B, N=N, global_n_nodes=rng.randint(21, 26, B).astype(np.int32), ctx=[89.8693, 210.7831, 217.7827],
                    mode="inpaint", resample=1, z_known=zk, fixed_mask=fm, n_forwards=201,
                    desc="C4 (configs[3]): inpaint, B=4096 samples, 21-25 atoms, 8 fixed fragment atoms, T=100, resample 1 "
                         "(201 EGNN forwards) + AdjMatSeer GCN")
    if name == "C1":
        return dict(B=20, N=19, global_n_nodes=rng.randint(15, 20, 20).astype(np.int32), ctx=CEYYAG_CONTEXT,
                    desc="C1 (configs[0]): B=20 samples, 15-19 atoms (ceyyag), T=100 + AdjMatSeer GCN")
    raise SystemExit("unknown workload " + name)


DUMP_BYTES = 64 * 10 ** 6


def dump_outputs(path, x, cls, bonds):
    """Writes what a caller of the timed path receives -- coordinates x (B,N,3), atom classes (B,N) (-1 = padding) and bond
    orders (B,42,42) -- as float32 .npy files, with the global sample id of each row (float64).  When all molecules
    exceed DUMP_BYTES, a fixed seeded sample of them is written, so that two builds can be compared file for file."""
    n = x.shape[0]
    per_mol = 4 * (x[0].numel() + cls[0].numel() + bonds[0].numel()) + 8
    keep = min(n, DUMP_BYTES // per_mol)
    ids = np.arange(n) if keep == n else np.sort(np.random.RandomState(0).choice(n, keep, replace=False))
    rows = torch.from_numpy(ids).to(x.device)
    os.makedirs(path, exist_ok=True)
    for name, t in (("x", x), ("atom_class", cls), ("bond_orders", bonds)):
        np.save(os.path.join(path, name + ".npy"), t.index_select(0, rows).float().cpu().numpy())
    np.save(os.path.join(path, "sample_id.npy"), ids.astype(np.float64))


def alg_flops_forward(n_nodes):
    n = np.asarray(n_nodes).astype(np.float64)
    return float((2 * 27 * MAC_PER_EDGE * n * (n - 1) + 2 * MAC_PER_NODE * n).sum())


def normed_ctx(raw, B):
    from ml_conformer_generator_b200.config import CONTEXT_NORMS
    c = (np.asarray(raw, np.float32) - np.asarray(CONTEXT_NORMS["mean"], np.float32)) / np.asarray(
        CONTEXT_NORMS["mad"], np.float32)
    return np.tile(c.reshape(1, 3), (B, 1)).astype(np.float32)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(burst=d["bf16_tflops"], sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    hbm=d["hbm_gbs"], source="measured")
    return dict(burst=1590.0, sustained=1400.0, hbm=6650.0, source="fallback")


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "200"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(", ") for r in open(self.f.name).read().strip().splitlines() if r.strip()]
        os.unlink(self.f.name)
        clk, mx, reasons = [], None, set()
        for r in rows:
            try:
                c, m = float(r[1]), float(r[2])
            except (ValueError, IndexError):
                continue
            mx = m
            clk.append(c)
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.strip().lower().startswith("active"):
                    reasons.add(name)
        load = [c for c in clk if mx and c > 0.5 * mx] or clk
        return {"sm_mhz": statistics.median(load) if load else None, "sm_max_mhz": mx, "samples": len(clk),
                "reasons": sorted(reasons)}


# ----------------------------------------------------------------------------------------------------------------
# reference arm: the reference's own torch implementation of the path, timed on the host cores (or, --ref-device cuda,
# its eager-torch path on the GPU as an extra labelled line)
# ----------------------------------------------------------------------------------------------------------------
def reference_modules(device):
    """The UNMODIFIED reference modules (oracle/_ref staged copy, or /root/reference in the build container) with the
    random-init weights of this bench, or None when the staged copy is missing (then the oracle port is timed)."""
    from oracle.reference_loader import load_reference, reference_available
    if not reference_available():
        return None
    load_reference()
    from mlconfgen.adj_mat_seer import AdjMatSeer
    from mlconfgen.egnn import EGNNDynamics
    from mlconfgen.equivariant_diffusion import EquivariantDiffusion, PredefinedNoiseSchedule
    from ml_conformer_generator_b200.weights import random_state_dicts
    sd, ssd = random_state_dicts(0)
    dyn = EGNNDynamics(in_node_nf=9, context_node_nf=3, hidden_nf=420, device=torch.device(device))  # conformer_generator.py:67-72
    edm = EquivariantDiffusion(dynamics=dyn, in_node_nf=8, timesteps=1000, noise_precision=1e-5)
    edm.load_state_dict(sd, strict=True)
    seer = AdjMatSeer(dimension=42, n_hidden=2048, embedding_dim=64, num_embeddings=36, num_bond_types=5,
                      device=torch.device(device))  # conformer_generator.py:81-88
    seer.load_state_dict(ssd, strict=True)
    edm.gamma = PredefinedNoiseSchedule(timesteps=T_STEPS, precision=1e-5)  # conformer_generator.py:104-113
    edm.time_steps = torch.flip(torch.arange(0, T_STEPS), dims=[0])
    edm.T = T_STEPS
    return edm.eval().to(device), seer.eval().to(device)


class ReferenceRunner:
    """Times reverse steps of the reference on a bounded sample of the workload and extrapolates to a whole molecule:
    n_forwards denoiser calls (the reference's cost per call does not depend on t) + one AdjMatSeer pass."""

    def __init__(self, wl, n_mols, threads, device="cpu"):
        from ml_conformer_generator_b200.config import CONTEXT_NORMS
        from oracle import edm_oracle as O
        torch.set_num_threads(threads)
        self.O, self.wl, self.n_mols, self.device = O, wl, n_mols, torch.device(device)
        self.mods = reference_modules(self.device)
        self.kind = "reference" if self.mods is not None else "port"
        n_nodes = torch.from_numpy(np.asarray(wl["global_n_nodes"][:n_mols]).astype(np.int64))
        self.n_nodes, self.N = n_nodes, wl["N"]
        self.nm, self.em = O.prepare_masks(n_nodes, self.N)
        self.ctx = O.batch_context(O.normalise_context(torch.tensor(wl["ctx"]), CONTEXT_NORMS), self.nm)
        if self.mods is None:
            from ml_conformer_generator_b200.weights import random_state_dicts
            self.sd, self.ssd = random_state_dicts(0)
            self.gamma = O.gamma_table(T_STEPS)
        g = torch.Generator().manual_seed(99)
        self.z0 = torch.randn(n_mols, self.N, 11, generator=g) * self.nm
        el, dist, adj = O.seer_inputs_from_samples(self.z0[:, :, :3] * 2, torch.argmax(self.z0[:, :, 3:10], dim=2), n_nodes)
        self.seer_in = (el, dist, adj)

    def _sync(self):
        if self.device.type == "cuda":
            torch.cuda.synchronize()

    @torch.no_grad()
    def step(self, s):
        """One reverse step p(z_s | z_t) on the sample; returns seconds."""
        dev, B = self.device, self.n_mols
        if self.mods is not None:
            edm = self.mods[0]
            s_arr = torch.full((B, 1), s, device=dev) / T_STEPS
            t_arr = torch.full((B, 1), s + 1, device=dev) / T_STEPS
            z, nm, em, ctx = self.z0.to(dev), self.nm.to(dev), self.em.to(dev), self.ctx.to(dev)
            self._sync()
            t0 = time.perf_counter()
            edm.sample_p_zs_given_zt(s_arr, t_arr, z, nm, em, ctx)
            self._sync()
            return time.perf_counter() - t0
        O = self.O
        s_arr, t_arr = O._times(s, T_STEPS, B)
        tape = O.NoiseTape.draw(1, B, self.N, 1)
        t0 = time.perf_counter()
        O.sample_p_zs_given_zt(self.sd, self.gamma, s_arr, t_arr, self.z0, self.nm, self.em, self.ctx, tape)
        return time.perf_counter() - t0

    @torch.no_grad()
    def seer(self):
        el, dist, adj = (t.to(self.device) for t in self.seer_in)
        self._sync()
        t0 = time.perf_counter()
        if self.mods is not None:
            logits = self.mods[1](el, dist, adj)
            torch.argmax(logits, dim=3)
        else:
            self.O.bond_orders(self.O.seer_forward(self.ssd, el, dist, adj))
        self._sync()
        return time.perf_counter() - t0

    def rate(self, step_s, seer_s):
        return self.n_mols / (step_s * self.wl.get("n_forwards", T_STEPS + 1) + seer_s)

    @torch.no_grad()
    def full_loop(self):
        """The reference's whole sampler (EquivariantDiffusion.forward: 100 reverse steps + decode, 101 denoiser calls) on
        the sample, no extrapolation; returns seconds.  Needs the reference modules."""
        edm = self.mods[0]
        dev = self.device
        nm, em, ctx = self.nm.to(dev), self.em.to(dev), self.ctx.to(dev)
        torch.manual_seed(1)
        self._sync()
        t0 = time.perf_counter()
        edm(nm, em, ctx, 0)
        self._sync()
        return time.perf_counter() - t0


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = workload(args.workload)
    threads = os.cpu_count() or 1
    on_gpu = args.ref_device == "cuda"
    n_mols = args.ref_mols or (256 if on_gpu else 32)
    run = ReferenceRunner(wl, n_mols, threads, args.ref_device)
    for i in range(args.warmup):
        run.step(T_STEPS - 1 - (i % T_STEPS))
    seer_s = min(run.seer(), run.seer())
    t0 = time.perf_counter()
    if args.ref_full and run.mods is not None:
        # whole reverse loop, no extrapolation (configs[0]: the reference's own CPU-runnable case)
        loops = [run.full_loop() for _ in range(max(args.steps, 1))]
        ms = (time.perf_counter() - t0) / max(args.steps, 1) * 1e3
        step_s = statistics.median(loops) / wl.get("n_forwards", T_STEPS + 1)
        value = n_mols / (statistics.median(loops) + seer_s)
    else:
        steps = [run.step(T_STEPS - 1 - (i % T_STEPS)) for i in range(args.steps)]
        ms = (time.perf_counter() - t0) / max(args.steps, 1) * 1e3
        step_s = statistics.median(steps)
        value = run.rate(step_s, seer_s)
    where = ("eager torch on the GPU (extra line, not the CPU baseline)" if on_gpu else "torch CPU, %d threads" % threads)
    from oracle.reference_loader import reference_path
    who = ("the reference's own modules, unmodified (%s)" % os.path.relpath(reference_path(), ROOT) if run.kind == "reference"
           else "oracle port of the reference CPU path (staged reference copy missing)")
    if args.ref_full and run.mods is not None:
        sample = ("%s (%s): each bench step = the reference's WHOLE sampler EquivariantDiffusion.forward (100 reverse steps + "
                  "decode) on the first %d molecules of the workload, padded to %d atoms; %.3f s per denoiser call; "
                  "mols/s = %d / (whole loop [%d forwards] + AdjMatSeer %.3f s), no extrapolation"
                  % (who, where, n_mols, wl["N"], step_s, n_mols, wl.get("n_forwards", T_STEPS + 1), seer_s))
    else:
        sample = ("%s (%s): each bench step = one reverse step p(z_s|z_t) (one EGNNDynamics forward + the posterior update) on "
                  "the first %d molecules of the workload, padded to %d atoms as the reference does; median %.3f s / step; "
                  "mols/s = %d / (%d forwards x step + AdjMatSeer %.3f s)"
                  % (who, where, n_mols, wl["N"], step_s, n_mols, wl.get("n_forwards", T_STEPS + 1), seer_s))
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value,
        "unit": "mols/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": wl["desc"], "precision": "fp32 (%s)" % where},
        "cpu_baseline": {"value": value, "unit": "mols/s", "cores": threads if not on_gpu else 0, "kind": run.kind,
                         "sample": sample},
        "e2e": {"value": value, "unit": "mols/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


# ----------------------------------------------------------------------------------------------------------------
# B200 arm
# ----------------------------------------------------------------------------------------------------------------
def parity_block(eng, precision):
    """Live parity of the bench precision against the committed golden run of the reference at config 2's molecule size
    (tests/golden/edm_forward_T100_n39.npz: 8 x 39 atoms, T = 100): teacher-forced eps over all 101 denoiser calls and
    the free-running argmax agreement.  Fixtures only -- no oracle, no reference."""
    from tools import parity_check as PC
    try:
        g = PC.load_golden("edm_forward_T100_n39")
    except OSError:
        return None
    errs = PC.teacher_forced(eng, g)
    xerr, agree, atoms = PC.free_running(eng, g)
    return {"golden": "edm_forward_T100_n39 (reference run: 8 x 39 atoms, T=100, 101 denoiser calls)",
            "teacher_forced_eps_rel_l2_max": max(errs), "teacher_forced_eps_rel_l2_median": float(np.median(errs)),
            "tolerance": PC.TOL[precision], "free_running_atom_type_agreement": agree, "free_running_atoms": atoms,
            "free_running_x_rel_l2": xerr,
            "note": "10k-atom argmax agreement and strict-lower-triangle bond agreement: profiles/r2_parity.txt (pytest -m gpu)"}


def kernel_breakdown(eng, wl_n_nodes, N, ctx_dev, pk, n_forwards):
    """Live per-kernel-class timing of one EGNN forward (CUDA event after every launch), the step kernel and the GCN."""
    import ctypes as C
    from ml_conformer_generator_b200 import _lib
    dev = eng.device
    B = len(wl_n_nodes)
    g = torch.Generator().manual_seed(1)
    mask = (torch.arange(N).view(1, N) < torch.as_tensor(wl_n_nodes).view(B, 1)).float().unsqueeze(-1)
    z = (torch.randn(B, N, 11, generator=g) * mask).to(dev)
    t = torch.full((B,), 0.5, device=dev)
    eng.egnn_forward_breakdown(t, z, ctx_dev)  # warm
    bd = eng.egnn_forward_breakdown(t, z, ctx_dev)
    M = int(np.asarray(wl_n_nodes).sum())
    out = {"egnn_forward_ms": bd["total_ms"], "classes": {k: v for k, v in bd.items() if k != "total_ms"}}
    for k, v in out["classes"].items():
        v["share"] = v["ms"] / bd["total_ms"] if bd["total_ms"] > 0 else None
    # HBM traffic of the node GEMMs per launch (algorithmic: operands in + results out; weights are L2-resident)
    if bd["node_mlp2"]["launches"]:
        nb = {"pq_projection": M * (448 * 2 + 896 * 2), "node_mlp1": M * (896 * 2 + 448 * 2),
              "node_mlp2": M * (448 * 2 + 448 * 4 * 2 + 448 * 2)}
        for k, b in nb.items():
            c = out["classes"][k]
            if c["launches"]:
                gbs = b / (c["ms"] / c["launches"] * 1e-3) / 1e9
                c["alg_gb_per_s"], c["frac_of_hbm_peak"] = gbs, gbs / pk["hbm"]
    # diffusion-step kernel: reads z, eps, writes z (3 x B*N*11 fp32)
    eps = torch.randn(B, N, 11, device=dev)
    sc = _lib.StepScalars(0.5, 0.99, 0.01, 0.01, 1.0, 0.0, 0.0)
    nz = _lib.Noise(None, 1, 1, 0, None)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for it in range(2):
        e0.record()
        for _ in range(50):
            eng.lib.mlcg_step(eng.h, z.data_ptr(), eps.data_ptr(), C.byref(sc), C.byref(nz), eng._stream())
        e1.record()
        torch.cuda.synchronize(dev)
    step_us = e0.elapsed_time(e1) / 50 * 1e3
    sb = 3.0 * M * 11 * 4
    out["k_step"] = {"us": step_us, "alg_gb_per_s": sb / (step_us * 1e-6) / 1e9, "frac_of_hbm_peak": sb / (step_us * 1e-6) / 1e9 / pk["hbm"],
                     "note": "one warp per molecule; Philox noise generated in the kernel"}
    # GCN (inputs + AdjMatSeer + argmax)
    x = z[:, :, :3].contiguous()
    cls = torch.zeros(B, N, dtype=torch.int32, device=dev)
    for it in range(2):
        e0.record()
        el, dmat, adj = eng.seer_inputs(x, cls)
        eng.seer_forward(el, dmat, adj, want_logits=False)
        e1.record()
        torch.cuda.synchronize(dev)
    gcn_ms = e0.elapsed_time(e1)
    out["gcn_ms"] = gcn_ms
    out["gcn_tflops"] = 1.871e9 * B / (gcn_ms * 1e-3) / 1e12
    out["gcn_share_of_step"] = gcn_ms / (gcn_ms + n_forwards * bd["total_ms"])
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--precision", default="fp16", choices=["fp16", "bf16", "tf32"])
    ap.add_argument("--workload", default="C3", choices=["C1", "C2", "C3", "C4", "C5"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip parity / breakdown / secondary workload")
    ap.add_argument("--ref-device", default="cpu", choices=["cpu", "cuda"])
    ap.add_argument("--ref-mols", type=int, default=0)
    ap.add_argument("--ref-full", action="store_true", help="reference arm: time the whole 100-step loop, no extrapolation")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the results of the last timed step to DIR/<name>.npy (float32, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the results of the b200 arm")
    if args.impl == "reference":
        run_reference(args)
        return

    import torch.distributed as dist
    from ml_conformer_generator_b200 import parallel as P
    from ml_conformer_generator_b200.engine import Engine
    from ml_conformer_generator_b200.weights import random_state_dicts

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: the CUDA extension has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    wl = workload(args.workload, world=world, rank=rank)
    N = wl["N"]
    gn = wl["global_n_nodes"]
    n_job = len(gn)
    shards = P.shard_indices(gn, world)
    mine = shards[rank]
    my_nodes = gn[mine]
    eng = Engine(dev, args.precision)
    sd, ssd = random_state_dicts(0)
    eng.load_edm_state_dict(sd)
    eng.load_seer_state_dict(ssd)
    del sd, ssd
    ctx_all = normed_ctx(wl["ctx"], n_job)
    mode = wl.get("mode", "forward")
    n_forwards = wl.get("n_forwards", T_STEPS + 1)
    max_batch = 8192

    # ---- device-timed arm -------------------------------------------------------------------------------------
    if world == 1:
        # inputs resident in HBM; sub-batches of <= 8192 molecules (one for every workload but C5)
        subs = [np.arange(s, min(s + max_batch, n_job)) for s in range(0, n_job, max_batch)]
        ctx_dev = [torch.from_numpy(ctx_all[ids]).to(dev) for ids in subs]
        zk_dev = torch.from_numpy(wl["z_known"]).to(dev) if mode != "forward" else None
        fm_dev = torch.from_numpy(wl["fixed_mask"]).to(dev) if mode != "forward" else None

        def device_step(seed):
            outs = []
            for ids, cdev in zip(subs, ctx_dev):
                if len(subs) > 1 or eng.B != len(ids):
                    eng.set_batch(gn[ids], N)   # the batch plan (edge-tile table) is part of the job when it changes
                x, cls = eng.sample(cdev, T_STEPS, mode, wl.get("resample", 0), z_known=zk_dev, fixed_mask=fm_dev, seed=seed,
                                    sample_ids=ids)
                el, dmat, adj = eng.seer_inputs(x, cls)
                _, bonds = eng.seer_forward(el, dmat, adj, want_logits=False)
                outs.append((x, cls, bonds))
            return outs
        eng.set_batch(gn[subs[0]], N)
    else:
        if mode != "forward":
            raise SystemExit("the fragment workload is a single-GPU bench line")

        def device_step(seed):
            # the multi-GPU product path: size-balanced shards by global id, one launch sequence per rank (CUDA graph
            # replay), results stay on the device, ONE packed NCCL all-gather
            return [P.generate_sharded_engine(eng, gn, N, ctx_all, T_STEPS, 0, seed=seed, max_batch=max_batch)]

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for i in range(args.warmup):
        device_step(100 + i)
    sync()
    sampler = ClockSampler(local) if rank == 0 else None
    l0 = eng.kernel_launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        outs = device_step(200 + i)
    e1.record()
    sync()
    ms = e0.elapsed_time(e1) / args.steps
    launches = eng.kernel_launches() - l0
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        # sub-batches are consecutive ranges of the global ids; the multi-GPU path returns the gathered job in id order
        dump_outputs(args.dump_outputs, *(torch.cat(t) for t in zip(*outs)))
    del outs

    # ---- end to end: host buffers in, pinned host buffers out, copies inside the timed region -----------------------
    e2e_ms = float("nan")
    h2d = d2h = 0
    if mode == "forward":
        e2e_steps = max(1, min(args.steps, 2))
        if world == 1:
            outs = [eng.generate_host(gn[ids], N, ctx_all[ids], T_STEPS, 0, seed=300, sample_ids=ids) for ids in subs]
            sync()
            t0 = time.perf_counter()
            for i in range(e2e_steps):
                for ids, o in zip(subs, outs):
                    eng.generate_host(gn[ids], N, ctx_all[ids], T_STEPS, 0, seed=400 + i, sample_ids=ids, out=o)
            sync()
        else:
            host = [torch.empty(n_job, N, 3).pin_memory(), torch.empty(n_job, N, dtype=torch.int32).pin_memory(),
                    torch.empty(n_job, 42, 42, dtype=torch.int8).pin_memory()]
            P.generate_sharded_engine(eng, gn, N, ctx_all, T_STEPS, 0, seed=300, max_batch=max_batch)
            sync()
            t0 = time.perf_counter()
            for i in range(e2e_steps):
                res = P.generate_sharded_engine(eng, gn, N, ctx_all, T_STEPS, 0, seed=400 + i, max_batch=max_batch)
                if rank == 0:  # the job's result lands in pinned host memory on rank 0
                    for hbuf, r in zip(host, res):
                        hbuf.copy_(r, non_blocking=True)
            sync()
        e2e_ms = (time.perf_counter() - t0) / e2e_steps * 1e3
        h2d = int(n_job * (4 + 3 * 4 + 8))
        d2h = int(n_job * (N * 3 * 4 + N * 4 + 42 * 42))

    # ---- dominant kernel: fused edge kernel (GCL variant), timed live with CUDA events on the launching stream -----------
    eng.set_batch(my_nodes[:max_batch], N)
    edge_ms = eng.time_edge_kernel(layer=0, iters=20)
    n_edges = eng.num_edges()

    t = torch.tensor([ms, e2e_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, e2e_ms = float(t[0]), float(t[1])

    if rank == 0:
        pk = peaks()
        edge_flops = 2.0 * MAC_PER_EDGE * n_edges
        achieved = edge_flops / (edge_ms * 1e-3) / 1e12
        step_flops = alg_flops_forward(my_nodes) * n_forwards + 1.871e9 * len(my_nodes)
        prof = os.path.join(ROOT, "profiles", "edge_kernel_traffic.json")
        traffic = None
        if os.path.exists(prof):  # measured with ncu --set full for one (workload, precision); null for any other
            traffic = json.load(open(prof)).get("%s/%s" % (args.workload, args.precision))
        res = {
            "metric": METRIC,
            "value": n_job / (ms * 1e-3), "unit": "mols/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "strong" if wl.get("strong") else "weak",
            "vs_baseline": None, "dtype": args.precision, "data": "synthetic",
            "config": {"workload": wl["desc"], "per_gpu_batch": len(mine), "max_atoms": N, "diffusion_steps": T_STEPS,
                       "weights": "random-init (seed 0) of the reference architecture",
                       "noise": "device Philox4x32-10 keyed by (seed, global sample id, atom, draw)",
                       "l2": "per-step working set (P/Q projections %.0f MB + operands) exceeds the 126 MB L2; no flush"
                             % (float(my_nodes.sum()) * 896 * 2 / 1e6),
                       "parallelism": ("dp%d: size-balanced shards by global sample id (parallel.generate_sharded_engine), no "
                                       "collective inside the loop, one packed NCCL all-gather of the results" % world)},
            "e2e": ({"value": n_job / (e2e_ms * 1e-3), "unit": "mols/s", "h2d_bytes_per_step": h2d,
                     "d2h_bytes_per_step": d2h} if e2e_ms == e2e_ms else None),
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": {"bound": "tensor", "kernel": "k_tc_edge3 (GCL sub-layer, %s)" % args.precision,
                         "achieved": achieved, "peak": pk["burst"], "unit": "TFLOP/s", "frac": achieved / pk["burst"],
                         "traffic": traffic, "peak_source": pk["source"] + " bf16 dense burst",
                         "launch_ms": edge_ms, "alg_flops_per_launch": edge_flops,
                         "step_achieved": step_flops / (ms * 1e-3) / 1e12,
                         "step_frac_of_sustained": step_flops / (ms * 1e-3) / 1e12 / pk["sustained"]},
        }
        if world == 1 and not args.no_extras:
            try:
                res["breakdown"] = kernel_breakdown(eng, my_nodes[:max_batch], N, torch.from_numpy(ctx_all[:len(my_nodes[:max_batch])]).to(dev), pk, n_forwards)
            except Exception as ex:  # measurement extras must never lose the headline line
                res["breakdown"] = {"error": repr(ex)}
            try:
                res["parity"] = parity_block(eng, args.precision)
            except Exception as ex:
                res["parity"] = {"error": repr(ex)}
            if args.workload == "C3":
                # continuity with round 1's headline: config 2 (1024 x 39 atoms), 2 timed steps
                try:
                    w2 = workload("C2")
                    eng.set_batch(w2["global_n_nodes"], 39)
                    c2 = torch.from_numpy(normed_ctx(w2["ctx"], 1024)).to(dev)

                    def c2_step(seed):
                        x, cls = eng.sample(c2, T_STEPS, "forward", 0, seed=seed)
                        el, dmat, adj = eng.seer_inputs(x, cls)
                        eng.seer_forward(el, dmat, adj, want_logits=False)
                    c2_step(1)
                    torch.cuda.synchronize(dev)
                    e0.record()
                    c2_step(2)
                    c2_step(3)
                    e1.record()
                    torch.cuda.synchronize(dev)
                    c2_ms = e0.elapsed_time(e1) / 2
                    c2_edge = eng.time_edge_kernel(layer=0, iters=20)
                    c2_fl = 2.0 * MAC_PER_EDGE * eng.num_edges()
                    res["other_workloads"] = {"C2 (configs[1]): 1024 x 39 atoms, T=100 + GCN": {
                        "value": 1024 / (c2_ms * 1e-3), "unit": "mols/s", "ms_per_step": c2_ms,
                        "edge_kernel_launch_ms": c2_edge, "edge_kernel_frac_of_bf16_burst": c2_fl / (c2_edge * 1e-3) / 1e12 / pk["burst"]}}
                except Exception as ex:
                    res["other_workloads"] = {"error": repr(ex)}
        if not args.no_cpu_baseline and world == 1:
            try:
                run = ReferenceRunner(wl, 32 if N > 30 else 64, os.cpu_count() or 1)
                run.step(99)
                steps = [run.step(98), run.step(97)]
                seer_s = run.seer()
                v = run.rate(min(steps), seer_s)
                res["cpu_baseline"] = {
                    "value": v, "unit": "mols/s", "cores": os.cpu_count() or 1, "kind": run.kind,
                    "sample": "%s, torch fp32 on the host cores: 2 timed reverse steps (best taken) + AdjMatSeer on %d molecules "
                              "of this workload, %.2f s / step, extrapolated to %d forwards"
                              % ("the reference's own modules (oracle/_ref)" if run.kind == "reference" else "oracle port",
                                 run.n_mols, min(steps), n_forwards)}
            except Exception as ex:
                res["cpu_baseline"] = {"error": repr(ex)}
        print(json.dumps(res))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
