"""Thin Python host over the C ABI: owns one `mlcg_handle`, keeps torch tensors alive across asynchronous calls, and
converts the reference's tensor conventions (float masks, (B,N,3) context) into the library's (atom counts, (B,3))."""
import ctypes as C
import os
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib
from .schedule import all_step_scalars, decode_scalars, forward_level_scalars, gamma_table

PRECISIONS = {"fp32": 0, "tf32": 1, "bf16": 2, "fp16": 3}


class MlcgError(RuntimeError):
    pass


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


class Engine:
    """One handle on one CUDA device.  Not thread-safe."""

    def __init__(self, device: torch.device = torch.device("cuda:0"), precision: str = "fp16"):
        device = torch.device(device)
        if device.type != "cuda":
            raise MlcgError("ml_conformer_generator_b200 runs on sm_100 CUDA devices only (got %s); there is no CPU "
                            "fallback" % device)
        if not torch.cuda.is_available():
            raise MlcgError("no CUDA device visible; ml_conformer_generator_b200 has no CPU fallback")
        self.lib = _lib.load()
        self.device = torch.device("cuda", device.index or 0)
        self.precision = precision
        torch.cuda.set_device(self.device)
        torch.cuda.init()
        torch.zeros(1, device=self.device)  # make sure the primary context exists
        self.h = C.c_void_p()
        rc = self.lib.mlcg_create(C.byref(self.h), self.device.index, PRECISIONS[precision])
        if rc != 0:
            raise MlcgError("mlcg_create failed (%d): no sm_100 device / bad arguments" % rc)
        self._keep: List[torch.Tensor] = []
        self.B = self.N = 0
        self.n_nodes: Optional[torch.Tensor] = None

    def close(self):
        if getattr(self, "h", None) is not None and self.h:
            torch.cuda.synchronize(self.device)
            self.lib.mlcg_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------------------------------------------------
    def _check(self, rc: int, what: str):
        if rc != 0:
            msg = self.lib.mlcg_last_error(self.h).decode()
            if rc < 0 and rc != -2:
                raise ValueError("%s: %s" % (what, msg))  # the reference raises ValueError on bad arguments
            raise MlcgError("%s failed (%d): %s" % (what, rc, msg))

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _descs(self, sd: Dict[str, torch.Tensor], prefix_filter=None):
        keep, arr = [], []
        for k, v in sd.items():
            if prefix_filter and not k.startswith(prefix_filter):
                continue
            t = v.detach().to(self.device, torch.float32).contiguous()
            keep.append(t)
            rows = t.shape[0] if t.dim() >= 1 else 1
            arr.append(_lib.WeightDesc(k.encode(), t.data_ptr(), rows, max(t.numel() // max(rows, 1), 1)))
        return keep, (_lib.WeightDesc * len(arr))(*arr), len(arr)

    def load_edm_state_dict(self, sd: Dict[str, torch.Tensor]):
        keep, arr, n = self._descs(sd, "dynamics.")
        self._check(self.lib.mlcg_load_egnn(self.h, arr, n), "load_egnn")

    def load_seer_state_dict(self, sd: Dict[str, torch.Tensor]):
        keep, arr, n = self._descs(sd)
        self._check(self.lib.mlcg_load_seer(self.h, arr, n), "load_seer")

    def set_batch(self, n_nodes: Sequence[int], max_n_nodes: int):
        nn = np.ascontiguousarray(np.asarray(n_nodes, dtype=np.int32).reshape(-1))
        self._check(self.lib.mlcg_set_batch(self.h, nn.ctypes.data_as(C.c_void_p), int(nn.size), int(max_n_nodes)),
                    "set_batch")
        self.B, self.N = int(nn.size), int(max_n_nodes)
        self.n_nodes = torch.from_numpy(nn.copy())

    # ------------------------------------------------------------------------------------------------------------
    def egnn_forward(self, t: torch.Tensor, z: torch.Tensor, ctx: torch.Tensor) -> torch.Tensor:
        """t (B,), z (B,N,11), ctx (B,3) on the device -> eps (B,N,11)."""
        t = t.reshape(-1).to(self.device, torch.float32).contiguous()
        z = z.to(self.device, torch.float32).contiguous()
        ctx = ctx.to(self.device, torch.float32).contiguous()
        if z.shape != (self.B, self.N, 11) or t.numel() != self.B or ctx.shape != (self.B, 3):
            raise ValueError("egnn_forward: shapes do not match the batch set with set_batch")
        eps = torch.empty_like(z)
        self._check(self.lib.mlcg_egnn_forward(self.h, _ptr(t), _ptr(z), _ptr(ctx), _ptr(eps), self._stream()),
                    "egnn_forward")
        return eps

    BREAKDOWN_CLASSES = ["prepare", "pq_projection", "edge_gcl", "edge_equiv", "edge_fixup", "node_mlp1", "node_mlp2",
                         "readout"]

    def egnn_forward_breakdown(self, t: torch.Tensor, z: torch.Tensor, ctx: torch.Tensor) -> dict:
        """One EGNN forward with a CUDA event after every launch: {class: (ms, launches)} + 'total' (measurement hook)."""
        t = t.reshape(-1).to(self.device, torch.float32).contiguous()
        z = z.to(self.device, torch.float32).contiguous()
        ctx = ctx.to(self.device, torch.float32).contiguous()
        eps = torch.empty_like(z)
        out = (C.c_double * 17)()
        self._check(self.lib.mlcg_egnn_forward_breakdown(self.h, _ptr(t), _ptr(z), _ptr(ctx), _ptr(eps), out, self._stream()),
                    "egnn_forward_breakdown")
        res = {n: {"ms": float(out[i]), "launches": int(out[9 + i])} for i, n in enumerate(self.BREAKDOWN_CLASSES)}
        res["total_ms"] = float(out[8])
        return res

    def _steps(self, T: int, blend_power: int):
        gamma = gamma_table(T)
        sc = all_step_scalars(gamma)
        arr = (_lib.StepScalars * T)()
        for s, d in enumerate(sc):
            blend = float(torch.pow(1 - torch.full([1], s, dtype=torch.int64) / T, blend_power))
            arr[s] = _lib.StepScalars(d["t"], d["alpha_ts"], d["c_eps"], d["c_sigma"], d["alpha_s"], d["sigma_s"], blend)
        return gamma, arr

    def _steps_cached(self, T: int, blend_power: int):
        key = (T, blend_power)
        cache = self.__dict__.setdefault("_steps_cache", {})
        if key not in cache:
            cache[key] = self._steps(T, blend_power)
        return cache[key]

    def sample(self, ctx: torch.Tensor, T: int, mode: str = "forward", resample_steps: int = 0,
               z_known: Optional[torch.Tensor] = None, fixed_mask: Optional[torch.Tensor] = None,
               diffusion_level: int = 50, blend_power: int = 3, noise_tape: Optional[torch.Tensor] = None,
               seed: int = 0, sample_offset: int = 0, trace: bool = False, sample_ids=None):
        """Runs the reverse loop for the batch set by set_batch.  Returns (x (B,N,3), atom_class (B,N) int32[, trace]).
        Device noise is keyed by (seed, global sample id): `sample_ids` (B int64) or `sample_offset + b`.  Modes:
        "forward", "inpaint", "merge" (merge_fragments) and "analogue" (the merge loop with nothing re-injected: z_known
        forward-diffused to `diffusion_level`, then denoised; fixed_mask is ignored)."""
        modes = {"forward": 0, "inpaint": 1, "merge": 2, "analogue": 3}
        gamma, steps = self._steps(T, blend_power)
        dec = decode_scalars(gamma)
        from_known = mode in ("merge", "analogue")
        lvl = forward_level_scalars(gamma, diffusion_level) if from_known else {"alpha": 0.0, "sigma": 0.0}
        B, N = self.B, self.N
        dev = self.device
        ctx = ctx.to(dev, torch.float32).contiguous()
        if ctx.shape != (B, 3):
            raise ValueError("sample: ctx must be (B,3)")
        zk = None if z_known is None else z_known.to(dev, torch.float32).contiguous()
        fm = None if fixed_mask is None else fixed_mask.to(dev, torch.float32).reshape(B, N).contiguous()
        tape = None if noise_tape is None else noise_tape.to(dev, torch.float32).contiguous()
        ids = None
        if sample_ids is not None:
            ids = torch.as_tensor(np.asarray(sample_ids, dtype=np.int64).reshape(-1)).to(dev).contiguous()
            if ids.numel() != B:
                raise ValueError("sample: sample_ids must hold one id per sample")
        r_eff = resample_steps if mode == "forward" else max(resample_steps, 1)
        n_active = T if not from_known else min(diffusion_level, T - 1) + 1
        if mode == "forward":
            n_fwd, n_draw = T * (r_eff + 1) + 1, 1 + T * (r_eff + 1) + 1
        elif mode == "inpaint":
            n_fwd, n_draw = T * (r_eff + 1) + 1, 1 + T * (2 * r_eff + 1) + 1
        elif mode == "merge":
            n_fwd, n_draw = n_active * r_eff + 1, 1 + n_active * 2 * r_eff + 1
        else:
            n_fwd, n_draw = n_active * r_eff + 1, 1 + n_active * r_eff + 1
        if tape is not None and tuple(tape.shape) != (n_draw, B, N, 11):
            raise ValueError("sample: noise tape must be (%d,%d,%d,11), got %s" % (n_draw, B, N, tuple(tape.shape)))
        z = torch.empty(B, N, 11, device=dev)
        x = torch.empty(B, N, 3, device=dev)
        cls = torch.empty(B, N, dtype=torch.int32, device=dev)
        tz = torch.empty(n_fwd, B, N, 11, device=dev) if trace else None
        te = torch.empty(n_fwd, B, N, 11, device=dev) if trace else None
        rc = self.lib.mlcg_sample(self.h, modes[mode], T, steps, resample_steps, diffusion_level, lvl["alpha"],
                                  lvl["sigma"], dec["sigma_0"], dec["alpha_0"], dec["sigma_x"], _ptr(ctx), _ptr(zk),
                                  _ptr(fm), _ptr(tape), seed, sample_offset, _ptr(ids), _ptr(z), _ptr(x), _ptr(cls),
                                  _ptr(tz), _ptr(te), self._stream())
        self._check(rc, "sample")
        self._keep = [ctx, zk, fm, tape, ids]
        if trace:
            return x, cls, (tz, te)
        return x, cls

    # ------------------------------------------------------------------------------------------------------------
    def seer_inputs(self, x: torch.Tensor, cls: torch.Tensor):
        B = self.B
        el = torch.empty(B, 42, dtype=torch.int32, device=self.device)
        dist = torch.empty(B, 42, 42, device=self.device)
        adj = torch.empty(B, 42, 42, device=self.device)
        x = x.to(self.device, torch.float32).contiguous()
        cls = cls.to(self.device, torch.int32).contiguous()
        self._check(self.lib.mlcg_seer_inputs(self.h, _ptr(x), _ptr(cls), _ptr(el), _ptr(dist), _ptr(adj),
                                              self._stream()), "seer_inputs")
        return el, dist, adj

    def seer_forward(self, elements: torch.Tensor, dist: torch.Tensor, adj: torch.Tensor, want_logits: bool = True):
        el = elements.to(self.device, torch.int32).contiguous()
        dist = dist.to(self.device, torch.float32).contiguous()
        adj = adj.to(self.device, torch.float32).contiguous()
        B = el.shape[0]
        logits = torch.empty(B, 42, 42, 5, device=self.device) if want_logits else None
        bonds = torch.empty(B, 42, 42, dtype=torch.int8, device=self.device)
        self._check(self.lib.mlcg_seer_forward(self.h, _ptr(el), _ptr(dist), _ptr(adj), _ptr(logits), _ptr(bonds), B,
                                               self._stream()), "seer_forward")
        self._keep = [el, dist, adj]
        return logits, bonds

    # ------------------------------------------------------------------------------------------------------------
    # inertial fragment matching on the device (reference utils/mol_utils.py:373-550)
    def ifm_context(self, fixed_fragment_x: torch.Tensor, reference_context: torch.Tensor, context_norms: Dict,
                    n_nodes: torch.Tensor):
        """Device version of ifm_prepare_gen_fragment_context after its batch-independent prologue.  n_nodes: (B) total
        atoms per sample.  Returns device tensors (ctx (B,3) normalised, shift (B,3), rotation (B,3,3), n_gen (B) i32)."""
        from .mol_utils import ifm_moi_prologue
        n_ff = int(fixed_fragment_x.size(0))
        moi0, com = ifm_moi_prologue(fixed_fragment_x, reference_context)
        mean = torch.as_tensor(context_norms["mean"], dtype=torch.float32).contiguous()
        mad = torch.as_tensor(context_norms["mad"], dtype=torch.float32).contiguous()
        nn = n_nodes.to(self.device, torch.int32).contiguous()
        B = int(nn.numel())
        ctx = torch.empty(B, 3, device=self.device)
        shift = torch.empty(B, 3, device=self.device)
        rot = torch.empty(B, 3, 3, device=self.device)
        n_gen = torch.empty(B, dtype=torch.int32, device=self.device)
        self._check(self.lib.mlcg_ifm_context(self.h, _ptr(moi0), _ptr(com), n_ff, _ptr(mean), _ptr(mad), _ptr(nn), B,
                                              _ptr(ctx), _ptr(shift), _ptr(rot), _ptr(n_gen), self._stream()), "ifm_context")
        return ctx, shift, rot, n_gen

    def ifm_merge_inputs(self, x_gen: torch.Tensor, cls_gen: torch.Tensor, shift: torch.Tensor, rot: torch.Tensor,
                         fixed_fragment_x: torch.Tensor, fixed_fragment_h: torch.Tensor, max_n_nodes: int):
        """Device version of inverse_coord_transform + ifm_prepare_fragments_for_merge: (z_known (B,N,11), fixed_mask (B,N))."""
        x_gen = x_gen.to(self.device, torch.float32).contiguous()
        cls_gen = cls_gen.to(self.device, torch.int32).contiguous()
        ffx = fixed_fragment_x.to(self.device, torch.float32).contiguous()
        ffh = fixed_fragment_h.to(self.device, torch.float32).contiguous()
        B, Ng = int(x_gen.shape[0]), int(x_gen.shape[1])
        zk = torch.empty(B, max_n_nodes, 11, device=self.device)
        fm = torch.empty(B, max_n_nodes, device=self.device)
        self._check(self.lib.mlcg_ifm_merge_inputs(self.h, _ptr(x_gen), _ptr(cls_gen), _ptr(shift.contiguous()),
                                                   _ptr(rot.contiguous()), _ptr(ffx), _ptr(ffh), int(ffx.shape[0]), B, Ng,
                                                   int(max_n_nodes), _ptr(zk), _ptr(fm), self._stream()), "ifm_merge_inputs")
        self._keep = [x_gen, cls_gen, ffx, ffh, shift, rot]
        return zk, fm

    def check_finite(self, what: str = "sample") -> bool:
        """True if every coordinate decoded since the last check was finite; otherwise warns and returns False.
        Synchronises the current stream."""
        if int(self.lib.mlcg_nonfinite(self.h, self._stream())):
            import warnings
            warnings.warn("%s: non-finite coordinates were generated -- the trajectory diverged%s" % (
                what, " or left the fp16 range (pairwise distances > ~1.6e4); precision='bf16' / 'tf32' have fp32's exponent "
                "range" if self.precision == "fp16" else ""), RuntimeWarning, stacklevel=2)
            return False
        return True

    def generate_host(self, n_nodes: np.ndarray, max_n_nodes: int, ctx: np.ndarray, T: int = 100,
                      resample_steps: int = 0, seed: int = 0, sample_offset: int = 0, out=None, sample_ids=None,
                      device_out: bool = False):
        """End-to-end with host inputs: returns (x (B,N,3) f32, atom_class (B,N) i32, bonds (B,42,42) i8) in pinned host
        buffers, or -- `device_out=True`, used by the multi-GPU driver whose gather runs on the device -- in device
        tensors.  `sample_ids` (B int64): global ids keying the device noise (default `sample_offset + b`)."""
        return self._generate("generate_host", "generate", self.lib.mlcg_generate, None, n_nodes, max_n_nodes, ctx, T, 3,
                              resample_steps, seed, sample_offset, sample_ids, out, device_out)

    def _generate(self, name, what, call, table, n_nodes, max_n_nodes, ctx, T, blend_power, resample_steps, seed,
                  sample_offset, sample_ids, out, device_out):
        """The host generation call `call` (an mlcg_generate* prototype) once its kind's table (a ctypes structure passed
        by reference, or None) is built: host inputs, schedule, errors and non-finite warnings under `what`, and the batch
        bookkeeping.  Argument errors found here name the public method `name`.  Returns the outputs: `out`, or new
        pinned host / device tensors (x (B,N,3), atom_class (B,N), bonds (B,42,42))."""
        nn = np.ascontiguousarray(np.asarray(n_nodes, dtype=np.int32).reshape(-1))
        B, N = int(nn.size), int(max_n_nodes)
        ctxh = torch.from_numpy(np.ascontiguousarray(ctx, dtype=np.float32).reshape(B, 3)).pin_memory()
        ids = None
        if sample_ids is not None:
            ids = np.ascontiguousarray(np.asarray(sample_ids, dtype=np.int64).reshape(-1))
            if ids.size != B:
                raise ValueError("%s: sample_ids must hold one id per sample" % name)
        if out is None:
            if device_out:
                out = (torch.empty(B, N, 3, device=self.device), torch.empty(B, N, dtype=torch.int32, device=self.device),
                       torch.empty(B, 42, 42, dtype=torch.int8, device=self.device))
            else:
                out = (torch.empty(B, N, 3).pin_memory(), torch.empty(B, N, dtype=torch.int32).pin_memory(),
                       torch.empty(B, 42, 42, dtype=torch.int8).pin_memory())
        gamma, steps = self._steps_cached(T, blend_power)
        dec = decode_scalars(gamma)
        head = (self.h,) if table is None else (self.h, C.byref(table))
        rc = call(*head, nn.ctypes.data_as(C.c_void_p), B, N, _ptr(ctxh), T, steps, resample_steps, dec["sigma_0"],
                  dec["alpha_0"], dec["sigma_x"], seed, sample_offset,
                  None if ids is None else ids.ctypes.data_as(C.c_void_p), _ptr(out[0]), _ptr(out[1]), _ptr(out[2]),
                  self._stream())
        self._check(rc, what)
        self.check_finite(what)
        self.B, self.N = B, N
        self.n_nodes = torch.from_numpy(nn.copy())
        return out

    @staticmethod
    def _pack_molecules(what, noun, mols):
        """(coordinates (n,3), one-hot (n,8)) pairs -> atom counts (int32) and the coordinates (sum n,3) and one-hots
        (sum n,8) back to back, float32."""
        xs, hs = [], []
        for x, h in mols:
            x = np.asarray(torch.as_tensor(x).detach().cpu().numpy(), dtype=np.float32)
            h = np.asarray(torch.as_tensor(h).detach().cpu().numpy(), dtype=np.float32)
            if x.ndim != 2 or x.shape[1] != 3 or h.shape != (x.shape[0], 8):
                raise ValueError("%s: %s must be coordinates (n,3) and a one-hot (n,8)" % (what, noun))
            xs.append(x)
            hs.append(h)
        return (np.array([x.shape[0] for x in xs], dtype=np.int32), np.ascontiguousarray(np.concatenate(xs).reshape(-1, 3)),
                np.ascontiguousarray(np.concatenate(hs).reshape(-1, 8)))

    def generate_fragment_host(self, n_nodes: np.ndarray, max_n_nodes: int, ctx: np.ndarray, fragment_x, fragment_h,
                               inertial_fragment_matching: bool = True, reference_context=None, context_norms=None,
                               T: int = 100, resample_steps: int = 0, blend_power: int = 3, diffusion_level: int = 50,
                               seed: int = 0, sample_offset: int = 0, sample_ids=None, out=None, device_out: bool = False):
        """generate_host around a fixed fragment (the reference's `fixed_fragment=`): fragment_x (n_ff,3) coordinates in
        the frame centred on the reference's centre of mass, fragment_h (n_ff,8) raw 0/1 one-hot.  With
        inertial_fragment_matching (the reference's default) the atoms still to be generated are sampled on their own in
        the frame of their inertia tensor -- which needs the raw `reference_context` (principal moments) and
        `context_norms` (default CONTEXT_NORMS) -- and merged with the fragment in a second loop at `diffusion_level`;
        otherwise the fragment is inpainted.  `ctx` (B,3) is the normalised reference context of every sample.  Same
        outputs, noise keys and graph replay as generate_host; the result equals the eager composition of
        MLConformerGenerator.edm_sample_tensors + the GCN bit for bit."""
        what = "generate_fragment_host"
        fj, keep = self._fragment_table(what, np.size(n_nodes), np.zeros(np.size(n_nodes), np.int32),
                                        [(fragment_x, fragment_h)], inertial_fragment_matching,
                                        None if reference_context is None else [reference_context], context_norms, T,
                                        blend_power, diffusion_level)
        return self._generate(what, "generate_fragment", self.lib.mlcg_generate_fragment_jobs, fj, n_nodes, max_n_nodes,
                              ctx, T, blend_power, resample_steps, seed, sample_offset, sample_ids, out, device_out)

    def generate_fragment_jobs_host(self, n_nodes: np.ndarray, max_n_nodes: int, ctx: np.ndarray, job_of_sample,
                                    fragments, inertial_fragment_matching: bool = True, reference_contexts=None,
                                    context_norms=None, T: int = 100, resample_steps: int = 0, blend_power: int = 3,
                                    diffusion_level: int = 50, seed: int = 0, sample_offset: int = 0, sample_ids=None,
                                    out=None, device_out: bool = False):
        """generate_fragment_host for many fragment jobs of one mode in one call: sample b runs with the fragment
        fragments[job_of_sample[b]] = (coordinates (n,3), one-hot (n,8)) and -- inertial fragment matching -- the raw
        reference context reference_contexts[job_of_sample[b]].  `ctx` (B,3) is every sample's normalised context; the
        loop settings are shared.  Same outputs, noise keys and graph replay as generate_fragment_host, and every sample
        equals a call holding only its own job with the same sample id, bit for bit."""
        what = "generate_fragment_jobs_host"
        fj, keep = self._fragment_table(what, np.size(n_nodes), job_of_sample, fragments, inertial_fragment_matching,
                                        reference_contexts, context_norms, T, blend_power, diffusion_level)
        return self._generate(what, "generate_fragment", self.lib.mlcg_generate_fragment_jobs, fj, n_nodes, max_n_nodes,
                              ctx, T, blend_power, resample_steps, seed, sample_offset, sample_ids, out, device_out)

    def _fragment_table(self, what, B, job_of_sample, fragments, inertial_fragment_matching, reference_contexts,
                        context_norms, T, blend_power, diffusion_level):
        """mlcg_fragment_jobs and the host arrays it points to, which must outlive the call."""
        job = np.ascontiguousarray(np.asarray(job_of_sample, dtype=np.int32).reshape(-1))
        if job.size != B:
            raise ValueError("%s: job_of_sample must hold one job per sample" % what)
        n_ff, packed_x, packed_h = self._pack_molecules(what, "the fragment", fragments)
        keep = [job, n_ff, packed_x, packed_h]
        fj = _lib.FragmentJobs(2 if inertial_fragment_matching else 1, n_ff.size, *(a.ctypes.data for a in keep))
        if inertial_fragment_matching:
            if reference_contexts is None or len(reference_contexts) != n_ff.size:
                raise ValueError("%s: inertial fragment matching needs the raw reference_context of every job" % what)
            from .config import CONTEXT_NORMS
            from .mol_utils import ifm_moi_prologue
            norms = CONTEXT_NORMS if context_norms is None else context_norms
            pro = [ifm_moi_prologue(torch.from_numpy(fx), ref)
                   for fx, ref in zip(np.split(packed_x, np.cumsum(n_ff)[:-1]), reference_contexts)]
            ifm = [torch.stack([p[0] for p in pro]).contiguous(), torch.stack([p[1] for p in pro]).contiguous()] + \
                [torch.as_tensor(norms[k], dtype=torch.float32).contiguous() for k in ("mean", "mad")]
            keep += ifm
            lvl = forward_level_scalars(self._steps_cached(T, blend_power)[0], diffusion_level)
            fj.diffusion_level, fj.merge_alpha, fj.merge_sigma = int(diffusion_level), lvl["alpha"], lvl["sigma"]
            fj.moi_gen_origin_host, fj.ff_weighted_com_host, fj.norm_mean_host, fj.norm_mad_host = (
                t.data_ptr() for t in ifm)
        return fj, keep

    @staticmethod
    def _analogue_table(what, job_of_sample, B, parents, fixed):
        """mlcg_analogue_jobs (diffusion level unset) and the host arrays it points to, which must outlive the call."""
        job = np.ascontiguousarray(np.asarray(job_of_sample, dtype=np.int32).reshape(-1))
        if job.size != B:
            raise ValueError("%s: job_of_sample must hold one job per sample" % what)
        if fixed is not None and len(fixed) != len(parents):
            raise ValueError("%s: fixed must hold one flag array per parent" % what)
        n_atoms, px, ph = Engine._pack_molecules(what, "a parent", parents)
        pf = []
        for j, n in enumerate(n_atoms):
            f = np.zeros(n, np.int32) if fixed is None or fixed[j] is None else np.asarray(fixed[j]).reshape(-1).astype(np.int32)
            if f.size != n:
                raise ValueError("%s: the fixed flags must hold one entry per parent atom" % what)
            pf.append(f)
        keep = [job, n_atoms, px, ph, np.ascontiguousarray(np.concatenate(pf))]
        return _lib.AnalogueJobs(n_atoms.size, *(a.ctypes.data for a in keep)), keep

    def analogue_inputs(self, job_of_sample, parents, fixed, max_n_nodes: int):
        """Device version of the analogue jobs' first step (mlcg_analogue_inputs): (z_known (B,N,11), fixed_mask (B,N)) with
        sample b holding parent job_of_sample[b] = (centred coordinates (n,3), one-hot (n,8)) and its fixed flags
        (fixed[j]: (n,) 0/1, or None for none)."""
        B, N = int(np.size(job_of_sample)), int(max_n_nodes)
        aj, keep = self._analogue_table("analogue_inputs", job_of_sample, B, parents, fixed)
        zk = torch.empty(B, N, 11, device=self.device)
        fm = torch.empty(B, N, device=self.device)
        self._check(self.lib.mlcg_analogue_inputs(self.h, C.byref(aj), B, N, _ptr(zk), _ptr(fm), self._stream()),
                    "analogue_inputs")
        del keep
        return zk, fm

    def generate_analogue_jobs_host(self, n_nodes: np.ndarray, max_n_nodes: int, ctx: np.ndarray, job_of_sample, parents,
                                    fixed=None, T: int = 100, resample_steps: int = 0, blend_power: int = 3,
                                    diffusion_level: int = 50, seed: int = 0, sample_offset: int = 0, sample_ids=None,
                                    out=None, device_out: bool = False):
        """Analogues of parent molecules in one call (mlcg_generate_analogue_jobs): sample b starts from parent
        parents[job_of_sample[b]] = (coordinates (n,3) centred on their mean, raw 0/1 one-hot (n,8)) forward-diffused to
        `diffusion_level` and is denoised from there; n_nodes[b] must be that parent's n.  fixed[j] ((n,) 0/1 or None)
        marks atoms re-injected at every step as merge_fragments re-injects a fragment; in one call every job has a fixed
        atom or none has.  `ctx` (B,3) is every sample's normalised context.  Same outputs, noise keys and graph replay as
        generate_fragment_jobs_host; every sample equals a call holding only its own job with the same id, bit for bit,
        and the result equals the eager composition analogue_inputs + sample + the GCN."""
        what = "generate_analogue_jobs_host"
        aj, keep = self._analogue_table(what, job_of_sample, np.size(n_nodes), parents, fixed)
        if not 1 <= int(diffusion_level) <= T:
            raise ValueError("generate_analogue_jobs_host: diffusion_level must lie in [1, T=%d]" % T)
        lvl = forward_level_scalars(self._steps_cached(T, blend_power)[0], int(diffusion_level))
        aj.diffusion_level, aj.merge_alpha, aj.merge_sigma = int(diffusion_level), lvl["alpha"], lvl["sigma"]
        return self._generate(what, "generate_analogue", self.lib.mlcg_generate_analogue_jobs, aj, n_nodes, max_n_nodes,
                              ctx, T, blend_power, resample_steps, seed, sample_offset, sample_ids, out, device_out)

    # ------------------------------------------------------------------------------------------------------------
    def num_edges(self) -> int:
        return int(self.lib.mlcg_num_edges(self.h))

    def num_edge_tiles(self) -> int:
        return int(self.lib.mlcg_num_edge_tiles(self.h))

    def kernel_launches(self) -> int:
        return int(self.lib.mlcg_kernel_launches(self.h))

    def graph_captures(self) -> int:
        """CUDA graphs captured by the host calls since the engine was created (a replay leaves it unchanged)."""
        return int(self.lib.mlcg_graph_captures(self.h))

    def time_edge_kernel(self, layer: int = 0, iters: int = 10) -> float:
        return float(self.lib.mlcg_time_edge_kernel(self.h, layer, iters, self._stream()))

    def edge_phase_profile(self, layer: int = 0):
        out = (C.c_double * 16)()
        self._check(self.lib.mlcg_edge_phase_profile(self.h, layer, out, self._stream()), "edge_phase_profile")
        names = ["rowinfo_pq_wait", "a_gen", "mma_tail", "pass1", "pass2", "a_ring_backpressure", "tiles",
                 "p2_wait_segmma", "p2_load_gate_pack", "p2_stage_arrive", "p2_readout", "a_handoff"]
        if self.precision in ("fp16", "bf16") and os.environ.get("MLCG_EDGE_V3", "1") != "0" and \
                os.environ.get("MLCG_EDGE_PAIR", "1") != "0":
            # k_tc_edge3 (mlcg_tc3.cuh): per tile, thread 0 of the compute warps (the highest-priority warp of its
            # sub-partition: it finishes the MUFU-bound phases first and waits at the barriers for the others).
            # Equivariant sub-layers: "gate_selector" holds the remaining A chunks of the next tile and "agen_rest" the
            # coordinate sums (they run in that order there); "wait_segsum" / "readout" are GCL only.
            names = ["wait_third0", "pass1_third0", "wait_third1", "pass1_third1", "barrier_pq_wait", "agen_early", "tiles",
                     "wait_third2", "pass1_third2", "gate_selector", "agen_rest", "wait_segsum", "readout", "end_barrier",
                     "unused14", "unused15"]
        return {n: float(out[i]) for i, n in enumerate(names)}

    def gemm_phase_profile(self, which: int) -> dict:
        """Cycle counters of one node-GEMM launch (0 = P/Q projection, 1 = SiLU GEMM, 2 = residual GEMM) on the current
        batch; see mlcg_gemm_phase_profile.  Diagnostics only (which = 2 modifies the residual stream)."""
        out = (C.c_double * 8)()
        self._check(self.lib.mlcg_gemm_phase_profile(self.h, which, out, self._stream()), "gemm_phase_profile")
        names = ["producer_wait_slot", "mma_wait_operands", "mma_wait_epilogue", "epi_wait_accumulator", "epilogue",
                 "tiles_per_cta", "cta_lifetime", "launch_ms"]
        return {n: float(out[i]) for i, n in enumerate(names)}

    def test_gemm(self, mode: str, bn: int, a: torch.Tensor, w: torch.Tensor, bias: torch.Tensor) -> torch.Tensor:
        a = a.to(self.device, torch.float32).contiguous()
        w = w.to(self.device, torch.float32).contiguous()
        bias = bias.to(self.device, torch.float32).contiguous()
        M, K = a.shape
        N = w.shape[0]
        c = torch.empty(M, N, device=self.device)
        self._check(self.lib.mlcg_test_gemm(self.h, PRECISIONS[mode], bn, _ptr(a), _ptr(w), _ptr(bias), _ptr(c), M, N,
                                            K, self._stream()), "test_gemm")
        return c
