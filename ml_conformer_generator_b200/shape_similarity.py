"""Gaussian shape similarity of generated conformers on the GPU -- host side.

Mirrors the tensor part of the reference's `evaluate_samples` (cheminformatics/pipeline.py:37-86) and the functions of
cheminformatics/shape_similarity.py it calls, with the same names where a counterpart exists.  The clique series and the
grid overlap run in `libmlcg_b200.so` (`mlcg_shape_moments`, `mlcg_shape_tanimoto`, `mlcg_shape_tanimoto_jobs`); the 3x3
eigen-decomposition stays on the host in torch, exactly as the reference does it (`torch.linalg.eigh`,
shape_similarity.py:139), so the principal-frame sign / order conventions are the reference's.  There is no CPU fallback.
"""
from typing import Dict, Optional, Sequence

import numpy as np
import torch

from .engine import Engine, _ptr

ATOM_RADIUS = 1.60   # reference shape_similarity.py:14
AMPLITUDE = 2.70     # reference shape_similarity.py:15
GRID_POINTS = 40     # tanimoto_score default, :470
MAX_ATOMS = 64
MAX_JOB_REFERENCES = 256  # references per mlcg_shape_tanimoto_jobs call: 64 MB of density workspace at 40^3


def get_alpha(atom_radius: float = ATOM_RADIUS, gaussian_amplitude: float = AMPLITUDE) -> float:
    """reference shape_similarity.py:322-329."""
    lyambda_ = 4 * np.pi / 3 / gaussian_amplitude
    k_a = np.pi / lyambda_ ** (2 / 3)
    return k_a / atom_radius ** 2


def orientation_matrices() -> torch.Tensor:
    """(4,3,3): identity and the three rotations by pi evaluate_samples tries (pipeline.py:46-51), built like
    rotate_coord (shape_similarity.py:422-436) from float32 cos/sin of float32 pi."""
    pi = torch.pi
    mats = [torch.eye(3)]
    for angles in (torch.tensor([pi, 0, 0]), torch.tensor([0, pi, 0]), torch.tensor([0, 0, pi])):
        c, s = torch.cos(angles), torch.sin(angles)
        rx = torch.tensor([[1, 0, 0], [0, c[0], -s[0]], [0, s[0], c[0]]])
        ry = torch.tensor([[c[1], 0, s[1]], [0, 1, 0], [-s[1], 0, c[1]]])
        rz = torch.tensor([[c[2], -s[2], 0], [s[2], c[2], 0], [0, 0, 1]])
        mats.append(rx @ ry @ rz)
    return torch.stack(mats).to(torch.float32)


def grid_axes(ref_pts: torch.Tensor, n: int = GRID_POINTS, bounds_scale: float = 6, max_sigma: float = ATOM_RADIUS) -> torch.Tensor:
    """(3,n) grid coordinates of the reference's Grid as tanimoto_score builds it (shape_similarity.py:476-480, 381-403).
    The reference reduces cat(ref, cand) over dim=1 -- the x/y/z components of each ATOM -- and reads entries 0, 1, 2, so
    the bounds of the x, y, z axes are the smallest / largest component of the first, second and third atom of the
    reference molecule (+- 6 * 1.6).  With at least three reference atoms the grid therefore does not depend on the
    candidate; that case is the one supported here."""
    if ref_pts.size(0) < 3:
        raise ValueError("the reference molecule needs at least 3 heavy atoms")
    p = ref_pts.detach().cpu().to(torch.float32)
    lo = p.min(dim=1).values - bounds_scale * max_sigma
    hi = p.max(dim=1).values + bounds_scale * max_sigma
    return torch.stack([torch.linspace(lo[k], hi[k], n) for k in range(3)])


class ShapeScorer:
    """Batched get_shape_quadrupole_for_molecule + tanimoto_score on one GPU."""

    def __init__(self, engine: Optional[Engine] = None, device: torch.device = torch.device("cuda:0"),
                 amplitude: float = AMPLITUDE, atom_radius: float = ATOM_RADIUS, n_terms: int = 6):
        self.engine = engine if engine is not None else Engine(device, "bf16")
        self.device = self.engine.device
        self.amplitude, self.atom_radius, self.n_terms = float(amplitude), float(atom_radius), int(n_terms)
        self._orient = orientation_matrices()

    # -- get_shape_quadrupole_for_molecule, batched ---------------------------------------------------------------
    def principal_frames(self, coords: torch.Tensor, n_nodes: torch.Tensor) -> Dict[str, torch.Tensor]:
        """coords (B,N,3), n_nodes (B).  Returns `moments` (B,3) descending principal shape-quadrupole moments, `frames`
        (B,12) = shift + rotation with principal = (x - shift) @ rotation, `points` (B,N,3) the principal-frame
        coordinates (zero beyond n_nodes), `volume` (B,), `tensor0` (B,3,3)."""
        e = self.engine
        coords = coords.to(self.device, torch.float32).contiguous()
        if coords.dim() != 3 or coords.size(2) != 3:
            raise ValueError("coords must be (B, N, 3)")
        B, N = coords.size(0), coords.size(1)
        n_nodes = torch.as_tensor(n_nodes).to(torch.int32).cpu()
        if n_nodes.numel() != B or int(n_nodes.min()) < 1 or int(n_nodes.max()) > min(N, MAX_ATOMS):
            raise ValueError("n_nodes must hold B values in [1, min(N, 64)]")
        nn_dev = n_nodes.to(self.device)
        out = torch.empty(B, 16, device=self.device)
        e._check(e.lib.mlcg_shape_moments(e.h, _ptr(coords), _ptr(nn_dev), B, N, self.amplitude, self.atom_radius,
                                          self.n_terms, _ptr(out), e._stream()), "shape_moments")
        o = out.cpu()
        t0 = o[:, 4:13].reshape(B, 3, 3).contiguous()
        # host: eigenvectors, moments in the rotated frame, descending order (reference :139-140, 193-201)
        _, vecs = torch.linalg.eigh(t0)
        rotated_t = vecs.transpose(1, 2) @ t0 @ vecs
        moments, order = torch.sort(torch.diagonal(rotated_t, dim1=1, dim2=2), descending=True, dim=1)
        rot = torch.gather(vecs, 2, order.unsqueeze(1).expand(B, 3, 3))
        shift = o[:, 13:16] + o[:, 1:4]
        frames = torch.cat([shift, rot.reshape(B, 9)], dim=1).contiguous()
        mask = (torch.arange(N).unsqueeze(0) < n_nodes.unsqueeze(1)).unsqueeze(-1)
        points = ((coords.cpu() - shift.unsqueeze(1)) @ rot) * mask
        return {"moments": moments, "frames": frames, "points": points, "volume": o[:, 0].clone(), "tensor0": t0,
                "first_moments": o[:, 1:4].clone()}

    # -- tanimoto_score over samples x orientations ---------------------------------------------------------------
    def tanimoto(self, ref_pts: torch.Tensor, coords: torch.Tensor, n_nodes: torch.Tensor, frames: torch.Tensor,
                 n: int = GRID_POINTS) -> Dict[str, torch.Tensor]:
        """ref_pts (n_ref,3): reference atoms in their principal frame.  Returns `scores` (B,4) for the orientations of
        orientation_matrices() and `aligned` (B,4,N,3) the candidate coordinates in each of them (device tensors)."""
        e = self.engine
        coords = coords.to(self.device, torch.float32).contiguous()
        B, N = coords.size(0), coords.size(1)
        ref = ref_pts.to(self.device, torch.float32).contiguous()
        if ref.size(0) > MAX_ATOMS:
            raise ValueError("at most 64 reference atoms")
        axes = grid_axes(ref_pts, n).to(self.device).contiguous()
        orient = self._orient.reshape(-1, 9).to(self.device).contiguous()
        nn_dev = torch.as_tensor(n_nodes).to(torch.int32).to(self.device)
        fr = frames.to(self.device, torch.float32).contiguous()
        work = torch.empty(n ** 3 + 1, device=self.device)
        scores = torch.empty(B, orient.size(0), device=self.device)
        aligned = torch.zeros(B, orient.size(0), N, 3, device=self.device)
        e._check(e.lib.mlcg_shape_tanimoto(e.h, _ptr(ref), ref.size(0), _ptr(coords), _ptr(nn_dev), B, N, _ptr(fr),
                                           _ptr(orient), orient.size(0), _ptr(axes), n, self.amplitude, self.atom_radius,
                                           _ptr(work), _ptr(scores), _ptr(aligned), e._stream()), "shape_tanimoto")
        return {"scores": scores, "aligned": aligned}

    # -- the tensor part of evaluate_samples ------------------------------------------------------------------------
    def evaluate(self, reference_coord: torch.Tensor, sample_coords: torch.Tensor, n_nodes: torch.Tensor) -> Dict[str, torch.Tensor]:
        """reference_coord (n_ref,3) heavy-atom coordinates of the reference conformer; sample_coords (B,N,3) / n_nodes
        (B) heavy atoms of the samples.  Returns `shape_tanimoto` (B,) the best of the four orientations (first strict
        maximum, pipeline.py:76-85), `best_orientation` (B,), `aligned_coords` (B,N,3) the sample in that orientation,
        `scores` (B,4), `reference_coords` (n_ref,3) the reference in its principal frame, `moments` (B,3)."""
        ref = reference_coord.to(torch.float32)
        rf = self.principal_frames(ref.unsqueeze(0), torch.tensor([ref.size(0)]))
        ref_pts = rf["points"][0]
        sf = self.principal_frames(sample_coords, n_nodes)
        t = self.tanimoto(ref_pts, sample_coords, n_nodes, sf["frames"])
        scores = t["scores"].cpu()
        best = torch.zeros(scores.size(0), dtype=torch.long)
        best_score = scores[:, 0].clone()
        for k in range(1, scores.size(1)):
            better = scores[:, k] > best_score
            best = torch.where(better, torch.full_like(best, k), best)
            best_score = torch.where(better, scores[:, k], best_score)
        aligned = t["aligned"].cpu()
        idx = best.view(-1, 1, 1, 1).expand(-1, 1, aligned.size(2), 3)
        return {"shape_tanimoto": best_score, "best_orientation": best, "aligned_coords": aligned.gather(1, idx).squeeze(1),
                "scores": scores, "reference_coords": ref_pts, "moments": sf["moments"], "reference_moments": rf["moments"][0]}

    # -- evaluate for many references at once ------------------------------------------------------------------------
    def evaluate_jobs(self, references: Sequence[torch.Tensor], coords: torch.Tensor, n_nodes: torch.Tensor,
                      job: torch.Tensor, n: int = GRID_POINTS) -> Dict[str, object]:
        """`evaluate` of every sample against its own reference: sample b (coords (B,N,3), n_nodes (B)) is scored against
        references[job[b]] (heavy-atom coordinates (n_ref,3), 3 <= n_ref <= 64).  Returns device tensors
        `shape_tanimoto` (B,), `best_orientation` (B,), `aligned_coords` (B,N,3), `scores` (B,4), `moments` (B,3), and
        per reference the lists `reference_coords` (n_ref,3) and `reference_moments` (3,).  Every value is bit-identical
        to `evaluate(references[j], samples of job j)`: the references go through evaluate's own host code one at a time,
        the kernels score each sample alone, and the best orientation uses evaluate's rule on the device.  B may be 0
        (the reference outputs only).  Calls hold at most MAX_JOB_REFERENCES references each, which bounds the density
        workspace (256 KB per reference at n = 40)."""
        e = self.engine
        refs = [torch.as_tensor(r).detach().to(torch.float32) for r in references]
        J = len(refs)
        for j, r in enumerate(refs):
            if r.dim() != 2 or r.size(1) != 3 or not 3 <= r.size(0) <= MAX_ATOMS:
                raise ValueError("reference %d must be (n_ref, 3) with 3 <= n_ref <= %d" % (j, MAX_ATOMS))
        coords = coords.to(self.device, torch.float32).contiguous()
        if coords.dim() != 3 or coords.size(2) != 3:
            raise ValueError("coords must be (B, N, 3)")
        B, N = coords.size(0), coords.size(1)
        n_nodes = torch.as_tensor(n_nodes).reshape(-1)
        job = torch.as_tensor(job).reshape(-1).to(torch.int64).cpu()
        if n_nodes.numel() != B or job.numel() != B:
            raise ValueError("coords, n_nodes and job must have the same length B")
        if B and (J == 0 or int(job.min()) < 0 or int(job.max()) >= J):
            raise ValueError("job indices must lie in [0, %d)" % J)
        # the references exactly as evaluate computes them (principal_frames of that one reference, then grid_axes)
        ref_pts = torch.zeros(J, MAX_ATOMS, 3)
        axes = torch.empty(J, 3, n)
        ref_coords, ref_moments = [], []
        for j, r in enumerate(refs):
            rf = self.principal_frames(r.unsqueeze(0), torch.tensor([r.size(0)]))
            pts = rf["points"][0]
            ref_pts[j, :pts.size(0)] = pts
            axes[j] = grid_axes(pts, n)
            ref_coords.append(pts.to(self.device))
            ref_moments.append(rf["moments"][0].to(self.device))
        out = {"reference_coords": ref_coords, "reference_moments": ref_moments}
        n_orient = self._orient.size(0)
        if B == 0:
            out.update(shape_tanimoto=torch.empty(0, device=self.device),
                       best_orientation=torch.empty(0, dtype=torch.long, device=self.device),
                       aligned_coords=torch.empty(0, N, 3, device=self.device),
                       scores=torch.empty(0, n_orient, device=self.device), moments=torch.empty(0, 3, device=self.device))
            return out
        sf = self.principal_frames(coords, n_nodes)
        frames = sf["frames"].to(self.device)
        nn_dev = n_nodes.to(torch.int32).to(self.device)
        job_dev = job.to(self.device)
        ref_pts, axes = ref_pts.to(self.device), axes.to(self.device)
        n_ref = torch.tensor([r.size(0) for r in refs], dtype=torch.int32, device=self.device)
        orient = self._orient.reshape(-1, 9).to(self.device).contiguous()
        work = torch.empty(min(J, MAX_JOB_REFERENCES) * (n ** 3 + 1), device=self.device)
        scores = torch.empty(B, n_orient, device=self.device)
        aligned = torch.zeros(B, n_orient, N, 3, device=self.device)
        for j0 in range(0, J, MAX_JOB_REFERENCES):
            j1 = min(J, j0 + MAX_JOB_REFERENCES)
            rows = torch.nonzero((job_dev >= j0) & (job_dev < j1)).view(-1)
            if rows.numel() == 0:
                continue
            c, nn, fr = coords[rows].contiguous(), nn_dev[rows].contiguous(), frames[rows].contiguous()
            jb = (job_dev[rows] - j0).to(torch.int32).contiguous()
            sc = torch.empty(rows.numel(), n_orient, device=self.device)
            al = torch.zeros(rows.numel(), n_orient, N, 3, device=self.device)
            e._check(e.lib.mlcg_shape_tanimoto_jobs(
                e.h, _ptr(ref_pts[j0:j1]), _ptr(n_ref[j0:j1]), _ptr(axes[j0:j1]), j1 - j0, _ptr(c), _ptr(nn), _ptr(jb),
                rows.numel(), N, _ptr(fr), _ptr(orient), n_orient, n, self.amplitude, self.atom_radius, _ptr(work),
                _ptr(sc), _ptr(al), e._stream()), "shape_tanimoto_jobs")
            scores[rows], aligned[rows] = sc, al
        # evaluate's rule: the first strict maximum over the orientations (a NaN never wins)
        best = torch.zeros(B, dtype=torch.long, device=self.device)
        best_score = scores[:, 0].clone()
        for k in range(1, n_orient):
            better = scores[:, k] > best_score
            best = torch.where(better, torch.full_like(best, k), best)
            best_score = torch.where(better, scores[:, k], best_score)
        idx = best.view(-1, 1, 1, 1).expand(-1, 1, N, 3)
        out.update(shape_tanimoto=best_score, best_orientation=best, aligned_coords=aligned.gather(1, idx).squeeze(1),
                   scores=scores, moments=sf["moments"].to(self.device))
        return out
