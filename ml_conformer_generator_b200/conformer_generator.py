"""Drop-in host API for the hot path: mirrors the reference's `MLConformerGenerator` (conformer_generator.py:19-399) --
same constructor and method signatures, same attribute names (`generative_model`, `adj_mat_seer`) -- with the EDM
reverse loop, the EGNN denoiser and the AdjMatSeer GCN running in libmlcg_b200.so on a B200.

RDKit-only stages (XYZ -> Mol, SMILES-order canonicalisation, bond editing, MMFF standardisation; reference
mol_utils.py:18-57,110-126,197-223 and standardizer.py) are not re-implemented: `generate_conformers` / `edm_samples`
call into RDKit exactly where the reference does and raise ImportError when it is not installed.  The tensor-level
entry points `edm_sample_tensors` / `generate_tensors` cover the accelerated path end to end without RDKit."""
import os
from typing import Dict, List, Optional, Tuple

import numpy as np
import torch

from .config import (ATOM_DECODER, CONTEXT_NORMS, DIMENSION, MAX_N_NODES, MIN_N_NODES, NUM_BOND_TYPES)
from .engine import Engine
from .mol_utils import (context_rows, counts_from_masks, get_context_shape, ifm_prepare_fragments_for_merge,
                        ifm_prepare_gen_fragment_context, inverse_coord_transform, normalise_context, prepare_edm_input,
                        prepare_fragment)
from .schedule import gamma_table


def _one_hot(atom_class: torch.Tensor) -> torch.Tensor:
    """(B,N) int classes (-1 = padding) -> (B,N,8) 0/1, the `h` the reference returns (equivariant_diffusion.py:283)."""
    h = torch.nn.functional.one_hot(atom_class.clamp_min(0).long(), 8)
    return h * (atom_class >= 0).unsqueeze(-1)


class EquivariantDiffusionB200:
    """Call-compatible stand-in for the reference's EquivariantDiffusion module (equivariant_diffusion.py:137-607)."""

    def __init__(self, engine: Engine, timesteps: int):
        self.engine = engine
        self.T = timesteps
        self.gamma = gamma_table(timesteps)
        self.time_steps = torch.flip(torch.arange(0, timesteps), dims=[0])
        self.noise_tape: Optional[torch.Tensor] = None  # parity hook: inject raw N(0,1) draws (n_draws,B,N,11)
        self.seed = 0

    def _setup(self, node_mask, edge_mask, context):
        counts = counts_from_masks(node_mask, edge_mask)
        self.engine.set_batch(counts.numpy(), node_mask.size(1))
        return context_rows(context, node_mask)

    def _finish(self, x, cls):
        return x, _one_hot(cls).to(x.device)

    def dynamics(self, t, xh, node_mask, edge_mask, context) -> torch.Tensor:
        """EGNNDynamics.forward (egnn.py:472-513)."""
        ctx = self._setup(node_mask, edge_mask, context)
        return self.engine.egnn_forward(t.reshape(-1), xh, ctx)

    def __call__(self, node_mask, edge_mask, context, resample_steps: int = 0):
        """EquivariantDiffusion.forward (equivariant_diffusion.py:365-421) -> (x (B,N,3), h (B,N,8))."""
        ctx = self._setup(node_mask, edge_mask, context)
        x, cls = self.engine.sample(ctx, self.T, "forward", resample_steps, noise_tape=self.noise_tape, seed=self.seed)
        return self._finish(x, cls)

    forward = __call__

    def inpaint(self, node_mask, edge_mask, context, z_known, fixed_mask, resample_steps: int = 1, blend_power: int = 3):
        """EquivariantDiffusion.inpaint (equivariant_diffusion.py:423-513)."""
        ctx = self._setup(node_mask, edge_mask, context)
        x, cls = self.engine.sample(ctx, self.T, "inpaint", resample_steps, z_known=z_known, fixed_mask=fixed_mask,
                                    blend_power=blend_power, noise_tape=self.noise_tape, seed=self.seed)
        return self._finish(x, cls)

    def merge_fragments(self, node_mask, edge_mask, fixed_mask, context, z_known, diffusion_level: int = 50,
                        resample_steps: int = 1, blend_power: int = 3):
        """EquivariantDiffusion.merge_fragments (equivariant_diffusion.py:515-607)."""
        ctx = self._setup(node_mask, edge_mask, context)
        x, cls = self.engine.sample(ctx, self.T, "merge", resample_steps, z_known=z_known, fixed_mask=fixed_mask,
                                    diffusion_level=diffusion_level, blend_power=blend_power,
                                    noise_tape=self.noise_tape, seed=self.seed)
        return self._finish(x, cls)


class AdjMatSeerB200:
    """Call-compatible stand-in for the reference's AdjMatSeer module (adj_mat_seer.py:60-165)."""

    def __init__(self, engine: Engine):
        self.engine = engine

    def __call__(self, elements, dist_mat, adj_mat) -> torch.Tensor:
        logits, _ = self.engine.seer_forward(elements, dist_mat, adj_mat, want_logits=True)
        return logits

    forward = __call__

    def bond_orders(self, elements, dist_mat, adj_mat) -> torch.Tensor:
        """Fused argmax of redefine_bonds (mol_utils.py:210-211): (B,42,42) int8, lower triangle."""
        _, bonds = self.engine.seer_forward(elements, dist_mat, adj_mat, want_logits=False)
        return bonds


class MLConformerGenerator:
    """Same public interface as the reference class (conformer_generator.py:25-37, 126-137, 269-282, 371-399).

    Additive keyword arguments: `precision` ("fp16" default: tcgen05 kind::f16 with fp16 operands -- tf32-class parity at
    full tensor-core rate; "bf16" 4 % faster, 8x coarser mantissa; "tf32"; "fp32" exact SIMT mode) and
    `edm_state_dict` / `adj_mat_seer_state_dict` to pass weights that are already in memory (the HuggingFace checkpoint
    files the reference downloads are not available offline)."""

    def __init__(self, diffusion_steps: int = 100, device: torch.device = torch.device("cuda:0"),
                 dimension: int = DIMENSION, num_bond_types: int = NUM_BOND_TYPES, min_n_nodes: int = MIN_N_NODES,
                 max_n_nodes: int = MAX_N_NODES, context_norms: dict = CONTEXT_NORMS, atom_decoder: dict = ATOM_DECODER,
                 edm_weights: str = "./edm_moi_chembl_15_39.pt",
                 adj_mat_seer_weights: str = "./adj_mat_seer_chembl_15_39.pt", precision: str = "fp16",
                 edm_state_dict: Optional[Dict[str, torch.Tensor]] = None,
                 adj_mat_seer_state_dict: Optional[Dict[str, torch.Tensor]] = None):
        if dimension != DIMENSION or num_bond_types != NUM_BOND_TYPES:
            raise ValueError("the B200 kernels are built for dimension=42 and num_bond_types=5")
        self.device = torch.device(device)
        self.dimension = dimension
        self.context_norms = {k: torch.tensor(v) for k, v in context_norms.items()}
        self.atom_decoder = atom_decoder
        self.min_n_nodes = min_n_nodes
        self.max_n_nodes = max_n_nodes
        if edm_state_dict is None:
            edm_state_dict = torch.load(edm_weights, map_location="cpu")["state_dict"]  # as conformer_generator.py:90-95
        if adj_mat_seer_state_dict is None:
            adj_mat_seer_state_dict = torch.load(adj_mat_seer_weights, map_location="cpu")["state_dict"]
        self.engine = Engine(self.device, precision)
        self.engine.load_edm_state_dict(edm_state_dict)
        self.engine.load_seer_state_dict(adj_mat_seer_state_dict)
        # the schedule is rebuilt for the requested number of steps (conformer_generator.py:104-113)
        self.generative_model = EquivariantDiffusionB200(self.engine, diffusion_steps)
        self.adj_mat_seer = AdjMatSeerB200(self.engine)

    # ------------------------------------------------------------------------------------------------------------
    # tensor-level path (no RDKit)
    # ------------------------------------------------------------------------------------------------------------
    @torch.no_grad()
    def edm_sample_tensors(self, reference_context: torch.Tensor, n_samples: int = 100, max_n_nodes: int = 32,
                           min_n_nodes: int = 25, resample_steps: int = 0,
                           fixed_fragment: Optional[Tuple[torch.Tensor, torch.Tensor]] = None,
                           inertial_fragment_matching: bool = True, blend_power: int = 3, ifm_diffusion_level: int = 50
                           ) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
        """Tensor part of edm_samples (conformer_generator.py:155-260): returns x (B,N,3), h (B,N,8), node_mask.
        `fixed_fragment` is (coords (n,3) in the frame centred on the reference's centre of mass, one-hot (n,8))."""
        min_n_nodes = max(min_n_nodes, self.min_n_nodes)
        max_n_nodes = min(max_n_nodes, self.max_n_nodes)
        node_mask, edge_mask, ctx = prepare_edm_input(n_samples, reference_context, self.context_norms, min_n_nodes,
                                                      max_n_nodes)
        gm = self.generative_model
        if fixed_fragment is None:
            x, h = gm(node_mask, edge_mask, ctx, resample_steps)
        elif inertial_fragment_matching:
            # Inertial fragment matching (conformer_generator.py:178-236).  Everything between the two reverse loops --
            # the per-sample context of the fragment to generate (inverse parallel-axis shift + 3x3 eigh), the inverse
            # coordinate transform and the assembly of z_known / fixed_mask -- runs on the device (mlcg_ifm_*): the first
            # loop's outputs never leave HBM.
            ff_x, ff_h = fixed_fragment
            n_ff = int(ff_x.size(0))
            from .mol_utils import _check_fragment_size
            _check_fragment_size(n_ff, min_n_nodes, max_n_nodes)
            eng = self.engine
            n_nodes = node_mask.sum(dim=(1, 2)).to(torch.int32)
            f_ctx, shift, rotation, n_gen = eng.ifm_context(ff_x, reference_context, self.context_norms, n_nodes)
            n_max_frag = max_n_nodes - n_ff
            eng.set_batch((n_nodes - n_ff).numpy(), n_max_frag)
            x_gen, cls_gen = eng.sample(f_ctx, gm.T, "forward", resample_steps, noise_tape=gm.noise_tape, seed=gm.seed)
            z_known, fixed_mask = eng.ifm_merge_inputs(x_gen, cls_gen, shift, rotation, ff_x, ff_h, max_n_nodes)
            x, h = gm.merge_fragments(node_mask, edge_mask, fixed_mask, ctx, z_known, ifm_diffusion_level,
                                      resample_steps, blend_power)
        else:
            z_known, fixed_mask = prepare_fragment(n_samples, fixed_fragment[0], fixed_fragment[1], max_n_nodes, min_n_nodes)
            x, h = gm.inpaint(node_mask, edge_mask, ctx, z_known, fixed_mask, resample_steps, blend_power)
        self.engine.check_finite("edm_samples")
        return x, h, node_mask

    @torch.no_grad()
    def generate_tensors(self, reference_context: torch.Tensor, n_atoms: int, n_samples: int = 10, variance: int = 2,
                         resample_steps: int = 0, **fragment_kwargs) -> Dict[str, torch.Tensor]:
        """The accelerated part of generate_conformers end to end: EDM samples -> GCN inputs (declared connectivity
        rule, DESIGN.md) -> AdjMatSeer -> bond orders.  Returns device tensors.

        PROVISIONAL `bonds` / `bond_logits`: coordinates and atom classes are the reference's (parity-tested), and
        AdjMatSeer itself is parity-tested on identical tensor inputs, but the inputs built here are NOT the ones the
        reference builds: it takes the 1st-order connectivity from RDKit's rdDetermineBonds.DetermineConnectivity and
        renumbers the atoms into SMILES output order (utils/mol_utils.py:110-126, 146-194) before the slot-dependent GCN
        (nodes_coord_fc couples the 42 slots); this path uses d <= 1.3 (Rcov_i + Rcov_j) and keeps generation order.  The
        bond orders a trained model gives for the same sample can therefore differ.  `generate_conformers` (RDKit
        canonicalisation, then AdjMatSeerB200) is the parity path for bonds."""
        x, h, node_mask = self.edm_sample_tensors(reference_context, n_samples, n_atoms + variance, n_atoms - variance,
                                                  resample_steps, **fragment_kwargs)
        n_nodes = node_mask.sum(dim=(1, 2)).long()
        cls = torch.where(h.sum(-1) > 0, h.argmax(-1), torch.full_like(h.argmax(-1), -1)).to(torch.int32)
        self.engine.set_batch(n_nodes.numpy(), x.size(1))
        el, dist, adj = self.engine.seer_inputs(x, cls)
        logits, bonds = self.engine.seer_forward(el, dist, adj, want_logits=True)
        return {"x": x, "atom_class": cls, "n_nodes": n_nodes, "elements": el, "dist_mat": dist, "adj_mat": adj,
                "bond_logits": logits, "bonds": bonds}

    def generate_sdf(self, reference_context: torch.Tensor, n_atoms: int, n_samples: int = 10, variance: int = 2,
                     resample_steps: int = 0, **fragment_kwargs) -> List[str]:
        """generate_tensors + an RDKit-free V2000 writer: one mol block per sample with the GCN's bond orders.  No
        sanitisation / hydrogens / MMFF (those are RDKit's, reference conformer_generator.py:357-368).  The bond orders
        are PROVISIONAL (see generate_tensors); every block says so in its comment line."""
        from .mol_utils import samples_to_sdf_blocks
        t = self.generate_tensors(reference_context, n_atoms, n_samples, variance, resample_steps, **fragment_kwargs)
        return samples_to_sdf_blocks(t["x"], t["atom_class"], t["bonds"], t["n_nodes"])

    def generate_stream(self, reference_context: torch.Tensor, n_atoms: int, n_samples: int, batch_size: int = 8192,
                        variance: int = 2, postprocess=None, n_workers: int = 8, seed: int = 0,
                        fixed_fragment: Optional[Tuple[torch.Tensor, torch.Tensor]] = None,
                        inertial_fragment_matching: bool = True, blend_power: int = 3, ifm_diffusion_level: int = 50):
        """Generates `n_samples` molecules in batches and post-processes batch k on a pool of CPU threads WHILE the GPU
        generates batch k + 1 (SURVEY.md 8f-3; `pipeline.GenerationPipeline`).  `postprocess(x (n,3), atom_class (n,),
        bonds (42,42), n, index)` -> result or None runs once per molecule; the default writes an RDKit-free V2000 block
        (provisional bond orders, see generate_tensors) -- where RDKit is installed pass a callable that builds the Mol and
        runs the reference's redefine_bonds + standardize_mol.  Yields one list of results per batch, in order.
        `fixed_fragment` and the IFM arguments are those of edm_sample_tensors (Engine.generate_fragment_host)."""
        import numpy as np

        from .mol_utils import _check_fragment_size
        from .pipeline import GenerationPipeline, engine_batches, sdf_postprocess
        lo, hi = max(n_atoms - variance, self.min_n_nodes), min(n_atoms + variance, self.max_n_nodes)
        if fixed_fragment is not None:
            _check_fragment_size(int(fixed_fragment[0].size(0)), lo, hi)
        g = torch.Generator().manual_seed(seed)
        sizes = torch.randint(lo, hi + 1, (n_samples,), generator=g).numpy().astype(np.int32)   # as prepare_edm_input
        ctx = normalise_context(reference_context, self.context_norms).numpy().reshape(1, 3)
        nn = [sizes[s:s + batch_size] for s in range(0, n_samples, batch_size)]
        cx = [np.tile(ctx, (len(b), 1)).astype(np.float32) for b in nn]
        gen = engine_batches(self.engine, nn, hi, cx, self.generative_model.T, seed, fixed_fragment,
                             inertial_fragment_matching, reference_context, self.context_norms, blend_power,
                             ifm_diffusion_level)
        pipe = GenerationPipeline(gen, postprocess or sdf_postprocess, n_workers=n_workers)
        yield from pipe.run(len(nn))

    @torch.no_grad()
    def generate_jobs(self, jobs: List[Dict], resample_steps: int = 0, blend_power: int = 3, ifm_diffusion_level: int = 50,
                      seed: int = 0, max_batch: int = 8192, keep_best: Optional[int] = None) -> List[Dict[str, torch.Tensor]]:
        """Many small generation jobs -- different references, atom counts and fixed fragments -- in few packed device
        calls (the GPU reaches its rate only with thousands of molecules per call).  A job is a dict:
          reference_context   raw principal moments (3)
          n_atoms, variance   atom counts uniform in [n_atoms - variance, n_atoms + variance] (variance default 2, clipped
                              to [min_n_nodes, max_n_nodes]), or
          n_nodes             explicit atom count of every sample
          n_samples           number of molecules (implied by n_nodes)
          fixed_fragment      optional (coordinates (n,3), one-hot (n,8)), as in edm_sample_tensors
          inertial_fragment_matching   default True
          job_id              default: the job's position in the list
          reference_conformer optional heavy-atom coordinates (n_ref,3), 3 <= n_ref <= 64, to score the molecules against
        An analogue job asks for molecules like a given one instead:
          parent_molecule     (coordinates (n,3), raw 0/1 one-hot (n,8)), the parent's n heavy atoms, 3 <= n <=
                              max_n_nodes; every sample has exactly these n atoms.  n_samples is required; n_atoms,
                              variance, n_nodes, fixed_fragment and inertial_fragment_matching cannot go with it
          fixed_atoms         optional distinct indices of at most n - 1 parent atoms, re-injected at every step as
                              merge_fragments re-injects a fragment (blend (1 - s/T)^blend_power, centre-of-mass alignment)
          diffusion_level     optional L in [1, T] (default `ifm_diffusion_level`): the parent is forward-diffused to level
                              L and denoised from there -- L = 1 gives the parent back, L = T a fresh sample
          reference_context   optional here: default the parent's own principal moments, get_context_shape of the centred
                              coordinates (as generate_conformers takes them from a reference conformer); another context
                              steers the analogues toward another shape
        The parent is centred on its mean before noising and the results are returned in its input frame.  Atom class 7
        (Br) is never emitted -- the decode reads 7 class channels -- and that holds for fixed atoms too.  Rows that
        keep_best returned can be fed back as parents: (x[k, :n], one_hot(atom_class[k, :n], 8)).
        Jobs are grouped by kind (plain / inpainting / inertial fragment matching / analogue, the last by (has fixed
        atoms, diffusion level)) and cut into calls of at most `max_batch` samples; the loop settings are shared.  A job's molecules depend only on `seed`, its job_id, its own
        fields and the shared settings (jobs.py), never on the other jobs or their order.  Returns one dict per job, in
        input order, of host tensors: x (n,N,3), atom_class (n,N) (-1 = padding), n_nodes (n,), bonds (n,42,42) (the
        provisional bond orders of generate_tensors), with N the job's own max atom count.

        The molecules of all jobs with a reference_conformer are scored on the GPU in one pass (ShapeScorer.evaluate_jobs,
        the tensor part of the reference's evaluate_samples), and their dicts gain shape_tanimoto (n,), best_orientation
        (n,), aligned_coords (n,N,3) and reference_coords (n_ref,3), each bit-identical to ShapeScorer.evaluate on that job.
        With `keep_best` = k (every job then needs a reference_conformer) each job keeps only its min(k, n) best molecules
        by shape_tanimoto, descending (NaN last, ties to the lower index), and gains sample_index: each row's position in
        the unfiltered job."""
        from .jobs import attach_scores, check_keep_best, flatten_jobs, run_packed, score_packed, split_jobs
        packed = flatten_jobs(jobs, seed, self.context_norms, self.min_n_nodes, self.max_n_nodes)
        check_keep_best(packed, keep_best)
        idx = np.arange(packed.ids.size)
        args = (self.engine, packed, idx, self.generative_model.T, resample_steps, blend_power, ifm_diffusion_level, seed,
                max_batch)
        if not packed.scored:
            return split_jobs(packed, *run_packed(*args, context_norms=self.context_norms))
        from .shape_similarity import ShapeScorer
        x, cls, bonds = run_packed(*args, device_out=True, context_norms=self.context_norms)
        scores = score_packed(ShapeScorer(self.engine), packed, idx, x)
        res = attach_scores(packed, split_jobs(packed, x, cls, bonds), *scores, keep_best)
        return [{k: v.cpu() for k, v in r.items()} for r in res]

    # ------------------------------------------------------------------------------------------------------------
    # RDKit-facing path, same signatures as the reference
    # ------------------------------------------------------------------------------------------------------------
    @staticmethod
    def _rdkit():
        try:
            from rdkit import Chem  # noqa: F401
            return Chem
        except ImportError as exc:
            raise ImportError("generate_conformers / edm_samples return RDKit Mol objects and need rdkit (the reference "
                              "depends on rdkit>=2023.9.5); use generate_tensors / edm_sample_tensors for the "
                              "accelerated path without RDKit") from exc

    @torch.no_grad()
    def edm_samples(self, reference_context: torch.Tensor, n_samples: int = 100, max_n_nodes: int = 32,
                    min_n_nodes: int = 25, resample_steps: int = 0, fixed_fragment=None,
                    inertial_fragment_matching: bool = True, blend_power: int = 3, ifm_diffusion_level: int = 50) -> List:
        """reference conformer_generator.py:126-266: list of RDKit Mol objects without bonds."""
        Chem = self._rdkit()
        frag = None
        if fixed_fragment is not None:
            ff = Chem.RemoveAllHs(fixed_fragment)
            from .mol_utils import symbols_to_one_hot
            frag = (torch.tensor(ff.GetConformer().GetPositions(), dtype=torch.float32),
                    symbols_to_one_hot([a.GetSymbol() for a in ff.GetAtoms()]))
        x, h, node_mask = self.edm_sample_tensors(reference_context, n_samples, max_n_nodes, min_n_nodes, resample_steps,
                                                  frag, inertial_fragment_matching, blend_power, ifm_diffusion_level)
        from .mol_utils import samples_to_xyz_blocks
        blocks = samples_to_xyz_blocks(x, h.argmax(-1), node_mask.sum(dim=(1, 2)).long())
        return [m for m in (Chem.MolFromXYZBlock(b) for b in blocks) if m is not None]

    @torch.no_grad()
    def generate_conformers(self, reference_conformer=None, n_samples: int = 10, variance: int = 2,
                            reference_context: torch.Tensor = None, n_atoms: int = None, optimise_geometry: bool = True,
                            resample_steps: int = 0, fixed_fragment=None, inertial_fragment_matching: bool = True,
                            blend_power: int = 3, ifm_diffusion_level: int = 50) -> List:
        """reference conformer_generator.py:268-368.  Argument validation is identical; the RDKit post-processing
        (canonicalise, redefine_bonds, standardize_mol) is delegated to the reference package when it is installed."""
        if reference_conformer:
            Chem = self._rdkit()
            ref = Chem.RemoveHs(reference_conformer)
            ref_n_atoms = ref.GetNumAtoms()
            coord = torch.tensor(ref.GetConformer().GetPositions(), dtype=torch.float32)
            ref_context, _ = get_context_shape(coord - coord.mean(dim=0))
        elif reference_context is not None:
            if n_atoms:
                ref_n_atoms = n_atoms
            else:
                raise ValueError("Reference Number of Atoms should be provided, when generating samples using context.")
            ref_context = reference_context
        else:
            raise ValueError(
                "Either a reference RDkit Mol object or context as torch.Tensor should be provided for generation.")
        self._rdkit()
        try:
            from mlconfgen.utils import prepare_adj_mat_seer_input, redefine_bonds, standardize_mol
        except ImportError as exc:
            raise ImportError("the RDKit post-processing of generate_conformers lives in the reference package "
                              "(mlconfgen.utils); install it next to rdkit, or use generate_tensors") from exc
        mols = self.edm_samples(ref_context, n_samples, ref_n_atoms + variance, ref_n_atoms - variance, resample_steps,
                                fixed_fragment, inertial_fragment_matching, blend_power, ifm_diffusion_level)
        el, dm, am, canon = prepare_adj_mat_seer_input(mols=mols, dimension=self.dimension, device=torch.device("cpu"))
        logits = self.adj_mat_seer(el, dm, am).to("cpu")
        out = []
        for i, adj in enumerate(logits):
            std = standardize_mol(mol=redefine_bonds(canon[i], adj), optimize_geometry=optimise_geometry)
            if std:
                out.append(std)
        return out

    forward = generate_conformers
    __call__ = generate_conformers
