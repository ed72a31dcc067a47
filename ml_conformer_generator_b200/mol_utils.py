"""Host-side tensor helpers that define the hot path's input / output layouts.

Mirrors the *tensor half* of the reference's `src/mlconfgen/utils/mol_utils.py` (same names, argument meaning and error
behaviour; file:line cited per function).  Everything that needs RDKit stays in the reference (SURVEY.md section 2,
rows 6-8); a fixed-column V2000 reader is provided so contexts / fragments can be taken from `.mol` files without it.
"""
from typing import Dict, List, Optional, Sequence, Tuple

import torch

from .config import ATOM_DECODER, DIMENSION, PERMITTED_ELEMENTS

_SYMBOL_TO_CLASS = {v: k for k, v in ATOM_DECODER.items()}


# ----------------------------------------------------------------------------------------------------------------
# masks / context
# ----------------------------------------------------------------------------------------------------------------
def prepare_masks(n_nodes: torch.Tensor, max_n_nodes: int, device: torch.device = torch.device("cpu")
                  ) -> Tuple[torch.Tensor, torch.Tensor]:
    """reference mol_utils.py:226-252 -- node_mask (B,N,1): first n_nodes[b] slots are 1; edge_mask (B*N*N,1):
    outer product of the node mask with a zero diagonal, rows ordered (b, i, j)."""
    counts = torch.as_tensor(n_nodes).reshape(-1).long()
    node = (torch.arange(max_n_nodes).unsqueeze(0) < counts.unsqueeze(1)).to(torch.float32)
    off_diag = 1.0 - torch.eye(max_n_nodes)
    edge = node.unsqueeze(2) * node.unsqueeze(1) * off_diag
    return node.unsqueeze(2).to(device), edge.reshape(-1, 1).to(device)


def counts_from_masks(node_mask: torch.Tensor, edge_mask: torch.Tensor = None) -> torch.Tensor:
    """Inverse of prepare_masks with validation: the CUDA path indexes atoms by count, so the masks must be exactly the
    prefix / outer-product form prepare_masks emits.  Raises ValueError otherwise (bit-exact mask contract)."""
    nm = node_mask.detach().to("cpu", torch.float32)
    if nm.dim() != 3 or nm.size(2) != 1:
        raise ValueError("node_mask must have shape (B, N, 1)")
    b, n, _ = nm.shape
    counts = nm.sum(dim=(1, 2)).round().long()
    expect, expect_edge = prepare_masks(counts, n)
    if not torch.equal(nm, expect):
        raise ValueError("node_mask is not a prefix mask (first n_nodes[b] slots set), as prepare_masks emits")
    if edge_mask is not None:
        em = edge_mask.detach().to("cpu", torch.float32).reshape(-1, 1)
        if em.shape != expect_edge.shape or not torch.equal(em, expect_edge):
            raise ValueError("edge_mask is not outer(node_mask, node_mask) with a zero diagonal")
    if int(counts.min()) < 1:
        raise ValueError("every sample needs at least one atom")
    return counts


def prepare_edm_input(n_samples: int, reference_context: torch.Tensor, context_norms: Dict[str, torch.Tensor],
                      min_n_nodes: int, max_n_nodes: int, device: torch.device = torch.device("cpu")
                      ) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """reference mol_utils.py:255-295 -- sizes ~ randint(min, max+1) from the global CPU generator, masks, and the
    normalised context broadcast over real atoms."""
    sizes = torch.randint(min_n_nodes, max_n_nodes + 1, (n_samples,))
    node_mask, edge_mask = prepare_masks(sizes, max_n_nodes, device)
    normed = normalise_context(reference_context, context_norms).to(device)
    ctx = normed.view(1, 1, 3).expand(n_samples, max_n_nodes, 3) * node_mask
    return node_mask, edge_mask, ctx


def normalise_context(reference_context: torch.Tensor, context_norms: Dict[str, torch.Tensor]) -> torch.Tensor:
    """(context - mean) / mad, reference mol_utils.py:283-285."""
    mean = torch.as_tensor(context_norms["mean"], dtype=torch.float32)
    mad = torch.as_tensor(context_norms["mad"], dtype=torch.float32)
    return (torch.as_tensor(reference_context, dtype=torch.float32).cpu() - mean) / mad


def context_rows(context: torch.Tensor, node_mask: torch.Tensor) -> torch.Tensor:
    """(B,N,3) masked per-atom context (reference layout) -> (B,3) per-sample context (library layout).  The rows of a
    sample must be identical over its real atoms, as prepare_edm_input / ifm_prepare_gen_fragment_context build them."""
    ctx = context.detach().to("cpu", torch.float32)
    first = ctx[:, 0, :]
    nm = node_mask.detach().to("cpu", torch.float32)
    if not torch.equal(ctx, first.unsqueeze(1) * nm):
        raise ValueError("context must be one 3-vector per sample broadcast over its real atoms")
    return first.contiguous()


# ----------------------------------------------------------------------------------------------------------------
# moments of inertia / principal frame
# ----------------------------------------------------------------------------------------------------------------
def get_moment_of_inertia_tensor(coord: torch.Tensor, weights: torch.Tensor) -> torch.Tensor:
    """reference mol_utils.py:60-85.  As in the reference, `weights` only enters the diagonal."""
    x, y, z = coord[:, 0], coord[:, 1], coord[:, 2]
    diag = torch.stack([(weights * (y * y + z * z)).sum(), (weights * (x * x + z * z)).sum(),
                        (weights * (x * x + y * y)).sum()])
    xy, xz, yz = -(x * y).sum(), -(x * z).sum(), -(y * z).sum()
    m = torch.zeros(3, 3, dtype=torch.float32)
    m[0, 0], m[1, 1], m[2, 2] = diag[0], diag[1], diag[2]
    m[0, 1] = m[1, 0] = xy
    m[0, 2] = m[2, 0] = xz
    m[1, 2] = m[2, 1] = yz
    return m


def get_context_shape(coord: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """reference mol_utils.py:88-107 -- principal moments (unit masses) and the coordinates in the principal frame."""
    coord = coord.to(torch.float32)
    ones = torch.ones(coord.size(0))
    _, vecs = torch.linalg.eigh(get_moment_of_inertia_tensor(coord, ones))
    rotated = coord @ vecs
    return torch.diag(get_moment_of_inertia_tensor(rotated, ones)), rotated


def shift_moi_to_com_batch(moi_origin: torch.Tensor, r_coms: torch.Tensor, masses: torch.Tensor) -> torch.Tensor:
    """reference mol_utils.py:527-550 -- inverse parallel-axis theorem, batched."""
    b = r_coms.size(0)
    r = r_coms.view(b, 3, 1)
    shift = masses.view(b, 1, 1) * ((r_coms ** 2).sum(1).view(b, 1, 1) * torch.eye(3).expand(b, 3, 3)
                                    - r @ r.transpose(1, 2))
    return moi_origin - shift


def inverse_coord_transform(coord: torch.Tensor, shift: torch.Tensor, rotation: torch.Tensor) -> torch.Tensor:
    """reference mol_utils.py:508-524 -- rotate by R^T then translate by -shift."""
    return torch.bmm(coord, rotation.transpose(1, 2)) - shift.view(-1, 1, 3)


# ----------------------------------------------------------------------------------------------------------------
# fragments
# ----------------------------------------------------------------------------------------------------------------
def _check_fragment_size(n_frag: int, min_n_nodes: int, max_n_nodes: int):
    # same messages as reference mol_utils.py:320-327 / 400-407
    if n_frag >= min_n_nodes:
        raise ValueError("Fragment must contain fewer atoms than minimum generation size.")
    if n_frag >= max_n_nodes:
        raise ValueError("Fragment has more atoms than the maximum number of atoms requested.")


def prepare_fragment(n_samples: int, fragment_x: torch.Tensor, fragment_h: torch.Tensor, max_n_nodes: int = DIMENSION,
                     min_n_nodes: int = 15, device: torch.device = torch.device("cpu")
                     ) -> Tuple[torch.Tensor, torch.Tensor]:
    """reference mol_utils.py:298-342 with the RDKit step (ifm_get_xh_from_fragment) factored out: takes the fragment's
    heavy-atom coordinates (n,3) and raw 0/1 one-hot classes (n,8).  Returns z_known (B,N,11), fixed_mask (B,N,1)."""
    n = fragment_x.size(0)
    _check_fragment_size(n, min_n_nodes, max_n_nodes)
    z = torch.zeros(n_samples, max_n_nodes, 11)
    z[:, :n, :3] = fragment_x.to(torch.float32)
    z[:, :n, 3:] = fragment_h.to(torch.float32)
    fixed = torch.zeros(n_samples, max_n_nodes, 1)
    fixed[:, :n] = 1.0
    return z.to(device), fixed.to(device)


def ifm_prepare_gen_fragment_context(fixed_fragment_x: torch.Tensor, reference_context: torch.Tensor,
                                     context_norms: Dict[str, torch.Tensor], n_nodes: torch.Tensor, max_n_nodes: int,
                                     min_n_nodes: int, device: torch.device = torch.device("cpu")):
    """reference mol_utils.py:373-457 -- per-sample context of the fragment still to be generated: reference MOI minus
    the fixed fragment's MOI, shifted to the generated fragment's centre of mass, diagonalised."""
    b = n_nodes.size(0)
    n_ff = fixed_fragment_x.size(0)
    _check_fragment_size(n_ff, min_n_nodes, max_n_nodes)
    ffx = fixed_fragment_x.detach().cpu().to(torch.float32)
    moi_gen_origin = (torch.diag(torch.as_tensor(reference_context, dtype=torch.float32).cpu())
                      - get_moment_of_inertia_tensor(ffx, torch.ones(n_ff))).unsqueeze(0).repeat(b, 1, 1)
    n_gen = n_nodes.detach().cpu().view(b, 1).float() - n_ff
    shift = (n_ff * ffx.mean(dim=0).view(1, 3)) / n_gen
    frag_context, rotation = torch.linalg.eigh(shift_moi_to_com_batch(moi_gen_origin, shift, n_gen))
    normed = (frag_context - torch.as_tensor(context_norms["mean"], dtype=torch.float32)) / torch.as_tensor(
        context_norms["mad"], dtype=torch.float32)
    n_max_frag = max_n_nodes - n_ff
    node_mask, edge_mask = prepare_masks(n_gen.long(), n_max_frag, device)
    ctx = normed.to(device).unsqueeze(1).repeat(1, n_max_frag, 1) * node_mask
    return node_mask, edge_mask, ctx, shift.to(device), rotation.to(device)


def ifm_moi_prologue(fixed_fragment_x: torch.Tensor, reference_context: torch.Tensor
                     ) -> Tuple[torch.Tensor, torch.Tensor]:
    """Batch-independent prologue of ifm_prepare_gen_fragment_context, in float32 as there (reference mol_utils.py:396-411):
    moi_gen_origin (3,3) = diag(reference_context) - MOI(fixed fragment), and ff_weighted_com (3) = n_ff * mean(fixed
    fragment coordinates).  The host inputs of mlcg_ifm_context / mlcg_generate_fragment."""
    ffx = fixed_fragment_x.detach().to("cpu", torch.float32)
    n_ff = int(ffx.size(0))
    moi0 = (torch.diag(torch.as_tensor(reference_context, dtype=torch.float32).cpu())
            - get_moment_of_inertia_tensor(ffx, torch.ones(n_ff))).contiguous()
    com = (n_ff * ffx.mean(dim=0)).to(torch.float32).contiguous()
    return moi0, com


def ifm_prepare_fragments_for_merge(fixed_fragment_x: torch.Tensor, fixed_fragment_h: torch.Tensor,
                                    gen_fragments_x: torch.Tensor, gen_fragments_h: torch.Tensor, max_n_nodes: int,
                                    device: torch.device = torch.device("cpu")):
    """reference mol_utils.py:460-505 -- fixed fragment first, generated fragment after it; fixed_mask over the first
    n_ff atoms."""
    b = gen_fragments_x.size(0)
    n_ff = fixed_fragment_x.size(0)
    x = torch.cat([fixed_fragment_x.to(device).unsqueeze(0).repeat(b, 1, 1), gen_fragments_x.to(device)], dim=1)
    h = torch.cat([fixed_fragment_h.to(device).unsqueeze(0).repeat(b, 1, 1).to(gen_fragments_h.dtype),
                   gen_fragments_h.to(device)], dim=1)
    fixed = torch.zeros(b, max_n_nodes, 1, device=device)
    fixed[:, :n_ff] = 1.0
    return torch.cat([x, h.to(x.dtype)], dim=2), fixed


# ----------------------------------------------------------------------------------------------------------------
# files / outputs
# ----------------------------------------------------------------------------------------------------------------
def read_mol_heavy_atoms(path: str) -> Tuple[List[str], torch.Tensor]:
    """Fixed-column V2000 molfile reader (counts line at row 4; x, y, z in columns 0-30, symbol in 31-34).  Returns the
    heavy-atom symbols and coordinates (n,3) -- what RemoveHs + GetPositions give the reference
    (conformer_generator.py:302-307)."""
    with open(path) as fh:
        lines = fh.read().splitlines()
    n_atoms = int(lines[3][0:3])
    symbols, xyz = [], []
    for line in lines[4:4 + n_atoms]:
        sym = line[31:34].strip()
        if sym == "H":
            continue
        symbols.append(sym)
        xyz.append([float(line[0:10]), float(line[10:20]), float(line[20:30])])
    return symbols, torch.tensor(xyz, dtype=torch.float32)


def symbols_to_one_hot(symbols: Sequence[str]) -> torch.Tensor:
    """Raw 0/1 one-hot over the 8 atom classes (reference molgraph one_hot_elements_encoding; utils/config.py:9-18)."""
    idx = []
    for s in symbols:
        if s not in _SYMBOL_TO_CLASS:
            raise ValueError("element %s is not permitted (allowed: %s)" % (s, sorted(_SYMBOL_TO_CLASS)))
        idx.append(_SYMBOL_TO_CLASS[s])
    return torch.nn.functional.one_hot(torch.tensor(idx), 8).to(torch.float32)


def reference_context_from_mol_file(path: str) -> Tuple[torch.Tensor, int, torch.Tensor]:
    """Context (principal moments), heavy-atom count and centred coordinates of a reference conformer, as
    generate_conformers computes them (reference conformer_generator.py:302-313)."""
    _, xyz = read_mol_heavy_atoms(path)
    centred = xyz - xyz.mean(dim=0)
    ctx, _ = get_context_shape(centred)
    return ctx, xyz.size(0), centred


def samples_to_xyz_blocks(x: torch.Tensor, atom_class: torch.Tensor, n_nodes: torch.Tensor) -> List[str]:
    """XYZ text blocks in the format the reference feeds to RDKit (mol_utils.py:39-51), built without RDKit."""
    x = x.detach().cpu()
    cls = atom_class.detach().cpu()
    out = []
    for b in range(x.size(0)):
        n = int(n_nodes[b])
        rows = ["%s %.9f %.9f %.9f" % (ATOM_DECODER[int(cls[b, i])], x[b, i, 0], x[b, i, 1], x[b, i, 2]) for i in range(n)]
        out.append("%d\n\n%s\n" % (n, "\n".join(rows)))
    return out


def bond_orders_from_logits(logits: torch.Tensor) -> torch.Tensor:
    """(B,42,42,5) AdjMatSeer logits -> (B,42,42) bond order 0..4 for i > j (lower triangle, zero diagonal), as the
    reference's redefine_bonds does per molecule (mol_utils.py:210-211)."""
    order = torch.argmax(logits, dim=-1)
    return torch.tril(order, diagonal=-1)


PROVISIONAL_BONDS_NOTE = ("bond orders PROVISIONAL: AdjMatSeer fed with distance-rule connectivity in generation order, "
                          "not RDKit DetermineConnectivity + SMILES-order atoms")


def samples_to_sdf_blocks(x: torch.Tensor, atom_class: torch.Tensor, bonds: torch.Tensor, n_nodes: torch.Tensor,
                          names: Optional[Sequence[str]] = None, comment: str = PROVISIONAL_BONDS_NOTE) -> List[str]:
    """V2000 mol blocks ("...M  END\n$$$$\n") from the accelerated path's tensors, without RDKit.

    x (B,N,3) coordinates, atom_class (B,N) (-1 = padding), bonds (B,D,D) bond order per pair as mlcg_seer_forward /
    bond_orders_from_logits return it (only i > j is read; 1 single, 2 double, 3 triple, 4 aromatic -- the reference's
    bond_type_dict, mol_utils.py:10-15).  This is the wire format of the reference's results (Chem.MolToMolBlock in
    cheminformatics/pipeline.py:88) minus RDKit's sanitisation: no implicit hydrogens, no charge / valence fix-up.
    `comment` goes to the block's comment line (line 3): by default it marks the bond orders of the RDKit-free path as
    provisional -- AdjMatSeer is slot-dependent and the reference feeds it RDKit connectivity with atoms renumbered into
    SMILES output order (utils/mol_utils.py:110-126, 146-194), which cannot be reproduced without RDKit."""
    x = x.detach().cpu()
    cls = atom_class.detach().cpu()
    bo = bonds.detach().cpu()
    out = []
    for b in range(x.size(0)):
        n = int(n_nodes[b])
        if n > 999:
            raise ValueError("V2000 mol blocks hold at most 999 atoms")
        pairs = [(i, j, int(bo[b, i, j])) for i in range(n) for j in range(i) if int(bo[b, i, j]) != 0]
        lines = [names[b] if names is not None else "mlcg_%d" % b, "  ml_conformer_generator_b200", comment[:200],
                 "%3d%3d  0  0  0  0  0  0  0  0999 V2000" % (n, len(pairs))]
        for i in range(n):
            lines.append("%10.4f%10.4f%10.4f %-3s 0  0  0  0  0  0  0  0  0  0  0  0"
                         % (float(x[b, i, 0]), float(x[b, i, 1]), float(x[b, i, 2]), ATOM_DECODER[int(cls[b, i])]))
        for i, j, order in pairs:
            lines.append("%3d%3d%3d  0" % (j + 1, i + 1, order))
        lines += ["M  END", "$$$$"]
        out.append("\n".join(lines) + "\n")
    return out


def read_mol_block(block: str) -> Tuple[List[str], torch.Tensor, List[Tuple[int, int, int]]]:
    """Inverse of samples_to_sdf_blocks for one V2000 block: symbols, coordinates (n,3), bonds [(a, b, order)] with
    0-based atom indices."""
    lines = block.splitlines()
    n_atoms, n_bonds = int(lines[3][0:3]), int(lines[3][3:6])
    symbols = [ln[31:34].strip() for ln in lines[4:4 + n_atoms]]
    xyz = torch.tensor([[float(ln[0:10]), float(ln[10:20]), float(ln[20:30])] for ln in lines[4:4 + n_atoms]],
                       dtype=torch.float32).view(-1, 3)
    bonds = [(int(ln[0:3]) - 1, int(ln[3:6]) - 1, int(ln[6:9])) for ln in lines[4 + n_atoms:4 + n_atoms + n_bonds]]
    return symbols, xyz, bonds


def atomic_numbers(atom_class: torch.Tensor) -> torch.Tensor:
    table = torch.tensor(PERMITTED_ELEMENTS, dtype=torch.long)
    return torch.where(atom_class >= 0, table[atom_class.clamp_min(0).long()], torch.zeros_like(atom_class, dtype=torch.long))
