"""CPU: host-side mirrors of the reference's tensor helpers against golden vectors produced by the reference."""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN, golden
from ml_conformer_generator_b200 import mol_utils as M
from ml_conformer_generator_b200.config import CONTEXT_NORMS

NORMS = {k: torch.tensor(v) for k, v in CONTEXT_NORMS.items()}


def test_context_of_demo_molecules():
    g = golden("host_utils")
    for name, expect in (("ceyyag", [50.5897, 105.3132, 133.5223]), ("yibfeu", [89.8693, 210.7831, 217.7827])):
        xyz = torch.from_numpy(g[name + "_xyz"])
        ctx, rot = M.get_context_shape(xyz - xyz.mean(dim=0))
        assert np.allclose(ctx.numpy(), g[name + "_context"], rtol=1e-5)
        assert np.allclose(ctx.numpy(), expect, rtol=1e-4)  # SURVEY.md 8d known answers
        assert np.allclose(np.abs(rot.numpy()), np.abs(g[name + "_rotated"]), atol=1e-3)


def test_prepare_edm_input_matches_reference_rng():
    g = golden("host_utils")
    torch.manual_seed(123)
    nm, em, ctx = M.prepare_edm_input(6, torch.from_numpy(g["ceyyag_context"]), NORMS, 15, 19)
    assert np.array_equal(nm.numpy(), g["edm_in_node_mask"]) and np.array_equal(em.numpy(), g["edm_in_edge_mask"])
    assert np.allclose(ctx.numpy(), g["edm_in_context"], atol=1e-7)
    assert torch.equal(M.counts_from_masks(nm, em), nm.sum(dim=(1, 2)).long())
    assert np.allclose(M.context_rows(ctx, nm).numpy(), g["edm_in_context"][:, 0, :])


def test_mask_validation():
    nm, em = M.prepare_masks(torch.tensor([3, 5]), 5)
    bad = nm.clone()
    bad[0, 0, 0], bad[0, 4, 0] = 0.0, 1.0  # not a prefix mask
    with pytest.raises(ValueError):
        M.counts_from_masks(bad, em)
    bad_e = em.clone()
    bad_e[1] = 0.0
    with pytest.raises(ValueError):
        M.counts_from_masks(nm, bad_e)
    with pytest.raises(ValueError):
        M.counts_from_masks(torch.zeros(2, 5, 1))  # empty samples


def test_inertial_fragment_matching_helpers():
    g = golden("host_utils")
    ff_x = torch.from_numpy(g["ifm_ff_x"])
    nm, em, ctx, shift, rot = M.ifm_prepare_gen_fragment_context(ff_x, torch.from_numpy(g["yibfeu_context"]), NORMS,
                                                                 torch.from_numpy(g["ifm_n_nodes"]), 25, 21)
    assert np.array_equal(nm.numpy(), g["ifm_node_mask"]) and np.array_equal(em.numpy(), g["ifm_edge_mask"])
    assert np.allclose(ctx.numpy(), g["ifm_context"], atol=2e-5)
    assert np.allclose(shift.numpy(), g["ifm_shift"], atol=1e-6)
    # eigenvectors are defined up to sign
    assert np.allclose(np.abs(rot.numpy()), np.abs(g["ifm_rotation"]), atol=1e-4)
    inv = M.inverse_coord_transform(torch.from_numpy(g["ifm_xg"]), torch.from_numpy(g["ifm_shift"]),
                                    torch.from_numpy(g["ifm_rotation"]))
    assert np.allclose(inv.numpy(), g["ifm_inv"], atol=1e-6)
    zk, fm = M.ifm_prepare_fragments_for_merge(ff_x, torch.from_numpy(g["ifm_ff_h"]), inv, torch.from_numpy(g["ifm_hg"]), 25)
    assert np.allclose(zk.numpy(), g["ifm_z_known"], atol=1e-6) and np.array_equal(fm.numpy(), g["ifm_fixed_mask"])
    with pytest.raises(ValueError, match="fewer atoms than minimum"):
        M.ifm_prepare_gen_fragment_context(ff_x, torch.from_numpy(g["yibfeu_context"]), NORMS, torch.tensor([9]), 25, 8)


def test_prepare_fragment_and_symbols():
    g = golden("host_utils")
    sym = [str(s) for s in g["frag_yibfeu_symbols"]]
    h = M.symbols_to_one_hot(sym)
    assert h.shape == (8, 8) and int(h[0].argmax()) == 6 and int(h[2].argmax()) == 0  # Cl = class 6, C = class 0
    zk, fm = M.prepare_fragment(3, torch.from_numpy(g["ifm_ff_x"]), h, 25, 21)
    assert zk.shape == (3, 25, 11) and float(zk[:, 8:].abs().max()) == 0 and float(fm[:, :8].min()) == 1
    assert float(zk[0, 0, 3 + 6]) == 1.0  # raw 0/1 one-hot, not divided by the norm value (reference mol_utils.py:329-335)
    with pytest.raises(ValueError, match="more atoms than the maximum"):
        M.prepare_fragment(1, torch.zeros(8, 3), h, 8, 20)
    with pytest.raises(ValueError):
        M.symbols_to_one_hot(["Si"])


def test_v2000_reader_on_reference_assets():
    """The heavy-atom rows of the reference's demo molfiles ceyyag.mol and yibfeu.mol, stored under tests/golden/, read
    back to the coordinates and context the reference computed from the originals."""
    g = golden("host_utils")
    sym, xyz = M.read_mol_heavy_atoms(os.path.join(GOLDEN, "ceyyag.mol"))
    assert len(sym) == 17 and sym == [str(s) for s in g["ceyyag_symbols"]] and np.allclose(xyz.numpy(), g["ceyyag_xyz"])
    ctx, n, _ = M.reference_context_from_mol_file(os.path.join(GOLDEN, "yibfeu.mol"))
    assert n == 23 and np.allclose(ctx.numpy(), g["yibfeu_context"], rtol=1e-5)


def test_xyz_blocks():
    x = torch.tensor([[[0.0, 1.0, 2.0], [3.0, 4.0, 5.5], [0, 0, 0]]])
    blocks = M.samples_to_xyz_blocks(x, torch.tensor([[0, 6, -1]]), torch.tensor([2]))
    assert blocks[0].splitlines()[0] == "2" and blocks[0].splitlines()[3].startswith("Cl 3.000000000 4.000000000 5.5")


def test_sdf_blocks_round_trip():
    """samples_to_sdf_blocks writes V2000 blocks that read back to the same atoms, coordinates (4 decimals) and bonds;
    the reference's demo molfile survives read -> write -> read as well."""
    x = torch.tensor([[[0.0, 1.0, 2.0], [1.2345678, -4.0, 5.5], [0.5, 0.25, -0.125], [9, 9, 9]]])
    cls = torch.tensor([[0, 2, 6, -1]])
    bonds = torch.zeros(1, 42, 42, dtype=torch.int32)
    bonds[0, 1, 0] = 2   # only the lower triangle is read
    bonds[0, 2, 1] = 4
    bonds[0, 0, 2] = 3   # upper triangle: ignored
    blocks = M.samples_to_sdf_blocks(x, cls, bonds, torch.tensor([3]), names=["probe"])
    assert blocks[0].startswith("probe\n") and blocks[0].endswith("M  END\n$$$$\n")
    sym, xyz, bl = M.read_mol_block(blocks[0])
    assert sym == ["C", "O", "Cl"] and bl == [(0, 1, 2), (1, 2, 4)]
    assert np.allclose(xyz.numpy(), x[0, :3].numpy(), atol=5e-5)
    logits = torch.zeros(1, 42, 42, 5)
    logits[0, 1, 0, 2] = 1.0
    logits[0, 0, 1, 2] = 1.0
    logits[0, 5, 5, 3] = 1.0   # diagonal is dropped
    bo = M.bond_orders_from_logits(logits)
    assert int(bo[0, 1, 0]) == 2 and int(bo.sum()) == 2



def test_shape_host_helpers_match_oracle():
    """Host-side pieces of the GPU shape scorer (grid axes incl. the reference's per-atom min/max quirk, orientation
    matrices, alpha) against the oracle restatement of shape_similarity.py -- no device needed."""
    from oracle import shape_oracle as S
    import importlib
    H = importlib.import_module("ml_conformer_generator_b200.shape_similarity")
    g = golden("shape")
    ref_pts = torch.from_numpy(g["ref_pts"])
    cand = torch.from_numpy(g["pts"][0, : int(g["n_nodes"][0])])
    ax = H.grid_axes(ref_pts)
    for k, a in enumerate(S.grid_axes(ref_pts, cand)):
        assert torch.equal(ax[k], a)
    assert abs(H.get_alpha() - S.ALPHA) < 1e-15
    mats = H.orientation_matrices()
    assert torch.equal(mats[0], torch.eye(3))
    for k, ang in enumerate(S.orientations()[1:]):
        assert torch.equal(cand @ mats[k + 1], S.rotate(cand, ang)) or torch.allclose(cand @ mats[k + 1], S.rotate(cand, ang), atol=1e-6)
    with pytest.raises(ValueError):
        H.grid_axes(ref_pts[:2])
