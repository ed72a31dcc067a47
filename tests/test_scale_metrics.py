"""CPU: the per-element GEMM check and the per-molecule eps check of test_gpu_scale.py catch a corruption confined to one
128-row tile of a 129 029-row GEMM output or to one molecule of an 8192-molecule batch, which a single rel-L2 over the
whole output at the bounds of test_gpu_parity.py lets through."""
import numpy as np
import torch

from conftest import rel_l2
from oracle import edm_oracle as O
from test_gpu_scale import C3_SIZES, N_MAX, TC_VS_FP32, gemm_error_bound, gemm_worst, rel_l2_per_molecule, representable


def test_gemm_check_flags_one_corrupt_tile():
    g = torch.Generator().manual_seed(0)
    M, N, K = 129029, 32, 32
    a = torch.randn(M, K, generator=g)
    w = torch.randn(N, K, generator=g) / K ** 0.5
    b = torch.randn(N, generator=g)
    a64, w64, b64 = a.double(), w.double(), b.double()
    ref = torch.addmm(b64, a64, w64.t())
    bound = gemm_error_bound(a64, w64, b64, "tf32")
    # what a correct tf32 kernel may return: operands truncated to tf32 (relative error < 2^-10), fp32 result
    c = (torch.addmm(b64, representable(a, "tf32").double(), representable(w, "tf32").double().t())).float()
    assert gemm_worst(c, ref, bound)[0] <= 1.0
    blk = 517
    c[blk * 128:(blk + 1) * 128] *= 1 + 1e-2
    worst, row, _ = gemm_worst(c, ref, bound)
    assert worst > 1.0 and row // 128 == blk
    assert rel_l2(c, ref) < 2e-3  # test_tc_gemm's tf32 bound misses it


def test_molecule_check_flags_one_corrupt_molecule():
    g = torch.Generator().manual_seed(1)
    n_nodes = torch.from_numpy(C3_SIZES.astype(np.int64))
    nm, _ = O.prepare_masks(n_nodes, N_MAX)
    ref = torch.randn(len(C3_SIZES), N_MAX, 11, generator=g) * nm
    out = ref + 3e-4 * torch.randn(ref.shape, generator=g) * nm  # tensor-core-like rounding noise
    assert float(rel_l2_per_molecule(out, ref).max()) < TC_VS_FP32["tf32"]
    mol = 4321
    out[mol] *= 1 + 1e-2
    err = rel_l2_per_molecule(out, ref)
    assert float(err.max()) > TC_VS_FP32["tf32"] and int(torch.argmax(err)) == mol
    assert rel_l2(out, ref) < 1e-3  # the whole-batch tf32 / fp16 bound of test_gpu_parity.py misses it
