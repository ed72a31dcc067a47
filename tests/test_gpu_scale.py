"""GPU: the node GEMM, the EGNN forward and the AdjMatSeer GCN at the batch sizes of the benchmark (config C3: 8192 molecules
of 15-39 atoms; C2: 1024 x 39 atoms) against float64 references.

Several code paths only run at these sizes: the persistent k_tc_gemm processes more than one tile per CTA (ring-phase
counters, accumulator hand-over, double-buffered bias, reuse of the staging slot), the fp32 SIMT path cuts the edge list
into chunks of 49 152 rows, and the GCN splits batches into chunks of 3072 molecules.  A single rel-L2 over a batch of
8192 molecules hides one wrong molecule or one wrong 128-row tile, so every check here is per element (GEMM) or per
molecule (EGNN, GCN), and reports where the worst error occurred."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from ml_conformer_generator_b200.config import CONTEXT_NORMS
from oracle import edm_oracle as O

pytestmark = pytest.mark.gpu

N_MAX = 39
ONNX_CONTEXT = [53.6424, 108.3042, 151.4399]
C3_SIZES = np.random.RandomState(5).randint(15, 40, 65536).astype(np.int32)[:8192]  # bench.py workload("C3")
TOL = {"fp32": 2e-5, "tf32": 1e-3, "fp16": 1e-3, "bf16": 2e-2}        # per molecule against the float64 oracle
TC_VS_FP32 = {"tf32": 2e-3, "fp16": 2e-3, "bf16": 3e-2}              # per molecule, tensor-core modes against fp32 CUDA
SEER_TOL = {"fp32": 1e-4, "tf32": 2e-3}                              # per molecule, logits against the float64 oracle
SIMT_CHUNK_ROWS = 49152                                              # mlcg_set_batch: edge rows per fp32 SIMT chunk
SEER_CHUNK = 3072                                                    # mlcg_seer_forward: molecules per GCN chunk
TILE_M = 128


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


# ---------------------------------------------------------------------------------------------------------------
# metrics (also exercised without a GPU by test_scale_metrics.py)
# ---------------------------------------------------------------------------------------------------------------
UNIT_ROUNDOFF = {"tf32": 2.0 ** -10, "bf16": 2.0 ** -8, "fp16": 2.0 ** -11}


def gemm_error_bound(a, w, b, mode, exact_operands=False):
    """Elementwise bound on |C - (A.W^T + b)| for C computed from `mode`-rounded operands with fp32 accumulation:
    gamma * ((|A|.|W|^T)_ij + |b_j|), gamma = 2u + K 2^-23 (one rounding of each operand, K fp32 additions and the bias
    add, each allowed a truncation's error).  fp16 adds the absolute error of operands that round to subnormals (at most
    2^-25 each): 2^-25 * (sum_k |a_ik| + sum_k |w_jk|).  `exact_operands`: the operands are exact in the mode's format, so
    only the accumulation error K 2^-23 remains.  Inputs in float64."""
    K = a.shape[1]
    gamma = (0 if exact_operands else 2 * UNIT_ROUNDOFF[mode]) + K * 2.0 ** -23
    bound = gamma * (a.abs() @ w.abs().t() + b.abs())
    if mode == "fp16" and not exact_operands:
        bound += 2.0 ** -25 * (a.abs().sum(1, keepdim=True) + w.abs().sum(1))
    return bound


def gemm_worst(c, ref, bound):
    """(largest |c - ref| / bound, its row, its column)."""
    excess = (c.double() - ref).abs() / bound
    k = int(torch.argmax(excess))
    return float(excess.view(-1)[k]), k // c.shape[1], k % c.shape[1]


def representable(x, mode):
    """x rounded to a float32 value that the mode's operand format holds exactly."""
    if mode == "tf32":
        return (x.view(torch.int32) & ~0x1FFF).view(torch.float32)
    return x.to(torch.bfloat16 if mode == "bf16" else torch.float16).float()


def rel_l2_per_molecule(out, ref):
    """Relative L2 error of every molecule (leading axis), in float64."""
    out, ref = out.double(), ref.double()
    return (out - ref).flatten(1).norm(dim=1) / ref.flatten(1).norm(dim=1).clamp_min(1e-30)


# ---------------------------------------------------------------------------------------------------------------
# A. generic GEMM with many tiles per CTA
# ---------------------------------------------------------------------------------------------------------------
# name -> (M, N, K, BN) as a function of the SM count.  K = 420 is not a multiple of the 32 / 64-element K chunk; N = 420
# leaves a column tail inside a 448-wide tile; K = 64 gives n_kc < NSTAGE (ring slot 0 never carries operands); K = 896
# and 2048 give chunk counts that are not multiples of NSTAGE, so the ring phases of a CTA's tiles drift against each other.
GEMM_SHAPES = {
    "tiles=sms,K=420": lambda s: (s * TILE_M - 37, 448, 420, 448),
    "tiles=sms+1,N=420": lambda s: ((s + 1) * TILE_M - 1, 420, 448, 448),
    "tiles~4sms,K=896": lambda s: (2 * s * TILE_M + 200, 896, 896, 448),
    "tiles~4sms,K=64": lambda s: (2 * s * TILE_M + 77, 512, 64, 256),
    "tiles~54sms,seer": lambda s: (129029, 2048, 2048, 256),
}
_GEMM_REF = {}


def _gemm_problem(name, sms):
    """Seeded inputs and float64 reference of one shape (the last shape's are kept for the next mode)."""
    if name not in _GEMM_REF:
        _GEMM_REF.clear()
        torch.cuda.empty_cache()
        M, N, K, bn = GEMM_SHAPES[name](sms)
        g = torch.Generator(device="cuda").manual_seed(M + N + K)
        a = torch.randn(M, K, device="cuda", generator=g)
        w = torch.randn(N, K, device="cuda", generator=g) / K ** 0.5
        b = torch.randn(N, device="cuda", generator=g)
        a64, w64, b64 = a.double(), w.double(), b.double()
        ref = torch.addmm(b64, a64, w64.t())
        _GEMM_REF[name] = (M, N, K, bn, a, w, b, a64, w64, b64, ref)
    return _GEMM_REF[name]


@pytest.mark.parametrize("mode", ["tf32", "bf16", "fp16"])
@pytest.mark.parametrize("name", list(GEMM_SHAPES))
def test_gemm_many_tiles_per_cta(engines, name, mode):
    """Every element within the rounding bound, for fp32 operands and -- a ~10-30x tighter bound that leaves only the
    accumulation error -- for operands the mode's format holds exactly."""
    sms = _sms()
    M, N, K, bn, a, w, b, a64, w64, b64, ref = _gemm_problem(name, sms)
    n_tiles = -(-M // TILE_M) * -(-N // bn)
    grid = min(n_tiles, sms)
    if name.startswith("tiles=sms,"):
        assert n_tiles == sms
    else:
        assert n_tiles > grid, "the shape must give some CTA a second tile"
    e = engines(mode)
    for operands in ("fp32", "representable"):
        if operands == "representable":
            a, w = representable(a, mode), representable(w, mode)
            a64, w64 = a.double(), w.double()
            ref = torch.addmm(b64, a64, w64.t())
        c = e.test_gemm(mode, bn, a, w, b)
        torch.cuda.synchronize()
        assert bool(torch.isfinite(c).all())
        bound = gemm_error_bound(a64, w64, b64, mode, exact_operands=operands == "representable")
        worst, r, col = gemm_worst(c, ref, bound)
        del bound, c
        tile = (r // TILE_M) * -(-N // bn) + col // bn
        where = "row %d col %d (tile %d, CTA %d of %d)" % (r, col, tile, tile % grid, grid)
        print("gemm %s %s, %s operands: M=%d N=%d K=%d BN=%d, %d tiles = %.2f per CTA; worst |c-ref|/bound %.3f at %s"
              % (name, mode, operands, M, N, K, bn, n_tiles, n_tiles / grid, worst, where))
        assert worst <= 1.0, "%s, %s operands: |c - ref| exceeds the rounding bound by %.2fx at %s" % (
            mode, operands, worst, where)


# ---------------------------------------------------------------------------------------------------------------
# B. EGNN forward at the C3 and C2 geometries
# ---------------------------------------------------------------------------------------------------------------
def simt_chunks(sizes, cap=SIMT_CHUNK_ROWS):
    """Python replica of the fp32 SIMT chunk rule of mlcg_set_batch: consecutive nodes, each contributing its n - 1 edge
    rows, until the next node would exceed `cap` rows.  Returns [(first node, end node)]."""
    deg = np.repeat(np.asarray(sizes) - 1, sizes)
    chunks, nb = [], 0
    while nb < len(deg):
        start, rows = nb, 0
        while nb < len(deg) and not (rows + deg[nb] > cap and rows > 0):
            rows += deg[nb]
            nb += 1
        chunks.append((start, nb))
    return chunks


def _spread(v, k):
    """At most k entries of v, evenly spaced."""
    v = np.unique(np.asarray(v, dtype=np.int64))
    return v if len(v) <= k else v[np.linspace(0, len(v) - 1, k).astype(np.int64)]


def _egnn_subset(sizes, sms, seed):
    """Molecules compared with the float64 oracle: the first and last, molecules that straddle a 128-row node tile,
    molecules at the first CTA wrap of the P/Q GEMM, molecules on both sides of SIMT chunk boundaries, molecules owning a
    target split between two CTAs of the edge kernel, and random ones."""
    from test_tile_plan import plan
    B = len(sizes)
    off = np.concatenate([[0], np.cumsum(sizes)])
    mol_of_node = np.repeat(np.arange(B), sizes)
    M = int(off[-1])
    pick = {"ends": [0, B - 1]}
    pick["straddle_node_tile"] = _spread(np.nonzero(off[:-1] // TILE_M != (off[1:] - 1) // TILE_M)[0], 12)
    n_mtiles = -(-M // TILE_M)
    grid = min(2 * n_mtiles, sms)  # P/Q GEMM: 2 column tiles per m-tile, tile = 2 * m-tile + n-tile
    wrap = []
    for tile in (grid - 1, grid):
        mt = tile // 2
        if mt < n_mtiles:
            wrap += list(np.unique(mol_of_node[mt * TILE_M:min(M, (mt + 1) * TILE_M)]))
    pick["pq_cta_wrap"] = wrap
    cut = [c[0] for c in simt_chunks(sizes)[1:]]
    pick["simt_chunk_boundary"] = _spread([mol_of_node[n - 1] for n in cut] + [mol_of_node[n] for n in cut], 24)
    tiles, _, _ = plan(sizes, N_MAX, sms)
    pick["split_target_between_ctas"] = _spread(tiles[tiles[:, 7] >= 0, 0], 16)
    pick["random"] = np.random.RandomState(seed).choice(B, 16, replace=False)
    idx = np.unique(np.concatenate([np.asarray(v, dtype=np.int64) for v in pick.values()]))
    return idx, {k: len(v) for k, v in pick.items()}


def _egnn_batch(sizes, seed):
    """z as in test_gpu_properties._batch, with t spread over [0, 1]."""
    B = len(sizes)
    g = torch.Generator().manual_seed(seed)
    n_nodes = torch.from_numpy(np.asarray(sizes, dtype=np.int64))
    nm, _ = O.prepare_masks(n_nodes, N_MAX)
    z = torch.randn(B, N_MAX, 11, generator=g) * nm
    z[:, :, :3] *= 1.7
    z[:, :, :3] = O.remove_mean_with_mask(z[:, :, :3], nm)
    ctx = O.normalise_context(torch.tensor(ONNX_CONTEXT), CONTEXT_NORMS).view(1, 3).repeat(B, 1)
    t = torch.linspace(0, 1, B)[torch.randperm(B, generator=g)]
    return nm, z, ctx, t


def _oracle_eps(sd, sizes, z, ctx, t, chunk=64):
    """float64 oracle eps of the given molecules on the GPU, in chunks of `chunk` molecules."""
    sd64 = {k: v.to("cuda", torch.float64) for k, v in sd.items()}
    out = []
    for s in range(0, len(sizes), chunk):
        n = torch.from_numpy(np.asarray(sizes[s:s + chunk], dtype=np.int64))
        nm, em = (m.to("cuda", torch.float64) for m in O.prepare_masks(n, N_MAX))
        c = ctx[s:s + chunk].to("cuda", torch.float64).view(-1, 1, 3) * nm
        with torch.no_grad():
            out.append(O.egnn_dynamics(sd64, t[s:s + chunk].to("cuda", torch.float64), z[s:s + chunk].to("cuda", torch.float64),
                                       nm, em, c))
    return torch.cat(out)


@pytest.fixture(scope="module", params=["C3", "C2"])
def egnn_case(request, engines, state_dicts):
    sizes = C3_SIZES if request.param == "C3" else np.full(1024, N_MAX, np.int32)
    nm, z, ctx, t = _egnn_batch(sizes, 31)
    e = engines("fp32")
    e.set_batch(sizes, N_MAX)
    eps32 = e.egnn_forward(t, z, ctx).clone()
    idx, picked = _egnn_subset(sizes, _sms(), 7)
    oracle = _oracle_eps(state_dicts[0], sizes[idx], z[idx], ctx[idx], t[idx])
    print("\n%s: %d molecules, %d nodes, %d SIMT chunks; oracle subset of %d molecules: %s"
          % (request.param, len(sizes), int(sizes.sum()), len(simt_chunks(sizes)), len(idx), picked))
    return dict(name=request.param, sizes=sizes, real=nm.squeeze(-1).cuda() > 0, z=z, ctx=ctx, t=t, eps32=eps32,
                idx=idx, oracle=oracle)


@pytest.mark.parametrize("mode", ["fp16", "bf16", "tf32", "fp32"])
def test_egnn_forward_at_scale(engines, egnn_case, mode):
    cs = egnn_case
    sizes, idx = cs["sizes"], cs["idx"]
    e = engines(mode)
    e.set_batch(sizes, N_MAX)
    eps = e.egnn_forward(cs["t"], cs["z"], cs["ctx"]).clone()
    if bool((~cs["real"]).any()):
        assert float(eps[~cs["real"]].abs().max()) == 0.0  # padded rows exactly zero
    if mode == "fp32":
        n_chunks = len(simt_chunks(sizes))
        print("%s fp32: %d SIMT chunks of <= %d edge rows" % (cs["name"], n_chunks, SIMT_CHUNK_ROWS))
        assert n_chunks >= 2
    else:
        tpc = e.gemm_phase_profile(0)["tiles_per_cta"]
        err = rel_l2_per_molecule(eps, cs["eps32"])
        b = int(torch.argmax(err))
        print("%s %s: P/Q GEMM %.2f tiles per CTA; worst per-molecule rel-L2 vs fp32 CUDA %.3e (molecule %d, %d atoms)"
              % (cs["name"], mode, tpc, float(err[b]), b, sizes[b]))
        assert tpc >= 4
        assert float(err[b]) < TC_VS_FP32[mode], "molecule %d (%d atoms)" % (b, sizes[b])
    err = rel_l2_per_molecule(eps[idx], cs["oracle"])
    k = int(torch.argmax(err))
    print("%s %s: worst per-molecule rel-L2 vs float64 oracle over %d molecules %.3e (molecule %d, %d atoms)"
          % (cs["name"], mode, len(idx), float(err[k]), idx[k], sizes[idx[k]]))
    assert float(err[k]) < TOL[mode], "molecule %d (%d atoms)" % (idx[k], sizes[idx[k]])
    if mode != "fp32":
        # the same molecules as a small batch: bit-identical rows (tiles never span molecules)
        e.set_batch(sizes[idx], N_MAX)
        sub = e.egnn_forward(cs["t"][idx], cs["z"][idx], cs["ctx"][idx])
        diff = (sub != eps[idx]).flatten(1).any(1).nonzero().flatten().tolist()
        assert not diff, "molecules %s differ between the big and the small batch" % [int(idx[i]) for i in diff]


# ---------------------------------------------------------------------------------------------------------------
# C. AdjMatSeer across the 3072-molecule chunk
# ---------------------------------------------------------------------------------------------------------------
SEER_BATCHES = (3072, 3073, 7000)


def _seer_samples(B=max(SEER_BATCHES)):
    """Ragged molecules (the C3 sizes) with random coordinates scaled to ~3 covalent neighbours per atom, classes 0-6."""
    g = torch.Generator().manual_seed(11)
    n = torch.from_numpy(C3_SIZES[:B].astype(np.int64))
    nm, _ = O.prepare_masks(n, N_MAX)
    scale = (1.75 * (n.double() / 27) ** (1 / 3)).float().view(-1, 1, 1)
    x = torch.randn(B, N_MAX, 3, generator=g) * scale * nm
    cls = torch.randint(0, 7, (B, N_MAX), generator=g)
    return n, x, cls


def _seer_subset(B, seed):
    """Molecules compared with the oracle: the chunk edges, the last one, molecules whose 42 rows straddle a 128-row tile
    of their chunk, and random ones."""
    b = np.arange(B)
    r = (b % SEER_CHUNK) * 42
    straddle = b[r // TILE_M != (r + 41) // TILE_M]
    pick = [0, SEER_CHUNK - 1, SEER_CHUNK, SEER_CHUNK + 1, B - 1, *_spread(straddle, 12),
            *np.random.RandomState(seed).choice(B, 8, replace=False)]
    return np.unique(np.asarray([p for p in pick if p < B], dtype=np.int64))


def seer_checks(e, seer_sd, n, el, dist, adj, tol):
    """Logits against the float64 oracle per molecule, bond orders against the oracle's argmax, and batch invariance, for
    every batch size of SEER_BATCHES.  Returns the report lines; raises AssertionError on a failure."""
    sd64 = {k: v.to("cuda", torch.float64) for k, v in seer_sd.items()}
    lines = []
    D = 42
    tri = torch.tril(torch.ones(D, D, dtype=torch.bool, device="cuda"), diagonal=-1)
    for B in SEER_BATCHES:
        logits, bonds = e.seer_forward(el[:B], dist[:B], adj[:B])
        torch.cuda.synchronize()
        idx = _seer_subset(B, B)
        with torch.no_grad():
            ref = O.seer_forward(sd64, el[idx].long(), dist[idx].double(), adj[idx].double())
        err = rel_l2_per_molecule(logits[idx], ref)
        k = int(torch.argmax(err))
        lines.append("B=%d: worst per-molecule logits rel-L2 %.3e (molecule %d) over %d molecules"
                     % (B, float(err[k]), idx[k], len(idx)))
        assert float(err[k]) < tol, lines[-1]
        # bond orders of real atom pairs (strict lower triangle): a flip must be a tie at the logit error
        abs_err = (logits[idx].double() - ref).flatten(1).abs().max(1).values
        top2 = torch.topk(ref, 2, dim=-1).values
        margin = top2[..., 0] - top2[..., 1]
        ar = torch.arange(D, device="cuda")
        nn = n[idx].to("cuda").view(-1, 1, 1)
        real = tri & (ar.view(1, D, 1) < nn) & (ar.view(1, 1, D) < nn)
        flip = real & (bonds[idx].long() != O.bond_orders(ref.cpu()).to("cuda"))
        bad = flip & (margin > 2 * abs_err.view(-1, 1, 1))
        lines.append("B=%d: %d bond flips among %d real pairs, all at oracle top-2 margins below twice the logit error"
                     % (B, int(flip.sum()), int(real.sum())))
        assert not bool(bad.any()), "B=%d: bond flips beyond the logit error in molecules %s" % (
            B, sorted({int(idx[i]) for i in bad.nonzero()[:, 0].tolist()}))
        # batch invariance: a molecule's logits do not depend on its chunk, its tile or its neighbours
        five = torch.from_numpy(np.asarray([0, SEER_CHUNK - 1, SEER_CHUNK, SEER_CHUNK + 1, B - 1]) % B)
        small, small_bonds = e.seer_forward(el[five], dist[five], adj[five])
        assert torch.equal(small, logits[five]) and torch.equal(small_bonds, bonds[five]), "B=%d: batch of 5 differs" % B
        del logits, bonds
    return lines


def _seer_inputs(e, n, x, cls):
    e.set_batch(n.numpy(), N_MAX)
    return e.seer_inputs(x, cls.int())


def test_seer_inputs_at_scale(engines):
    n, x, cls = _seer_samples()
    el, dist, adj = (v.cpu() for v in _seer_inputs(engines("tf32"), n, x, cls))
    el_r, dist_r, adj_r = O.seer_inputs_from_samples(x, cls, n)
    assert torch.equal(el.long(), el_r)
    derr = float((dist - dist_r).abs().max())
    assert derr < 1e-5
    # connectivity: equal except for pairs within 1e-5 of the covalent threshold
    r = torch.tensor(O.COV_RADII)[cls]
    thr = O.COV_FACTOR * (r[:, :, None] + r[:, None, :])
    thr = torch.nn.functional.pad(thr, (0, 3, 0, 3), value=-1.0)  # 39 -> 42 slots
    near = (dist_r - thr).abs() < 1e-5
    mism = (adj != adj_r) & ~near
    deg = float((adj_r.sum((1, 2)) - 42).sum() / n.sum())
    print("seer inputs, B=%d: max |dist err| %.2e, %.2f bonds per atom, %d pairs within 1e-5 of the threshold excluded"
          % (len(n), derr, deg, int(near.sum())))
    assert deg > 1.0
    assert not bool(mism.any()), "adjacency differs in molecules %s" % sorted(set(mism.nonzero()[:, 0].tolist()))[:20]


@pytest.mark.parametrize("mode", ["fp32", "tf32"])
def test_seer_forward_across_chunks(engines, state_dicts, mode):
    e = engines(mode)
    n, x, cls = _seer_samples()
    el, dist, adj = _seer_inputs(e, n, x, cls)
    for ln in seer_checks(e, state_dicts[1], n, el, dist, adj, SEER_TOL[mode]):
        print("seer", mode, ln)


_SEER_SCRIPT = r"""
import sys, torch
sys.path.insert(0, sys.argv[1]); sys.path.insert(0, sys.argv[1] + "/tests")
import test_gpu_scale as S
from ml_conformer_generator_b200.engine import Engine
from ml_conformer_generator_b200.weights import random_state_dicts
_, seer_sd = random_state_dicts(0)
e = Engine(torch.device("cuda:0"), "tf32"); e.load_seer_state_dict(seer_sd)
n, x, cls = S._seer_samples()
el, dist, adj = S._seer_inputs(e, n, x, cls)
for ln in S.seer_checks(e, seer_sd, n, el, dist, adj, S.SEER_TOL["tf32"]):
    print(ln)
e.close()
print("OK")
"""


def test_seer_plain_tf32_across_chunks():
    """MLCG_SEER_3XTF32=0 (read once per process, hence the subprocess): the single-pass TF32 GCN passes the same checks."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, "-c", _SEER_SCRIPT, root], env=dict(os.environ, MLCG_SEER_3XTF32="0"),
                         capture_output=True, text=True, timeout=900)
    print(out.stdout)
    assert out.returncode == 0, out.stderr[-3000:]
    assert out.stdout.splitlines()[-1] == "OK"


def test_seer_fp16_engine_equals_tf32(engines):
    """The GCN always runs TF32 on the tensor cores, whatever the engine's precision."""
    n, x, cls = _seer_samples()
    el, dist, adj = _seer_inputs(engines("tf32"), n, x, cls)
    a = engines("tf32").seer_forward(el, dist, adj)
    b = engines("fp16").seer_forward(el, dist, adj)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


# ---------------------------------------------------------------------------------------------------------------
# D. the product path at C3
# ---------------------------------------------------------------------------------------------------------------
def test_generate_at_c3(engines):
    """generate_host at the C3 geometry: the first call runs eagerly, the second captures and replays a CUDA graph; both
    give the same outputs, and the bonds equal the GCN entry points applied to the returned coordinates and classes."""
    e = engines("fp16")
    B = len(C3_SIZES)
    ctx = np.tile(np.asarray(O.normalise_context(torch.tensor(ONNX_CONTEXT), CONTEXT_NORMS)), (B, 1))
    e.set_batch(C3_SIZES, N_MAX)  # drops any graph captured earlier, so the next call is an eager first call
    eager = [t.clone() for t in e.generate_host(C3_SIZES, N_MAX, ctx, T=2, seed=3)]
    graph = [t.clone() for t in e.generate_host(C3_SIZES, N_MAX, ctx, T=2, seed=3)]
    assert all(torch.equal(u, v) for u, v in zip(eager, graph))
    x, cls, bonds = eager
    el, dist, adj = e.seer_inputs(x, cls)
    _, bonds_again = e.seer_forward(el, dist, adj)
    diff = (bonds_again.cpu() != bonds).flatten(1).any(1).nonzero().flatten().tolist()
    print("C3 generate, T=2: eager and graph replay identical; bonds recomputed through seer_inputs / seer_forward, %d "
          "molecules differ" % len(diff))
    assert not diff, "bonds differ for molecules %s" % diff[:20]
