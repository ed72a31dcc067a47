"""GPU: the noise the product path draws, checked end to end against a float64 oracle.

The host generation calls (plain, inpainting, inertial fragment matching, analogue jobs with and without fixed atoms)
draw their noise on the device from Philox4x32-10 keyed by the seed, the global sample id and the draw number
(DESIGN section 4.3; oracle/philox_oracle.py restates it).  Here every kind runs through its host call in fp32 (the exact
SIMT path) with device noise, ragged atom counts and sample ids with a non-zero high word, two of them as packed jobs whose
ids (job_id * 2**32 + k) come from jobs.flatten_jobs.  The oracle rebuilds the noise tape from
philox_oracle.raw_noise(seed, ids, N, d) for d = 0, 1, ... and runs the reference sampler (oracle/edm_oracle.py) in
float64: a wrong draw index, a wrong id or a wrong atom slot changes a molecule by O(1).

Inertial fragment matching is composed as the reference composes it: the host prologue and
ifm_prepare_gen_fragment_context with the eigenvectors signed by the device rule (largest component positive, DESIGN
section 2.2), the first loop on the n - n_ff atoms still to be generated padded to N - min n_ff, inverse_coord_transform
and the merge inputs, then a merge loop whose draws start again at 0 (kMergeDrawBase).  Its coordinates are compared after
centring each molecule: the padded rows of z_known leak into the reference's centre of mass (DESIGN section 2.2).

Per molecule: coordinates by rel-L2 over the real atoms; atom classes equal except at argmax ties of the oracle's final
class logits (top-2 margin below TIE); bond orders against the float64 GCN on the same coordinates and classes, a flip
allowed only where the oracle's top-2 logit margin is below twice the GCN's measured logit error (the rule of
test_gpu_scale.seer_checks).

Measured on one B200 (1000 W power limit), worst / median per-molecule x rel-L2 over 5 molecules per kind: plain
1.68e-7 / 1.60e-7, inpainting 2.73e-7 / 2.62e-7, inertial fragment matching 2.45e-7 / 1.93e-7, analogue without fixed
atoms 1.50e-6 / 1.21e-6, with fixed atoms 1.41e-6 / 1.24e-6; no class ties, no bond flips, GCN logit error <= 1.5e-7.
X_TOL is ten times the worst of these (1.50e-6), well inside 1e-3."""
import contextlib

import numpy as np
import pytest
import torch

from analogue_oracle import edm_analogue
from ml_conformer_generator_b200 import jobs as J
from ml_conformer_generator_b200.config import CONTEXT_NORMS
from ml_conformer_generator_b200.mol_utils import ifm_moi_prologue, inverse_coord_transform, shift_moi_to_com_batch
from oracle import edm_oracle as O
from oracle import philox_oracle as PH

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not torch.cuda.is_available(), reason="needs a B200")]
T, L, SEED = 4, 2, 11
N_DRAWS = 2 + 3 * T  # the most any loop here draws: inpainting, 1 + T * (2 * 1 + 1) + 1
X_TOL = 1.5e-5
TIE = 1e-4  # class-logit margin below which an argmax flip counts as a tie (~100x the coordinate error)


@contextlib.contextmanager
def _f64_cuda():
    """The oracle in float64 on the GPU: its factory calls default to float64 on cuda (its schedule stays float32, as the
    host computes the step scalars)."""
    old = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    try:
        with torch.device("cuda"), torch.no_grad():
            yield
    finally:
        torch.set_default_dtype(old)


def _tape(ids, n):
    """The draws d = 0 .. N_DRAWS-1 of samples `ids` over n atom slots, in the layout the oracle consumes."""
    pairs = []
    for d in range(N_DRAWS):
        r = torch.from_numpy(PH.raw_noise(SEED, ids, n, d)).to("cuda")
        pairs.append((r[..., :3], r[..., 3:]))
    return O.NoiseTape(pairs)


def _masks(nn, N):
    return O.prepare_masks(torch.as_tensor(np.asarray(nn, np.int64), device="cuda"), N)


def _bctx(ctx, nm):
    return torch.as_tensor(np.asarray(ctx), dtype=torch.float64, device="cuda").view(-1, 1, 3) * nm


class _LastZ:
    """Oracle hook: keeps the latent of the last network call, the z0 whose class channels the decode argmaxes."""

    def __call__(self, z, t, eps):
        self.z = z


@pytest.fixture(scope="module")
def sd64(state_dicts):
    return tuple({k: v.to("cuda", torch.float64) for k, v in sd.items()} for sd in state_dicts)


def _compare(e, seer64, what, out, nn, x_ref, z0_ref, centred=False):
    """Checks one call's outputs against the oracle (module docstring).  Returns the per-molecule rel-L2 errors."""
    x, cls, bonds = (t.cpu() for t in out)
    B, N = x.shape[:2]
    errs = []
    for b in range(B):
        n = int(nn[b])
        a, r = x[b, :n].double(), x_ref[b, :n].double().cpu()
        if centred:
            a, r = a - a.mean(0), r - r.mean(0)
        errs.append(float((a - r).norm() / r.norm()))
    real = torch.arange(N).view(1, N) < torch.as_tensor(np.asarray(nn)).view(B, 1)
    logits = z0_ref[:, :, 3:10].double().cpu()
    top = torch.topk(logits, 2, dim=-1).values
    flips = real & (cls.long() != logits.argmax(-1))
    # bonds: the float64 GCN on the same coordinates and classes
    el, dist, adj = e.seer_inputs(x.cuda(), cls.cuda())
    dev_logits, dev_bonds = e.seer_forward(el, dist, adj)
    assert torch.equal(dev_bonds.cpu(), bonds), "%s: the call's bonds differ from the GCN entry points'" % what
    with torch.no_grad():
        ref = O.seer_forward(seer64, el.long(), dist.double(), adj.double())
    abs_err = (dev_logits.double() - ref).flatten(1).abs().max(1).values.cpu()
    ref = ref.cpu()
    top2 = torch.topk(ref, 2, dim=-1).values
    D = 42
    ar = torch.arange(D)
    nn_t = torch.as_tensor(np.asarray(nn)).view(-1, 1, 1)
    pairs = torch.tril(torch.ones(D, D, dtype=torch.bool), -1) & (ar.view(1, D, 1) < nn_t) & (ar.view(1, 1, D) < nn_t)
    bflip = pairs & (bonds.long() != O.bond_orders(ref))
    bad = bflip & (top2[..., 0] - top2[..., 1] > 2 * abs_err.view(-1, 1, 1))
    print("%s: x rel-L2 worst %.3e median %.3e over %d molecules; %d class ties; %d bond flips at ties (GCN logit error "
          "%.1e)" % (what, max(errs), float(np.median(errs)), B, int(flips.sum()), int(bflip.sum()), float(abs_err.max())))
    assert not bool((flips & (top[..., 0] - top[..., 1] > TIE)).any()), "%s: atom classes differ beyond argmax ties" % what
    assert bool((cls[~real] == -1).all())
    assert not bool(bad.any()), "%s: bond orders differ beyond the GCN logit error" % what
    assert max(errs) < X_TOL, "%s: x rel-L2 %.3e (per molecule %s)" % (what, max(errs), ["%.1e" % v for v in errs])
    return errs


def _ids(high, lows):
    return (np.int64(high) << 32) + np.asarray(lows, np.int64)


def _frag(n, seed):
    g = torch.Generator().manual_seed(seed)
    return 1.4 * torch.randn(n, 3, generator=g), torch.eye(8)[torch.randint(0, 6, (n,), generator=g)]


def _parent(n, seed):
    g = torch.Generator().manual_seed(seed)
    st = torch.randn(n, 3, generator=g)
    x = torch.cumsum(1.5 * st / st.norm(dim=1, keepdim=True), 0) * 0.6
    return x - x.mean(0), torch.eye(8)[torch.randint(0, 7, (n,), generator=g)]


def _ctx(B, seed):
    return (0.5 * np.random.RandomState(seed).randn(B, 3)).astype(np.float32)


def _known(nn, N, job, mols, flags=None):
    """z_known (B,N,11) and fixed_mask (B,N,1): sample b holds mols[job[b]] in its first rows, fixed where flagged (all its
    rows when flags is None)."""
    B = len(nn)
    zk, fm = torch.zeros(B, N, 11, device="cuda", dtype=torch.float64), torch.zeros(B, N, 1, device="cuda", dtype=torch.float64)
    for b, j in enumerate(job):
        x, h = mols[j]
        n = x.shape[0]
        zk[b, :n, :3], zk[b, :n, 3:] = torch.as_tensor(x).cuda(), torch.as_tensor(h).cuda()
        fm[b, :n, 0] = 1.0 if flags is None else torch.as_tensor(flags[j]).cuda().double()
    return zk, fm


def test_plain_jobs_match_the_float64_oracle(engines, sd64):
    """Two plain jobs through jobs.run_packed (what generate_jobs runs): ids job_id * 2**32 + k from flatten_jobs."""
    e = engines("fp32")
    jobs = [dict(reference_context=[60.0, 120.0, 170.0], n_atoms=17, variance=2, n_samples=3, job_id=7),
            dict(reference_context=[45.0, 90.0, 160.0], n_atoms=16, variance=1, n_samples=2, job_id=123456)]
    packed = J.flatten_jobs(jobs, seed=SEED)
    out = J.run_packed(e, packed, np.arange(packed.ids.size), T, 0, 3, L, SEED)
    nn, N = packed.n_nodes, packed.N
    hook = _LastZ()
    with _f64_cuda():
        nm, em = _masks(nn, N)
        x_ref, _ = O.edm_forward(sd64[0], O.gamma_table(T), nm, em, _bctx(packed.ctx, nm), _tape(packed.ids, N), 0,
                                 hook=hook)
    _compare(e, sd64[1], "plain", out, nn, x_ref, hook.z)


def test_inpainting_matches_the_float64_oracle(engines, sd64):
    e = engines("fp32")
    frags = [_frag(3, 0), _frag(5, 1)]
    job = np.array([0, 1, 1, 0, 1], np.int32)
    nn = np.array([15, 19, 17, 18, 16], np.int32)
    N, ids, ctx = 19, _ids(5, [3, 17, 4, 90, 41]), _ctx(5, 0)
    out = e.generate_fragment_jobs_host(nn, N, ctx, job, frags, False, T=T, resample_steps=0, seed=SEED, sample_ids=ids)
    hook = _LastZ()
    with _f64_cuda():
        nm, em = _masks(nn, N)
        zk, fm = _known(nn, N, job, frags)
        x_ref, _ = O.edm_inpaint(sd64[0], O.gamma_table(T), nm, em, _bctx(ctx, nm), zk, fm, _tape(ids, N), 0, 3, hook=hook)
    _compare(e, sd64[1], "inpaint", out, nn, x_ref, hook.z)


def test_inertial_fragment_matching_jobs_match_the_float64_oracle(engines, sd64):
    """Two IFM jobs with fragments of 3 and 5 atoms through jobs.run_packed: ids from flatten_jobs, the first loop padded
    to N - min n_ff."""
    e = engines("fp32")
    jobs = [dict(reference_context=[70.0, 140.0, 190.0], n_atoms=17, variance=2, n_samples=3, job_id=31,
                 fixed_fragment=_frag(3, 2), inertial_fragment_matching=True),
            dict(reference_context=[55.0, 110.0, 150.0], n_atoms=18, variance=1, n_samples=2, job_id=2 ** 30 + 5,
                 fixed_fragment=_frag(5, 3), inertial_fragment_matching=True)]
    packed = J.flatten_jobs(jobs, seed=SEED)
    out = J.run_packed(e, packed, np.arange(packed.ids.size), T, 0, 3, L, SEED)
    nn, N, job, ids = packed.n_nodes, packed.N, packed.job, packed.ids
    B = nn.size
    n_ff = np.array([packed.fragments[j][0].shape[0] for j in job])
    Ng = N - int(n_ff.min())
    pro = [ifm_moi_prologue(packed.fragments[j][0], packed.references[j]) for j in job]  # the host inputs, float32
    hook = _LastZ()
    with _f64_cuda():
        # ifm_prepare_gen_fragment_context in float64, eigenvectors signed by the device rule
        n_gen = torch.as_tensor(nn - n_ff, dtype=torch.float64, device="cuda")
        shift = torch.stack([p[1].cuda().double() for p in pro]) / n_gen.view(B, 1)
        moi = shift_moi_to_com_batch(torch.stack([p[0].cuda().double() for p in pro]), shift, n_gen)
        vals, rot = torch.linalg.eigh(moi)
        big = rot.abs().argmax(dim=1, keepdim=True)
        rot = rot * torch.sign(rot.gather(1, big))
        mean, mad = (torch.as_tensor(CONTEXT_NORMS[k], dtype=torch.float64, device="cuda") for k in ("mean", "mad"))
        nm1, em1 = _masks(nn - n_ff, Ng)
        xg, hg = O.edm_forward(sd64[0], O.gamma_table(T), nm1, em1, ((vals - mean) / mad).view(B, 1, 3) * nm1,
                               _tape(ids, Ng), 0)
        # back to the reference frame next to the fixed fragment: the merge inputs
        xg = inverse_coord_transform(xg.double(), shift, rot)
        zk, fm = _known(nn, N, job, packed.fragments)
        for b in range(B):
            m = N - int(n_ff[b])
            zk[b, n_ff[b]:, :3], zk[b, n_ff[b]:, 3:] = xg[b, :m], hg[b, :m].double()
        nm, em = _masks(nn, N)
        x_ref, _ = O.edm_merge_fragments(sd64[0], O.gamma_table(T), nm, em, fm, _bctx(packed.ctx, nm), zk, _tape(ids, N),
                                         L, 0, 3, hook=hook)
    _compare(e, sd64[1], "ifm", out, nn, x_ref, hook.z, centred=True)


@pytest.mark.parametrize("fixed", [False, True])
def test_analogue_jobs_match_the_float64_oracle(engines, sd64, fixed):
    e = engines("fp32")
    parents = [_parent(13, 4), _parent(16, 5)]
    flags = [np.isin(np.arange(p[0].shape[0]), [0, 3, 6]).astype(np.int32) for p in parents] if fixed else None
    job = np.array([1, 0, 1, 1, 0], np.int32)
    nn = np.array([parents[j][0].shape[0] for j in job], np.int32)
    N, ids, ctx = 17, _ids(9, [8, 1, 77, 23, 6]), _ctx(5, 1)
    out = e.generate_analogue_jobs_host(nn, N, ctx, job, parents, flags, T, 0, 3, L, seed=SEED, sample_ids=ids)
    hook = _LastZ()
    with _f64_cuda():
        nm, em = _masks(nn, N)
        zk, fm = _known(nn, N, job, parents, flags or [np.zeros(p[0].shape[0]) for p in parents])
        x_ref, _ = edm_analogue(sd64[0], O.gamma_table(T), nm, em, fm, _bctx(ctx, nm), zk, _tape(ids, N), L, 0, 3,
                                hook=hook)
    _compare(e, sd64[1], "analogue fixed=%s" % fixed, out, nn, x_ref, hook.z)
