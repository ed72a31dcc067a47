"""GPU: the CUDA graph of the host generation calls (generate_graphed in csrc/mlcg_api.cu) against fresh eager runs.

A host generation call runs eagerly on the first call with a graph key, captures a CUDA graph on the second and replays it
from then on.  The key (graph_key) must hold everything the captured launches bake in, and nothing else:
  * changing one key field must force an eager call -- no capture on that call -- that equals, bit for bit, a first call
    with the same arguments on a new Engine; the next two calls capture and replay and equal it too;
  * changing an input that is not in the key (context, seed, sample_offset, sample ids, the job table's contents at the
    same sizes) must replay the graph and still equal a fresh eager call.
And a captured graph must survive every other entry point run on the same handle between capture and replay, or be
dropped when one of them reallocates a buffer it references (the GCN workspaces grow with mlcg_seer_forward's batch).

Every call is made through ctypes, so every key field -- each of the seven step scalars, the decode scalars, the IFM
norms -- can be moved by one ulp.  Comparisons are of float bit patterns, so NaN positions count (random-init 16-bit
trajectories may leave the finite range, DESIGN section 3)."""
import ctypes as C

import numpy as np
import pytest
import torch

from ml_conformer_generator_b200 import _lib
from ml_conformer_generator_b200.config import CONTEXT_NORMS
from ml_conformer_generator_b200.mol_utils import ifm_moi_prologue
from ml_conformer_generator_b200.schedule import decode_scalars, forward_level_scalars, gamma_table

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not torch.cuda.is_available(), reason="needs a B200")]
T, L = 4, 2
KINDS = ["plain", "inpaint", "ifm", "analogue_fixed", "analogue_free"]
STEP_FIELDS = [f for f, _ in _lib.StepScalars._fields_]


# ---------------------------------------------------------------------------------------------------------------
# one host generation call, described by a dict of host arrays ("spec") and made through ctypes
# ---------------------------------------------------------------------------------------------------------------
def _up(v):
    """The next float32 above v: a one-ulp change."""
    return np.nextafter(np.float32(v), np.float32(np.inf))


def _schedule(T_):
    """Step scalars (T,7) f32 as Engine builds them, decode scalars (3) f32 and the gamma table."""
    gamma = gamma_table(T_)
    from ml_conformer_generator_b200.schedule import all_step_scalars
    rows = []
    for s, d in enumerate(all_step_scalars(gamma)):
        blend = float(torch.pow(1 - torch.full([1], s, dtype=torch.int64) / T_, 3))
        rows.append([d["t"], d["alpha_ts"], d["c_eps"], d["c_sigma"], d["alpha_s"], d["sigma_s"], blend])
    dec = decode_scalars(gamma)
    return np.asarray(rows, np.float32), np.asarray([dec["sigma_0"], dec["alpha_0"], dec["sigma_x"]], np.float32), gamma


def _set_T(s, T_, level=None):
    s["T"] = T_
    s["steps"], s["dec"], gamma = _schedule(T_)
    if "level" in s:
        s["level"] = s["level"] if level is None else level
        lv = forward_level_scalars(gamma, s["level"])
        s["malpha"], s["msigma"] = np.float32(lv["alpha"]), np.float32(lv["sigma"])
    return s


def _frag(n, seed):
    g = torch.Generator().manual_seed(seed)
    return (1.4 * torch.randn(n, 3, generator=g)).numpy(), torch.eye(8)[torch.randint(0, 6, (n,), generator=g)].numpy()


def _parent(n, seed):
    """A compact random skeleton of n atoms, centred on its mean, classes 0..6."""
    g = torch.Generator().manual_seed(seed)
    st = torch.randn(n, 3, generator=g)
    x = torch.cumsum(1.5 * st / st.norm(dim=1, keepdim=True), 0) * 0.6
    return (x - x.mean(0)).numpy(), torch.eye(8)[torch.randint(0, 7, (n,), generator=g)].numpy()


def _set_fragments(s, n_ff, seed=0, ref_shift=0.0):
    """The packed fragment table of `n_ff` (one entry per job) and, for IFM, its moment-of-inertia prologue."""
    s["n_ff"] = np.asarray(n_ff, np.int32)
    fr = [_frag(int(n), seed + 10 * k) for k, n in enumerate(n_ff)]
    s["ffx"] = np.concatenate([f[0] for f in fr]).astype(np.float32)
    s["ffh"] = np.concatenate([f[1] for f in fr]).astype(np.float32)
    refs = [torch.tensor([60.0, 120.0, 170.0]) * (1 + 0.07 * k + ref_shift) for k in range(len(n_ff))]
    pro = [ifm_moi_prologue(torch.from_numpy(f[0]), r) for f, r in zip(fr, refs)]
    s["moi"] = np.stack([p[0].numpy().reshape(9) for p in pro]).astype(np.float32)
    s["com"] = np.stack([p[1].numpy() for p in pro]).astype(np.float32)
    return s


def _set_parents(s, sizes, fixed_at, seed=0):
    """The packed parent table of jobs with `sizes` atoms; n_nodes follow the samples' jobs."""
    s["n_atoms"] = np.asarray(sizes, np.int32)
    pr = [_parent(int(n), seed + k) for k, n in enumerate(sizes)]
    s["px"] = np.concatenate([p[0] for p in pr]).astype(np.float32)
    s["ph"] = np.concatenate([p[1] for p in pr]).astype(np.float32)
    fl = []
    for n in sizes:
        f = np.zeros(int(n), np.int32)
        f[[a for a in fixed_at if a < n]] = 1
        fl.append(f)
    s["fixed"] = np.concatenate(fl)
    s["nn"] = s["n_atoms"][s["job"]].astype(np.int32)
    return s


def _base(kind):
    """B = 6 ragged samples of two jobs, N = 18 (analogue: 16), T = 4."""
    g = np.random.RandomState(1)
    s = dict(kind=kind, nn=np.array([15, 18, 16, 17, 15, 18], np.int32), N=18, r=0, seed=5, offset=0, ids=None,
             ctx=(0.5 * g.randn(6, 3)).astype(np.float32), job=np.array([0, 1, 0, 1, 1, 0], np.int32))
    if kind in ("inpaint", "ifm"):
        _set_fragments(s, [3, 4])
        s["level"] = L
        s["mean"] = np.asarray(CONTEXT_NORMS["mean"], np.float32)
        s["mad"] = np.asarray(CONTEXT_NORMS["mad"], np.float32)
    elif kind.startswith("analogue"):
        s["N"], s["level"] = 16, L
        _set_parents(s, [12, 15], [1, 4] if kind == "analogue_fixed" else [])
    return _set_T(s, T)


def _call(e, s):
    """The host generation call of `s` on engine e: (x (B,N,3), atom_class (B,N), bonds (B,42,42)) on the host."""
    B, N, T_ = len(s["nn"]), s["N"], s["T"]
    nn = np.ascontiguousarray(s["nn"], np.int32)
    ctx = np.ascontiguousarray(s["ctx"], np.float32)
    steps = (_lib.StepScalars * T_)(*[_lib.StepScalars(*[float(v) for v in row]) for row in s["steps"]])
    ids = None if s["ids"] is None else np.ascontiguousarray(s["ids"], np.int64)
    out = [torch.empty(B, N, 3), torch.empty(B, N, dtype=torch.int32), torch.empty(B, 42, 42, dtype=torch.int8)]
    kind = s["kind"]
    keep = []
    if kind == "plain":
        fn, head = e.lib.mlcg_generate, (e.h,)
    elif kind in ("inpaint", "ifm"):
        keep = [np.ascontiguousarray(s[k]) for k in ("job", "n_ff", "ffx", "ffh", "moi", "com", "mean", "mad")]
        p = [a.ctypes.data for a in keep]
        tab = _lib.FragmentJobs(2 if kind == "ifm" else 1, len(s["n_ff"]), p[0], p[1], p[2], p[3], int(s["level"]),
                                float(s["malpha"]), float(s["msigma"]), p[4], p[5], p[6], p[7])
        fn, head = e.lib.mlcg_generate_fragment_jobs, (e.h, C.byref(tab))
    else:
        keep = [np.ascontiguousarray(s[k]) for k in ("job", "n_atoms", "px", "ph", "fixed")]
        p = [a.ctypes.data for a in keep]
        tab = _lib.AnalogueJobs(len(s["n_atoms"]), p[0], p[1], p[2], p[3], p[4], int(s["level"]), float(s["malpha"]),
                                float(s["msigma"]))
        fn, head = e.lib.mlcg_generate_analogue_jobs, (e.h, C.byref(tab))
    rc = fn(*head, nn.ctypes.data_as(C.c_void_p), B, N, ctx.ctypes.data, T_, steps, int(s["r"]), *[float(v) for v in s["dec"]],
            int(s["seed"]), int(s["offset"]), None if ids is None else ids.ctypes.data, out[0].data_ptr(),
            out[1].data_ptr(), out[2].data_ptr(), e._stream())
    e._check(rc, "generate (%s)" % kind)
    e.lib.mlcg_nonfinite(e.h, e._stream())  # clear the flag: random-init trajectories may diverge
    e.B, e.N, e.n_nodes = B, N, torch.from_numpy(nn.copy())
    del keep
    return out


def _bits(t):
    t = torch.as_tensor(t).detach().cpu()
    return t.view(torch.int32) if t.dtype == torch.float32 else t


def _same(got, want, what):
    for a, b, k in zip(got, want, ("x", "atom_class", "bonds")):
        u, v = _bits(a), _bits(b)
        assert u.shape == v.shape and torch.equal(u, v), "%s: %s differs from a fresh eager call" % (what, k)


# ---------------------------------------------------------------------------------------------------------------
# the changes: one key field each, then inputs outside the key
# ---------------------------------------------------------------------------------------------------------------
def _permute_samples(s, perm):
    for k in ("nn", "ctx", "job"):
        s[k] = s[k][perm]
    if s["ids"] is not None:
        s["ids"] = s["ids"][perm]
    return s


def _drop_last(s):
    for k in ("nn", "ctx", "job"):
        s[k] = s[k][:-1]
    return s


def _step(field):
    def f(s):
        s["steps"] = s["steps"].copy()
        c = STEP_FIELDS.index(field)
        s["steps"][1, c] = _up(s["steps"][1, c])
        return s
    return f


def _dec(i):
    def f(s):
        s["dec"] = s["dec"].copy()
        s["dec"][i] = _up(s["dec"][i])
        return s
    return f


def _vec_up(key):
    def f(s):
        s[key] = s[key].copy()
        s[key][0] = _up(s[key][0])
        return s
    return f


KEY_CHANGES = {
    "B": _drop_last,
    "N": lambda s: dict(s, N=s["N"] + 1),
    "n_nodes_order": lambda s: _permute_samples(s, np.array([1, 0, 3, 2, 5, 4])),
    "T": lambda s: _set_T(s, s["T"] + 1),
    "resample_steps": lambda s: dict(s, r=2),
    **{"step_" + f: _step(f) for f in STEP_FIELDS},
    "sigma_0": _dec(0), "alpha_0": _dec(1), "sigma_x": _dec(2),
}
LEVEL_CHANGES = {
    "diffusion_level": lambda s: _set_T(s, s["T"], s["level"] + 1),
    "merge_alpha": lambda s: dict(s, malpha=_up(s["malpha"])),
    "merge_sigma": lambda s: dict(s, msigma=_up(s["msigma"])),
}
FRAGMENT_CHANGES = {
    "n_ff_per_job": lambda s: _set_fragments(s, [4, 3]),                                  # same packed length
    "job_count": lambda s: _set_fragments(dict(s, job=np.array([0, 1, 2, 1, 2, 0], np.int32)), [3, 2, 2]),  # same length
    "packed_length": lambda s: _set_fragments(s, [3, 5]),
}
ANALOGUE_CHANGES = {
    "job_count": lambda s: _set_parents(dict(s, job=np.array([0, 1, 2, 1, 2, 0], np.int32)), [12, 8, 7],
                                        [1, 4] if s["kind"] == "analogue_fixed" else []),  # same packed length
    "packed_length": lambda s: _set_parents(s, [12, 16], [1, 4] if s["kind"] == "analogue_fixed" else []),
}


def _key_changes(kind):
    ch = dict(KEY_CHANGES)
    if kind in ("ifm", "analogue_fixed", "analogue_free"):
        ch.update(LEVEL_CHANGES)
    if kind == "ifm":
        ch.update(norm_mean=_vec_up("mean"), norm_mad=_vec_up("mad"))
    if kind in ("inpaint", "ifm"):
        ch.update(FRAGMENT_CHANGES)
    if kind.startswith("analogue"):
        ch.update(ANALOGUE_CHANGES)
    return ch


def _table_contents(s):
    """Other fragments / parents (and flags) of the same sizes, and for IFM other reference contexts."""
    if s["kind"] in ("inpaint", "ifm"):
        return _set_fragments(s, s["n_ff"], seed=7, ref_shift=0.3)
    if s["kind"].startswith("analogue"):
        return _set_parents(s, s["n_atoms"], [0, 2, 5] if s["kind"] == "analogue_fixed" else [], seed=9)
    return s


OTHER_CHANGES = {
    "context": lambda s: dict(s, ctx=s["ctx"][::-1].copy() + np.float32(0.25)),
    "seed": lambda s: dict(s, seed=s["seed"] + 1),
    "sample_offset": lambda s: dict(s, offset=1000),
    "sample_ids": lambda s: dict(s, ids=(np.int64(3) << 32) + np.array([9, 2, 40, 7, 11, 5], np.int64)),
    "table_contents": _table_contents,
}


def _other_changes(kind):
    ch = dict(OTHER_CHANGES)
    if kind == "plain":
        del ch["table_contents"]
    if kind == "inpaint":  # inpainting starts from noise: the level and its scalars are not part of its call
        ch.update({"ignored_" + k: v for k, v in LEVEL_CHANGES.items()})
    return ch


# ---------------------------------------------------------------------------------------------------------------
# fixtures
# ---------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def gpu_state_dicts(state_dicts):
    return tuple({k: v.to("cuda") for k, v in sd.items()} for sd in state_dicts)


def _new_engine(sds, precision):
    from ml_conformer_generator_b200.engine import Engine
    e = Engine(torch.device("cuda:0"), precision)
    e.load_edm_state_dict(sds[0])
    e.load_seer_state_dict(sds[1])
    return e


@pytest.fixture(scope="module")
def tested(gpu_state_dicts):
    """One engine per precision that every call of this module's key tests goes through."""
    made = {}

    def get(precision):
        if precision not in made:
            made[precision] = _new_engine(gpu_state_dicts, precision)
        return made[precision]

    yield get
    for e in made.values():
        e.close()


@pytest.fixture(scope="module")
def fresh(gpu_state_dicts):
    """fresh(precision, spec): the call of `spec` as the first call on a new engine (an eager run)."""
    def run(precision, s):
        e = _new_engine(gpu_state_dicts, precision)
        try:
            out = _call(e, s)
            assert e.graph_captures() == 0
            return out
        finally:
            e.close()
    return run


def _capture_base(e, s):
    """Drops whatever graph e holds, then makes the eager and the capturing call of `s`."""
    e.set_batch([1], 1)
    caps = []
    for _ in range(2):
        c0 = e.graph_captures()
        out = _call(e, s)
        caps.append(e.graph_captures() - c0)
    assert caps == [0, 1]
    return out


def _expect(e, s, want, captures, what):
    """Calls `s` len(captures) times: each equals `want`, with the given number of new captures per call."""
    got = []
    for _ in captures:
        c0 = e.graph_captures()
        out = _call(e, s)
        got.append(e.graph_captures() - c0)
        _same(out, want, what)
    assert got == list(captures), "%s: captures per call %s, expected %s" % (what, got, list(captures))
    return out


# ---------------------------------------------------------------------------------------------------------------
# 1. key coverage
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind,field", [(k, f) for k in KINDS for f in _key_changes(k)])
@pytest.mark.parametrize("precision", ["fp16", "fp32"])
def test_a_changed_key_field_runs_eagerly_then_captures_anew(tested, fresh, precision, kind, field):
    e = tested(precision)
    base = _base(kind)
    _capture_base(e, base)
    s = _key_changes(kind)[field](dict(base))
    want = fresh(precision, s)
    _expect(e, s, want, [0, 1, 0], "%s %s" % (kind, field))  # eager, captured, replayed


@pytest.mark.parametrize("kind,field", [(k, f) for k in KINDS for f in _other_changes(k)])
@pytest.mark.parametrize("precision", ["fp16", "fp32"])
def test_inputs_outside_the_key_replay_the_graph_with_the_new_values(tested, fresh, precision, kind, field):
    e = tested(precision)
    base = _base(kind)
    first = _capture_base(e, base)
    s = _other_changes(kind)[field](dict(base))
    want = fresh(precision, s)
    _expect(e, s, want, [0, 0], "%s %s" % (kind, field))  # both replays
    if not field.startswith("ignored_") and bool(torch.isfinite(first[0]).all()):
        assert not torch.equal(_bits(want[0]), _bits(first[0])), "%s: the change did not reach the outputs" % field


# ---------------------------------------------------------------------------------------------------------------
# 2. every other entry point between capture and replay
# ---------------------------------------------------------------------------------------------------------------
def _run_other_entry_points(e, s):
    """Calls once each, on the batch the generation call left set, every entry point that keeps the batch plan."""
    B, N = len(s["nn"]), s["N"]
    dev, st, lib = e.device, e._stream(), e.lib
    g = torch.Generator().manual_seed(3)
    ctx = torch.randn(B, 3, generator=g).to(dev)
    z = (0.5 * torch.randn(B, N, 11, generator=g)).to(dev)
    t = torch.full((B,), 0.5, device=dev)
    e.egnn_forward(t, z, ctx)
    e.egnn_forward_breakdown(t, z, ctx)
    zk = torch.zeros(B, N, 11, device=dev)
    zk[:, :3, :3] = torch.randn(B, 3, 3, generator=g).to(dev)
    zk[:, :3, 3] = 1.0
    fm = torch.zeros(B, N, device=dev)
    fm[:, :3] = 1.0
    for mode in ("forward", "inpaint", "merge", "analogue"):
        e.sample(ctx, 3, mode, 0, z_known=zk, fixed_mask=fm, diffusion_level=2, seed=2)
    # the single-step entry points
    steps = e._steps(3, 3)[1]
    noise = _lib.Noise(None, 7, 1, 0, None)
    zz, eps = torch.empty(B, N, 11, device=dev), torch.zeros(B, N, 11, device=dev)
    x, cls = torch.empty(B, N, 3, device=dev), torch.empty(B, N, dtype=torch.int32, device=dev)
    p = lambda a: C.c_void_p(a.data_ptr())
    assert lib.mlcg_noise_init(e.h, p(zz), C.byref(noise), st) == 0
    assert lib.mlcg_step(e.h, p(zz), p(eps), C.byref(steps[1]), C.byref(noise), st) == 0
    assert lib.mlcg_reinject(e.h, p(zz), p(zk), p(fm), C.byref(steps[1]), C.byref(noise), st) == 0
    assert lib.mlcg_forward_diffuse(e.h, p(zz), p(zk), 0.5, 0.5, C.byref(noise), st) == 0
    assert lib.mlcg_decode(e.h, p(zz), p(eps), 1.0, 1.0, 1.0, C.byref(noise), p(x), p(cls), st) == 0
    el, dist, adj = e.seer_inputs(x, cls)
    # the IFM and analogue hooks
    ffx, ffh = (torch.from_numpy(a) for a in _frag(3, 1))
    f_ctx, shift, rot, _ = e.ifm_context(ffx, torch.tensor([60.0, 120.0, 170.0]), CONTEXT_NORMS, torch.from_numpy(s["nn"]))
    e.ifm_merge_inputs(x[:, :N - 3], cls[:, :N - 3], shift, rot, ffx, ffh, N)
    e.analogue_inputs([0] * B, [_parent(int(min(s["nn"])), 4)], [np.eye(1, int(min(s["nn"])), 0, dtype=np.int32)[0]], N)
    # measurement and test hooks
    a, w = torch.randn(200, 96, generator=g), torch.randn(256, 96, generator=g)
    e.test_gemm("bf16", 256, a, w, torch.randn(256, generator=g))
    if e.precision != "fp32":
        assert e.time_edge_kernel(0, 2) > 0
        e.gemm_phase_profile(0)
    lib.mlcg_nonfinite(e.h, st)
    torch.cuda.synchronize()
    return el, dist, adj


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("precision", ["fp16", "fp32"])
def test_graph_survives_other_entry_points_or_is_dropped_when_they_grow_its_buffers(gpu_state_dicts, fresh, precision,
                                                                                      kind):
    e = _new_engine(gpu_state_dicts, precision)  # its own engine: no GCN workspace grown beyond this test's batch yet
    try:
        s = _base(kind)
        _capture_base(e, s)
        # (a) entry points that keep the batch plan and every buffer the graph holds: the next call replays
        el, dist, adj = _run_other_entry_points(e, s)
        s1 = OTHER_CHANGES["context"](OTHER_CHANGES["seed"](dict(s)))
        _expect(e, s1, fresh(precision, s1), [0], "%s after the other entry points" % kind)
        # (b) the GCN on more molecules than the graph's batch grows its workspaces: the graph is dropped, so the next
        # call runs eagerly (a replay would write into freed memory), the one after captures again
        big = 7 * len(s["nn"])
        logits, bonds = e.seer_forward(el.repeat(7, 1), dist.repeat(7, 1, 1), adj.repeat(7, 1, 1))
        assert logits.shape[0] == big
        s2 = dict(s1, seed=s1["seed"] + 1, ctx=s1["ctx"] * np.float32(0.5))
        _expect(e, s2, fresh(precision, s2), [0, 1, 0], "%s after seer_forward on %d molecules" % (kind, big))
        # (c) a generation call of another kind takes over the handle's plan and graph
        other = _base("analogue_free" if kind == "plain" else "plain")
        _call(e, other)
        s3 = dict(s2, seed=s2["seed"] + 1)
        _expect(e, s3, fresh(precision, s3), [0, 1, 0], "%s after a call of kind %s" % (kind, other["kind"]))
    finally:
        e.close()
