"""GPU: fragment-conditioned generation through the graph-replayed host call (Engine.generate_fragment_host ->
mlcg_generate_fragment), the id-keyed shards, the streaming pipeline and two GPUs.  The reference result is the eager
composition MLConformerGenerator.edm_sample_tensors runs (set_batch + Engine.sample per loop, the device IFM steps between
them) followed by the GCN entry points; every comparison is bit for bit (float bit patterns, so NaN positions count)."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import golden
from ml_conformer_generator_b200 import _lib
from ml_conformer_generator_b200.config import CONTEXT_NORMS
from ml_conformer_generator_b200.mol_utils import normalise_context, prepare_fragment

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
T, L, N = 8, 4, 25  # small T: random-init inpainting trajectories diverge at large T


def _fragment():
    g = golden("host_utils")
    return torch.from_numpy(g["ifm_ff_x"]), torch.from_numpy(g["ifm_ff_h"]).float(), torch.from_numpy(g["yibfeu_context"])


def _other_fragment(ffx, ffh):
    """A different fragment of the same size: moved atoms, classes rotated by one."""
    g = torch.Generator().manual_seed(3)
    return ffx + 0.3 * torch.randn(ffx.shape, generator=g), torch.roll(ffh, 1, dims=0)


def _ctx(ref, B):
    return np.tile(normalise_context(ref, CONTEXT_NORMS).numpy().reshape(1, 3), (B, 1)).astype(np.float32)


def _sizes(B, seed):
    return np.random.RandomState(seed).randint(21, 26, B).astype(np.int32)  # ragged, 21-25 atoms


def _eager(e, ifm, n_nodes, ffx, ffh, ref, seed, ids, r=1):
    """The eager composition of edm_sample_tensors (mode 1: inpaint; mode 2: the IFM sequence) + the GCN."""
    B, n_ff = len(n_nodes), ffx.shape[0]
    ctx = torch.from_numpy(_ctx(ref, B))
    if ifm:
        f_ctx, shift, rot, _ = e.ifm_context(ffx, ref, CONTEXT_NORMS, torch.from_numpy(n_nodes))
        e.set_batch(n_nodes - n_ff, N - n_ff)
        xg, cg = e.sample(f_ctx, T, "forward", r, seed=seed, sample_ids=ids)
        zk, fm = e.ifm_merge_inputs(xg, cg, shift, rot, ffx, ffh, N)
        e.set_batch(n_nodes, N)
        x, cls = e.sample(ctx, T, "merge", r, z_known=zk, fixed_mask=fm, diffusion_level=L, seed=seed, sample_ids=ids)
    else:
        zk, fm = prepare_fragment(B, ffx, ffh, N, n_ff + 1)
        e.set_batch(n_nodes, N)
        x, cls = e.sample(ctx, T, "inpaint", r, z_known=zk, fixed_mask=fm, seed=seed, sample_ids=ids)
    el, dist, adj = e.seer_inputs(x, cls)
    _, bonds = e.seer_forward(el, dist, adj, want_logits=False)
    e.check_finite()
    return x.cpu(), cls.cpu(), bonds.cpu()


def _fast(e, ifm, n_nodes, ffx, ffh, ref, seed, ids, r=1, device_out=False):
    out = e.generate_fragment_host(n_nodes, N, _ctx(ref, len(n_nodes)), ffx, ffh, ifm, ref, None, T, r, 3, L, seed=seed,
                                   sample_ids=ids, device_out=device_out)
    return [t.cpu().clone() for t in out]


def _assert_same(a, b):
    for u, v in zip(a, b):
        assert u.dtype == v.dtype and u.shape == v.shape
        if u.dtype == torch.float32:
            u, v = u.view(torch.int32), v.view(torch.int32)
        assert torch.equal(u, v)


@pytest.mark.parametrize("precision", ["fp16", "bf16"])
@pytest.mark.parametrize("ifm", [False, True], ids=["inpaint", "ifm"])
def test_matches_eager_composition_on_eager_capture_and_replay_calls(engines, precision, ifm):
    e = engines(precision)
    ffx, ffh, ref = _fragment()
    n_nodes = _sizes(24, 0)
    ids = np.arange(24)
    calls = []
    for _ in range(3):  # 1st call eager, 2nd captured into a CUDA graph, 3rd a replay
        l0 = e.kernel_launches()
        calls.append(_fast(e, ifm, n_nodes, ffx, ffh, ref, 11, ids, r=0))
        assert e.kernel_launches() > l0
    want = _eager(e, ifm, n_nodes, ffx, ffh, ref, 11, ids, r=0)
    for got in calls:
        _assert_same(got, want)
    if precision == "bf16" or ifm:
        # with the random-init weights, fp16 inpainting leaves the fp16 range (mlcg_nonfinite); there the comparison
        # covers the NaN positions, the atom classes and the bonds
        assert bool(torch.isfinite(want[0]).all())
    if ifm:  # the merge loop ends with a re-injection: the fixed atoms keep the fragment's classes
        assert bool((want[1][:, :ffx.shape[0]].long() == ffh.argmax(-1).view(1, -1)).all())


@pytest.mark.parametrize("ifm", [False, True], ids=["inpaint", "ifm"])
def test_replay_uses_the_new_inputs(engines, ifm):
    """With the graph captured, a call with another seed and other sample ids, and one with another fragment of the same
    size, equal the eager composition for those inputs (bf16: finite trajectories, so the results differ visibly)."""
    e = engines("bf16")
    ffx, ffh, ref = _fragment()
    n_nodes = _sizes(20, 1)
    first = None
    for _ in range(2):
        first = _fast(e, ifm, n_nodes, ffx, ffh, ref, 1, np.arange(20))
    ids = np.random.RandomState(4).choice(10 ** 6, 20, replace=False)
    got = _fast(e, ifm, n_nodes, ffx, ffh, ref, 2, ids)
    assert not torch.equal(got[0], first[0])
    ffx2, ffh2 = _other_fragment(ffx, ffh)
    got2 = _fast(e, ifm, n_nodes, ffx2, ffh2, ref, 2, ids)
    _assert_same(got, _eager(e, ifm, n_nodes, ffx, ffh, ref, 2, ids))
    _assert_same(got2, _eager(e, ifm, n_nodes, ffx2, ffh2, ref, 2, ids))
    assert bool(torch.isfinite(got2[0]).all()) and not torch.equal(got2[0], got[0])


@pytest.mark.parametrize("ifm", [False, True], ids=["inpaint", "ifm"])
def test_sharding_by_arbitrary_id_subsets_is_bit_exact(engines, ifm):
    e = engines("bf16")
    ffx, ffh, ref = _fragment()
    n_nodes = _sizes(14, 2)
    full = _fast(e, ifm, n_nodes, ffx, ffh, ref, 5, None)
    perm = np.random.RandomState(1).permutation(14)
    outs = [torch.empty_like(t) for t in full]
    for ids in (np.sort(perm[:5]), np.sort(perm[5:6]), np.sort(perm[6:])):
        res = _fast(e, ifm, n_nodes[ids], ffx, ffh, ref, 5, ids, device_out=True)
        for o, r in zip(outs, res):
            o[torch.as_tensor(ids)] = r
    _assert_same(outs, full)


def test_generate_stream_with_a_fragment_equals_one_call(state_dicts):
    from ml_conformer_generator_b200 import MLConformerGenerator
    gen = MLConformerGenerator(diffusion_steps=T, device=torch.device("cuda:0"), edm_state_dict=state_dicts[0],
                               adj_mat_seer_state_dict=state_dicts[1])
    ffx, ffh, ref = _fragment()

    def post(x, cls, bonds, n, index):
        return index, np.array(x), np.array(cls), np.array(bonds)

    got = [m for batch in gen.generate_stream(ref, n_atoms=23, n_samples=40, batch_size=16, variance=2, postprocess=post,
                                              n_workers=3, seed=5, fixed_fragment=(ffx, ffh), ifm_diffusion_level=L)
           for m in batch]
    assert [m[0] for m in got] == list(range(40))
    sizes = torch.randint(21, 26, (40,), generator=torch.Generator().manual_seed(5)).numpy().astype(np.int32)
    x, cls, bonds = gen.engine.generate_fragment_host(sizes, N, _ctx(ref, 40), ffx, ffh, True, ref, gen.context_norms, T, 0,
                                                      3, L, seed=5)
    for i, (_, xi, ci, bi) in enumerate(got):
        n = int(sizes[i])
        assert np.array_equal(xi.view(np.int32), x[i, :n].numpy().view(np.int32))
        assert np.array_equal(ci, cls[i, :n].numpy()) and np.array_equal(bi, bonds[i].numpy())
    with pytest.raises(ValueError, match="fewer atoms than minimum"):
        next(gen.generate_stream(ref, n_atoms=23, n_samples=4, variance=2,
                                 fixed_fragment=(torch.zeros(21, 3), torch.eye(8)[[0] * 21])))
    gen.engine.close()


def test_plain_generation_is_unaffected_by_fragment_calls(engines):
    e = engines("fp16")
    ffx, ffh, ref = _fragment()
    n_nodes = np.random.RandomState(6).randint(15, 40, 30).astype(np.int32)
    ctx = _ctx(ref, 30)
    plain = [[t.clone() for t in e.generate_host(n_nodes, 39, ctx, T=T, seed=3)] for _ in range(2)]
    _assert_same(plain[1], plain[0])
    for ifm in (True, False, True):
        _fast(e, ifm, _sizes(30, 7), ffx, ffh, ref, 3, None)
    for _ in range(3):  # eager after the key change, captured, replayed
        _assert_same([t.clone() for t in e.generate_host(n_nodes, 39, ctx, T=T, seed=3)], plain[0])


def _raw_call(e, frag, n_nodes, n=N, ctx=None):
    B = len(n_nodes)
    nn = np.ascontiguousarray(n_nodes, dtype=np.int32)
    ctx = _ctx(torch.tensor([89.87, 210.78, 217.78]), B) if ctx is None else ctx
    steps = e._steps_cached(T, 3)[1]
    out = [torch.empty(B, n, 3), torch.empty(B, n, dtype=torch.int32), torch.empty(B, 42, 42, dtype=torch.int8)]
    rc = e.lib.mlcg_generate_fragment(e.h, C.byref(frag), nn.ctypes.data_as(C.c_void_p), B, n, ctx.ctypes.data, T, steps, 0,
                                      1.0, 1.0, 1.0, 0, 0, None, out[0].data_ptr(), out[1].data_ptr(), out[2].data_ptr(),
                                      e._stream())
    e._check(rc, "generate_fragment")


def test_argument_errors(engines, state_dicts):
    e = engines("fp16")
    ffx, ffh, ref = _fragment()
    x, h = ffx.numpy().copy(), ffh.numpy().copy()
    n_nodes = _sizes(6, 8)
    with pytest.raises(ValueError, match="mode must be 1"):
        _raw_call(e, _lib.Fragment(3, 8, x.ctypes.data, h.ctypes.data), n_nodes)
    with pytest.raises(ValueError, match="null pointer"):
        _raw_call(e, _lib.Fragment(1, 8, None, h.ctypes.data), n_nodes)
    with pytest.raises(ValueError, match="null pointer"):
        _raw_call(e, _lib.Fragment(2, 8, x.ctypes.data, h.ctypes.data), n_nodes)  # IFM without its prologue
    with pytest.raises(ValueError, match="at least one atom"):
        _raw_call(e, _lib.Fragment(1, 0, x.ctypes.data, h.ctypes.data), n_nodes)
    with pytest.raises(ValueError, match="fewer atoms than N"):
        _raw_call(e, _lib.Fragment(1, 8, x.ctypes.data, h.ctypes.data), np.full(6, 8, np.int32), n=8)
    for ifm in (False, True):
        with pytest.raises(ValueError, match="fewer atoms than every sample"):
            _fast(e, ifm, np.array([21, 8, 25], np.int32), ffx, ffh, ref, 0, None)
        with pytest.raises(ValueError, match="fewer atoms than every sample"):
            _fast(e, ifm, np.array([21, 9, 25], np.int32), torch.zeros(9, 3), torch.eye(8)[[0] * 9], ref, 0, None)
    with pytest.raises(ValueError, match="reference_context"):
        e.generate_fragment_host(n_nodes, N, _ctx(ref, 6), ffx, ffh, True, None, T=T)
    with pytest.raises(ValueError, match="one-hot"):
        e.generate_fragment_host(n_nodes, N, _ctx(ref, 6), ffx, ffh[:, :7], False, T=T)
    from ml_conformer_generator_b200.engine import Engine
    bare = Engine(torch.device("cuda:0"), "fp16")
    with pytest.raises(ValueError, match="load both weight sets"):
        bare.generate_fragment_host(n_nodes, N, _ctx(ref, 6), ffx, ffh, False, T=T)
    bare.close()
    # a failed call leaves the handle usable
    _assert_same(_fast(e, False, n_nodes, ffx, ffh, ref, 0, None), _eager(e, False, n_nodes, ffx, ffh, ref, 0, None))


_TWO_RANK = r"""
import os, sys, numpy as np, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from ml_conformer_generator_b200.config import CONTEXT_NORMS
from ml_conformer_generator_b200.engine import Engine
from ml_conformer_generator_b200.mol_utils import normalise_context
from ml_conformer_generator_b200.weights import random_state_dicts
from ml_conformer_generator_b200 import parallel as P
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(rank)
dev = torch.device("cuda", rank)
dist.init_process_group("nccl", device_id=dev)
sd, ssd = random_state_dicts(0)
e = Engine(dev, "bf16"); e.load_edm_state_dict(sd); e.load_seer_state_dict(ssd)
g = dict(np.load(os.path.join(sys.argv[1], "tests", "golden", "host_utils.npz")))
ffx, ffh, ref = torch.from_numpy(g["ifm_ff_x"]), torch.from_numpy(g["ifm_ff_h"]).float(), torch.from_numpy(g["yibfeu_context"])
n_nodes = np.random.RandomState(2).randint(21, 26, 41).astype(np.int32)
ctx = np.tile(normalise_context(ref, CONTEXT_NORMS).numpy().reshape(1, 3), (41, 1)).astype(np.float32)
ok = True
for ifm in (True, False):
    stats = {}
    x, cls, bonds = P.generate_sharded_engine(e, n_nodes, 25, ctx, T=5, resample_steps=1, seed=9, stats=stats,
                                              fixed_fragment=(ffx, ffh), inertial_fragment_matching=ifm,
                                              reference_context=ref, ifm_diffusion_level=3)
    assert stats["calls"] == 1
    if rank == 0:
        xs, cs, bs = e.generate_fragment_host(n_nodes, 25, ctx, ffx, ffh, ifm, ref, None, 5, 1, 3, 3, seed=9)
        ok = ok and torch.equal(x.cpu().view(torch.int32), xs.view(torch.int32)) and torch.equal(cls.cpu(), cs) \
            and torch.equal(bonds.cpu(), bs)
if rank == 0:
    print("SHARDED_FRAGMENT_EQUALS_SINGLE", ok)
dist.barrier()
dist.destroy_process_group()
"""


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_rank_sharded_fragment_generation_equals_single_gpu(tmp_path):
    script = tmp_path / "two_rank_fragment.py"
    script.write_text(_TWO_RANK)
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
                          "127.0.0.1", "--master-port", "29537", str(script), ROOT], capture_output=True, text=True,
                         timeout=900)
    assert out.returncode == 0, out.stderr[-3000:]
    assert "SHARDED_FRAGMENT_EQUALS_SINGLE True" in out.stdout
