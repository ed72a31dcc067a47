"""CPU: the host logic of fragment-conditioned generation -- sharding (gloo, world size 2) and streaming batches with a
stand-in engine that records its calls -- and the inertial-fragment-matching prologue shared by the device entry points."""
import os

import numpy as np
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import golden
from ml_conformer_generator_b200 import parallel as P
from ml_conformer_generator_b200.config import CONTEXT_NORMS
from ml_conformer_generator_b200.mol_utils import ifm_moi_prologue, ifm_prepare_gen_fragment_context, shift_moi_to_com_batch
from ml_conformer_generator_b200.pipeline import engine_batches

N_MAX = 25
FRAG = (torch.arange(12, dtype=torch.float32).view(4, 3), torch.eye(8)[[6, 6, 0, 0]])
REF = [89.8693, 210.7831, 217.7827]


class FakeEngine:
    """Stand-in for Engine: every output row is a pure function of (global sample id, atom count, call arguments), like
    the keyed device RNG; only generate_fragment_host exists, so a plain call fails."""
    device = torch.device("cpu")

    def __init__(self):
        self.calls = []

    def generate_fragment_host(self, n_nodes, max_n_nodes, ctx, fragment_x, fragment_h, inertial_fragment_matching=True,
                               reference_context=None, context_norms=None, T=100, resample_steps=0, blend_power=3,
                               diffusion_level=50, seed=0, sample_offset=0, sample_ids=None, out=None, device_out=False):
        ids = np.asarray(sample_ids)
        self.calls.append(dict(ids=ids.copy(), n_ff=int(fragment_x.shape[0]), ifm=inertial_fragment_matching,
                               ref=reference_context, T=T, r=resample_steps, bp=blend_power, L=diffusion_level, seed=seed,
                               reuse=out is not None, device_out=device_out))
        tag = float(seed + 10 * diffusion_level + 1000 * inertial_fragment_matching + fragment_x.sum())
        ids_t = torch.as_tensor(ids, dtype=torch.float32).view(-1, 1, 1)
        x = ids_t + tag + torch.as_tensor(ctx, dtype=torch.float32)[:, :1].view(-1, 1, 1) * torch.ones(len(ids), max_n_nodes, 3)
        cls = (torch.as_tensor(ids).view(-1, 1) + torch.as_tensor(n_nodes).view(-1, 1)).repeat(1, max_n_nodes).to(torch.int32)
        bonds = (torch.as_tensor(ids).view(-1, 1, 1) % 5).repeat(1, 42, 42).to(torch.int8)
        if out is not None:
            for o, r in zip(out, (x, cls, bonds)):
                o.copy_(r)
            return out
        return x, cls, bonds


def _sharded(n_nodes, max_batch, ifm):
    e = FakeEngine()
    ctx = np.arange(len(n_nodes) * 3, dtype=np.float32).reshape(-1, 3)
    res = P.generate_sharded_engine(e, n_nodes, N_MAX, ctx, T=7, resample_steps=1, seed=3, max_batch=max_batch,
                                    fixed_fragment=FRAG, inertial_fragment_matching=ifm, reference_context=REF,
                                    blend_power=2, ifm_diffusion_level=4)
    return res, e.calls


def _worker(rank, world, port, n_nodes, tmp, max_batch):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.save([_sharded(n_nodes, max_batch, ifm) for ifm in (True, False)], tmp + ".%d" % rank)
    dist.barrier()
    dist.destroy_process_group()


def _run(tmp_path, n_nodes, port, max_batch=8192):
    single = [_sharded(n_nodes, max_batch, ifm) for ifm in (True, False)]
    out_file = str(tmp_path / "gathered.pt")
    mp.spawn(_worker, args=(2, port, n_nodes, out_file, max_batch), nprocs=2, join=True)
    ranks = [torch.load(out_file + ".%d" % r, weights_only=False) for r in range(2)]
    shards = P.shard_indices(n_nodes, 2)
    for m, (want, single_calls) in enumerate(single):
        assert [c["ids"].tolist() for c in single_calls] == [list(range(s, min(s + max_batch, len(n_nodes))))
                                                             for s in range(0, len(n_nodes), max_batch)]
        for r in range(2):
            got, calls = ranks[r][m]
            for a, b in zip(want, got):  # every rank holds the whole job in global order
                assert a.dtype == b.dtype and torch.equal(a, b)
            # each rank ran its own shard, in sub-batches of at most max_batch ids, with the fragment arguments
            assert np.array_equal(np.concatenate([c["ids"] for c in calls] or [np.zeros(0, np.int64)]), shards[r])
            assert all(len(c["ids"]) <= max_batch for c in calls)
            for c in calls:
                assert (c["n_ff"], c["ifm"], c["ref"], c["T"], c["r"], c["bp"], c["L"], c["seed"], c["device_out"]) == \
                    (4, m == 0, REF, 7, 1, 2, 4, 3, True)
    return [[len(ranks[r][m][1]) for r in range(2)] for m in range(2)]


def test_sharded_fragment_generation_matches_single_process(tmp_path):
    n_nodes = np.random.RandomState(1).randint(21, 26, size=37)
    assert _run(tmp_path, n_nodes, 29527) == [[1, 1], [1, 1]]


def test_sharded_fragment_generation_sub_batches(tmp_path):
    assert _run(tmp_path, np.full(64, 25), 29528, max_batch=10) == [[4, 4], [4, 4]]


def test_sharded_fragment_generation_with_an_empty_shard(tmp_path):
    assert [sorted(c) for c in _run(tmp_path, np.array([23]), 29529)] == [[0, 1], [0, 1]]


def test_engine_batches_with_a_fragment():
    e = FakeEngine()
    nn = [np.array([21, 22, 23]), np.array([24, 25]), np.array([21])]
    cx = [np.full((len(b), 3), k, np.float32) for k, b in enumerate(nn)]
    gen = engine_batches(e, nn, N_MAX, cx, T=9, seed=4, fixed_fragment=FRAG, inertial_fragment_matching=False,
                         reference_context=REF, context_norms=CONTEXT_NORMS, blend_power=2, ifm_diffusion_level=6)
    first = gen(0, None)
    second = gen(1, None)
    again = gen(2, first)      # other batch size: new buffers
    reused = gen(0, first)     # same batch size: the ring slot's buffers are reused
    assert [c["ids"].tolist() for c in e.calls] == [[0, 1, 2], [3, 4], [5], [0, 1, 2]]
    assert [c["reuse"] for c in e.calls] == [False, False, False, True]
    assert all((c["n_ff"], c["ifm"], c["T"], c["r"], c["bp"], c["L"], c["seed"]) == (4, False, 9, 0, 2, 6, 4) for c in e.calls)
    assert reused[0] is first[0] and np.array_equal(reused[3], nn[0])
    assert second[0].shape == (2, N_MAX, 3) and again[0].shape == (1, N_MAX, 3)
    assert float(second[0][1, 0, 0]) == 4 + 4 + 60 + float(FRAG[0].sum()) + 1  # id 4, ctx of batch 1


def test_ifm_moi_prologue_equals_the_reference_host_values():
    g = golden("host_utils")
    ffx, ref = torch.from_numpy(g["ifm_ff_x"]), torch.from_numpy(g["yibfeu_context"])
    n_nodes = torch.from_numpy(g["ifm_n_nodes"])
    moi0, com = ifm_moi_prologue(ffx, ref)
    assert moi0.shape == (3, 3) and com.shape == (3,) and moi0.dtype == com.dtype == torch.float32
    _, _, ctx, shift, rot = ifm_prepare_gen_fragment_context(ffx, ref, CONTEXT_NORMS, n_nodes, 25, 21)
    n_gen = n_nodes.view(-1, 1).float() - ffx.shape[0]
    assert torch.equal(com.view(1, 3) / n_gen, shift)
    b = n_nodes.numel()
    w, v = torch.linalg.eigh(shift_moi_to_com_batch(moi0.unsqueeze(0).repeat(b, 1, 1), shift, n_gen))
    mean, mad = (torch.as_tensor(CONTEXT_NORMS[k], dtype=torch.float32) for k in ("mean", "mad"))
    assert torch.equal((w - mean) / mad, ctx[:, 0, :]) and torch.equal(v, rot)
    # and the golden values the reference itself produced
    assert float((shift - torch.from_numpy(g["ifm_shift"])).abs().max()) < 1e-6
