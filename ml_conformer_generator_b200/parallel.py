"""Multi-GPU host logic.  Samples are independent through the whole reverse loop and the GCN (SURVEY.md 8e), so a batch
is sharded across ranks with NO collective inside the loop; the only exchange is ONE all-gather of the packed results
(coordinates, atom classes, bond matrices: ~2.4 kB per molecule).  One process per GPU; `torch.distributed` (NCCL on
GPUs, gloo in the CPU tests of this logic) is the plumbing.

The device noise is keyed by (seed, global sample id) with a per-sample id array (`mlcg_noise.sample_ids`), so a shard
may be ANY subset of the samples: every rank runs its whole shard as one launch sequence (sub-batched only to bound
memory) and the sharded result equals the single-GPU result bit for bit."""
from typing import Callable, List, Optional, Sequence, Tuple

import numpy as np
import torch
import torch.distributed as dist

SEER_D = 42


def sample_cost(n_nodes: np.ndarray) -> np.ndarray:
    """Relative cost of a sample: edge work n(n-1) dominates (F_alg, SURVEY.md 8d), plus the per-node term."""
    n = np.asarray(n_nodes, dtype=np.float64)
    return 9_593_640.0 * n * (n - 1) + 38_122_560.0 * n


def shard_indices(n_nodes: Sequence[int], world_size: int) -> List[np.ndarray]:
    """Deterministic, cost-balanced partition of the sample ids over the ranks: samples sorted by cost (stable) are dealt
    in snake order (0..W-1, W-1..0, ...), so every rank gets the same number of samples (+-1) of every size class and
    the same total cost to within one sample.  Each rank's ids are returned sorted ascending.  Every rank computes the
    same partition from `n_nodes` alone -- no communication."""
    n_nodes = np.asarray(n_nodes)
    order = np.argsort(-sample_cost(n_nodes), kind="stable")
    pos = np.arange(order.size)
    lap, k = pos // world_size, pos % world_size
    rank_of = np.where(lap % 2 == 0, k, world_size - 1 - k)
    return [np.sort(order[rank_of == r]).astype(np.int64) for r in range(world_size)]


def result_bytes(max_n_nodes: int) -> int:
    return max_n_nodes * 3 * 4 + max_n_nodes * 4 + SEER_D * SEER_D


def pack_results(x: torch.Tensor, cls: torch.Tensor, bonds: torch.Tensor) -> torch.Tensor:
    """(n,N,3) f32, (n,N) i32, (n,42,42) i8 -> (n, result_bytes(N)) uint8: one buffer, one collective."""
    n = x.shape[0]
    return torch.cat([x.contiguous().view(torch.uint8).reshape(n, -1), cls.contiguous().view(torch.uint8).reshape(n, -1),
                      bonds.contiguous().view(torch.uint8).reshape(n, -1)], dim=1)


def unpack_results(buf: torch.Tensor, max_n_nodes: int) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    n, N = buf.shape[0], max_n_nodes
    a, b = N * 12, N * 16
    x = buf[:, :a].clone().view(torch.float32).reshape(n, N, 3)
    cls = buf[:, a:b].clone().view(torch.int32).reshape(n, N)
    bonds = buf[:, b:].clone().view(torch.int8).reshape(n, SEER_D, SEER_D)
    return x, cls, bonds


def gather_packed(local: torch.Tensor, shards: List[np.ndarray], total: int, group=None) -> torch.Tensor:
    """The single collective of the path.  `local` (len(shards[rank]), W) holds this rank's rows in the order of
    shards[rank]; returns (total, W) in global sample order on every rank.  Shards may differ in size (or be empty): they
    are padded to the largest shard for the fixed-size all-gather; the shard lists are known on every rank."""
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    width = local.shape[1]
    full = torch.zeros((total, width), dtype=local.dtype, device=local.device)
    if world == 1:
        full[torch.as_tensor(shards[0], device=local.device)] = local
        return full
    cap = max(len(s) for s in shards)
    if cap == 0:
        return full
    pad = torch.zeros((cap, width), dtype=local.dtype, device=local.device)
    pad[: local.shape[0]] = local
    allp = torch.empty((world * cap, width), dtype=local.dtype, device=local.device)
    dist.all_gather_into_tensor(allp, pad, group=group)
    allp = allp.view(world, cap, width)
    for r in range(world):
        k = len(shards[r])
        if k:
            full[torch.as_tensor(shards[r], device=local.device)] = allp[r, :k]
    assert local.shape[0] == len(shards[rank])
    return full


def generate_sharded(run_shard: Callable[[np.ndarray, np.ndarray], Sequence[torch.Tensor]], n_nodes: Sequence[int],
                     max_n_nodes: int, group=None, max_batch: int = 8192, device: Optional[torch.device] = None,
                     stats: Optional[dict] = None) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """Shards `n_nodes` over the ranks of `group`; this rank calls `run_shard(ids, n_nodes[ids])` -- the per-GPU hot path,
    e.g. `Engine.generate_host(..., sample_ids=ids, device_out=True)` -- once per sub-batch of at most `max_batch` of its
    samples (one call for a shard that fits), packs the results and runs the one all-gather.  Returns
    (x (B,N,3) f32, atom_class (B,N) i32, bonds (B,42,42) i8) for ALL samples in global order, on every rank."""
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    n_nodes = np.asarray(n_nodes)
    shards = shard_indices(n_nodes, world)
    mine = shards[rank]
    pieces = []
    for s in range(0, len(mine), max_batch):
        ids = mine[s:s + max_batch]
        x, cls, bonds = run_shard(ids, n_nodes[ids])
        pieces.append(pack_results(x, cls, bonds))
    if stats is not None:
        stats["calls"] = len(pieces)
        stats["shard"] = len(mine)
    if pieces:
        local = torch.cat(pieces, dim=0) if len(pieces) > 1 else pieces[0]
    else:
        local = torch.zeros((0, result_bytes(max_n_nodes)), dtype=torch.uint8, device=device or torch.device("cpu"))
    full = gather_packed(local, shards, len(n_nodes), group)
    return unpack_results(full, max_n_nodes)


def generate_sharded_engine(engine, n_nodes: Sequence[int], max_n_nodes: int, ctx: np.ndarray, T: int = 100,
                            resample_steps: int = 0, seed: int = 0, group=None, max_batch: int = 8192,
                            stats: Optional[dict] = None, fixed_fragment=None, inertial_fragment_matching: bool = True,
                            reference_context=None, blend_power: int = 3, ifm_diffusion_level: int = 50):
    """`generate_sharded` driving `Engine.generate_host` (device outputs): the multi-GPU product path.  ctx: (B,3)
    normalised context of every sample.  With `fixed_fragment` = (coordinates (n,3), one-hot (n,8)) every shard runs
    `Engine.generate_fragment_host` instead (inertial fragment matching needs the raw `reference_context`); the cost of a
    sample still rises with its atom count, so the same size-balanced shards apply."""
    ctx = np.asarray(ctx, dtype=np.float32).reshape(-1, 3)

    def run_shard(ids, nn):
        if fixed_fragment is not None:
            return engine.generate_fragment_host(nn, max_n_nodes, ctx[ids], fixed_fragment[0], fixed_fragment[1],
                                                 inertial_fragment_matching, reference_context, None, T, resample_steps,
                                                 blend_power, ifm_diffusion_level, seed=seed, sample_ids=ids,
                                                 device_out=True)
        return engine.generate_host(nn, max_n_nodes, ctx[ids], T, resample_steps, seed=seed, sample_ids=ids, device_out=True)

    return generate_sharded(run_shard, n_nodes, max_n_nodes, group, max_batch, engine.device, stats)


def generate_jobs_sharded(engine, jobs, T: int = 100, resample_steps: int = 0, blend_power: int = 3,
                          ifm_diffusion_level: int = 50, seed: int = 0, group=None, max_batch: int = 8192,
                          stats: Optional[dict] = None, context_norms=None, min_n_nodes: Optional[int] = None,
                          max_n_nodes: Optional[int] = None):
    """MLConformerGenerator.generate_jobs over the ranks of `group`: the jobs are flattened as there (jobs.flatten_jobs),
    the flat samples dealt with `shard_indices`, and each rank runs the per-kind packed calls of its samples
    (jobs.run_packed, device outputs).  One packed all-gather, then the split per job: every rank returns one dict per
    job, equal bit for bit to the single-GPU result."""
    from .config import CONTEXT_NORMS, MAX_N_NODES, MIN_N_NODES
    from .jobs import flatten_jobs, run_packed, split_jobs
    norms = CONTEXT_NORMS if context_norms is None else context_norms
    packed = flatten_jobs(jobs, seed, norms, MIN_N_NODES if min_n_nodes is None else min_n_nodes,
                          MAX_N_NODES if max_n_nodes is None else max_n_nodes)

    def run_shard(ids, nn):
        return run_packed(engine, packed, ids, T, resample_steps, blend_power, ifm_diffusion_level, seed, max_batch,
                          device_out=True, context_norms=norms)

    x, cls, bonds = generate_sharded(run_shard, packed.n_nodes, packed.N, group, max_batch, engine.device, stats)
    return split_jobs(packed, x, cls, bonds)
