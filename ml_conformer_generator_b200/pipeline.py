"""Host-side overlap of CPU post-processing with GPU generation (SURVEY.md 8f-3).

In the reference, everything after the two GPU models -- bond editing, sanitisation, MMFF, mol-block writing
(conformer_generator.py:357-368, utils/standardizer.py:83-111) -- runs in the calling thread, one molecule at a time, after
the whole batch has been generated.  Once the generation itself takes ~1 ms per molecule that CPU stage is what bounds a
"valid molecules per second" figure.  `GenerationPipeline` runs it in a pool of worker threads on batch k while the GPU
generates batch k + 1:

  * the generator call (e.g. `Engine.generate_host`) blocks inside the C library with the GIL released, so one feeder
    thread keeps the GPU busy;
  * results land in a small ring of output buffers (pinned host memory when the generator provides it); a buffer is handed
    back to the generator only after every worker has finished with it;
  * the post-processing callable gets one molecule's tensors at a time and may be anything -- the RDKit-free V2000 writer of
    this package (default), or RDKit's `redefine_bonds` + `standardize_mol` where RDKit is installed (those release the GIL
    in their C++ parts).  Molecules the callable maps to `None` are dropped, as the reference drops invalid ones.

Nothing here touches CUDA: the class is plain threading around two callables, and is tested on the CPU with stand-ins.
"""
import threading
from concurrent.futures import ThreadPoolExecutor
from typing import Callable, Iterator, List, Optional, Sequence, Tuple

import numpy as np


def _as_numpy(t):
    return t.numpy() if hasattr(t, "numpy") else np.asarray(t)


class GenerationPipeline:
    """generate(k, out) -> (x (B,N,3), atom_class (B,N), bonds (B,42,42), n_nodes (B,)) for batch k, writing into / returning
    host buffers (`out` is the buffer set to reuse, or None on first use); postprocess(x_i, cls_i, bonds_i, n_i, global_index)
    -> result or None for one molecule."""

    def __init__(self, generate: Callable, postprocess: Callable, n_workers: int = 8, depth: int = 2, chunk: int = 64):
        if depth < 2:
            raise ValueError("depth must be >= 2: one buffer is being filled while another is being post-processed")
        self.generate, self.postprocess = generate, postprocess
        self.n_workers, self.depth, self.chunk = max(1, n_workers), depth, max(1, chunk)
        self.stats = {"batches": 0, "molecules": 0, "kept": 0}

    def _post_chunk(self, bufs, lo, hi, base):
        x, cls, bonds, n_nodes = bufs
        out = []
        for i in range(lo, hi):
            n = int(n_nodes[i])
            out.append(self.postprocess(x[i, :n], cls[i, :n], bonds[i], n, base + i))
        return out

    def run(self, n_batches: int) -> Iterator[List]:
        """Yields, batch by batch and in order, the list of post-processed molecules (None results dropped)."""
        free = threading.Semaphore(self.depth)
        ready: List[Optional[Tuple]] = [None] * n_batches
        events = [threading.Event() for _ in range(n_batches)]
        slots = [None] * self.depth
        err: List[BaseException] = []

        def feeder():
            try:
                for k in range(n_batches):
                    free.acquire()
                    if err:
                        return
                    s = k % self.depth
                    res = self.generate(k, slots[s])
                    slots[s] = res
                    ready[k] = tuple(_as_numpy(t) for t in res)
                    events[k].set()
            except BaseException as e:  # surface generator errors in the consumer
                err.append(e)
                for ev in events:
                    ev.set()

        th = threading.Thread(target=feeder, name="mlcg-generate", daemon=True)
        th.start()
        base = 0
        with ThreadPoolExecutor(max_workers=self.n_workers, thread_name_prefix="mlcg-post") as pool:
            for k in range(n_batches):
                events[k].wait()
                if ready[k] is None:      # the generator failed at (or before) this batch
                    raise err[0]
                bufs = ready[k]
                B = int(bufs[0].shape[0])
                futs = [pool.submit(self._post_chunk, bufs, lo, min(lo + self.chunk, B), base)
                        for lo in range(0, B, self.chunk)]
                results = [r for f in futs for r in f.result()]   # GPU is already generating batch k + 1 meanwhile
                ready[k] = None
                free.release()                                    # the buffer set of batch k may be overwritten now
                kept = [r for r in results if r is not None]
                self.stats["batches"] += 1
                self.stats["molecules"] += B
                self.stats["kept"] += len(kept)
                base += B
                yield kept
        th.join()


def sdf_postprocess(x, cls, bonds, n, index) -> str:
    """Default post-processing: one RDKit-free V2000 block (provisional bond orders, see mol_utils.samples_to_sdf_blocks)."""
    import torch

    from .mol_utils import samples_to_sdf_blocks
    return samples_to_sdf_blocks(torch.from_numpy(np.ascontiguousarray(x)).unsqueeze(0),
                                 torch.from_numpy(np.ascontiguousarray(cls)).unsqueeze(0),
                                 torch.from_numpy(np.ascontiguousarray(bonds)).unsqueeze(0), [n], names=["mlcg_%d" % index])[0]


def engine_batches(engine, n_nodes_per_batch: Sequence[np.ndarray], max_n_nodes: int, ctx_per_batch: Sequence[np.ndarray],
                   T: int = 100, seed: int = 0, fixed_fragment=None, inertial_fragment_matching: bool = True,
                   reference_context=None, context_norms=None, blend_power: int = 3,
                   ifm_diffusion_level: int = 50) -> Callable:
    """`generate` callable over `Engine.generate_host`: batch k gets global sample ids following the previous batches (so the
    whole run equals one big batch, bit for bit) and reuses the pinned output buffers of its ring slot.  With
    `fixed_fragment` = (coordinates (n,3), one-hot (n,8)) it calls `Engine.generate_fragment_host` instead."""
    offsets = np.concatenate([[0], np.cumsum([len(n) for n in n_nodes_per_batch])])

    def generate(k, out):
        nn = np.asarray(n_nodes_per_batch[k], dtype=np.int32)
        reuse = None
        if out is not None and tuple(out[0].shape) == (len(nn), max_n_nodes, 3):
            reuse = out[:3]
        ids = np.arange(offsets[k], offsets[k + 1])
        if fixed_fragment is not None:
            x, cls, bonds = engine.generate_fragment_host(nn, max_n_nodes, ctx_per_batch[k], fixed_fragment[0],
                                                          fixed_fragment[1], inertial_fragment_matching, reference_context,
                                                          context_norms, T, 0, blend_power, ifm_diffusion_level, seed=seed,
                                                          sample_ids=ids, out=reuse)
        else:
            x, cls, bonds = engine.generate_host(nn, max_n_nodes, ctx_per_batch[k], T, 0, seed=seed, sample_ids=ids,
                                                 out=reuse)
        return x, cls, bonds, nn

    return generate
