"""Doc-id-range sharding across GPUs and the cross-shard top-k merge.

The corpus is split into contiguous doc-id ranges, rank r owning ``[N*r//R, N*(r+1)//R)`` - the
split the reference already uses to shard corpus *encoding* (mfar/modeling/contrastive.py:470).
Queries / W / mask are replicated.  Each rank scores its shard with GLOBAL doc ids, the packed
(score,id) keys [Q,k] are exchanged with ONE all-gather (NCCL over NVLink), and every rank runs
the same merge kernel - replacing the reference's ``{rank}.qres`` files + barrier + rank-0 merge
(contrastive.py:616-631).
"""
from __future__ import annotations

from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch
import torch.distributed as dist

from . import _native as nv


def shard_range(n_docs: int, rank: int, world: int) -> Tuple[int, int]:
    return n_docs * rank // world, n_docs * (rank + 1) // world


def weighted_shard_ranges(n_docs: int, weights: Sequence[float], align: int = 128) -> List[Tuple[int, int]]:
    """Contiguous doc-id ranges with sizes proportional to ``weights`` (one per rank, e.g. measured docs/s of each
    GPU), boundaries rounded to ``align`` docs.  Every step of a sharded search ends with an exchange that waits for the
    slowest rank, so on a node whose GPUs settle at different clocks under the power cap an equal split runs at the pace
    of the slowest GPU; a speed-weighted split lets every rank finish together.  Equal weights reproduce
    ``shard_range`` up to the rounding."""
    w = [max(float(x), 1e-12) for x in weights]
    total = sum(w)
    cuts, acc = [0], 0.0
    for x in w[:-1]:
        acc += x
        c = int(round(n_docs * acc / total / align)) * align
        cuts.append(min(max(c, cuts[-1]), n_docs))
    cuts.append(n_docs)
    return [(cuts[i], cuts[i + 1]) for i in range(len(w))]


def held_ranges(cuts: Sequence[int], margin: int, n_docs: int) -> List[Tuple[int, int]]:
    """Doc ranges each rank keeps RESIDENT when its active range may move by up to ``margin`` docs at either end:
    rank r holds ``[cuts[r] - margin, cuts[r+1] + margin)`` clipped to the corpus."""
    return [(max(0, cuts[r] - margin), min(n_docs, cuts[r + 1] + margin)) for r in range(len(cuts) - 1)]


def rebalanced_boundaries(cuts: Sequence[int], step_ms: Sequence[float], base_cuts: Sequence[int], margin: int,
                          align: int = 128, damping: float = 0.8) -> List[int]:
    """One step of shard-boundary tuning.  ``cuts`` = current boundaries (``R+1`` doc ids, ``cuts[0] = 0``,
    ``cuts[R] = n_docs``), ``step_ms[r]`` = the time rank r just needed for its range.  Ranges are resized towards
    sizes proportional to the measured docs/ms (``damping`` of the way), boundaries rounded to ``align`` docs (a window
    of a tile-major corpus starts on a tile) and kept within ``margin`` docs of ``base_cuts`` - the ranges the ranks
    hold resident (``held_ranges``), so moving a boundary is a pointer offset on both sides, never a copy.

    Why: the job runs at the pace of its slowest rank, and the GPUs of a node differ by a few per cent under the power
    cap - persistently enough that a calibration on another kernel size or moment mis-predicts it; the real step,
    measured and corrected a few times at start-up, does not."""
    R = len(cuts) - 1
    n_docs = cuts[-1]
    sizes = [cuts[r + 1] - cuts[r] for r in range(R)]
    speed = [sizes[r] / max(float(step_ms[r]), 1e-9) for r in range(R)]
    total = sum(speed)
    target = [n_docs * v / total for v in speed]
    new_sizes = [(1.0 - damping) * sizes[r] + damping * target[r] for r in range(R)]
    out, acc = [0], 0.0
    for r in range(R - 1):
        acc += new_sizes[r]
        c = int(round(acc / align)) * align
        c = min(max(c, base_cuts[r + 1] - margin), base_cuts[r + 1] + margin)     # stay inside what both sides hold
        c = min(max(c, out[-1] + align), n_docs - align * (R - 1 - r))            # ranges stay non-empty and ordered
        out.append(c)
    out.append(n_docs)
    return out


# ---- host-side mirror of the device key packing (csrc/common.cuh) - used by tests and debugging
NAN_ORDERED = 0xFFC00000          # the one score word of every NaN (sign and payload ignored): above +inf's 0xFF800000


def encode_keys(scores: np.ndarray, ids: np.ndarray) -> np.ndarray:
    f = np.ascontiguousarray(scores, dtype=np.float32)
    u = f.view(np.uint32).astype(np.uint64)
    neg = (u & np.uint64(0x80000000)) != 0
    o = np.where(neg, (~u) & np.uint64(0xFFFFFFFF), u | np.uint64(0x80000000))
    o = np.where(np.isnan(f), np.uint64(NAN_ORDERED), o)
    low = (~np.asarray(ids).astype(np.uint64)) & np.uint64(0xFFFFFFFF)
    return (o << np.uint64(32)) | low


def decode_keys(keys: np.ndarray) -> Tuple[np.ndarray, np.ndarray]:
    keys = np.asarray(keys).astype(np.uint64)
    o = (keys >> np.uint64(32)).astype(np.uint32)
    u = np.where((o & np.uint32(0x80000000)) != 0, o & np.uint32(0x7FFFFFFF), ~o)
    scores = u.astype(np.uint32).view(np.float32)
    ids = ((~keys) & np.uint64(0xFFFFFFFF)).astype(np.int64)
    empty = keys == 0
    return np.where(empty, -np.inf, scores).astype(np.float32), np.where(empty, -1, ids)


def all_gather_keys(keys: torch.Tensor, group=None) -> torch.Tensor:
    """keys: int64 view of the packed uint64 keys [Q,k] -> [R,Q,k] (same on every rank)."""
    world = dist.get_world_size(group)
    keys = keys.contiguous()
    out = torch.empty((world * keys.shape[0],) + tuple(keys.shape[1:]), dtype=keys.dtype, device=keys.device)
    dist.all_gather_into_tensor(out, keys, group=group)          # concatenated along dim 0 (gloo and nccl)
    return out.view((world,) + tuple(keys.shape))


def merge_keys(all_keys: torch.Tensor, k: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """[R,Q,k_in] packed keys (device) -> global (scores [Q,k], ids [Q,k]) via mfar_topk_merge."""
    nv.require_device(all_keys, "all_keys")
    R, Q, k_in = all_keys.shape
    scores = torch.empty((Q, k), dtype=torch.float32, device=all_keys.device)
    ids = torch.empty((Q, k), dtype=torch.int64, device=all_keys.device)
    nv.check(nv.lib().mfar_topk_merge(nv.ptr(all_keys.contiguous()), R, Q, k_in, k, 0, nv.ptr(scores), nv.ptr(ids),
                                      nv.stream()), "topk_merge")
    return scores, ids


class PeerExchange:
    """Per-shard [Q,k] key lists exchanged and merged by ONE kernel over NVLink peer memory
    (``mfar_topk_exchange_merge``): every rank stores its keys straight into all peers' exchange buffers, spins on
    per-query flags, merges locally.  No NCCL call on the data path; ``torch.distributed._symmetric_memory`` is only
    the plumbing that maps the peers' buffers into this process (CUDA VMM handles exchanged at rendezvous)."""

    def __init__(self, q_cap: int, k_cap: int = 128, group=None, device=None, peer_buffers=None, rank=None, world=None):
        self.q_cap, self.k_cap = int(q_cap), int(k_cap)
        self.epoch = 0
        self._last_shape = None           # (Q, k_in) of the last push
        if peer_buffers is not None:                      # explicit buffers (tests: "virtual ranks" on one device)
            self.rank, self.world = int(rank), int(world)
            self._bufs = peer_buffers
            self.ptrs = [int(b.data_ptr()) for b in peer_buffers]
        else:
            import torch.distributed._symmetric_memory as symm_mem
            group = group or dist.group.WORLD
            self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
            n = nv.lib().mfar_exchange_buffer_bytes(self.world, self.q_cap, self.k_cap)
            buf = symm_mem.empty(n, dtype=torch.uint8, device=device or torch.device("cuda", torch.cuda.current_device()))
            buf.zero_()
            self._hdl = symm_mem.rendezvous(buf, group.group_name if hasattr(group, "group_name") else group)
            self._bufs = [buf]
            self.ptrs = [int(p) for p in self._hdl.buffer_ptrs]
            torch.cuda.synchronize()
            dist.barrier(group)                           # every rank's flags are zero before anyone pushes
        import ctypes
        self._ptr_arr = (ctypes.c_uint64 * self.world)(*self.ptrs)
        # the call counter lives on the device and is incremented by a one-thread kernel in front of every exchange, so a
        # merge call is identical from launch to launch and can be replayed from a CUDA graph
        dev = peer_buffers[self.rank].device if peer_buffers is not None else self._bufs[0].device
        self.epoch_dev = torch.zeros(1 + 4, dtype=torch.int32, device=dev)   # counter + batch size per exchange slot

    @staticmethod
    def buffer_bytes(world: int, q_cap: int, k_cap: int = 128) -> int:
        return nv.lib().mfar_exchange_buffer_bytes(world, q_cap, k_cap)

    def merge(self, keys: torch.Tensor, k: int) -> Tuple[torch.Tensor, torch.Tensor]:
        """keys: int64 view of this rank's packed keys [Q,k_in] (device) -> global (scores [Q,k], ids [Q,k])."""
        import ctypes
        nv.require_device(keys, "keys")
        Q, k_in = keys.shape
        if Q > self.q_cap or k_in > self.k_cap:
            raise ValueError(f"exchange buffers sized for [{self.q_cap},{self.k_cap}], got [{Q},{k_in}]")
        self.epoch += 1                                   # bookkeeping only (calls issued or captured so far)
        self._last_shape = (Q, k_in)
        scores = torch.empty((Q, k), dtype=torch.float32, device=keys.device)
        ids = torch.empty((Q, k), dtype=torch.int64, device=keys.device)
        nv.check(nv.lib().mfar_topk_exchange_merge_dev_epoch(
            nv.ptr(keys.contiguous()), Q, k_in, k, self.rank, self.world, ctypes.addressof(self._ptr_arr), self.q_cap,
            self.k_cap, nv.ptr(self.epoch_dev), 0, nv.ptr(scores), nv.ptr(ids), nv.stream()), "topk_exchange_merge")
        return scores, ids


    # ---- the exchange in two halves (pipelined sharded step)
    def push(self, keys: torch.Tensor) -> None:
        """Open a new epoch and store this rank's packed keys [Q,k_in] into every rank's buffer; waits for nobody."""
        import ctypes
        nv.require_device(keys, "keys")
        Q, k_in = keys.shape
        if Q > self.q_cap or k_in > self.k_cap:
            raise ValueError(f"exchange buffers sized for [{self.q_cap},{self.k_cap}], got [{Q},{k_in}]")
        self.epoch += 1
        self._last_shape = (Q, k_in)
        nv.check(nv.lib().mfar_topk_exchange_push(nv.ptr(keys.contiguous()), Q, k_in, self.rank, self.world,
                                                  ctypes.addressof(self._ptr_arr), self.q_cap, self.k_cap,
                                                  nv.ptr(self.epoch_dev), nv.stream()), "topk_exchange_push")

    def wait_merge(self, k: int, lag: int = 0) -> Tuple[torch.Tensor, torch.Tensor]:
        """Merge the keys all ranks pushed ``lag`` epochs ago (0: the epoch just pushed, 1: the one before - its peer
        pushes landed a whole step ago, so nothing waits).  Epoch 0 (nothing pushed yet) gives (-inf, -1) rows."""
        import ctypes
        Q, k_in = self._last_shape
        dev = self.epoch_dev.device
        scores = torch.empty((Q, k), dtype=torch.float32, device=dev)
        ids = torch.empty((Q, k), dtype=torch.int64, device=dev)
        nv.check(nv.lib().mfar_topk_exchange_wait_merge(Q, k_in, k, self.rank, self.world,
                                                        ctypes.addressof(self._ptr_arr), self.q_cap, self.k_cap,
                                                        nv.ptr(self.epoch_dev), int(lag), 0, nv.ptr(scores), nv.ptr(ids),
                                                        nv.stream()), "topk_exchange_wait_merge")
        return scores, ids


class ShardedRetriever:
    """One process per GPU; wraps the rank-local ``MultiFieldRetriever`` (built over this rank's doc
    range with ``doc_id_base = shard_range(...)[0]``)."""

    def __init__(self, local, group=None, exchange: Optional[PeerExchange] = None, pipelined: bool = False):
        """``pipelined`` (needs ``exchange``): every ``search`` pushes its own keys and returns the merged result of
        the PREVIOUS call (the first call returns (-inf, -1) rows); ``flush()`` returns the last batch's result.  No
        rank then waits for the slowest rank of the current step - throughput mode for a stream of batches."""
        self.local = local
        self.group = group
        self.exchange = exchange          # None: NCCL/gloo all-gather + merge kernel; else the fused NVLink kernel
        self.pipelined = bool(pipelined) and exchange is not None
        self._k = None

    @torch.no_grad()
    def search(self, q_vecs, q_emb=None, sparse_local=None, top_k: Optional[int] = None, sparse_tokens=None,
               doc_filter=None):
        """``sparse_local``: this shard's columns of the precomputed sparse scores; ``sparse_tokens``: the (replicated)
        query tokens when the local retriever holds this shard's BM25 postings (``DeviceBM25.shard``).
        ``doc_filter``: the GLOBAL doc bitmap of ``MultiFieldRetriever.search`` (the same tensor on every rank: its
        bits are indexed by global doc id, so each shard reads its own range)."""
        k = top_k or self.local.top_k
        k_local = min(k, self.local.n_docs)
        extra = {} if doc_filter is None else {"doc_filter": doc_filter}
        _, _, keys = self.local.search(q_vecs, q_emb, sparse_local, top_k=k_local, return_keys=True,
                                       sparse_tokens=sparse_tokens, **extra)
        if k_local < k:                                   # tiny shard: pad with empty keys
            keys = torch.nn.functional.pad(keys, (0, k - k_local))
        if not dist.is_initialized() or dist.get_world_size(self.group) == 1:
            return merge_keys(keys.unsqueeze(0), k)
        if self.pipelined:
            self._k = k
            self.exchange.push(keys)
            return self.exchange.wait_merge(k, lag=1)
        if self.exchange is not None:
            return self.exchange.merge(keys, k)
        return merge_keys(all_gather_keys(keys, self.group), k)

    def flush(self):
        """Pipelined mode: the merged result of the last ``search`` call."""
        if not self.pipelined or self._k is None:
            raise RuntimeError("flush() belongs to a pipelined ShardedRetriever after at least one search")
        return self.exchange.wait_merge(self._k, lag=0)
