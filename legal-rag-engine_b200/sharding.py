"""Multi-GPU layout of the hybrid index: one process per GPU (torchrun), aligned row shards,
one exchange of candidate records per query batch (SURVEY.md 8e).

GPU g owns the contiguous global id range ``shard_range(N, g, G)`` of BOTH the fp16 chunk
matrix and the BM25 postings (doc ids local, ``id_base`` added on the way out).  idf / avgdl
are whole-corpus statistics (``global_bm25_stats``: two all-reduces at build time), so a
shard's BM25 scores equal the unsharded ones bit for bit.  Per query batch each rank runs
K2 + K3 on its shard, the packed blocks ``[B][2][2k] records | [B] max | [B] flags`` (~1 KB per
sub-query per rank -- latency-bound) are exchanged, and every rank runs the same deterministic
merge + fusion.  The exchange is ``lrx_search_sharded``: a kernel of the chain stores the block
straight into every peer's memory over NVLink and the fusion kernel acquires the peers' sequence
flags; no collective call per batch (the IPC handles are swapped once).
"""
from __future__ import annotations

from typing import Tuple

import numpy as np
import torch
import torch.distributed as dist

RECORD = np.dtype([("id", "<i8"), ("dense", "<f8"), ("bm25", "<f8")])


def shard_range(n: int, rank: int, world: int) -> Tuple[int, int]:
    per = -(-n // world)
    return min(n, rank * per), min(n, (rank + 1) * per)


def global_bm25_stats(df_local: torch.Tensor, total_len_local: int, group=None):
    """Sum document frequencies and token counts over the shards (in place on ``df_local``'s
    device: CUDA tensors go over NCCL, CPU tensors over gloo).  Returns (df_global, total_len)."""
    df = df_local.clone()
    tl = torch.tensor([int(total_len_local)], dtype=torch.int64, device=df.device)
    if dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(df, group=group)
        dist.all_reduce(tl, group=group)
    return df, int(tl.item())


def packed_layout(B: int, k: int):
    """Byte offsets of the packed per-shard block (must equal packed_layout in csrc/api.cu)."""
    rec = B * 2 * (2 * k) * RECORD.itemsize
    o_max = rec
    o_flags = rec + B * 8
    total = (o_flags + B * 4 + 15) // 16 * 16
    return o_max, o_flags, total


def unpack(block: np.ndarray, B: int, k: int):
    """uint8 [total] -> (records [B,2,2k] structured, max f64 [B], flags i32 [B]) views."""
    o_max, o_flags, total = packed_layout(B, k)
    assert block.dtype == np.uint8 and block.size == total
    rec = block[:o_max].view(RECORD).reshape(B, 2, 2 * k)
    return rec, block[o_max:o_max + 8 * B].view("<f8"), block[o_flags:o_flags + 4 * B].view("<i4")


class ShardedSearcher:
    """K2+K3 local -> peer exchange -> K4, for device-resident query batches."""

    exchange = "peer"          # the only cross-shard path; bench.py reports it

    def __init__(self, dev, group=None, B_max: int = 64, k_max: int = 128):
        self.dev = dev
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self._bufs = {}
        if self.world > 1 and not dev.exchange_setup(B_max, k_max, group):
            raise RuntimeError("the GPUs of this box cannot map each other's memory (CUDA IPC / peer "
                               "access): the sharded engine needs it")

    def buffers(self, B: int, k: int):
        # a 3-tuple whose third item is the output tuple: the layout bench.py reads
        key = (B, k)
        if key not in self._bufs:
            self._bufs[key] = (None, None, self.dev.alloc_outputs(B, k))
        return self._bufs[key]

    def search(self, q_fp16: torch.Tensor, q_terms: torch.Tensor, q_ptr: torch.Tensor, k: int, mode: int,
               weights: torch.Tensor, width: int = 0):
        """-> (ids, score, semantic, keyword, status) device tensors [B,k] (replicated on every
        rank).  Asynchronous on torch's current stream; `status` must be looked at by the caller
        (`search_checked` does) -- 0 ok, 1 = exactness guard (rerun wider), 2 = token capacity,
        -1 = a peer's block did not arrive in time."""
        outs = self.buffers(int(q_fp16.shape[0]), k)[2]
        return self.dev.search_sharded(q_fp16, q_terms, q_ptr, k, mode, weights, outs, width)

    def search_checked(self, q_fp16, q_terms, q_ptr, k: int, mode: int, weights):
        """`search` + a synchronising look at the status words: widens the dense candidate lists
        (x2 up to 512) while the exactness guard trips, raises on a lost peer or on a query longer
        than the token capacity.  The status is the OR over all shards and the result is
        replicated, so every rank takes the same branch (SPMD)."""
        from ._lib import LRX_E_AMBIGUOUS, LRX_E_PEER, LrxError
        width = 0
        while True:
            outs = self.search(q_fp16, q_terms, q_ptr, k, mode, weights, width)
            st = outs[4].cpu().numpy()
            if (st < 0).any():
                raise LrxError(LRX_E_PEER, "a peer shard did not publish its candidates in time")
            if (st & 2).any():
                raise LrxError(-1, "a shard saw more query tokens than its capacity")
            if not st.any():
                return outs
            if width == 0:                                   # the library's default for this depth
                width = 64
                while width < 2 * k + 32:
                    width *= 2
            width *= 2
            if width > 512:
                raise LrxError(LRX_E_AMBIGUOUS, "dense candidates are not separable at width 512")
