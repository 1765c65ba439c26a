"""world_size-2 gloo test (CPU) of the multi-GPU host logic: aligned shard ranges, global BM25
statistics by all-reduce, the per-shard packed record block exchanged between the ranks, and the
merge rule -- with the CPU oracle standing in for the per-shard kernels.  The result on every rank
must equal the unsharded oracle search."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from legal_rag_engine_b200 import sharding, synth
from legal_rag_engine_b200.bm25_index import okapi_idf
from oracle import bm25 as obm25
from oracle import flat_ip, fusion
from oracle.search import OracleIndex

N, B, K_TOP, VOCAB = 5000, 3, 10, 1500
WEIGHTS = [0.5, 0.6, 0.5]


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _inputs():
    x = synth.host_vectors(N, seed=61, dup_frac=0.01)
    idx = synth.host_bm25(N, seed=62, vocab=VOCAB)
    q = synth.host_queries(B, seed=63)
    terms, ptr = synth.host_query_terms(B, 8, seed=64, vocab=VOCAB)
    return x, idx, q, [terms[ptr[b]:ptr[b + 1]].tolist() for b in range(B)]


def _oracle_local_block(x_sh, csr_sh, lo, q, lists, k, mode):
    """The packed block one shard's K2 + K3 emit, computed by the oracle."""
    o_max, o_flags, total = sharding.packed_layout(B, k)
    block = np.zeros(total, dtype=np.uint8)
    rec, mx, flags = sharding.unpack(block, B, k)
    rec["id"] = -1
    rec["dense"] = -np.inf
    K = 2 * k
    for b in range(B):
        s = flat_ip.exact_scores(x_sh, q[b][None])
        E, _, I = flat_ip.topk_from_scores(s, K, id_base=lo)
        bm = csr_sh.get_scores_ids(lists[b])
        n = int((I[0] >= 0).sum())
        rec[b, 0, :n]["id"] = I[0, :n]
        rec[b, 0, :n]["dense"] = E[0, :n]
        rec[b, 0, :n]["bm25"] = bm[I[0, :n] - lo]
        mx[b] = max(float(bm.max()), 0.0) if len(bm) else 0.0
        if mode == "rrf":
            bs, bi = obm25.topk_positive(bm, K, id_base=lo)
            rec[b, 1, :len(bi)]["id"] = bi
            rec[b, 1, :len(bi)]["bm25"] = bs
            rec[b, 1, :len(bi)]["dense"] = s[0, bi - lo]
    return block


def _oracle_finish(blocks, world, k, mode, weights):
    """The merge rule of K4 (fuse_kernel): (score desc, id asc) over the union."""
    K = 2 * k
    out = []
    parts = [sharding.unpack(blocks[r], B, k) for r in range(world)]
    for b in range(B):
        dense = [(float(r["dense"]), int(r["id"]), float(r["bm25"])) for p in parts for r in p[0][b, 0] if r["id"] >= 0]
        dense.sort(key=lambda t: (-t[0], t[1]))
        dense = dense[:K]
        mx = max(float(p[1][b]) for p in parts)
        mx = mx if mx > 0 else 1.0
        if mode == "linear":
            D = np.array([np.float32(d) for d, _, _ in dense], dtype=np.float32)
            I = np.array([i for _, i, _ in dense], dtype=np.int64)
            bm = {i: s for _, i, s in dense}
            out.append(fusion.linear_fuse(D, I, bm, mx, k, weights[b]))
        else:
            sparse = [(float(r["bm25"]), int(r["id"]), float(r["dense"])) for p in parts for r in p[0][b, 1] if r["id"] >= 0]
            sparse.sort(key=lambda t: (-t[0], t[1]))
            sparse = sparse[:K]
            out.append(fusion.rrf_fuse([(i, d, s) for d, i, s in dense], [(i, d, s) for s, i, d in sparse], mx, k))
    return out


def _worker(rank, world, port, mode, ret):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        x, idx, q, lists = _inputs()
        lo, hi = sharding.shard_range(N, rank, world)
        sh = idx.shard(lo, hi)
        # global statistics from the shards alone: df and token counts all-reduced
        df_local = torch.from_numpy(np.diff(sh.term_ptr.astype(np.int64)))
        df, total_len = sharding.global_bm25_stats(df_local, int(sh.doc_len.astype(np.int64).sum()))
        idf, _ = okapi_idf(df.numpy(), N)
        np.testing.assert_array_equal(idf, idx.idf)
        assert total_len / N == idx.avgdl
        csr_sh = obm25.BM25OkapiCSR(hi - lo, sh.doc_len, sh.term_ptr.astype(np.int64), sh.postings[:, 0],
                                    sh.postings[:, 1])
        csr_sh.idf, csr_sh.avgdl = idf, total_len / N        # global statistics on the shard
        csr_sh.doc_norm = csr_sh.k1 * (1 - csr_sh.b + csr_sh.b * csr_sh.doc_len / csr_sh.avgdl)
        mine = torch.from_numpy(_oracle_local_block(x[lo:hi], csr_sh, lo, q, lists, K_TOP, mode))
        every = torch.empty(mine.numel() * world, dtype=torch.uint8)
        dist.all_gather_into_tensor(every, mine)              # the one exchange per query batch
        blocks = every.numpy().reshape(world, -1)
        ret[rank] = _oracle_finish(blocks, world, K_TOP, mode, WEIGHTS)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("mode", ["linear", "rrf"])
def test_two_rank_exchange_equals_unsharded(mode):
    x, idx, q, lists = _inputs()
    csr = obm25.BM25OkapiCSR.from_postings(N, idx.doc_len, idx.term_ptr.astype(np.int64),
                                           idx.postings[:, 0], idx.postings[:, 1])
    want = OracleIndex(x, csr).search_batch_vec(q, lists, K_TOP, WEIGHTS, mode)
    port = _free_port()
    with mp.Manager() as mgr:
        ret = mgr.dict()
        mp.spawn(_worker, args=(2, port, mode, ret), nprocs=2, join=True)
        got0, got1 = ret[0], ret[1]
    assert got0 == got1 == want


def test_shard_ranges_tile_the_corpus():
    for n in (0, 1, 7, 1000, 10_000_000):
        for world in (1, 2, 3, 8):
            cuts = [sharding.shard_range(n, r, world) for r in range(world)]
            assert cuts[0][0] == 0 and cuts[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(cuts[:-1], cuts[1:]))
