"""Two real GPUs, one process each over NCCL: the sharded search (ShardedSearcher) must equal
the unsharded oracle.  Skipped on single-GPU boxes (run with `gpurun --gpus 2`)."""
import os
import socket
import time

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

N, B, K_TOP, VOCAB = 60000, 4, 10, 3000
WEIGHTS = [0.5, 0.6, 0.5, 0.6]


def _inputs():
    from legal_rag_engine_b200 import synth
    x = synth.host_vectors(N, seed=71, dup_frac=0.01)
    idx = synth.host_bm25(N, seed=72, vocab=VOCAB)
    q = synth.host_queries(B, seed=73)
    terms, ptr = synth.host_query_terms(B, 8, seed=74, vocab=VOCAB)
    return x, idx, q, terms, ptr


def _worker(rank, world, port, mode, ret):
    import torch.distributed as dist
    from legal_rag_engine_b200 import sharding
    from legal_rag_engine_b200.device_index import DeviceIndex, FUSION
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        x, idx, q, terms, ptr = _inputs()
        lo, hi = sharding.shard_range(N, rank, world)
        sh = idx.shard(lo, hi)
        dev = DeviceIndex(rank, rank, world)
        dev.set_corpus(torch.from_numpy(x[lo:hi]).cuda(), lo)
        dev.set_postings(sh.term_ptr, sh.postings, sh.doc_len, sh.idf, sh.avgdl)
        s = sharding.ShardedSearcher(dev)
        c = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
        # several batches back to back: the exchange slots and flags are reused every second call;
        # a different (reversed) batch in between must not leak into the last one
        dq, dt, dp, dw = c(q), c(terms), c(ptr), c(np.array(WEIGHTS))
        dq2 = c(q[::-1])
        for i in range(5):
            s.search(dq2 if i % 2 else dq, dt, dp, K_TOP, FUSION[mode], dw)
        torch.cuda.synchronize()
        if rank == 1:
            time.sleep(0.05)                                  # ranks drift apart: flags must hold
        outs = s.search(dq, dt, dp, K_TOP, FUSION[mode], dw)
        torch.cuda.synchronize()
        ret[rank] = [t.cpu().numpy() for t in outs]
        dist.barrier()                                        # nobody unmaps while a peer may store
        dev.close()
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("exchange", ["peer"])
@pytest.mark.parametrize("mode", ["linear", "rrf"])
def test_two_gpu_sharded_search_equals_oracle(mode, exchange):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    from oracle import bm25 as obm25
    from oracle.search import OracleIndex
    x, idx, q, terms, ptr = _inputs()
    csr = obm25.BM25OkapiCSR.from_postings(N, idx.doc_len, idx.term_ptr.astype(np.int64),
                                           idx.postings[:, 0], idx.postings[:, 1])
    lists = [terms[ptr[b]:ptr[b + 1]].tolist() for b in range(B)]
    want = OracleIndex(x, csr).search_batch_vec(q, lists, K_TOP, WEIGHTS, mode)
    with socket.socket() as so:
        so.bind(("127.0.0.1", 0))
        port = so.getsockname()[1]
    with mp.Manager() as mgr:
        ret = mgr.dict()
        mp.spawn(_worker, args=(2, port, mode, ret), nprocs=2, join=True)
        r0, r1 = ret[0], ret[1]
    for a, b in zip(r0, r1):
        np.testing.assert_array_equal(a, b)                   # replicated result
    ids, score, sem, kw, status = r0
    assert status.sum() == 0
    for b in range(B):
        assert ids[b][:len(want[b])].tolist() == [r[0] for r in want[b]]
        assert score[b][:len(want[b])].tolist() == [r[1] for r in want[b]]


# ------------------------------------------------------------------ host buffers, two in flight
def _worker_host(rank, world, port, mode, ret):
    import torch.distributed as dist
    from legal_rag_engine_b200 import sharding, synth
    from legal_rag_engine_b200.device_index import DeviceIndex
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        x, idx, q, terms, ptr = _inputs()
        lo, hi = sharding.shard_range(N, rank, world)
        sh = idx.shard(lo, hi)
        dev = DeviceIndex(rank, rank, world)
        dev.set_corpus(torch.from_numpy(x[lo:hi]).cuda(), lo)
        dev.set_postings(sh.term_ptr, sh.postings, sh.doc_len, sh.idf, sh.avgdl)
        devs = [dev, dev.clone_view()]
        streams = [torch.cuda.Stream(), torch.cuda.Stream()]
        for d, st in zip(devs, streams):
            with torch.cuda.stream(st):
                d.use_current_stream()
            assert d.exchange_setup(8, 16)
        lists = [terms[ptr[b]:ptr[b + 1]].tolist() for b in range(B)]
        lists[1] = lists[1] * 12                               # 96 tokens: past the old 64-slot limit
        got = []
        n_calls = 9                                           # replays of the captured chain included
        for i in range(n_calls):
            d = devs[i % 2]
            if i >= 2:
                got.append(d.search_host_end())
            qq = q if i % 3 else q[::-1].copy()
            d.search_host_begin(qq, lists, K_TOP, WEIGHTS, mode)
            if rank == 1 and i == 4:
                time.sleep(0.05)                              # ranks drift apart: flags must hold
        for i in (n_calls - 2, n_calls - 1):
            got.append(devs[i % 2].search_host_end())
        ret[rank] = got
        dist.barrier()
        for d in devs[::-1]:
            d.close()
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("mode", ["linear", "rrf"])
def test_two_gpu_host_begin_end_pipelined(mode):
    """lrx_search_host_begin/_end on a 2-shard index, two batches in flight per rank, captured chains
    replayed, a 96-token sub-query: every call equals the unsharded oracle on both ranks."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    from oracle import bm25 as obm25
    from oracle.search import OracleIndex
    x, idx, q, terms, ptr = _inputs()
    csr = obm25.BM25OkapiCSR.from_postings(N, idx.doc_len, idx.term_ptr.astype(np.int64),
                                           idx.postings[:, 0], idx.postings[:, 1])
    lists = [terms[ptr[b]:ptr[b + 1]].tolist() for b in range(B)]
    lists[1] = lists[1] * 12
    oracle = OracleIndex(x, csr)
    want_fwd = oracle.search_batch_vec(q, lists, K_TOP, WEIGHTS, mode)
    want_rev = oracle.search_batch_vec(q[::-1].copy(), lists, K_TOP, WEIGHTS, mode)
    with socket.socket() as so:
        so.bind(("127.0.0.1", 0))
        port = so.getsockname()[1]
    with mp.Manager() as mgr:
        ret = mgr.dict()
        mp.spawn(_worker_host, args=(2, port, mode, ret), nprocs=2, join=True)
        r0, r1 = ret[0], ret[1]
    assert len(r0) == len(r1) == 9
    for i, (a, b) in enumerate(zip(r0, r1)):
        want = want_fwd if i % 3 else want_rev
        for g in (a, b):
            ids, score, sem, kw = g
            for bq in range(B):
                assert ids[bq][:len(want[bq])].tolist() == [r[0] for r in want[bq]]
                assert score[bq][:len(want[bq])].tolist() == [r[1] for r in want[bq]]
                assert kw[bq][:len(want[bq])].tolist() == [r[3] for r in want[bq]]


# ------------------------------------------------------------------ the drop-in engine, sharded
def _worker_engine(rank, world, port, tmp, ret):
    import json
    import torch.distributed as dist
    from legal_rag_engine_b200 import synth
    from legal_rag_engine_b200.engine import RetrievalEngine, create_vector_store
    from legal_rag_engine_b200.tokenizer import HashTokenizer
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    os.environ["LOCAL_RANK"] = str(rank)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        sd = synth.bert_state_dict(42, 0.05, ln_jitter=0.1)
        tok = HashTokenizer(30522)
        # data-parallel index build: each rank embeds its chunk range, rank 0 writes the store
        create_vector_store(os.path.join(tmp, "legal_chunks.json"), os.path.join(tmp, "vs"),
                            encoder_state_dict=sd, tokenizer=tok)
        queries = ["What is the procedure for Zero FIR?", "How to file FIR for robbery BNSS procedure",
                   "Victim compensation rights for robbery NALSA scheme", "zzzz-not-in-vocabulary qqqq"]
        weights = [0.5, 0.6, 0.5, 0.6]
        strip = lambda res: [[(r["chunk"]["canonical_header"], r["score"], r["semantic"], r["keyword"])
                              for r in rs] for rs in res]
        single = None
        if rank == 0:
            one = RetrievalEngine(os.path.join(tmp, "vs"), encoder_state_dict=sd, tokenizer=tok,
                                  sharded=False, device=0)
            single = {f: strip(one.search_batch(queries, 5, weights, f)) for f in ("linear", "rrf")}
            xs = np.load(os.path.join(tmp, "vs", "vectors.f16.npy"))
            one_x = one.encode([c["text"] for c in one.chunks[300:364]])   # rank 1's range
            one.close()
        eng = RetrievalEngine(os.path.join(tmp, "vs"), encoder_state_dict=sd, tokenizer=tok)
        assert eng.world == 2 and eng.hi - eng.lo == eng._x.shape[0]
        if rank == 0:
            sharded = {f: strip(eng.search_batch(queries, 5, weights, f)) for f in ("linear", "rrf")}
            sharded["single_again"] = strip([eng.search(queries[0], k=5, hybrid_weight=0.5)])
            ret["single"], ret["sharded"] = single, sharded
            # the rows rank 1 embedded in the data-parallel build equal a one-GPU embedding
            ret["build_ok"] = bool(np.abs(xs[300:364].astype(np.float32) - one_x).max() <= 2e-3)
        else:
            eng.worker_loop()
        eng.close()
    finally:
        dist.destroy_process_group()


def test_two_gpu_sharded_engine_equals_single_gpu(tmp_path, legal_chunks):
    """RetrievalEngine under a 2-rank job (rank 0 serves, rank 1 in worker_loop) returns exactly what
    the one-GPU engine returns -- text in, dicts out -- on a store built data-parallel by both."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import json
    import torch.multiprocessing as mp
    (tmp_path / "legal_chunks.json").write_text(json.dumps(legal_chunks[:600]), encoding="utf-8")
    with socket.socket() as so:
        so.bind(("127.0.0.1", 0))
        port = so.getsockname()[1]
    with mp.Manager() as mgr:
        ret = mgr.dict()
        mp.spawn(_worker_engine, args=(2, port, str(tmp_path), ret), nprocs=2, join=True)
        single, sharded, build_ok = ret["single"], ret["sharded"], ret["build_ok"]
    assert build_ok
    for f in ("linear", "rrf"):
        assert sharded[f] == single[f]
        assert any(len(r) == 5 for r in sharded[f])
    assert sharded["single_again"][0] == single["linear"][0]
