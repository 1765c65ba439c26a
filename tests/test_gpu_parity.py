"""Parity of the CUDA path (through the C ABI) with the CPU oracle: bit-exact ids,
scores and fused order.  Runs on the B200 box (`-m gpu`)."""
import numpy as np
import pytest
import torch

from oracle import bm25 as obm25
from oracle import flat_ip
from oracle.search import OracleIndex

from legal_rag_engine_b200 import synth
from legal_rag_engine_b200.bm25_index import BM25Index, tokenize

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    from legal_rag_engine_b200.device_index import DeviceIndex
    d = DeviceIndex(0)
    yield d
    d.close()


def _csr_of(idx: BM25Index):
    return obm25.BM25OkapiCSR.from_postings(idx.n_docs, idx.doc_len, idx.term_ptr.astype(np.int64),
                                            idx.postings[:, 0], idx.postings[:, 1])


def _set_postings(dev, idx: BM25Index):
    dev.set_postings(idx.term_ptr, idx.postings, idx.doc_len, idx.idf, idx.avgdl, idx.k1, idx.b)


def _cuda(a, dt=None):
    t = torch.from_numpy(np.ascontiguousarray(a)).cuda()
    return t if dt is None else t.to(dt)


# ------------------------------------------------------------------ K2 dense
@pytest.mark.parametrize("n", [1, 5, 63, 64, 65, 1000, 20011, 300000])
@pytest.mark.parametrize("B", [1, 2, 3, 4, 5, 7, 8])     # 5..8: the 8-queries-per-pass instantiation
def test_dense_topk_matches_oracle(dev, n, B):
    x = synth.host_vectors(n, seed=100 + n, dup_frac=0.01)
    q = synth.host_queries(B, seed=7 + B)
    if n > 10:
        q[0] = synth.host_planted_queries(x, [n // 3], seed=1)[0]
    dev.set_corpus(_cuda(x), id_base=1000)
    s = flat_ip.exact_scores(x, q)
    for K in (1, 20, 200):
        Eo, Do, Io = flat_ip.topk_from_scores(s, K, id_base=1000)
        E, D, I, flags = dev.dense_topk(_cuda(q), K)
        assert flags.cpu().numpy().sum() == 0
        np.testing.assert_array_equal(I.cpu().numpy(), Io)
        np.testing.assert_array_equal(E.cpu().numpy(), Eo)        # exact float64, bit for bit
        np.testing.assert_array_equal(D.cpu().numpy(), Do)
    if n > 10:
        assert I[0, 0].item() == 1000 + n // 3 or s[0].argmax() != n // 3


def test_dense_topk_exact_duplicates_order_by_id(dev):
    x = synth.host_vectors(5000, seed=5, dup_frac=0.0)
    x[10:40] = x[4000]                       # 31 identical rows
    q = synth.host_planted_queries(x, [4000], seed=2)
    dev.set_corpus(_cuda(x), 0)
    E, D, I, flags = dev.dense_topk(_cuda(q), 20)
    assert flags.item() == 0
    Eo, Do, Io = flat_ip.topk_from_scores(flat_ip.exact_scores(x, q), 20)
    np.testing.assert_array_equal(I.cpu().numpy(), Io)
    assert I[0, :20].tolist() == list(range(10, 30))


def test_dense_guard_flags_unseparable_candidates(dev):
    # 600 identical rows tie at the top: width 64 cannot prove exactness -> flag set
    x = synth.host_vectors(4000, seed=6, dup_frac=0.0)
    x[100:700] = x[0]
    q = synth.host_planted_queries(x, [0], seed=3)
    dev.set_corpus(_cuda(x), 0)
    E, D, I, flags = dev.dense_topk(_cuda(q), 20, width=64)
    assert flags.item() == 1


def test_dense_at(dev):
    x = synth.host_vectors(3000, seed=8)
    q = synth.host_queries(2, seed=9)
    dev.set_corpus(_cuda(x), 500)
    ids = np.array([[500, 3499, 499, -1, 3500, 777], [1000, 1001, 1002, 1003, 1004, 1005]], dtype=np.int64)
    out = dev.dense_at(_cuda(q), _cuda(ids)).cpu().numpy()
    s = flat_ip.exact_scores(x, q)
    for b in range(2):
        for j, i in enumerate(ids[b]):
            if 500 <= i < 3500:
                assert out[b, j] == s[b, i - 500]
            else:
                assert out[b, j] == -np.inf


# ------------------------------------------------------------------- K3 bm25
def _check_bm25(dev, idx, csr, term_lists, id_base=0, K=20, n_cand=16, seed=0):
    rng = np.random.default_rng(seed)
    B = len(term_lists)
    ptr = np.zeros(B + 1, dtype=np.int32)
    for i, t in enumerate(term_lists):
        ptr[i + 1] = ptr[i] + len(t)
    terms = np.array([x for t in term_lists for x in t] or [0], dtype=np.int32)
    cand = rng.integers(id_base - 2, id_base + idx.n_docs + 2, size=(B, n_cand)).astype(np.int64)
    cand[:, 0] = -1
    cs, mx, ts, ti = dev.bm25(_cuda(terms), _cuda(ptr), _cuda(cand), K)
    cs, mx, ts, ti = cs.cpu().numpy(), mx.cpu().numpy(), ts.cpu().numpy(), ti.cpu().numpy()
    for b in range(B):
        s = csr.get_scores_ids(term_lists[b])
        pos = s[s > 0]
        assert mx[b] == (pos.max() if len(pos) else 0.0)
        for j in range(n_cand):
            i = cand[b, j] - id_base
            want = s[i] if (cand[b, j] >= 0 and 0 <= i < idx.n_docs) else 0.0
            assert cs[b, j] == want                        # bit for bit
        so, io = obm25.topk_positive(s, K, id_base)
        np.testing.assert_array_equal(ti[b, :len(io)], io)
        np.testing.assert_array_equal(ts[b, :len(io)], so)
        assert (ti[b, len(io):] == -1).all()


def test_bm25_real_corpus_bit_exact(dev, legal_texts, reference_queries):
    idx = BM25Index.from_texts(legal_texts)
    csr = obm25.BM25OkapiCSR.from_corpus([obm25.tokenize(t) for t in legal_texts])
    dev.set_corpus(_cuda(synth.host_vectors(idx.n_docs, seed=1)), 0)
    _set_postings(dev, idx)
    lists = [idx.term_ids(tokenize(q)) for q in reference_queries]
    _check_bm25(dev, idx, csr, lists, K=20)
    _check_bm25(dev, idx, csr, lists[:4], K=200)
    _check_bm25(dev, idx, csr, lists[:3], K=0)


@pytest.mark.parametrize("n,vocab", [(1, 10), (2047, 300), (2048, 300), (16385, 1000), (120000, 5000)])
def test_bm25_synthetic_bit_exact(dev, n, vocab):
    idx = synth.host_bm25(n, seed=n, vocab=vocab)
    csr = _csr_of(idx)
    dev.set_corpus(_cuda(synth.host_vectors(n, seed=2)), 77)
    _set_postings(dev, idx)
    terms, ptr = synth.host_query_terms(5, 8, seed=n + 1, vocab=vocab)
    lists = [terms[ptr[b]:ptr[b + 1]].tolist() for b in range(5)]
    lists[1] = lists[1] + [lists[1][0], -1, lists[1][0]]      # repeats + OOV
    lists[4] = []
    _check_bm25(dev, idx, csr, lists, id_base=77, K=20, seed=n)


def test_bm25_long_queries_any_length(dev):
    """More than 32 token slots: the scan walks a unit once per 32 slots.  EVERY token counts, as in
    the reference (retrieval_engine.py:67-68 scores all of query.lower().split()): 33, 64, 65 and
    200 tokens, repeats and out-of-vocabulary ids included."""
    n, vocab = 50000, 2000
    idx = synth.host_bm25(n, seed=5, vocab=vocab)
    csr = _csr_of(idx)
    dev.set_corpus(_cuda(synth.host_vectors(n, seed=2)), 0)
    _set_postings(dev, idx)
    terms, ptr = synth.host_query_terms(4, 200, seed=11, vocab=vocab)
    lists = [terms[ptr[b]:ptr[b + 1]].tolist() for b in range(4)]
    lists[0] = lists[0][:33]
    lists[1] = lists[1][:64]
    lists[2] = lists[2][:62] + [-1, lists[2][0], lists[2][40]]     # 65
    _check_bm25(dev, idx, csr, lists, K=20, seed=1)                # lists[3]: 200 tokens
    _check_bm25(dev, idx, csr, [lists[3], lists[3][:100]], K=0, seed=2)


def test_bm25_token_capacity_is_never_exceeded_silently(dev):
    """Device-pointer entry: a batch with more tokens than lrx_set_query_capacity is flagged (NaN
    maxima), not scored short."""
    n, vocab = 20000, 1000
    idx = synth.host_bm25(n, seed=6, vocab=vocab)
    dev.set_corpus(_cuda(synth.host_vectors(n, seed=2)), 0)
    _set_postings(dev, idx)
    terms, ptr = synth.host_query_terms(2, 40, seed=3, vocab=vocab)
    try:
        dev._capacity = 48
        dev._ck(dev.lib.lrx_set_query_capacity(dev.h, 48))           # 80 tokens > 48
        import ctypes as C
        mx = torch.empty(2, dtype=torch.float64, device="cuda")
        t, p = _cuda(terms), _cuda(ptr)
        dev._ck(dev.lib.lrx_bm25(dev.h, C.c_void_p(t.data_ptr()), C.c_void_p(p.data_ptr()), 2, None, 0, None,
                                 C.c_void_p(mx.data_ptr()), 0, None, None))
        assert torch.isnan(mx).all()
    finally:
        dev._capacity = 0
        dev._ck(dev.lib.lrx_set_query_capacity(dev.h, 0))


def test_bm25_division_matches_ddiv_rn(dev):
    """The scan's branch-free float64 division (csrc/bm25.cu okapi_div) gives the bits of the IEEE
    division for every (tf, len) a posting can hold, at several average lengths.  An average below 1
    (a corpus of mostly empty chunks) puts the divisor tf + k1*(1 - b + b*len/avgdl) far above 2^17."""
    import ctypes as C
    for avgdl in (104.35572519083969, 80.0, 1.0, 517.3, 3.0e4, 0.05, 0.3337):
        bad = C.c_uint64(123)
        dev._ck(dev.lib.lrx_debug_bm25_divcheck(dev.h, avgdl, 1.5, 0.75, 4096, 65536, C.byref(bad)))
        assert bad.value == 0, (avgdl, bad.value)
    bad = C.c_uint64(123)
    dev._ck(dev.lib.lrx_debug_bm25_divcheck(dev.h, 104.35572519083969, 1.5, 0.75, 65536, 4096, C.byref(bad)))
    assert bad.value == 0


def test_bm25_massive_ties(dev):
    """Thousands of documents with EXACTLY the same score: the list is decided by id."""
    n = 6000
    docs = [["common", f"u{i}"] for i in range(n)]
    docs[4000] = ["common", "common", "u4000"]           # one clear winner
    idx = BM25Index.from_token_lists(docs)
    csr = obm25.BM25OkapiCSR.from_corpus(docs)
    assert csr.idf[csr.vocab["common"]] > 0              # floored idf: epsilon * mean idf
    dev.set_corpus(_cuda(synth.host_vectors(n, seed=3)), 10)
    _set_postings(dev, idx)
    lists = [idx.term_ids(["common"]), idx.term_ids(["common", "u17", "common"]), idx.term_ids(["u5"])]
    for K in (20, 200):
        _check_bm25(dev, idx, csr, lists, id_base=10, K=K, seed=K)


# -------------------------------------------------- K4/K5 whole search, host API
def _oracle_search(x, csr, q, lists, k, weights, fusion):
    oi = OracleIndex(x, csr)
    return oi.search_batch_vec(q, lists, k, weights, fusion)


def _assert_results(got, want, k):
    ids, score, sem, kw = got
    for b, res in enumerate(want):
        assert ids[b, :len(res)].tolist() == [r[0] for r in res]
        assert (ids[b, len(res):] == -1).all()
        for j, r in enumerate(res):
            assert score[b, j] == r[1] and sem[b, j] == r[2] and kw[b, j] == r[3]


@pytest.mark.parametrize("fusion", ["linear", "rrf"])
@pytest.mark.parametrize("n", [7, 3000, 70000])
def test_search_batch_host_matches_oracle(dev, n, fusion):
    x = synth.host_vectors(n, seed=n + 1, dup_frac=0.01)
    idx = synth.host_bm25(n, seed=n + 2, vocab=3000)
    csr = _csr_of(idx)
    dev.set_corpus(_cuda(x), 0)
    _set_postings(dev, idx)
    B = 4
    q = synth.host_queries(B, seed=n + 3)
    q[1] = synth.host_planted_queries(x, [n // 2], seed=4)[0]
    terms, ptr = synth.host_query_terms(B, 8, seed=n + 4, vocab=3000)
    lists = [terms[ptr[b]:ptr[b + 1]].tolist() for b in range(B)]
    lists[2] = [-1, -1]                                        # all out-of-vocabulary
    weights = [0.5, 0.6, 0.5, 0.6]
    for k in (1, 5, 10):
        want = _oracle_search(x, csr, q, lists, k, weights, fusion)
        got = dev.search_batch_host(q, lists, k, weights, fusion)
        _assert_results(got, want, k)


@pytest.mark.parametrize("fusion", ["linear", "rrf"])
def test_search_top100_config_c5_depth(dev, fusion):
    """Config C5's depth (top-100: dense top-200, width 256, BM25 list of 200) on one shard."""
    n = 120000
    x = synth.host_vectors(n, seed=91, dup_frac=0.005)
    idx = synth.host_bm25(n, seed=92, vocab=4000)
    csr = _csr_of(idx)
    dev.set_corpus(_cuda(x), 0)
    _set_postings(dev, idx)
    B = 3
    q = synth.host_queries(B, seed=93)
    terms, ptr = synth.host_query_terms(B, 8, seed=94, vocab=4000)
    lists = [terms[ptr[b]:ptr[b + 1]].tolist() for b in range(B)]
    weights = [0.5, 0.6, 0.5]
    want = _oracle_search(x, csr, q, lists, 100, weights, fusion)
    got = dev.search_batch_host(q, lists, 100, weights, fusion)
    _assert_results(got, want, 100)


def test_clone_view_two_batches_in_flight(dev):
    """A second handle over the same resident index (DeviceIndex.clone_view), each on its own stream:
    batches interleaved on the two streams give the oracle's results."""
    n = 50000
    x = synth.host_vectors(n, seed=17, dup_frac=0.01)
    idx = synth.host_bm25(n, seed=18, vocab=3000)
    csr = _csr_of(idx)
    dev.set_corpus(_cuda(x), 0)
    _set_postings(dev, idx)
    other = dev.clone_view()
    try:
        from legal_rag_engine_b200.device_index import FUSION
        from legal_rag_engine_b200.sharding import ShardedSearcher
        streams = [torch.cuda.Stream(), torch.cuda.Stream()]
        devs = [dev, other]
        for d, st in zip(devs, streams):
            with torch.cuda.stream(st):
                d.use_current_stream()
        searchers = [ShardedSearcher(d) for d in devs]
        B, k, weights = 4, 10, [0.5, 0.6, 0.5, 0.6]
        batches = []
        for i in range(6):
            q = synth.host_queries(B, seed=100 + i)
            terms, ptr = synth.host_query_terms(B, 8, seed=200 + i, vocab=3000)
            lists = [terms[ptr[b]:ptr[b + 1]].tolist() for b in range(B)]
            batches.append((q, terms, ptr, lists))
        torch.cuda.synchronize()
        w = _cuda(np.array(weights))
        got = []
        for i, (q, terms, ptr, lists) in enumerate(batches):
            j = i % 2
            with torch.cuda.stream(streams[j]):
                outs = searchers[j].search(_cuda(q), _cuda(terms), _cuda(ptr), k, FUSION["rrf"], w)
                got.append([t.clone() for t in outs])            # clone on the same stream
        torch.cuda.synchronize()
        for (q, terms, ptr, lists), outs in zip(batches, got):
            want = _oracle_search(x, csr, q, lists, k, weights, "rrf")
            ids, score, sem, kw, status = [t.cpu().numpy() for t in outs]
            assert status.sum() == 0
            _assert_results((ids, score, sem, kw), want, k)
    finally:
        dev.use_current_stream()
        other.close()


def test_real_corpus_hybrid_search(dev, legal_texts, reference_queries):
    """Config C1 minus the encoder: real BM25 side, seeded stand-in vectors."""
    idx = BM25Index.from_texts(legal_texts)
    csr = obm25.BM25OkapiCSR.from_corpus([obm25.tokenize(t) for t in legal_texts])
    x = synth.host_vectors(idx.n_docs, seed=42, dup_frac=0.004)
    dev.set_corpus(_cuda(x), 0)
    _set_postings(dev, idx)
    qs = reference_queries[:8]
    q = synth.host_planted_queries(x, list(range(100, 100 + len(qs))), seed=5, noise=0.5)
    lists = [idx.term_ids(tokenize(s)) for s in qs]
    weights = [0.6 if "procedure" in s.lower() else 0.5 for s in qs]
    for fusion in ("linear", "rrf"):
        want = _oracle_search(x, csr, q, lists, 10, weights, fusion)
        got = dev.search_batch_host(q, lists, 10, weights, fusion)
        _assert_results(got, want, 10)


def test_one_million_rows(dev):
    """Config C3 size: 1 M x 384, batch 1 and 4, top-20 -- still bit-exact."""
    n = 1_000_000
    x = synth.host_vectors(n, seed=1234)
    q = synth.host_queries(4, seed=4321)
    dev.set_corpus(_cuda(x), 0)
    s = flat_ip.exact_scores(x, q)
    Eo, Do, Io = flat_ip.topk_from_scores(s, 20)
    E, D, I, flags = dev.dense_topk(_cuda(q), 20)
    assert flags.sum().item() == 0
    np.testing.assert_array_equal(I.cpu().numpy(), Io)
    np.testing.assert_array_equal(E.cpu().numpy(), Eo)
    E1, D1, I1, f1 = dev.dense_topk(_cuda(q[:1]), 20)
    np.testing.assert_array_equal(I1.cpu().numpy(), Io[:1])


# ------------------------------------------------ K2b: tensor-core batched scoring
@pytest.mark.parametrize("n,B,K", [(300, 5, 20), (1000, 64, 20), (20011, 130, 10), (300000, 256, 20),
                                   (100000, 1024, 200)])
def test_dense_topk_batched_matches_oracle(dev, n, B, K):
    x = synth.host_vectors(n, seed=n + 7, dup_frac=0.01)
    q = synth.host_queries(B, seed=B + n)
    q[0] = x[n // 2]                                   # a planted exact hit
    dev.set_corpus(_cuda(x), 1000)
    E, D, I, flags = dev.dense_topk_batched(_cuda(q), K)
    assert int(flags.sum().item()) == 0
    s = flat_ip.exact_scores(x, q)
    Eo, Do, Io = flat_ip.topk_from_scores(s, K, id_base=1000)
    np.testing.assert_array_equal(I.cpu().numpy(), Io)
    np.testing.assert_array_equal(E.cpu().numpy(), Eo)
    np.testing.assert_array_equal(D.cpu().numpy(), Do)


def test_dense_topk_batched_one_million_rows_b1024(dev):
    """Config C3: 1 M x 384, query batch 1024, top-20 -- bit-exact against the oracle on a sample
    of the queries, and against the small-batch kernel on all of them."""
    n, B, K = 1_000_000, 1024, 20
    x = synth.host_vectors(n, seed=1234)
    q = synth.host_queries(B, seed=4321)
    dev.set_corpus(_cuda(x), 0)
    E, D, I, flags = dev.dense_topk_batched(_cuda(q), K)
    assert int(flags.sum().item()) == 0
    pick = [0, 1, 511, 1023]
    s = flat_ip.exact_scores(x, q[pick])
    Eo, _, Io = flat_ip.topk_from_scores(s, K)
    np.testing.assert_array_equal(I.cpu().numpy()[pick], Io)
    np.testing.assert_array_equal(E.cpu().numpy()[pick], Eo)
    for b0 in range(0, 64, 4):                         # K2a on the first 64 queries
        E2, _, I2, f2 = dev.dense_topk(_cuda(q[b0:b0 + 4]), K)
        assert int(f2.sum().item()) == 0
        np.testing.assert_array_equal(I.cpu().numpy()[b0:b0 + 4], I2.cpu().numpy())
        np.testing.assert_array_equal(E.cpu().numpy()[b0:b0 + 4], E2.cpu().numpy())


def test_search_host_200_token_query(dev):
    """The host-buffer call sizes the token capacity from the batch: a 200-token sub-query beside
    short ones equals the oracle (the reference has no token limit)."""
    n = 30000
    x = synth.host_vectors(n, seed=31)
    idx = synth.host_bm25(n, seed=32, vocab=1500)
    csr = _csr_of(idx)
    dev.set_corpus(_cuda(x), 0)
    _set_postings(dev, idx)
    q = synth.host_queries(3, seed=33)
    terms, ptr = synth.host_query_terms(3, 200, seed=34, vocab=1500)
    lists = [terms[ptr[b]:ptr[b + 1]].tolist() for b in range(3)]
    lists[1] = lists[1][:5]
    lists[2] = lists[2][:70]
    for fusion in ("linear", "rrf"):
        want = _oracle_search(x, csr, q, lists, 10, [0.5, 0.6, 0.5], fusion)
        got = dev.search_batch_host(q, lists, 10, [0.5, 0.6, 0.5], fusion)
        _assert_results(got, want, 10)


def test_captured_chain_replays_equal_first_call(dev):
    """The launch chain is captured into a CUDA graph on the second call with the same buffers and
    replayed afterwards: calls 1 (direct), 2 (capture + replay), 3.. (replay) give the oracle's
    result, with NEW query contents in the same buffers every time."""
    from legal_rag_engine_b200.device_index import FUSION
    from legal_rag_engine_b200.sharding import ShardedSearcher
    n = 40000
    x = synth.host_vectors(n, seed=41, dup_frac=0.01)
    idx = synth.host_bm25(n, seed=42, vocab=2500)
    csr = _csr_of(idx)
    dev.set_corpus(_cuda(x), 0)
    _set_postings(dev, idx)
    s = ShardedSearcher(dev)
    B, k, weights = 4, 10, [0.5, 0.6, 0.5, 0.6]
    dq = torch.empty((B, 384), dtype=torch.float16, device="cuda")
    dt = torch.empty(B * 8, dtype=torch.int32, device="cuda")
    dp = _cuda((np.arange(B + 1) * 8).astype(np.int32))
    w = _cuda(np.array(weights))
    for fusion in ("rrf", "linear"):
        l0 = dev.launches
        per_call = []
        for i in range(5):
            q = synth.host_queries(B, seed=500 + i)
            terms, ptr = synth.host_query_terms(B, 8, seed=600 + i, vocab=2500)
            dq.copy_(_cuda(q)); dt.copy_(_cuda(terms))
            before = dev.launches
            outs = s.search_checked(dq, dt, dp, k, FUSION[fusion], w)
            per_call.append(dev.launches - before)
            ids, score, sem, kw, status = [t.cpu().numpy() for t in outs]
            lists = [terms[ptr[b]:ptr[b + 1]].tolist() for b in range(B)]
            _assert_results((ids, score, sem, kw), _oracle_search(x, csr, q, lists, k, weights, fusion), k)
        assert len(set(per_call)) == 1 and per_call[0] >= 6, per_call   # replays count their kernels
    # host-buffer call: same chain with the copies inside, also replayed
    for i in range(4):
        q = synth.host_queries(B, seed=700 + i)
        terms, ptr = synth.host_query_terms(B, 8, seed=800 + i, vocab=2500)
        lists = [terms[ptr[b]:ptr[b + 1]].tolist() for b in range(B)]
        got = dev.search_batch_host(q, lists, k, weights, "rrf")
        _assert_results(got, _oracle_search(x, csr, q, lists, k, weights, "rrf"), k)


def test_host_begin_end_two_handles_pipelined(dev):
    """lrx_search_host_begin / _end on two handles over one index: two batches in flight, results in
    order, a second begin on a busy handle is refused."""
    from legal_rag_engine_b200._lib import LrxError
    n = 30000
    x = synth.host_vectors(n, seed=51)
    idx = synth.host_bm25(n, seed=52, vocab=2000)
    csr = _csr_of(idx)
    dev.set_corpus(_cuda(x), 0)
    _set_postings(dev, idx)
    other = dev.clone_view()
    try:
        streams = [torch.cuda.Stream(), torch.cuda.Stream()]
        devs = [dev, other]
        for d, st in zip(devs, streams):
            with torch.cuda.stream(st):
                d.use_current_stream()
        B, k, weights = 4, 10, [0.5, 0.6, 0.5, 0.6]
        batches = []
        for i in range(7):
            q = synth.host_queries(B, seed=900 + i)
            terms, ptr = synth.host_query_terms(B, 8, seed=950 + i, vocab=2000)
            batches.append((q, [terms[ptr[b]:ptr[b + 1]].tolist() for b in range(B)]))
        got = [None] * len(batches)
        for i, (q, lists) in enumerate(batches):
            d = devs[i % 2]
            if i >= 2:
                got[i - 2] = d.search_host_end()
            d.search_host_begin(q, lists, k, weights, "rrf")
            if i == 0:
                with pytest.raises(LrxError):
                    d.search_host_begin(q, lists, k, weights, "rrf")
        for i in (len(batches) - 2, len(batches) - 1):
            got[i] = devs[i % 2].search_host_end()
        for (q, lists), g in zip(batches, got):
            _assert_results(g, _oracle_search(x, csr, q, lists, k, weights, "rrf"), k)
    finally:
        dev.use_current_stream()
        other.close()


@pytest.mark.parametrize("fusion", ["linear", "rrf"])
@pytest.mark.parametrize("B", [5, 8, 9, 33, 64])
def test_search_batch_routes_larger_batches_to_tensor_core_scoring(dev, B, fusion):
    """Up to 8 sub-queries share one streaming pass of the matrix (K2a, 8 query columns); from 9 on
    the search chain scores the batch with the tensor-core kernel (K2b), still in one pass: same
    exact results either way."""
    n = 90000
    x = synth.host_vectors(n, seed=61, dup_frac=0.01)
    idx = synth.host_bm25(n, seed=62, vocab=3000)
    csr = _csr_of(idx)
    dev.set_corpus(_cuda(x), 0)
    _set_postings(dev, idx)
    q = synth.host_queries(B, seed=63 + B)
    q[B // 2] = synth.host_planted_queries(x, [n // 3], seed=4)[0]
    terms, ptr = synth.host_query_terms(B, 8, seed=64 + B, vocab=3000)
    lists = [terms[ptr[b]:ptr[b + 1]].tolist() for b in range(B)]
    weights = [0.5 + 0.1 * (b % 2) for b in range(B)]
    want = _oracle_search(x, csr, q, lists, 10, weights, fusion)
    for _ in range(3):                                          # direct, captured, replayed
        got = dev.search_batch_host(q, lists, 10, weights, fusion)
        _assert_results(got, want, 10)
