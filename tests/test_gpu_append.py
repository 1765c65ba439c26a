"""RetrievalEngine.add_chunks / save and the device postings merge (lrx_bm25_append_postings): an
index grown by appends answers exactly as one rebuilt from all its chunks -- same chunks, bit-identical
float64 scores -- with the pre-filter on and off, at the reference corpus and at 1 M synthetic rows."""
import json
import threading

import numpy as np
import pytest
import torch

from legal_rag_engine_b200 import synth

pytestmark = pytest.mark.gpu

SPLITS = (2000, 2001, 2300)          # the store holds chunks[:2000]; adds [2000:2001], [2001:2300], [2300:]


def _strip(res):
    return [[(r["chunk"], r["score"], r["semantic"], r["keyword"]) for r in rs] for rs in res]


def _answers(eng, queries):
    """search_batch over every (pre-filter, k, fusion) combination, in batches of the orchestrator's
    fan-out size (4).  Larger coalesced batches, which take the tensor-core dense path, are checked
    on the whole corpus by test_gpu_dense_batched.py."""
    out = {}
    for pf in (True, False):
        eng.dev.set_prefilter(pf)
        for k in (5, 10):
            for fusion in ("linear", "rrf"):
                res = []
                for s in range(0, len(queries), 4):
                    part = queries[s:s + 4]
                    res += eng.search_batch(part, k=k, hybrid_weights=[0.6] * len(part), fusion=fusion)
                out[pf, k, fusion] = _strip(res)
    eng.dev.set_prefilter(True)
    return out


@pytest.fixture(scope="module")
def env(tmp_path_factory, legal_chunks):
    from legal_rag_engine_b200.engine import create_vector_store
    from legal_rag_engine_b200.tokenizer import HashTokenizer
    d = tmp_path_factory.mktemp("append")
    src = d / "first.json"
    src.write_text(json.dumps(legal_chunks[:SPLITS[0]]), encoding="utf-8")
    sd = synth.bert_state_dict(42, 0.05, ln_jitter=0.1)
    tok = HashTokenizer(30522)
    create_vector_store(str(src), str(d / "vs"), encoder_state_dict=sd, tokenizer=tok)
    return d, sd, tok


def _engine(env, path=None):
    from legal_rag_engine_b200.engine import RetrievalEngine
    d, sd, tok = env
    return RetrievalEngine(str(path or d / "vs"), encoder_state_dict=sd, tokenizer=tok)


def _rebuilt_store(path, chunks, x16, texts):
    from legal_rag_engine_b200.bm25_index import BM25Index
    from legal_rag_engine_b200.store import save_store
    save_store(path, chunks, x16.astype(np.float32), BM25Index.from_texts(texts))


@pytest.fixture(scope="module")
def grown(env, legal_chunks, reference_queries):
    """The engine after each of the three adds, beside an engine over a store rebuilt from the same
    chunks with the grown engine's own rows (the encoder is not claimed batch-invariant)."""
    d = env[0]
    eng = _engine(env)
    texts = [c["text"] for c in legal_chunks]
    steps, batches = [], []
    bounds = list(SPLITS) + [len(legal_chunks)]
    for lo, hi in zip(bounds[:-1], bounds[1:]):
        ids = eng.add_chunks(legal_chunks[lo:hi])
        assert ids == range(lo, hi) and eng.n_total == hi and len(eng.chunks) == hi
        batches.append((lo, hi))
        x16 = eng._x.cpu().numpy()
        assert x16.shape == (hi, 384)
        _rebuilt_store(d / f"rebuilt{hi}", legal_chunks[:hi], x16, texts[:hi])
        ref = _engine(env, d / f"rebuilt{hi}")
        try:
            steps.append((hi, _answers(eng, reference_queries), _answers(ref, reference_queries)))
        finally:
            ref.close()
    yield eng, steps, batches
    eng.close()


def test_grown_index_answers_as_a_rebuild(grown):
    _, steps, _ = grown
    for n, got, want in steps:
        for key in want:
            assert got[key] == want[key], (n, key)


@pytest.mark.parametrize("fusion", ["linear", "rrf"])
def test_grown_index_matches_oracle(grown, reference_queries, fusion):
    from oracle import bm25 as obm25
    from oracle.bm25 import tokenize
    from oracle.search import OracleIndex
    eng = grown[0]
    b = eng.bm25
    assert b.n_docs == eng.n_total == len(b.doc_len)
    csr = obm25.BM25OkapiCSR(b.n_docs, b.doc_len, b.term_ptr.astype(np.int64), b.postings[:, 0],
                             b.postings[:, 1], vocab=b.vocab)
    oracle = OracleIndex(eng._x.cpu().numpy(), csr)
    for q in reference_queries:
        for k, w in ((5, 0.5), (10, 0.6)):
            got = eng.search(q, k=k, hybrid_weight=w, fusion=fusion)
            qh = eng.encode([q]).astype(np.float16)[0]
            want = oracle.search_vec(qh, csr.term_ids(tokenize(q)), k, w, fusion)
            assert [(r["chunk"] is eng.chunks[i], r["score"], r["semantic"], r["keyword"]) for r, (i, *_) in
                    zip(got, want)] == [(True, s, sem, kw) for _, s, sem, kw in want]
            assert len(got) == len(want)


def test_device_postings_equal_a_full_build(grown, legal_texts):
    from legal_rag_engine_b200.bm25_index import BM25Index
    from legal_rag_engine_b200.device_index import DeviceIndex
    eng = grown[0]
    full = BM25Index.from_texts(legal_texts)
    fresh = DeviceIndex(0)
    try:
        fresh.set_postings(full.term_ptr, full.postings, full.doc_len, full.idf, full.avgdl)
        tp, p8, idf = eng.dev._post
        ftp, fp8, fidf = fresh._post
        nnz = full.nnz
        assert eng.dev._post_args == fresh._post_args and eng.dev.n_terms == full.n_terms
        assert torch.equal(tp, ftp) and torch.equal(idf, fidf)
        assert torch.equal(p8[:nnz], fp8[:nnz])
        if nnz % 2:
            assert not p8[nnz].any()                          # the zeroed pad of the last 16-byte unit
        assert torch.equal(eng.dev.doc_len, fresh.doc_len)
    finally:
        fresh.close()


def test_appended_embeddings(grown, env, legal_chunks, tmp_path):
    """Rows of each add = float16 of SentenceEncoder.encode over that add's texts, bit for bit; against
    create_vector_store over the whole corpus: cosine >= 0.9999 (the bulk encoder is not claimed
    batch-invariant, so rows encoded in other batches may differ in the last bits)."""
    from legal_rag_engine_b200.engine import create_vector_store
    eng, _, batches = grown
    x = eng._x.cpu().numpy()
    for lo, hi in batches:
        want = eng.model.encode([c["text"] for c in legal_chunks[lo:hi]]).astype(np.float16)
        np.testing.assert_array_equal(x[lo:hi].view(np.uint16), want.view(np.uint16))
    src = tmp_path / "all.json"
    src.write_text(json.dumps(legal_chunks), encoding="utf-8")
    _, sd, tok = env
    create_vector_store(str(src), str(tmp_path / "vs"), encoder_state_dict=sd, tokenizer=tok)
    full = np.load(tmp_path / "vs" / "vectors.f16.npy").astype(np.float64)
    got = x.astype(np.float64)
    cos = (got * full).sum(1) / np.linalg.norm(got, axis=1) / np.linalg.norm(full, axis=1)
    assert cos.min() >= 0.9999
    print(f"appended rows bit-equal to the whole-corpus build: {(x == full.astype(np.float16)).all(1).mean():.4f}")


def test_save_round_trip(grown, env, reference_queries, tmp_path):
    eng, steps, _ = grown
    d = env[0]
    n = eng.n_total
    out = eng.save(tmp_path / "saved")
    assert sorted(p.name for p in out.parent.iterdir()) == ["saved"]       # no temporary left behind
    reb = d / f"rebuilt{n}"
    np.testing.assert_array_equal(np.load(out / "vectors.f16.npy").view(np.uint16),
                                  np.load(reb / "vectors.f16.npy").view(np.uint16))
    za, zb = np.load(out / "bm25.npz"), np.load(reb / "bm25.npz")
    assert sorted(za.files) == sorted(zb.files)
    for f in za.files:
        assert za[f].dtype == zb[f].dtype, f
        np.testing.assert_array_equal(za[f], zb[f], err_msg=f)
    assert json.loads((out / "metadata.json").read_text()) == json.loads((reb / "metadata.json").read_text())
    eng.save(tmp_path / "saved")                                 # over an existing store
    again = _engine(env, tmp_path / "saved")
    try:
        assert _answers(again, reference_queries) == steps[-1][1]
    finally:
        again.close()


def test_added_chunk_is_found_after_captured_chains(env, legal_chunks):
    """Same-shape searches run direct, then captured, then replayed; an add must retire those chains."""
    eng = _engine(env)
    try:
        q = "quokka tribunal zebra amendment ordinance"
        first = [eng.search(q, k=5) for _ in range(3)]
        assert first[0] == first[1] == first[2]
        (new_id,) = eng.add_chunks([{"text": q, "canonical_header": "added"}])
        top = eng.search(q, k=5)[0]
        assert top["chunk"] is eng.chunks[new_id] and top["chunk"]["canonical_header"] == "added"
    finally:
        eng.close()


def _same_index(a, b):
    assert a.n_docs == b.n_docs
    assert list(a.vocab.items()) == list(b.vocab.items())            # ids AND insertion order
    for name in ("term_ptr", "postings", "doc_len"):
        x, y = getattr(a, name), getattr(b, name)
        assert x.dtype == y.dtype and x.shape == y.shape, name
        np.testing.assert_array_equal(x, y, err_msg=name)
    np.testing.assert_array_equal(a.idf.view(np.uint64), b.idf.view(np.uint64))
    assert a.avgdl == b.avgdl and (a.k1, a.b, a.epsilon) == (b.k1, b.b, b.epsilon)


def test_failed_add_changes_nothing(env, reference_queries, monkeypatch):
    """A failure after the postings are staged -- here the matrix append raising -- leaves the engine
    as it was.  The state is checked before any search, so no search runs over a handle whose
    postings and matrix could disagree."""
    eng = _engine(env)
    try:
        before = _answers(eng, reference_queries)
        b = eng.bm25
        post, n_docs, n_local, n = eng.dev._post, eng.dev.n_docs, eng.dev.n_local, eng.n_total

        def fail(*args, **kwargs):
            raise RuntimeError("injected failure of the matrix append")
        monkeypatch.setattr(eng.dev, "append_rows", fail)
        with pytest.raises(RuntimeError, match="injected"):
            eng.add_chunks([{"text": "quokka tribunal zebra amendment ordinance"}])
        monkeypatch.undo()
        assert eng.dev._post is post and eng.dev.n_docs == n_docs and eng.dev.n_local == n_local
        assert eng.n_total == n and len(eng.chunks) == n
        _same_index(eng.bm25, b)
        assert _answers(eng, reference_queries) == before
    finally:
        eng.close()


def test_bm25_is_a_snapshot(env, legal_chunks):
    """engine.bm25 taken before an add and a removal still describes the index it was taken from;
    read again, it equals a rebuild."""
    import copy
    from legal_rag_engine_b200.bm25_index import BM25Index
    eng = _engine(env)
    try:
        b = eng.bm25
        kept = copy.deepcopy(b)
        eng.add_chunks(legal_chunks[2000:2010])
        eng.remove_chunks([0, 5, 2003])
        _same_index(b, kept)
        _same_index(eng.bm25, BM25Index.from_texts([c["text"] for c in eng.chunks]))
    finally:
        eng.close()


def test_rejected_input_changes_nothing(env, reference_queries):
    eng = _engine(env)
    try:
        before = _answers(eng, reference_queries)
        n, x_ptr = eng.n_total, eng._x.data_ptr()
        with pytest.raises(ValueError):
            eng.add_chunks([{"text": "zero fir"}, {"body": "no text"}])
        with pytest.raises(ValueError):
            eng.add_chunks([{"text": "word " * 70000}])
        assert eng.add_chunks([]) == range(n, n)
        assert eng.n_total == n and len(eng.chunks) == n and eng._x.data_ptr() == x_ptr
        assert _answers(eng, reference_queries) == before
    finally:
        eng.close()


def test_concurrent_searches_see_before_or_after(env, legal_chunks):
    from legal_rag_engine_b200.serving import MicroBatchingEngine
    queries = ["What is the procedure for Zero FIR?", "Compensation for victims of acid attack",
               "Definition of a public servant under BNS", "What is the punishment for murder?",
               "How to file FIR for robbery BNSS procedure", "bail for non-bailable offence"]
    new = legal_chunks[2000:2300]
    key = lambda rs: [(r["chunk"]["canonical_header"], r["score"], r["semantic"], r["keyword"]) for r in rs]
    ref = _engine(env)
    try:
        before = {q: key(ref.search(q, k=5, hybrid_weight=0.6)) for q in queries}
        ref.add_chunks(new)
        after = {q: key(ref.search(q, k=5, hybrid_weight=0.6)) for q in queries}
    finally:
        ref.close()
    assert before != after
    mb = MicroBatchingEngine(_engine(env), max_batch=8, max_wait_ms=1.0)       # the K2a path, as _answers
    try:
        got, stop = [], threading.Event()

        def client(i):
            j = 0
            while not stop.is_set() or j < 4:
                q = queries[(i + j) % len(queries)]
                got.append((q, key(mb.search(q, k=5, hybrid_weight=0.6))))
                j += 1
        ts = [threading.Thread(target=client, args=(i,)) for i in range(8)]
        for t in ts:
            t.start()
        while len(got) < 40:
            threading.Event().wait(0.005)
        mb.add_chunks(new)                                        # forwarded to the engine
        n_mid = len(got)
        while len(got) < n_mid + 40:
            threading.Event().wait(0.005)
        stop.set()
        for t in ts:
            t.join()
        assert all(res in (before[q], after[q]) for q, res in got)
        assert any(res == after[q] != before[q] for q, res in got[n_mid:])
    finally:
        mb.close()


def test_one_million_rows_append_and_grow(tmp_path):
    """1 M synthetic rows + Zipf BM25; append 37 rows, then 100 000 (the matrix buffer grows both
    times: the index is loaded without slack, and 100 000 rows exceed the 1/16 slack).  After each
    append: search_batch_host bit-exact against the oracle over the concatenated data, pre-filter on
    and off; shadow bounds and postings equal a fresh build's."""
    from oracle import bm25 as obm25
    from oracle.search import OracleIndex
    from legal_rag_engine_b200.bm25_index import okapi_idf
    from legal_rag_engine_b200.device_index import DeviceIndex
    n0, steps = 1_000_000, (37, 100_000)
    total = n0 + sum(steps)
    x = synth.host_vectors(total, seed=61)
    full = synth.host_bm25(total, seed=62)
    B, k = 8, 10
    q = synth.host_queries(B, seed=63)
    q[0] = synth.host_planted_queries(x, [total - 5], seed=64)[0]             # an appended row on top
    terms, ptr = synth.host_query_terms(B, 8, seed=65)
    lists = [terms[ptr[b]:ptr[b + 1]].tolist() for b in range(B)]
    w = [0.5, 0.6] * (B // 2)

    def prefix_stats(n):
        p = full.shard(0, n)
        idf, _ = okapi_idf(np.diff(p.term_ptr.astype(np.int64)), n)
        return p, idf, int(p.doc_len.astype(np.int64).sum()) / n

    dev = DeviceIndex(0)
    try:
        p, idf, avgdl = prefix_stats(n0)
        dev.set_corpus(torch.from_numpy(x[:n0]).cuda(), 0, prefilter=True)
        dev.set_postings(p.term_ptr, p.postings, p.doc_len, idf, avgdl)
        n = n0
        for m in steps:
            cap = dev.capacity
            add = full.shard(n, n + m)
            post = add.postings.copy()
            post[:, 0] += np.uint32(n)
            dev.append_postings(add.term_ptr.astype(np.int64), post, add.doc_len, *prefix_stats(n + m)[1:])
            dev.append_rows(torch.from_numpy(x[n:n + m]).cuda())
            n += m
            assert dev.n_local == n and dev.capacity > cap
            p, idf, avgdl = prefix_stats(n)
            csr = obm25.BM25OkapiCSR.from_postings(n, p.doc_len, p.term_ptr.astype(np.int64), p.postings[:, 0],
                                                   p.postings[:, 1])
            for fusion in ("linear", "rrf"):
                want = OracleIndex(x[:n], csr).search_batch_vec(q, lists, k, w, fusion)
                for on in (True, False):
                    dev.set_prefilter(on)
                    ids, score, sem, kw = dev.search_batch_host(q, lists, k, w, fusion)
                    for b in range(B):
                        assert ids[b].tolist() == [r[0] for r in want[b]], (n, fusion, on, b)
                        assert score[b].tolist() == [r[1] for r in want[b]]
                        assert sem[b].tolist() == [r[2] for r in want[b]]
                        assert kw[b].tolist() == [r[3] for r in want[b]]
            fresh = DeviceIndex(0)
            try:
                fresh.set_corpus(torch.from_numpy(x[:n]).cuda(), 0, prefilter=True)
                assert dev.prefilter_bounds == fresh.prefilter_bounds
                fresh.set_postings(p.term_ptr, p.postings, p.doc_len, idf, avgdl)
                nnz = p.nnz
                assert torch.equal(dev._post[0], fresh._post[0])
                assert torch.equal(dev._post[1][:nnz], fresh._post[1][:nnz])
                assert torch.equal(dev._post[2], fresh._post[2])
            finally:
                fresh.close()
    finally:
        dev.close()
