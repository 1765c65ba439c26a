"""RetrievalEngine.remove_chunks and the device postings compaction (lrx_bm25_remove_postings): an
index shrunk by removals answers exactly as one rebuilt from the remaining chunks -- same chunks,
bit-identical float64 scores -- with the pre-filter on and off, at the reference corpus and at 1 M
synthetic rows."""
import json
import threading

import numpy as np
import pytest
import torch

from legal_rag_engine_b200 import synth

pytestmark = pytest.mark.gpu

LRX_E_ARG = -1


def _strip(res):
    return [[(r["chunk"], r["score"], r["semantic"], r["keyword"]) for r in rs] for rs in res]


def _answers(eng, queries):
    """search_batch over every (pre-filter, k, fusion) combination, in batches of at most 4 queries
    (the K2a path, as in test_gpu_append.py)."""
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
    d = tmp_path_factory.mktemp("remove")
    sd = synth.bert_state_dict(42, 0.05, ln_jitter=0.1)
    tok = HashTokenizer(30522)
    for name, chunks in (("all", legal_chunks), ("first", legal_chunks[:2000])):
        src = d / f"{name}.json"
        src.write_text(json.dumps(chunks), encoding="utf-8")
        create_vector_store(str(src), str(d / name), encoder_state_dict=sd, tokenizer=tok)
    return d, sd, tok


def _engine(env, path="all"):
    from legal_rag_engine_b200.engine import RetrievalEngine
    d, sd, tok = env
    return RetrievalEngine(str(d / path), encoder_state_dict=sd, tokenizer=tok)


def _rebuilt(env, name, chunks, x16):
    """An engine over a store rebuilt from `chunks` with the rows x16 (float16)."""
    from legal_rag_engine_b200.bm25_index import BM25Index
    from legal_rag_engine_b200.store import save_store
    save_store(env[0] / name, chunks, x16.astype(np.float32), BM25Index.from_texts([c["text"] for c in chunks]))
    return _engine(env, name)


def _rare_word_ids(chunks):
    from legal_rag_engine_b200.bm25_index import BM25Index, tokenize
    docs = [tokenize(c["text"]) for c in chunks]
    full = BM25Index.from_token_lists(docs)
    df = np.diff(full.term_ptr.astype(np.int64))
    word = next(w for w, t in full.vocab.items() if df[t] == 3)
    return word, [i for i, t in enumerate(docs) if word in t]


def _removal_sets(chunks):
    n = len(chunks)
    rng = np.random.default_rng(20)
    return {"chunk0": [0], "first50": list(range(50)),
            "random10pct": sorted(rng.choice(n, n // 10, replace=False).tolist()),
            "every_other": list(range(1, n, 2)), "rare_word": _rare_word_ids(chunks)[1], "last": [n - 1]}


def _assert_device_equals_fresh(eng):
    """Postings, term_ptr, idf, doc_len and the shadow's bounds byte-equal to a fresh set_postings /
    set_corpus of the rebuilt data."""
    from legal_rag_engine_b200.bm25_index import BM25Index
    from legal_rag_engine_b200.device_index import DeviceIndex
    full = BM25Index.from_texts([c["text"] for c in eng.chunks])
    fresh = DeviceIndex(0)
    try:
        fresh.set_corpus(eng._x.clone(), 0, prefilter=True)
        assert eng.dev.prefilter_bounds == fresh.prefilter_bounds
        fresh.set_postings(full.term_ptr, full.postings, full.doc_len, full.idf, full.avgdl)
        tp, p8, idf = eng.dev._post
        ftp, fp8, fidf = fresh._post
        nnz = full.nnz
        assert eng.dev._post_args == fresh._post_args and eng.dev.n_terms == full.n_terms
        assert eng.dev.n_docs == fresh.n_docs == len(eng.chunks)
        assert torch.equal(tp, ftp) and torch.equal(idf, fidf)
        assert torch.equal(p8[:nnz], fp8[:nnz])
        if nnz % 2:
            assert not p8[nnz].any()                          # the zeroed pad of the last 16-byte unit
        assert torch.equal(eng.dev.doc_len, fresh.doc_len)
    finally:
        fresh.close()


def _assert_matches_oracle(eng, queries):
    from oracle import bm25 as obm25
    from oracle.bm25 import tokenize
    from oracle.search import OracleIndex
    b = eng.bm25
    assert b.n_docs == eng.n_total == len(b.doc_len)
    csr = obm25.BM25OkapiCSR(b.n_docs, b.doc_len, b.term_ptr.astype(np.int64), b.postings[:, 0],
                             b.postings[:, 1], vocab=b.vocab)
    oracle = OracleIndex(eng._x.cpu().numpy(), csr)
    for fusion in ("linear", "rrf"):
        for q in queries:
            for k, w in ((5, 0.5), (10, 0.6)):
                got = eng.search(q, k=k, hybrid_weight=w, fusion=fusion)
                qh = eng.encode([q]).astype(np.float16)[0]
                want = oracle.search_vec(qh, csr.term_ids(tokenize(q)), k, w, fusion)
                assert [(r["chunk"] is eng.chunks[i], r["score"], r["semantic"], r["keyword"])
                        for r, (i, *_) in zip(got, want)] == [(True, s, sem, kw) for _, s, sem, kw in want]
                assert len(got) == len(want)


@pytest.mark.parametrize("which", ["chunk0", "first50", "random10pct", "every_other", "rare_word", "last"])
def test_removal_answers_as_a_rebuild(env, legal_chunks, reference_queries, which):
    from legal_rag_engine_b200.bm25_index import BM25Index
    removed = _removal_sets(legal_chunks)[which]
    eng = _engine(env)
    try:
        x_before = eng._x.cpu().numpy()
        ids_map = eng.remove_chunks(removed)
        keep = np.setdiff1d(np.arange(len(legal_chunks)), removed)
        want_map = np.full(len(legal_chunks), -1, dtype=np.int64)
        want_map[keep] = np.arange(len(keep))
        assert ids_map.dtype == np.int64 and np.array_equal(ids_map, want_map)
        remaining = [legal_chunks[i] for i in keep]
        assert eng.chunks == remaining and eng.n_total == len(keep)
        np.testing.assert_array_equal(eng._x.cpu().numpy().view(np.uint16), x_before[keep].view(np.uint16))
        ref = _rebuilt(env, f"rebuilt_{which}", remaining, eng._x.cpu().numpy())
        try:
            assert _answers(eng, reference_queries) == _answers(ref, reference_queries)
        finally:
            ref.close()
        want = BM25Index.from_texts([c["text"] for c in remaining])
        b = eng.bm25
        assert list(b.vocab.items()) == list(want.vocab.items())
        for name in ("term_ptr", "postings", "doc_len"):
            np.testing.assert_array_equal(getattr(b, name), getattr(want, name), err_msg=name)
        np.testing.assert_array_equal(b.idf.view(np.uint64), want.idf.view(np.uint64))
        assert b.avgdl == want.avgdl and b.n_docs == want.n_docs
        _assert_device_equals_fresh(eng)
        _assert_matches_oracle(eng, reference_queries)
    finally:
        eng.close()


def test_interleaved_adds_and_removals(env, legal_chunks, reference_queries, tmp_path):
    """Store of 2 000 chunks; add 300; remove old and just-appended chunks (every holder of a rare
    word among them); add a chunk bringing the vanished word back; after each step the engine answers
    as a rebuild, and save() writes the rebuilt store's files."""
    word, holders = _rare_word_ids(legal_chunks[:2300])
    eng = _engine(env, "first")
    try:
        live = list(legal_chunks[:2000])

        def check(step):
            assert eng.chunks == live
            ref = _rebuilt(env, f"rebuilt_seq{step}", live, eng._x.cpu().numpy())
            try:
                assert _answers(eng, reference_queries) == _answers(ref, reference_queries), step
            finally:
                ref.close()
            _assert_device_equals_fresh(eng)

        assert eng.add_chunks(legal_chunks[2000:2300]) == range(2000, 2300)
        live += legal_chunks[2000:2300]
        check(1)
        drop = sorted(set(holders) | {0, 1999, 2000, 2150, 2299})
        assert any(i >= 2000 for i in drop)
        eng.remove_chunks(drop)
        live = [c for i, c in enumerate(live) if i not in set(drop)]
        assert word not in eng.bm25.vocab
        check(2)
        back = {"text": f"{word} returns in an amended section", "canonical_header": "amended"}
        n_words = len(eng.bm25.vocab)
        (new_id,) = eng.add_chunks([back])
        live.append(back)
        assert eng.bm25.vocab[word] == n_words                          # numbered at its new first appearance
        check(3)
        eng.remove_chunks([3, new_id - 1])
        live = [c for i, c in enumerate(live) if i not in (3, new_id - 1)]
        check(4)
        out = eng.save(tmp_path / "saved")
        reb = env[0] / "rebuilt_seq4"
        np.testing.assert_array_equal(np.load(out / "vectors.f16.npy").view(np.uint16),
                                      np.load(reb / "vectors.f16.npy").view(np.uint16))
        za, zb = np.load(out / "bm25.npz"), np.load(reb / "bm25.npz")
        assert sorted(za.files) == sorted(zb.files)
        for f in za.files:
            assert za[f].dtype == zb[f].dtype, f
            np.testing.assert_array_equal(za[f], zb[f], err_msg=f)
        assert json.loads((out / "metadata.json").read_text()) == json.loads((reb / "metadata.json").read_text())
        again = _engine(env, tmp_path / "saved")
        try:
            assert _answers(again, reference_queries) == _answers(eng, reference_queries)
        finally:
            again.close()
    finally:
        eng.close()


def test_removed_chunk_is_gone_after_captured_chains(env):
    """Same-shape searches run direct, then captured, then replayed; a removal must retire those chains."""
    eng = _engine(env)
    try:
        q = "What is the procedure for Zero FIR?"
        first = [eng.search(q, k=5) for _ in range(3)]
        assert first[0] == first[1] == first[2]
        top = first[0][0]["chunk"]
        top_id = next(i for i, c in enumerate(eng.chunks) if c is top)
        eng.remove_chunks([top_id])
        after = eng.search(q, k=5)
        assert len(after) == 5 and all(r["chunk"] is not top for r in after)
    finally:
        eng.close()


def test_rejected_input_changes_nothing(env, reference_queries):
    eng = _engine(env)
    try:
        before = _answers(eng, reference_queries)
        n, x_ptr, post = eng.n_total, eng._x.data_ptr(), eng.dev._post
        for bad, exc in (([n], ValueError), ([-1], ValueError), ([3, 3], ValueError),
                         (list(range(n)), ValueError), ([1.0], TypeError), (["2"], TypeError), ([True], TypeError)):
            with pytest.raises(exc):
                eng.remove_chunks(bad)
        assert np.array_equal(eng.remove_chunks([]), np.arange(n))
        assert eng.n_total == n and len(eng.chunks) == n and eng._x.data_ptr() == x_ptr and eng.dev._post is post
        assert _answers(eng, reference_queries) == before
    finally:
        eng.close()


def _synthetic(n, seed, planted_block, planted_terms=6):
    """Zipf BM25 over n documents (synth.host_bm25's distribution) plus `planted_terms` extra terms that
    occur only inside the document range `planted_block` and in the first and last document."""
    from legal_rag_engine_b200.bm25_index import BM25Index
    rng = np.random.default_rng(seed)
    lens = synth.host_doc_lengths(n, rng)
    cdf = synth._zipf_cdf(synth.VOCAB)
    terms = np.minimum(np.searchsorted(cdf, rng.random(int(lens.sum())), side="right"), synth.VOCAB - 1)
    docs = np.repeat(np.arange(n, dtype=np.int64), lens)
    lo, hi = planted_block
    p_docs = np.concatenate([rng.integers(lo, hi, 40 * planted_terms), [0, n - 1]])
    p_terms = np.concatenate([synth.VOCAB + np.arange(40 * planted_terms) % planted_terms, [synth.VOCAB] * 2])
    return BM25Index.from_token_arrays(np.concatenate([docs, p_docs]), np.concatenate([terms, p_terms]), n,
                                       synth.VOCAB + planted_terms)


def _plan(idx, removed, rng):
    """A removal plan over an index without a string vocabulary, surviving terms numbered by a
    random permutation (the kernel takes any bijection)."""
    from legal_rag_engine_b200.bm25_index import BM25Remove, BM25Stats, okapi_idf
    tp = idx.term_ptr.astype(np.int64)
    V = idx.n_terms
    doc = idx.postings[:, 0].astype(np.int64)
    gone = np.isin(doc, removed)
    term_of = np.repeat(np.arange(V), np.diff(tp))
    r = np.bincount(term_of[gone], minlength=V)
    rem_ptr = np.zeros(V + 1, dtype=np.int64)
    np.cumsum(r, out=rem_ptr[1:])
    df = np.diff(tp) - r
    alive = np.nonzero(df > 0)[0]
    order = rng.permutation(alive)
    term_map = np.full(V, -1, dtype=np.int32)
    term_map[order] = np.arange(len(order), dtype=np.int32)
    df_out = df[order]
    term_ptr = np.zeros(len(order) + 1, dtype=np.int64)
    np.cumsum(df_out, out=term_ptr[1:])
    n_out = idx.n_docs - len(removed)
    doc_len = np.delete(idx.doc_len, removed)
    total = int(doc_len.astype(np.int64).sum())
    idf, _ = okapi_idf(df_out, n_out)
    return BM25Remove(np.asarray(removed, dtype=np.int64), rem_ptr, doc[gone].astype(np.uint32), term_map, term_ptr,
                      BM25Stats({}, df_out, np.zeros(0, np.int64), n_out, total, idf, total / n_out)), doc_len


def test_one_million_rows_remove(tmp_path):
    """1 M synthetic rows + Zipf BM25; remove 37 scattered rows, then 100 000 more (a block spanning
    whole posting tiles, plus the first and the last row; some terms lose every posting).  After each
    step: search_batch_host bit-exact against the oracle over the remaining data, pre-filter on and
    off; postings and shadow bounds equal a fresh build's."""
    from oracle import bm25 as obm25
    from oracle.search import OracleIndex
    from legal_rag_engine_b200.bm25_index import BM25Index, remove_csr
    from legal_rag_engine_b200.device_index import DeviceIndex
    n0 = 1_000_000
    rng = np.random.default_rng(71)
    x = synth.host_vectors(n0, seed=61)
    idx = _synthetic(n0, 62, (420_000, 480_000))
    B, k = 8, 10
    q = synth.host_queries(B, seed=63)
    q[0] = synth.host_planted_queries(x, [n0 - 2], seed=64)[0]
    terms, ptr = synth.host_query_terms(B, 8, seed=65)
    lists = [terms[ptr[b]:ptr[b + 1]].tolist() for b in range(B)]
    lists[1] = [synth.VOCAB, synth.VOCAB + 1] + lists[1][:4]              # planted terms
    w = [0.5, 0.6] * (B // 2)
    steps = (lambda n: np.sort(rng.choice(np.arange(1, n - 1), 37, replace=False)),
             lambda n: np.concatenate([[0], np.arange(400_000, 499_998), [n - 1]]))
    dev = DeviceIndex(0)
    try:
        dev.set_corpus(torch.from_numpy(x).cuda(), 0, prefilter=True)
        dev.set_postings(idx.term_ptr, idx.postings, idx.doc_len, idx.idf, idx.avgdl)
        for step, pick in enumerate(steps):
            n = idx.n_docs
            removed = pick(n)
            assert len(removed) in (37, 100_000)
            rem, doc_len = _plan(idx, removed, rng)
            if step == 1:
                assert (rem.term_map == -1).sum() >= 6
            dev.remove_postings(rem)
            keep = np.ones(n, dtype=bool)
            keep[removed] = False
            dev.remove_rows(keep)
            x = x[keep]
            tp, po = remove_csr(idx.term_ptr, idx.postings, rem)
            idx = BM25Index(rem.stats.n_docs, doc_len, tp, po, rem.stats.idf, rem.stats.avgdl)
            lists = [[int(rem.term_map[t]) for t in l if rem.term_map[t] >= 0] for l in lists]
            assert dev.n_local == n - len(removed) == idx.n_docs
            csr = obm25.BM25OkapiCSR.from_postings(idx.n_docs, idx.doc_len, tp.astype(np.int64), po[:, 0], po[:, 1])
            for fusion in ("linear", "rrf"):
                want = OracleIndex(x, csr).search_batch_vec(q, lists, k, w, fusion)
                for on in (True, False):
                    dev.set_prefilter(on)
                    ids, score, sem, kw = dev.search_batch_host(q, lists, k, w, fusion)
                    for b in range(B):
                        assert ids[b].tolist() == [r[0] for r in want[b]], (step, fusion, on, b)
                        assert score[b].tolist() == [r[1] for r in want[b]]
                        assert sem[b].tolist() == [r[2] for r in want[b]]
                        assert kw[b].tolist() == [r[3] for r in want[b]]
            fresh = DeviceIndex(0)
            try:
                fresh.set_corpus(torch.from_numpy(x).cuda(), 0, prefilter=True)
                assert dev.prefilter_bounds == fresh.prefilter_bounds
                fresh.set_postings(tp, po, doc_len, rem.stats.idf, rem.stats.avgdl)
                nnz = rem.nnz
                assert dev._post_args == fresh._post_args
                assert torch.equal(dev._post[0], fresh._post[0])
                assert torch.equal(dev._post[1][:nnz], fresh._post[1][:nnz])
                if nnz % 2:
                    assert not dev._post[1][nnz].any()
                assert torch.equal(dev._post[2], fresh._post[2])
                assert torch.equal(dev.doc_len, fresh.doc_len)
            finally:
                fresh.close()
    finally:
        dev.close()


def test_inconsistent_plan_is_refused_and_the_index_keeps_answering(legal_texts):
    """A plan whose removed list or term_map does not describe the postings: LRX_E_ARG, and the
    resident index answers as before."""
    from legal_rag_engine_b200._lib import LrxError
    from legal_rag_engine_b200.bm25_index import BM25Index, _ranges, csr_remove, tokenize
    from legal_rag_engine_b200.device_index import DeviceIndex
    docs = [tokenize(t) for t in legal_texts]
    full = BM25Index.from_token_lists(docs)
    tp = full.term_ptr.astype(np.int64)
    x = synth.host_vectors(len(docs), seed=5)
    q = synth.host_queries(4, seed=6)
    lists = [full.term_ids(tokenize(s)) for s in ("zero fir procedure", "the of and section 2023 bharatiya",
                                                  "victim compensation", "bail")]
    lists = [[t for t in l if t >= 0] for l in lists]

    def plan():
        return csr_remove(full.stats(), [0, 5, 17, 900], docs.__getitem__, lambda t, c: full.postings[_ranges(tp[t], c), 0])

    def unsorted_list(p):
        t = int(np.nonzero(np.diff(p.rem_ptr) >= 2)[0][0])
        a = int(p.rem_ptr[t])
        p.rem_doc[a], p.rem_doc[a + 1] = p.rem_doc[a + 1], p.rem_doc[a]

    def foreign_doc(p):                                  # an id that is not among the term's postings
        t = int(np.nonzero(np.diff(p.rem_ptr) == 1)[0][0])
        p.rem_doc[p.rem_ptr[t]] = 17 if p.rem_doc[p.rem_ptr[t]] != 17 else 5

    def missing_entry(p):                                # a removed posting absent from its list: the
        t = int(np.nonzero(np.diff(p.rem_ptr) == 1)[0][0])   # removed count no longer matches the output
        p.rem_doc = np.delete(p.rem_doc, p.rem_ptr[t])       # size (the host end check refuses it)
        p.rem_ptr[t + 1:] -= 1

    def missing_entry_consistent_tables(p):              # the same, with t's output range one longer, so
        t = int(np.nonzero((np.diff(p.rem_ptr) == 1) & (p.term_map >= 0))[0][0])   # every count adds up:
        p.rem_doc = np.delete(p.rem_doc, p.rem_ptr[t])       # only the copy kernel sees that a removed
        p.rem_ptr[t + 1:] -= 1                               # posting is not its term's next listed one
        p.term_ptr[p.term_map[t] + 1:] += 1

    def term_map_not_bijective(p):
        live = np.nonzero(p.term_map >= 0)[0]
        p.term_map[live[1]] = p.term_map[live[0]]

    def term_map_swapped(p):                             # a bijection whose ranges have the wrong lengths
        live = np.nonzero(p.term_map >= 0)[0]
        a, b = live[0], next(t for t in live if p.stats.df[p.term_map[t]] != p.stats.df[p.term_map[live[0]]])
        p.term_map[a], p.term_map[b] = p.term_map[b], p.term_map[a]

    def removed_unsorted(p):
        p.removed = p.removed[::-1].copy()

    dev = DeviceIndex(0)
    try:
        dev.set_corpus(torch.from_numpy(x).cuda(), 0, prefilter=True)
        dev.set_postings(full.term_ptr, full.postings, full.doc_len, full.idf, full.avgdl)
        before = dev.search_batch_host(q, lists, 10, [0.5] * 4)
        post = dev._post
        for corrupt in (unsorted_list, foreign_doc, missing_entry, missing_entry_consistent_tables,
                        term_map_not_bijective, term_map_swapped, removed_unsorted):
            p = plan()
            corrupt(p)
            with pytest.raises(LrxError) as e:
                dev.remove_postings(p)
            assert e.value.code == LRX_E_ARG, corrupt.__name__
            assert dev._post is post and dev.n_docs == full.n_docs
            after = dev.search_batch_host(q, lists, 10, [0.5] * 4)
            assert all(np.array_equal(u, v) for u, v in zip(before, after)), corrupt.__name__
        dev.remove_postings(plan())                          # the intact plan goes through
        assert dev.n_docs == full.n_docs - 4
    finally:
        dev.close()


def test_concurrent_searches_see_before_or_after(env, legal_chunks):
    from legal_rag_engine_b200.serving import MicroBatchingEngine
    queries = ["What is the procedure for Zero FIR?", "Compensation for victims of acid attack",
               "Definition of a public servant under BNS", "What is the punishment for murder?",
               "How to file FIR for robbery BNSS procedure", "bail for non-bailable offence"]
    key = lambda rs: [(r["chunk"]["canonical_header"], r["chunk"]["text"], r["score"], r["semantic"], r["keyword"])
                      for r in rs]
    ref = _engine(env)
    try:
        before = {q: key(ref.search(q, k=5, hybrid_weight=0.6)) for q in queries}
        tops = sorted({next(i for i, c in enumerate(ref.chunks) if c is ref.search(q, k=5, hybrid_weight=0.6)[0]["chunk"])
                       for q in queries})
        drop = sorted(set(tops) | set(range(0, 2620, 3)))
        ref.remove_chunks(drop)
        after = {q: key(ref.search(q, k=5, hybrid_weight=0.6)) for q in queries}
    finally:
        ref.close()
    assert all(before[q] != after[q] for q in queries)
    mb = MicroBatchingEngine(_engine(env), max_batch=8, max_wait_ms=1.0)
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
        mb.remove_chunks(drop)                                    # forwarded to the engine
        n_mid = len(got)
        while len(got) < n_mid + 40:
            threading.Event().wait(0.005)
        stop.set()
        for t in ts:
            t.join()
        assert all(res in (before[q], after[q]) for q, res in got)
        assert any(res == after[q] for q, res in got[n_mid:])
    finally:
        mb.close()
