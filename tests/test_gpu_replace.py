"""RetrievalEngine.replace_chunks and the device postings merge (lrx_bm25_replace_postings): an index
whose chunks were replaced in place answers exactly as one rebuilt from the edited chunk list -- same
chunks at the same positions, bit-identical float64 scores -- with the pre-filter on and off, at the
reference corpus and at 1 M synthetic rows."""
import json
import threading

import numpy as np
import pytest
import torch

from legal_rag_engine_b200 import synth

from test_gpu_remove import (_answers, _assert_device_equals_fresh, _assert_matches_oracle, _engine,  # noqa: F401
                             _rebuilt, _synthetic, env)

pytestmark = pytest.mark.gpu

LRX_E_ARG = -1


def _amend(chunk, how):
    """A new version of a chunk: same metadata, edited text."""
    words = chunk["text"].split()
    text = {"reverse": " ".join(words[::-1]), "empty": "",
            "trim": " ".join(w for w in words if w.lower() not in ("the", "section", "of")) + " amended quokka"}[how]
    return dict(chunk, text=text)


def _replacement_sets(chunks):
    """name -> (ids, new chunks)."""
    n = len(chunks)
    rng = np.random.default_rng(23)
    rand = sorted(rng.choice(n, n // 10, replace=False).tolist())
    return {"one": ([17], [_amend(chunks[17], "reverse")]),
            "block50": (list(range(100, 150)), [_amend(chunks[i], "reverse") for i in range(100, 150)]),
            "random10pct": (rand, [dict(chunks[(i * 7 + 3) % n]) for i in rand]),
            "chunk0": ([0], [_amend(chunks[0], "trim")]),
            "last": ([n - 1], [_amend(chunks[n - 1], "reverse")]),
            "empty": ([5], [_amend(chunks[5], "empty")])}


_SETS = ["one", "block50", "random10pct", "chunk0", "last", "empty"]


@pytest.mark.parametrize("which", _SETS)
def test_replacement_answers_as_a_rebuild(env, legal_chunks, reference_queries, which):
    from legal_rag_engine_b200.bm25_index import BM25Index
    ids, new = _replacement_sets(legal_chunks)[which]
    eng = _engine(env)
    try:
        x_before = eng._x.cpu().numpy()
        assert eng.replace_chunks(ids, new) is None
        edited = list(legal_chunks)
        for i, c in zip(ids, new):
            edited[i] = c
        assert eng.chunks == edited and eng.n_total == len(legal_chunks)
        x_after = eng._x.cpu().numpy()
        others = np.setdiff1d(np.arange(len(legal_chunks)), ids)
        np.testing.assert_array_equal(x_after[others].view(np.uint16), x_before[others].view(np.uint16))
        np.testing.assert_array_equal(x_after[ids].view(np.uint16),
                                      eng.encode([c["text"] for c in new]).astype(np.float16).view(np.uint16))
        ref = _rebuilt(env, f"rebuilt_rep_{which}", edited, x_after)
        try:
            assert _answers(eng, reference_queries) == _answers(ref, reference_queries)
        finally:
            ref.close()
        want = BM25Index.from_texts([c["text"] for c in edited])
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


def test_old_text_is_gone_after_captured_chains(env, legal_chunks):
    """Same-shape searches run direct, then captured, then replayed; a replacement must retire those
    chains, and a word only the old text held finds nothing afterwards."""
    from legal_rag_engine_b200.bm25_index import BM25Index, tokenize
    docs = [tokenize(c["text"]) for c in legal_chunks]
    full = BM25Index.from_token_lists(docs)
    df = np.diff(full.term_ptr.astype(np.int64))
    word = next(w for w, t in full.vocab.items() if df[t] == 1 and w.isalpha())
    holder = next(i for i, d in enumerate(docs) if word in d)
    eng = _engine(env)
    try:
        # rrf fuses the BM25 top list itself (linear fusion only re-weights the dense candidates)
        first = [eng.search(word, k=5, fusion="rrf") for _ in range(3)]
        assert first[0] == first[1] == first[2]
        assert [r["keyword"] > 0 for r in first[0]].count(True) == 1
        assert next(r for r in first[0] if r["keyword"] > 0)["chunk"] is eng.chunks[holder]
        new = dict(legal_chunks[holder], text=" ".join(w for w in legal_chunks[holder]["text"].split()
                                                        if w.lower() != word))
        eng.replace_chunks([holder], [new])
        for _ in range(3):
            after = eng.search(word, k=5, fusion="rrf")
            assert len(after) == 5 and all(r["keyword"] == 0.0 for r in after)
        assert word not in eng.bm25.vocab
    finally:
        eng.close()


def test_rejected_input_changes_nothing(env, reference_queries):
    eng = _engine(env)
    try:
        before = _answers(eng, reference_queries)
        n, x_ptr, post = eng.n_total, eng._x.data_ptr(), eng.dev._post
        x = eng._x.clone()
        c = {"text": "amended"}
        for ids, chunks, exc in (([n], [c], ValueError), ([-1], [c], ValueError), ([3, 3], [c, c], ValueError),
                                 ([1], [c, c], ValueError), ([True], [c], TypeError), ([1.0], [c], TypeError),
                                 ([1], [{"text": None}], ValueError), ([1], [{"text": "a " * 65536}], ValueError)):
            with pytest.raises(exc):
                eng.replace_chunks(ids, chunks)
        assert eng.replace_chunks([], []) is None
        assert eng.n_total == n and eng._x.data_ptr() == x_ptr and eng.dev._post is post
        assert torch.equal(eng._x, x)
        assert _answers(eng, reference_queries) == before
    finally:
        eng.close()


def test_interleaved_adds_removals_and_replacements(env, legal_chunks, reference_queries, tmp_path):
    """Store of 2 000 chunks; add, replace (old and just-added chunks), remove, replace again; after each
    step the engine answers as a rebuild, and save() writes the rebuilt store's files."""
    eng = _engine(env, "first")
    try:
        live = list(legal_chunks[:2000])

        def check(step):
            assert eng.chunks == live
            ref = _rebuilt(env, f"rebuilt_rseq{step}", live, eng._x.cpu().numpy())
            try:
                assert _answers(eng, reference_queries) == _answers(ref, reference_queries), step
            finally:
                ref.close()
            _assert_device_equals_fresh(eng)

        eng.add_chunks(legal_chunks[2000:2200])
        live += legal_chunks[2000:2200]
        check(1)
        ids = [0, 3, 1999, 2000, 2199]
        new = [_amend(live[i], "trim") for i in ids]
        eng.replace_chunks(ids, new)
        for i, c in zip(ids, new):
            live[i] = c
        check(2)
        drop = [1, 2000, 2100]
        eng.remove_chunks(drop)
        live = [c for i, c in enumerate(live) if i not in drop]
        check(3)
        ids = [0, 500, len(live) - 1]
        new = [_amend(live[500], "reverse"), dict(live[0]), _amend(live[-1], "empty")]
        eng.replace_chunks(ids, new)
        for i, c in zip(ids, new):
            live[i] = c
        check(4)
        out = eng.save(tmp_path / "saved")
        reb = env[0] / "rebuilt_rseq4"
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


def test_inconsistent_plan_is_refused_and_the_index_keeps_answering(legal_texts):
    """A plan whose lists or maps do not describe the postings: LRX_E_ARG, and the resident index
    answers as before."""
    from legal_rag_engine_b200._lib import LrxError
    from legal_rag_engine_b200.bm25_index import BM25Index, _ranges, csr_replace, tokenize
    from legal_rag_engine_b200.device_index import DeviceIndex
    docs = [tokenize(t) for t in legal_texts]
    full = BM25Index.from_token_lists(docs)
    tp = full.term_ptr.astype(np.int64)
    x = synth.host_vectors(len(docs), seed=5)
    q = synth.host_queries(4, seed=6)
    lists = [full.term_ids(tokenize(s)) for s in ("zero fir procedure", "the of and section 2023 bharatiya",
                                                  "victim compensation", "bail")]
    lists = [[t for t in l if t >= 0] for l in lists]
    ids = [0, 5, 17, 900]

    def plan():
        new = [docs[900][::-1], ["amended", "quokka"] + docs[5], docs[17], docs[0]]
        p = csr_replace(full.stats(), ids, new, docs.__getitem__, lambda t, c: full.postings[_ranges(tp[t], c), 0])
        dl = full.doc_len.copy()
        dl[p.replaced] = p.doc_len
        return p, dl

    def unsorted_list(p):
        t = int(np.nonzero(np.diff(p.rem_ptr) >= 2)[0][0])
        a = int(p.rem_ptr[t])
        p.rem_doc[a], p.rem_doc[a + 1] = p.rem_doc[a + 1], p.rem_doc[a]

    def foreign_doc(p):                                  # a replaced document that is not among the term's postings
        t = next(t for t in np.nonzero(np.diff(p.rem_ptr) == 1)[0]
                 if 17 not in full.postings[tp[t]:tp[t + 1], 0])
        p.rem_doc[p.rem_ptr[t]] = 17

    def missing_entry(p):                                # a dropped posting absent from its list, the output
        t = int(np.nonzero((np.diff(p.rem_ptr) == 1) & (p.term_map >= 0))[0][0])   # range one longer so that
        p.rem_doc = np.delete(p.rem_doc, p.rem_ptr[t])   # every count adds up: only the copy kernel sees it
        p.rem_ptr[t + 1:] -= 1
        p.term_ptr[p.term_map[t] + 1:] += 1

    def term_map_not_injective(p):
        live = np.nonzero(p.term_map >= 0)[0]
        p.term_map[live[1]] = p.term_map[live[0]]

    def wrong_range_length(p):
        p.term_ptr[1:-1] += 1                            # the first new term's range one longer, the last one shorter

    def inserted_not_replaced(p):                        # an inserted entry for a document that is not replaced
        j = int(p.ins_ptr[1]) - 1
        p.ins_postings[j, 0] = 1 if p.ins_postings[j, 0] != 1 else 2

    dev = DeviceIndex(0)
    try:
        dev.set_corpus(torch.from_numpy(x).cuda(), 0, prefilter=True)
        dev.set_postings(full.term_ptr, full.postings, full.doc_len, full.idf, full.avgdl)
        before = dev.search_batch_host(q, lists, 10, [0.5] * 4)
        post = dev._post
        for corrupt in (unsorted_list, foreign_doc, missing_entry, term_map_not_injective, wrong_range_length,
                        inserted_not_replaced):
            p, dl = plan()
            corrupt(p)
            with pytest.raises(LrxError) as e:
                dev.stage_replace(p, dl)
            assert e.value.code == LRX_E_ARG, corrupt.__name__
            assert dev._post is post and dev.n_docs == full.n_docs
            after = dev.search_batch_host(q, lists, 10, [0.5] * 4)
            assert all(np.array_equal(u, v) for u, v in zip(before, after)), corrupt.__name__
        p, dl = plan()
        dev.commit_postings(dev.stage_replace(p, dl))     # the intact plan goes through
        assert dev.n_terms == p.n_terms
    finally:
        dev.close()


def test_concurrent_searches_see_before_or_after(env, legal_chunks):
    from legal_rag_engine_b200.serving import MicroBatchingEngine
    queries = ["What is the procedure for Zero FIR?", "Compensation for victims of acid attack",
               "Definition of a public servant under BNS", "What is the punishment for murder?",
               "How to file FIR for robbery BNSS procedure", "bail for non-bailable offence"]
    key = lambda rs: [(r["chunk"]["canonical_header"], r["chunk"]["text"], r["score"], r["semantic"], r["keyword"])
                      for r in rs]
    n = len(legal_chunks)
    ref = _engine(env)
    try:
        before = {q: key(ref.search(q, k=5, hybrid_weight=0.6)) for q in queries}
        tops = sorted({next(i for i, c in enumerate(ref.chunks) if c is ref.search(q, k=5, hybrid_weight=0.6)[0]["chunk"])
                       for q in queries})
        ids = sorted(set(tops) | set(range(0, n, 3)))
        new = [_amend(legal_chunks[i], "reverse") if i in tops else dict(legal_chunks[(i + 1) % n]) for i in ids]
        ref.replace_chunks(ids, new)
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
        mb.replace_chunks(ids, new)                                   # forwarded to the engine
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


def synthetic_plan(idx, replaced, rng, new_terms=5, mean_len=60):
    """A replacement plan over an index without a string vocabulary: each replaced document gets Zipf
    text over the old terms plus `new_terms` new ones; the surviving terms are numbered by a random
    permutation (the kernel takes any injective map).  Returns (plan, doc_len after the edit)."""
    from legal_rag_engine_b200.bm25_index import BM25Replace, BM25Stats, okapi_idf
    tp = idx.term_ptr.astype(np.int64)
    V, n = idx.n_terms, idx.n_docs
    doc = idx.postings[:, 0].astype(np.int64)
    gone = np.isin(doc, replaced)
    term_of = np.repeat(np.arange(V), np.diff(tp))
    r = np.bincount(term_of[gone], minlength=V)
    rem_ptr = np.zeros(V + 1, dtype=np.int64)
    np.cumsum(r, out=rem_ptr[1:])
    lens = rng.integers(0, 2 * mean_len, len(replaced))
    cdf = synth._zipf_cdf(V)
    toks = np.minimum(np.searchsorted(cdf, rng.random(int(lens.sum())), side="right"), V - 1)
    toks = np.where(rng.random(len(toks)) < 0.01, V + rng.integers(0, new_terms, len(toks)), toks)
    tok_doc = np.repeat(np.asarray(replaced, dtype=np.int64), lens)
    W = V + new_terms
    uniq, tf = np.unique(toks * n + tok_doc, return_counts=True)
    it, idd = uniq // n, uniq % n
    df_ext = np.concatenate([np.diff(tp) - r, np.zeros(new_terms, np.int64)]) + np.bincount(it, minlength=W)
    order = rng.permutation(np.nonzero(df_ext > 0)[0])
    ext = np.full(W, -1, dtype=np.int32)
    ext[order] = np.arange(len(order), dtype=np.int32)
    df_out = df_ext[order]
    term_ptr = np.zeros(len(order) + 1, dtype=np.int64)
    np.cumsum(df_out, out=term_ptr[1:])
    nt = ext[it].astype(np.int64)
    o = np.lexsort((idd, nt))
    ins = np.stack([idd[o], tf[o]], axis=1).astype(np.uint32)
    ins_ptr = np.zeros(len(order) + 1, dtype=np.int64)
    np.cumsum(np.bincount(nt, minlength=len(order)), out=ins_ptr[1:])
    doc_len = idx.doc_len.copy()
    doc_len[replaced] = lens
    total = int(doc_len.astype(np.int64).sum())
    idf, _ = okapi_idf(df_out, n)
    plan = BM25Replace(np.asarray(replaced, dtype=np.int64), lens.astype(np.uint32), rem_ptr,
                       doc[gone].astype(np.uint32), ext[:V], [f"new{i}" for i in range(new_terms)], ext[V:], ins_ptr,
                       ins, term_ptr, BM25Stats({}, df_out, np.zeros(0, np.int64), n, total, idf, total / n))
    return plan, doc_len


def test_one_million_rows_replace():
    """1 M synthetic rows + Zipf BM25; replace 37 scattered documents, then a block of 100 000 plus the
    first and the last.  After each step the device postings equal replace_csr byte for byte (as a fresh
    build packs them), and search_batch_host answers as a handle set up from scratch."""
    from legal_rag_engine_b200.bm25_index import BM25Index, replace_csr
    from legal_rag_engine_b200.device_index import DeviceIndex
    n = 1_000_000
    rng = np.random.default_rng(81)
    x = synth.host_vectors(n, seed=61)
    idx = _synthetic(n, 62, (420_000, 480_000))
    B, k = 8, 10
    q = synth.host_queries(B, seed=63)
    terms, ptr = synth.host_query_terms(B, 8, seed=65)
    lists = [terms[ptr[b]:ptr[b + 1]].tolist() for b in range(B)]
    w = [0.5, 0.6] * (B // 2)
    steps = (np.sort(rng.choice(np.arange(1, n - 1), 37, replace=False)),
             np.concatenate([[0], np.arange(400_000, 500_000), [n - 1]]))
    dev = DeviceIndex(0)
    try:
        dev.set_corpus(torch.from_numpy(x).cuda(), 0, prefilter=True)
        dev.set_postings(idx.term_ptr, idx.postings, idx.doc_len, idx.idf, idx.avgdl)
        for replaced in steps:
            rep, doc_len = synthetic_plan(idx, replaced, rng)
            dev.commit_postings(dev.stage_replace(rep, doc_len))
            x_new = synth.host_vectors(len(replaced), seed=int(replaced[0]) + 7)
            dev.replace_rows(replaced, torch.from_numpy(x_new).cuda(), prefilter=True)
            x[replaced] = x_new
            tp, po = replace_csr(idx.term_ptr, idx.postings, rep)
            idx = BM25Index(n, doc_len, tp, po, rep.stats.idf, rep.stats.avgdl)
            lists = [[int(rep.term_map[t]) for t in l if rep.term_map[t] >= 0] for l in lists]
            fresh = DeviceIndex(0)
            try:
                fresh.set_corpus(torch.from_numpy(x).cuda(), 0, prefilter=True)
                assert dev.prefilter_bounds == fresh.prefilter_bounds
                fresh.set_postings(tp, po, doc_len, rep.stats.idf, rep.stats.avgdl)
                nnz = rep.nnz
                assert dev._post_args == fresh._post_args
                assert torch.equal(dev._post[0], fresh._post[0])
                assert torch.equal(dev._post[1][:nnz], fresh._post[1][:nnz])
                if nnz % 2:
                    assert not dev._post[1][nnz].any()
                assert torch.equal(dev._post[2], fresh._post[2])
                assert torch.equal(dev.doc_len, fresh.doc_len)
                for fusion in ("linear", "rrf"):
                    for on in (True, False):
                        dev.set_prefilter(on)
                        fresh.set_prefilter(on)
                        got = dev.search_batch_host(q, lists, k, w, fusion)
                        want = fresh.search_batch_host(q, lists, k, w, fusion)
                        assert all(np.array_equal(u, v) for u, v in zip(got, want)), (fusion, on)
            finally:
                fresh.close()
    finally:
        dev.close()
