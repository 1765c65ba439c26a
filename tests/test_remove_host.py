"""Removing documents from a BM25 index on the host: BM25Index.remove must equal a from-scratch build
over the remaining documents, field by field and bit for bit -- vocabulary order, CSR, lengths, idf
bits, avgdl -- and csr_remove must read no more documents than its complexity bound allows."""
import numpy as np
import pytest

from legal_rag_engine_b200.bm25_index import BM25Index, _ranges, csr_remove, okapi_idf, remove_csr, tokenize


def _same(a: BM25Index, b: BM25Index):
    assert a.n_docs == b.n_docs
    assert list(a.vocab.items()) == list(b.vocab.items())            # ids AND insertion order
    for name in ("term_ptr", "postings", "doc_len"):
        x, y = getattr(a, name), getattr(b, name)
        assert x.dtype == y.dtype and x.shape == y.shape, name
        np.testing.assert_array_equal(x, y, err_msg=name)
    assert a.idf.dtype == np.float64
    np.testing.assert_array_equal(a.idf.view(np.uint64), b.idf.view(np.uint64))
    assert a.avgdl == b.avgdl and (a.k1, a.b, a.epsilon) == (b.k1, b.b, b.epsilon)


def _stats_copy(s):
    return list(s.vocab.items()), s.df.copy(), s.first_doc.copy(), s.idf.view(np.uint64).copy()


def _assert_stats_unchanged(s, kept):
    """A plan leaves the statistics it was given as they were: vocabulary items and order, df,
    first_doc, idf bits."""
    items, df, first, idf = kept
    assert list(s.vocab.items()) == items
    np.testing.assert_array_equal(s.df, df)
    np.testing.assert_array_equal(s.first_doc, first)
    np.testing.assert_array_equal(s.idf.view(np.uint64), idf)


@pytest.fixture(scope="module")
def docs(legal_texts):
    return [tokenize(t) for t in legal_texts]


def _rare_word_docs(docs):
    """Every document holding some word of document frequency 3 (the word vanishes with them)."""
    full = BM25Index.from_token_lists(docs)
    df = np.diff(full.term_ptr.astype(np.int64))
    word = next(w for w, t in full.vocab.items() if df[t] == 3)
    return word, [d for d, toks in enumerate(docs) if word in toks]


def _removal_sets(docs):
    n = len(docs)
    rng = np.random.default_rng(20)
    return {"chunk0": [0], "first50": list(range(50)),
            "random10pct": sorted(rng.choice(n, n // 10, replace=False).tolist()),
            "every_other": list(range(1, n, 2)), "rare_word": _rare_word_docs(docs)[1], "last": [n - 1]}


class _Tokens:
    """A doc_tokens stub that counts the documents it is asked for."""
    def __init__(self, docs):
        self.docs, self.calls = docs, []

    def __call__(self, d):
        self.calls.append(d)
        return self.docs[d]


@pytest.mark.parametrize("which", ["chunk0", "first50", "random10pct", "every_other", "rare_word", "last"])
def test_remove_equals_rebuild_on_the_real_corpus(docs, which):
    removed = _removal_sets(docs)[which]
    gone = set(removed)
    full = BM25Index.from_token_lists(docs)
    want = BM25Index.from_token_lists([t for d, t in enumerate(docs) if d not in gone])
    tok = _Tokens(docs)
    got = full.remove(removed, tok)
    _same(got, want)
    # reads: each removed document once, then only new first documents of affected terms
    tp = full.term_ptr.astype(np.int64)
    first = full.postings[tp[:-1], 0]
    r = np.bincount([full.vocab[w] for d in removed for w in set(docs[d])], minlength=full.n_terms)
    affected = {t for t in np.nonzero(r)[0].tolist() if first[t] in gone and np.diff(tp)[t] > r[t]}
    assert tok.calls[:len(removed)] == sorted(removed)
    extra = tok.calls[len(removed):]
    assert len(extra) == len(set(extra)) <= len(affected)
    assert not gone & set(extra)
    if which == "chunk0":
        assert len(affected) > 0 and len(extra) > 0                  # every distinct token of chunk 0 is first seen there


def test_csr_remove_plan_and_host_compaction(docs):
    full = BM25Index.from_token_lists(docs)
    removed = list(range(50))
    tp = full.term_ptr.astype(np.int64)
    stats = full.stats()
    kept = _stats_copy(stats)
    rem = csr_remove(stats, removed, docs.__getitem__, lambda t, c: full.postings[_ranges(tp[t], c), 0])
    _assert_stats_unchanged(stats, kept)
    want = BM25Index.from_token_lists(docs[50:])
    s = rem.stats
    assert s.n_docs == want.n_docs and s.avgdl == want.avgdl
    assert s.total_len == int(want.doc_len.sum())
    np.testing.assert_array_equal(rem.term_ptr, want.term_ptr.astype(np.int64))
    np.testing.assert_array_equal(s.df, np.diff(want.term_ptr.astype(np.int64)))
    np.testing.assert_array_equal(s.first_doc, want.postings[want.term_ptr[:-1].astype(np.int64), 0])
    np.testing.assert_array_equal(s.idf.view(np.uint64), want.idf.view(np.uint64))
    # per-term removed lists: exactly the postings of the removed documents, ascending
    term_of = np.repeat(np.arange(full.n_terms), np.diff(tp))
    hit = full.postings[:, 0] < 50
    np.testing.assert_array_equal(np.diff(rem.rem_ptr), np.bincount(term_of[hit], minlength=full.n_terms))
    np.testing.assert_array_equal(rem.rem_doc, full.postings[hit, 0])
    assert sorted(rem.term_map[rem.term_map >= 0].tolist()) == list(range(rem.n_terms))
    tp_out, po = remove_csr(full.term_ptr, full.postings, rem)
    np.testing.assert_array_equal(tp_out, want.term_ptr)
    np.testing.assert_array_equal(po, want.postings)
    rem.commit_vocab()
    assert s.vocab is stats.vocab and list(s.vocab.items()) == list(want.vocab.items())


def test_old_id_order_would_change_the_floored_idf_bits(docs):
    """After removing chunks 0-49, the mean idf summed in the old term-id order differs in the last
    bits from the rebuild's: every floored idf would be wrong if the vocabulary kept its old order."""
    full = BM25Index.from_token_lists(docs)
    want = BM25Index.from_token_lists(docs[50:])
    got = full.remove(range(50), docs.__getitem__)
    df_new = np.diff(want.term_ptr.astype(np.int64))
    old_order = np.argsort([full.vocab[w] for w in want.vocab], kind="stable")
    naive, _ = okapi_idf(df_new[old_order], want.n_docs)
    naive_by_term = np.empty_like(naive)
    naive_by_term[old_order] = naive
    raw = np.array([np.log(want.n_docs - f + 0.5) - np.log(f + 0.5) for f in df_new])
    floored = raw < 0
    assert floored.sum() >= 10
    assert (naive_by_term[floored] != want.idf[floored]).all()
    np.testing.assert_array_equal(got.idf.view(np.uint64), want.idf.view(np.uint64))


def test_remove_append_remove_sequence(docs):
    """A word that vanishes and comes back is numbered at its new first appearance."""
    word, holders = _rare_word_docs(docs)
    live = list(range(len(docs)))
    idx = BM25Index.from_token_lists(docs)
    idx = idx.remove(holders, lambda d: docs[live[d]])
    live = [d for d in live if d not in set(holders)]
    _same(idx, BM25Index.from_token_lists([docs[d] for d in live]))
    assert word not in idx.vocab
    back = [["a", "new", word, "document"], docs[holders[0]]]
    idx = idx.append(back)
    corpus = [docs[d] for d in live] + back
    _same(idx, BM25Index.from_token_lists(corpus))
    assert idx.vocab[word] > max(idx.vocab[w] for w in docs[live[-1]])
    drop = [0, 7, len(corpus) - 2]                                   # includes a just-appended document
    idx = idx.remove(drop, corpus.__getitem__)
    _same(idx, BM25Index.from_token_lists([c for i, c in enumerate(corpus) if i not in drop]))


def test_small_corpora_and_rejected_input():
    corpus = [["zero", "fir", "zero"], ["bail", "fir"], ["bail"], ["quokka", "zero"]]
    full = BM25Index.from_token_lists(corpus)
    for drop in ([], [0], [1, 2], [0, 3], [0, 1, 2]):
        _same(full.remove(drop, corpus.__getitem__),
              BM25Index.from_token_lists([c for i, c in enumerate(corpus) if i not in drop]))
    for bad in ([4], [-1], [1, 1], [0, 1, 2, 3]):
        with pytest.raises(ValueError):
            full.remove(bad, corpus.__getitem__)
    with pytest.raises(ValueError):                                   # text that does not match the index
        full.remove([0], lambda d: ["unknown"])


def test_remove_chunks_on_a_sharded_engine_raises_before_touching_anything():
    from legal_rag_engine_b200.engine import RetrievalEngine
    eng = RetrievalEngine.__new__(RetrievalEngine)                   # no GPU: a stub with the state it reads
    eng.world, eng.rank = 2, 0
    eng.chunks = [{"text": "a"}, {"text": "b"}]
    eng.n_total = 2
    with pytest.raises(NotImplementedError):
        eng.remove_chunks([0])
    assert eng.chunks == [{"text": "a"}, {"text": "b"}] and eng.n_total == 2
