"""Appending documents to a BM25 index on the host: BM25Index.append must equal a from-scratch
build over old + new documents, field by field and bit for bit (vocabulary order, CSR, lengths,
idf bits, avgdl), and csr_append must describe the appended documents alone."""
import numpy as np
import pytest

from legal_rag_engine_b200.bm25_index import BM25Index, csr_append, merge_csr, tokenize


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


@pytest.mark.parametrize("split", [1, 1310, 2000, 2619])
def test_append_equals_rebuild_on_the_real_corpus(docs, split):
    _same(BM25Index.from_token_lists(docs[:split]).append(docs[split:]), BM25Index.from_token_lists(docs))


def test_repeated_appends_equal_rebuild(docs):
    idx = BM25Index.from_token_lists(docs[:2000])
    for lo, hi in ((2000, 2001), (2001, 2300), (2300, len(docs))):
        idx = idx.append(docs[lo:hi])
    _same(idx, BM25Index.from_token_lists(docs))


def test_append_of_new_terms_only_empty_document_and_nothing():
    old = [["zero", "fir", "zero"], ["bail", "fir"]]
    for new in ([["novel", "words", "novel"], ["only", "words"]],      # every term is new
                [[], ["fir", "late"], []],                           # empty documents
                []):                                                 # nothing appended
        _same(BM25Index.from_token_lists(old).append(new), BM25Index.from_token_lists(old + new))


def test_csr_append_is_the_appended_documents_alone(docs):
    old = BM25Index.from_token_lists(docs[:2000])
    stats = old.stats()
    kept = _stats_copy(stats)
    app = csr_append(stats, docs[2000:2100])
    _assert_stats_unchanged(stats, kept)
    full = BM25Index.from_token_lists(docs[:2100])
    assert app.n_terms == full.n_terms and app.stats.n_docs == 2100 and app.nnz == len(app.postings)
    assert app.new_words == list(full.vocab)[old.n_terms:]
    np.testing.assert_array_equal(app.stats.df, np.diff(full.term_ptr.astype(np.int64)))
    np.testing.assert_array_equal(app.stats.first_doc, full.postings[full.term_ptr[:-1].astype(np.int64), 0])
    np.testing.assert_array_equal(app.stats.idf.view(np.uint64), full.idf.view(np.uint64))
    assert app.stats.avgdl == full.avgdl and app.stats.total_len == int(full.doc_len.sum())
    # its own CSR = the rebuild's postings of documents >= 2000
    keep = full.postings[:, 0] >= 2000
    np.testing.assert_array_equal(app.postings, full.postings[keep])
    term_of = np.repeat(np.arange(full.n_terms), np.diff(full.term_ptr.astype(np.int64)))
    np.testing.assert_array_equal(np.diff(app.term_ptr), np.bincount(term_of[keep], minlength=full.n_terms))
    tp, po = merge_csr(old.term_ptr, old.postings, app)
    np.testing.assert_array_equal(tp, full.term_ptr)
    np.testing.assert_array_equal(po, full.postings)
    app.commit_vocab()
    assert stats.vocab is app.stats.vocab and list(stats.vocab.items()) == list(full.vocab.items())


def test_add_chunks_on_a_sharded_engine_raises_before_touching_anything():
    from legal_rag_engine_b200.engine import RetrievalEngine
    eng = RetrievalEngine.__new__(RetrievalEngine)                   # no GPU: a stub with the state add_chunks reads
    eng.world, eng.rank = 2, 0
    eng.chunks = [{"text": "a"}]
    eng.n_total = 1
    with pytest.raises(NotImplementedError):
        eng.add_chunks([{"text": "zero fir"}])
    with pytest.raises(NotImplementedError):
        eng.save()
    assert eng.chunks == [{"text": "a"}] and eng.n_total == 1
