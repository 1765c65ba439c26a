"""Replacing documents' text in place in a BM25 index on the host: BM25Index.replace must equal a
from-scratch build over the edited documents, field by field and bit for bit -- vocabulary order,
CSR, lengths, idf bits, avgdl -- and RetrievalEngine.replace_chunks must refuse bad input before
anything changes."""
import numpy as np
import pytest

from legal_rag_engine_b200.bm25_index import BM25Index, _ranges, csr_replace, replace_csr, tokenize
from legal_rag_engine_b200 import synth


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
    return list(s.vocab.items()), s.df.copy(), s.first_doc.copy(), s.idf.view(np.uint64).copy(), s.total_len


def _assert_stats_unchanged(s, kept):
    items, df, first, idf, total = kept
    assert list(s.vocab.items()) == items
    np.testing.assert_array_equal(s.df, df)
    np.testing.assert_array_equal(s.first_doc, first)
    np.testing.assert_array_equal(s.idf.view(np.uint64), idf)
    assert s.total_len == total


@pytest.fixture(scope="module")
def docs(legal_texts):
    return [tokenize(t) for t in legal_texts]


def _late_word(docs, start):
    """A word first seen at or after document `start` and absent from documents 0..4."""
    early = set(w for d in docs[:5] for w in d)
    seen = set(w for d in docs[:start] for w in d)
    return next(w for d in docs[start:] for w in d if w not in seen and w not in early)


def _replacement_sets(docs):
    """name -> (ids, new token lists).  Covers the cases a rebuild numbers differently."""
    n = len(docs)
    rng = np.random.default_rng(31)
    full = BM25Index.from_token_lists(docs)
    df = np.diff(full.term_ptr.astype(np.int64))
    rare = next(w for w, t in full.vocab.items() if df[t] == 2)
    holders = [d for d, t in enumerate(docs) if rare in t]
    late = _late_word(docs, n // 2)
    rand = sorted(rng.choice(n, n // 10, replace=False).tolist())
    return {
        "identity": ([0, 7, n - 1], [docs[0], docs[7], docs[n - 1]]),
        "new_words": ([3, 11], [["zqxv", "amended"] + docs[3], ["amended", "yyzzy", "zqxv"]]),
        "vanish": (holders, [[w for w in docs[d] if w != rare] for d in holders]),
        "chunk0_loses_common": ([0], [[w for w in docs[0] if w not in ("the", "section")] + ["amended"]]),
        "first_moves_earlier": ([2], [[late] + docs[2]]),
        "shared_new_words": ([5, 9, 40], [["novelword", "w2"] + docs[5], docs[9] + ["w2", "novelword"],
                                          ["w2", "w3"]]),
        "empty": ([4], [[]]),
        "reversed_block": (list(range(50)), [docs[d][::-1] for d in range(50)]),
        "random10pct": (rand, [docs[(d * 7 + 3) % n] for d in rand]),
        "unsorted_ids": ([30, 1, 17], [docs[17], docs[30], ["tail", "of", "the"]]),
        "every": (list(range(n)), [docs[(d + 1) % n] for d in range(n)]),
    }


_SETS = ["identity", "new_words", "vanish", "chunk0_loses_common", "first_moves_earlier", "shared_new_words",
         "empty", "reversed_block", "random10pct", "unsorted_ids", "every"]


def _edited(docs, ids, new):
    out = list(docs)
    for i, t in zip(ids, new):
        out[i] = t
    return out


@pytest.mark.parametrize("which", _SETS)
def test_replace_equals_rebuild_on_the_real_corpus(docs, which):
    ids, new = _replacement_sets(docs)[which]
    full = BM25Index.from_token_lists(docs)
    want = BM25Index.from_token_lists(_edited(docs, ids, new))
    _same(full.replace(ids, new, docs.__getitem__), want)
    if which == "chunk0_loses_common":
        assert "the" in docs[0] and "section" in docs[0]             # chunk 0 held them first
        assert want.vocab["the"] > full.vocab["the"] and want.vocab["section"] > full.vocab["section"]
    if which == "first_moves_earlier":
        late = new[0][0]
        assert want.vocab[late] < full.vocab[late]                  # its id moved
    if which == "vanish":
        gone = next(w for w in full.vocab if w not in want.vocab)
        assert gone and len(want.vocab) < len(full.vocab)


def test_plan_and_host_compaction(docs):
    full = BM25Index.from_token_lists(docs)
    ids, new = _replacement_sets(docs)["reversed_block"]
    ids, new = ids + [60, 61], new + [["zqxv"] + docs[60], []]
    tp = full.term_ptr.astype(np.int64)
    stats = full.stats()
    kept = _stats_copy(stats)
    rep = csr_replace(stats, ids, new, docs.__getitem__, lambda t, c: full.postings[_ranges(tp[t], c), 0])
    _assert_stats_unchanged(stats, kept)
    want = BM25Index.from_token_lists(_edited(docs, ids, new))
    s = rep.stats
    assert s.n_docs == want.n_docs and s.avgdl == want.avgdl and s.total_len == int(want.doc_len.sum())
    np.testing.assert_array_equal(rep.term_ptr, want.term_ptr.astype(np.int64))
    np.testing.assert_array_equal(s.df, np.diff(want.term_ptr.astype(np.int64)))
    np.testing.assert_array_equal(s.first_doc, want.postings[want.term_ptr[:-1].astype(np.int64), 0])
    np.testing.assert_array_equal(s.idf.view(np.uint64), want.idf.view(np.uint64))
    # dropped lists: exactly the postings of the replaced documents, ascending
    term_of = np.repeat(np.arange(full.n_terms), np.diff(tp))
    hit = np.isin(full.postings[:, 0], ids)
    np.testing.assert_array_equal(np.diff(rep.rem_ptr), np.bincount(term_of[hit], minlength=full.n_terms))
    np.testing.assert_array_equal(rep.rem_doc, full.postings[hit, 0])
    # inserted entries: exactly the postings of the replaced documents in the rebuild
    wtp = want.term_ptr.astype(np.int64)
    whit = np.isin(want.postings[:, 0], ids)
    np.testing.assert_array_equal(np.diff(rep.ins_ptr),
                                  np.bincount(np.repeat(np.arange(want.n_terms), np.diff(wtp))[whit],
                                              minlength=want.n_terms))
    np.testing.assert_array_equal(rep.ins_postings, want.postings[whit])
    tp_out, po = replace_csr(full.term_ptr, full.postings, rep)
    np.testing.assert_array_equal(tp_out, want.term_ptr)
    np.testing.assert_array_equal(po, want.postings)
    rep.commit_vocab()
    assert s.vocab is stats.vocab and list(s.vocab.items()) == list(want.vocab.items())


def test_remove_then_add_is_not_the_edited_store(docs):
    """Why replacement exists: remove + add of chunks 0-49 with their tokens reversed gives another
    vocabulary order and, through okapi_idf's sequential mean, 22 different floored idf values."""
    full = BM25Index.from_token_lists(docs)
    new = [d[::-1] for d in docs[:50]]
    want = BM25Index.from_token_lists(new + docs[50:])
    ra = full.remove(range(50), docs.__getitem__).append(new)
    assert list(ra.vocab) != list(want.vocab)
    by_word = {w: ra.idf[t] for w, t in ra.vocab.items()}
    differ = sum(by_word[w] != want.idf[t] for w, t in want.vocab.items())
    assert differ == 22
    _same(full.replace(range(50), new, docs.__getitem__), want)


def _zipf_docs(n, seed):
    rng = np.random.default_rng(seed)
    lens = synth.host_doc_lengths(n, rng)
    cdf = synth._zipf_cdf(synth.VOCAB)
    words = np.array([f"w{i}" for i in range(synth.VOCAB)])
    toks = words[np.minimum(np.searchsorted(cdf, rng.random(int(lens.sum())), side="right"), synth.VOCAB - 1)]
    return [t.tolist() for t in np.split(toks, np.cumsum(lens)[:-1])], rng


def test_replace_equals_rebuild_on_a_zipf_corpus():
    docs, rng = _zipf_docs(3000, 5)
    idx = BM25Index.from_token_lists(docs)
    live = list(docs)
    for step in range(4):
        ids = sorted(rng.choice(len(live), [1, 40, 300, 3000][step], replace=False).tolist())
        new = [live[int(rng.integers(len(live)))][::-1][: int(rng.integers(0, 80))] + [f"n{step}_{i % 7}"]
               for i in range(len(ids))]
        idx = idx.replace(ids, new, live.__getitem__)
        live = _edited(live, ids, new)
        _same(idx, BM25Index.from_token_lists(live))


def test_replace_mixed_with_adds_and_removals(docs):
    idx = BM25Index.from_token_lists(docs[:500])
    live = list(docs[:500])
    idx = idx.append(docs[500:600]); live += docs[500:600]
    idx = idx.replace([0, 550], [["fresh", "text"], docs[0]], live.__getitem__)
    live = _edited(live, [0, 550], [["fresh", "text"], docs[0]])
    _same(idx, BM25Index.from_token_lists(live))
    idx = idx.remove([1, 599], live.__getitem__)
    live = [t for i, t in enumerate(live) if i not in (1, 599)]
    idx = idx.replace([0, 1], [docs[2], ["fresh"]], live.__getitem__)
    live = _edited(live, [0, 1], [docs[2], ["fresh"]])
    _same(idx, BM25Index.from_token_lists(live))


def test_rejected_plans_change_nothing():
    corpus = [["zero", "fir", "zero"], ["bail", "fir"], ["bail"], ["quokka", "zero"]]
    full = BM25Index.from_token_lists(corpus)
    stats = full.stats()
    kept = _stats_copy(stats)
    tp = full.term_ptr.astype(np.int64)
    gather = lambda t, c: full.postings[_ranges(tp[t], c), 0]
    for ids, new in (([1, 1], [["a"], ["b"]]), ([4], [["a"]]), ([-1], [["a"]]), ([0], [["a"], ["b"]]),
                     ([0, 1, 2, 3], [[], [], [], []])):
        with pytest.raises(ValueError):
            csr_replace(stats, ids, new, corpus.__getitem__, gather)
        _assert_stats_unchanged(stats, kept)
    with pytest.raises(ValueError):                                   # text that does not match the index
        csr_replace(stats, [0], [["a"]], lambda d: ["unknown"], gather)
    _assert_stats_unchanged(stats, kept)
    _same(full.replace([], [], corpus.__getitem__), full)
    _same(full.replace([0, 1, 2, 3], [[], [], [], ["x"]], corpus.__getitem__),
          BM25Index.from_token_lists([[], [], [], ["x"]]))


class _HostDev:
    """The DeviceIndex calls replace_chunks makes before its first device step."""
    def __init__(self, idx):
        self.idx = idx

    def posting_docs(self, terms, counts):
        tp = self.idx.term_ptr.astype(np.int64)
        return self.idx.postings[_ranges(tp[terms], counts), 0].astype(np.int64)

    def __getattr__(self, name):
        raise AssertionError(f"replace_chunks reached the device ({name}) on rejected input")


class _Model:
    def encode(self, texts):
        return np.zeros((len(texts), 384), dtype=np.float32)


def _stub_engine(texts):
    import threading
    from legal_rag_engine_b200.engine import RetrievalEngine
    eng = RetrievalEngine.__new__(RetrievalEngine)                   # no GPU: a stub with the state it reads
    eng.world, eng.rank = 1, 0
    eng.chunks = [{"text": t} for t in texts]
    eng.n_total = len(texts)
    eng._lock = threading.RLock()
    idx = BM25Index.from_texts(texts)
    eng._stats = idx.stats()
    eng.dev = _HostDev(idx)
    eng.model = _Model()
    return eng


def test_replace_chunks_rejects_bad_input_before_touching_anything():
    texts = ["zero fir zero", "bail fir", "bail"]
    eng = _stub_engine(texts)
    kept = _stats_copy(eng._stats)
    cases = (([1, 1], [{"text": "a"}] * 2, ValueError), ([3], [{"text": "a"}], ValueError),
             ([-1], [{"text": "a"}], ValueError), ([True], [{"text": "a"}], TypeError),
             ([1.0], [{"text": "a"}], TypeError), (["0"], [{"text": "a"}], TypeError),
             ([0], [{"text": "a"}, {"text": "b"}], ValueError), ([0], [{"text": 3}], ValueError),
             ([0], ["zero"], ValueError), ([0], [{"text": "w " * 65536}], ValueError),
             ([0, 1, 2], [{"text": ""}, {"text": " "}, {"text": "\n"}], ValueError))
    for ids, chunks, exc in cases:
        with pytest.raises(exc):
            eng.replace_chunks(ids, chunks)
        assert eng.chunks == [{"text": t} for t in texts] and eng.n_total == 3
        _assert_stats_unchanged(eng._stats, kept)
    assert eng.replace_chunks([], []) is None
    assert eng.chunks == [{"text": t} for t in texts]


def test_replace_chunks_on_a_sharded_engine_raises_before_touching_anything():
    from legal_rag_engine_b200.engine import RetrievalEngine
    eng = RetrievalEngine.__new__(RetrievalEngine)                   # no GPU: a stub with the state it reads
    eng.world, eng.rank = 2, 0
    eng.chunks = [{"text": "a"}, {"text": "b"}]
    eng.n_total = 2
    with pytest.raises(NotImplementedError):
        eng.replace_chunks([0], [{"text": "c"}])
    assert eng.chunks == [{"text": "a"}, {"text": "b"}] and eng.n_total == 2
