"""BM25Okapi index build: statistics + term-major CSR postings for the K3 kernel.

Host side of the index build the reference does with
``BM25Okapi([text.lower().split() for text in texts])``
(create_vector_store.py:60-61).  The statistics keep rank_bm25's float64
semantics exactly (idf with the epsilon floor, average idf summed sequentially in
vocabulary insertion order, avgdl), because the CUDA kernel reproduces
``get_scores`` bit for bit from them.
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence

import numpy as np

K1 = 1.5
B = 0.75
EPSILON = 0.25


def tokenize(text: str) -> List[str]:
    """Corpus and query side alike: ``text.lower().split()``
    (create_vector_store.py:60, retrieval_engine.py:67)."""
    return text.lower().split()


def okapi_idf(df: np.ndarray, n_docs: int, epsilon: float = EPSILON):
    """rank_bm25 ``BM25Okapi._calc_idf``: ``ln(N-df+0.5) - ln(df+0.5)`` per term
    (libm log, as ``math.log``), negative values replaced by ``epsilon * mean``; the
    mean is a left-to-right float64 sum in term-id (= vocabulary insertion) order."""
    raw = np.fromiter((math.log(n_docs - int(f) + 0.5) - math.log(int(f) + 0.5) for f in df),
                      dtype=np.float64, count=len(df))
    total = float(np.add.accumulate(raw)[-1]) if len(raw) else 0.0   # sequential sum
    average_idf = total / max(len(raw), 1)
    eps = epsilon * average_idf
    return np.where(raw < 0, eps, raw), average_idf


@dataclass
class BM25Append:
    """Documents appended to an index: their own term-major CSR over the extended vocabulary, and
    the whole corpus's statistics after the append."""
    new_words: List[str]         # vocabulary extension, first-appearance order: ids n_terms, n_terms + 1, ...
    term_ptr: np.ndarray         # int64 [V_out+1]
    postings: np.ndarray         # uint32 [nnz_add, 2] = (doc id, tf), doc ids >= the old n_docs
    doc_len: np.ndarray          # uint32 [m]
    df: np.ndarray               # int64 [V_out] document frequencies, old + appended documents
    n_docs: int                  # after the append
    total_len: int               # tokens after the append
    idf: np.ndarray              # float64 [V_out]
    avgdl: float

    @property
    def n_terms(self) -> int:
        return len(self.term_ptr) - 1

    @property
    def nnz(self) -> int:
        return int(self.term_ptr[-1])


def csr_append(vocab: Dict[str, int], df: np.ndarray, n_docs: int, total_len: int,
               token_lists: Sequence[Sequence[str]], epsilon: float = EPSILON) -> BM25Append:
    """The appended documents' CSR and the updated statistics, in O(new tokens + V): no pass over
    the existing postings.  ``vocab`` is read, not changed.  A rebuild numbers terms in first
    appearance order over all documents in order; the old documents come first, so it keeps every
    old id and numbers the new terms in first-appearance order over the appended documents -- the
    order used here -- and okapi_idf's sequential mean, hence every idf bit, comes out the same."""
    new: Dict[str, int] = {}
    n_old = len(vocab)
    t_l, d_l, f_l, lens = [], [], [], []
    for d, document in enumerate(token_lists, start=n_docs):
        lens.append(len(document))
        freqs: Dict[str, int] = {}
        for word in document:
            freqs[word] = freqs.get(word, 0) + 1
        for word, f in freqs.items():
            t = vocab.get(word)
            if t is None:
                t = new.get(word)
                if t is None:
                    t = new[word] = n_old + len(new)
            t_l.append(t); d_l.append(d); f_l.append(f)
    n_out = n_old + len(new)
    t = np.asarray(t_l, dtype=np.int64)
    d = np.asarray(d_l, dtype=np.int64)
    f = np.asarray(f_l, dtype=np.int64)
    order = np.lexsort((d, t))
    t, d, f = t[order], d[order], f[order]
    count = np.bincount(t, minlength=n_out)
    term_ptr = np.zeros(n_out + 1, dtype=np.int64)
    np.cumsum(count, out=term_ptr[1:])
    postings = np.empty((len(d), 2), dtype=np.uint32)
    postings[:, 0] = d
    postings[:, 1] = f
    df_out = np.zeros(n_out, dtype=np.int64)
    df_out[:n_old] = df
    df_out += count
    n_all = int(n_docs) + len(lens)
    len_all = int(total_len) + sum(lens)
    idf, _ = okapi_idf(df_out, n_all, epsilon)
    return BM25Append(list(new), term_ptr, postings, np.asarray(lens, dtype=np.uint32), df_out, n_all,
                      len_all, idf, len_all / n_all)


def merge_csr(term_ptr: np.ndarray, postings: np.ndarray, app: BM25Append):
    """Host merge (the device does the same in lrx_bm25_append_postings): term t's old postings,
    then its appended ones.  Returns (term_ptr uint64 [V_out+1], postings uint32 [nnz + nnz_add, 2])."""
    old_ptr = np.asarray(term_ptr, dtype=np.int64)
    n_old = len(old_ptr) - 1
    add_ptr = app.term_ptr
    old_at = old_ptr[np.minimum(np.arange(app.n_terms + 1), n_old)]
    out = np.empty((len(postings) + len(app.postings), 2), dtype=np.uint32)
    shift = np.repeat(add_ptr[:n_old], np.diff(old_ptr))                   # old posting i of t -> i + add_ptr[t]
    out[np.arange(len(postings), dtype=np.int64) + shift] = postings
    ends = old_at[1:]                                                      # appended j of t -> old_end(t) + j
    out[np.repeat(ends, np.diff(add_ptr)) + np.arange(len(app.postings), dtype=np.int64)] = app.postings
    return (old_at + add_ptr).astype(np.uint64), out


@dataclass
class BM25Index:
    n_docs: int
    doc_len: np.ndarray          # uint32 [n_docs]
    term_ptr: np.ndarray         # uint64 [V+1]
    postings: np.ndarray         # uint32 [nnz, 2] = (doc id, tf), doc ascending per term
    idf: np.ndarray              # float64 [V]
    avgdl: float
    vocab: Optional[Dict[str, int]] = None
    k1: float = K1
    b: float = B
    epsilon: float = EPSILON

    @property
    def n_terms(self) -> int:
        return len(self.term_ptr) - 1

    @property
    def nnz(self) -> int:
        return int(self.term_ptr[-1])

    # ------------------------------------------------------------------ build
    @classmethod
    def from_postings(cls, n_docs, doc_len, term_ptr, post_doc, post_tf, vocab=None,
                      k1=K1, b=B, epsilon=EPSILON, total_docs=None, total_len=None, df=None):
        """From integer postings.  For a shard, pass the GLOBAL ``total_docs``,
        ``total_len`` and ``df`` so idf/avgdl are the whole-corpus statistics."""
        doc_len = np.ascontiguousarray(doc_len, dtype=np.uint32)
        term_ptr = np.ascontiguousarray(term_ptr, dtype=np.uint64)
        postings = np.empty((len(post_doc), 2), dtype=np.uint32)
        postings[:, 0] = post_doc
        postings[:, 1] = post_tf
        n_all = int(total_docs) if total_docs is not None else int(n_docs)
        len_all = int(total_len) if total_len is not None else int(doc_len.astype(np.int64).sum())
        df_all = np.asarray(df) if df is not None else np.diff(term_ptr.astype(np.int64))
        idf, _ = okapi_idf(df_all, n_all, epsilon)
        return cls(int(n_docs), doc_len, term_ptr, postings, idf, len_all / n_all, vocab, k1, b,
                   epsilon)

    @classmethod
    def from_token_lists(cls, corpus: Sequence[Sequence[str]], **kw):
        """From tokenised documents; term ids in first-appearance order."""
        vocab: Dict[str, int] = {}
        t_l, d_l, f_l, doc_len = [], [], [], []
        for d, document in enumerate(corpus):
            doc_len.append(len(document))
            freqs: Dict[str, int] = {}
            for word in document:
                freqs[word] = freqs.get(word, 0) + 1
            for word, f in freqs.items():
                t = vocab.get(word)
                if t is None:
                    t = vocab[word] = len(vocab)
                t_l.append(t); d_l.append(d); f_l.append(f)
        t = np.asarray(t_l, dtype=np.int64)
        d = np.asarray(d_l, dtype=np.int64)
        f = np.asarray(f_l, dtype=np.int64)
        order = np.lexsort((d, t))
        t, d, f = t[order], d[order], f[order]
        term_ptr = np.zeros(len(vocab) + 1, dtype=np.int64)
        np.add.at(term_ptr, t + 1, 1)
        term_ptr = np.cumsum(term_ptr)
        return cls.from_postings(len(corpus), doc_len, term_ptr, d, f, vocab=vocab, **kw)

    @classmethod
    def from_texts(cls, texts: Sequence[str], **kw):
        return cls.from_token_lists([tokenize(t) for t in texts], **kw)

    @classmethod
    def from_token_arrays(cls, doc_of_token: np.ndarray, term_of_token: np.ndarray, n_docs: int,
                          n_terms: int, **kw):
        """Vectorised build from flat (doc, term) token arrays (synthetic corpora)."""
        doc_of_token = np.asarray(doc_of_token, dtype=np.int64)
        term_of_token = np.asarray(term_of_token, dtype=np.int64)
        doc_len = np.bincount(doc_of_token, minlength=n_docs)
        key = term_of_token * n_docs + doc_of_token
        uniq, tf = np.unique(key, return_counts=True)
        t = uniq // n_docs
        d = uniq - t * n_docs
        term_ptr = np.zeros(n_terms + 1, dtype=np.int64)
        np.add.at(term_ptr, t + 1, 1)
        term_ptr = np.cumsum(term_ptr)
        return cls.from_postings(n_docs, doc_len, term_ptr, d, tf, **kw)

    # ------------------------------------------------------------------ append
    def append(self, token_lists: Sequence[Sequence[str]]) -> "BM25Index":
        """This index with the tokenised documents appended (ids n_docs, n_docs + 1, ...): equal,
        field by field and bit for bit, to ``from_token_lists(old documents + token_lists)``."""
        if self.vocab is None:
            raise ValueError("index has no string vocabulary")
        app = csr_append(self.vocab, np.diff(self.term_ptr.astype(np.int64)), self.n_docs,
                         int(self.doc_len.astype(np.int64).sum()), token_lists, self.epsilon)
        term_ptr, postings = merge_csr(self.term_ptr, self.postings, app)
        vocab = dict(self.vocab)
        vocab.update((w, len(self.vocab) + i) for i, w in enumerate(app.new_words))
        return BM25Index(app.n_docs, np.concatenate([self.doc_len, app.doc_len]), term_ptr, postings,
                         app.idf, app.avgdl, vocab, self.k1, self.b, self.epsilon)

    # ------------------------------------------------------------------ query
    def term_ids(self, tokens: Sequence[str]) -> List[int]:
        """Query tokens -> term ids; -1 = out of vocabulary (``idf.get(q) or 0``)."""
        if self.vocab is None:
            raise ValueError("index has no string vocabulary")
        return [self.vocab.get(tok, -1) for tok in tokens]

    # ------------------------------------------------------------------ shard
    def shard(self, lo: int, hi: int) -> "BM25Index":
        """Postings restricted to documents [lo, hi), doc ids made local.  idf and
        avgdl stay global, so shard scores equal whole-corpus scores bit for bit."""
        doc = self.postings[:, 0].astype(np.int64)
        keep = (doc >= lo) & (doc < hi)
        term_of = np.repeat(np.arange(self.n_terms, dtype=np.int64),
                            np.diff(self.term_ptr.astype(np.int64)))
        kept_terms = term_of[keep]
        term_ptr = np.zeros(self.n_terms + 1, dtype=np.int64)
        np.add.at(term_ptr, kept_terms + 1, 1)
        term_ptr = np.cumsum(term_ptr).astype(np.uint64)
        postings = self.postings[keep].copy()
        postings[:, 0] -= np.uint32(lo)
        return BM25Index(hi - lo, self.doc_len[lo:hi].copy(), term_ptr, postings, self.idf,
                         self.avgdl, self.vocab, self.k1, self.b, self.epsilon)
