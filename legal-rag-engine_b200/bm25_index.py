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
from typing import Callable, Dict, List, Optional, Sequence

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
class BM25Stats:
    """What planning an add or a removal reads.  A plan's ``stats`` describe the corpus after the
    change except its ``vocab``, the planner's input dict left as it was (an abandoned plan changes
    nothing, and a small plan does not pay for a copy of a large dict): ``commit_vocab`` updates it."""
    vocab: Dict[str, int]
    df: np.ndarray               # int64 [V]
    first_doc: np.ndarray        # int64 [V] each term's first document (postings[term_ptr[t]])
    n_docs: int
    total_len: int               # tokens
    idf: np.ndarray              # float64 [V]
    avgdl: float
    k1: float = K1
    b: float = B
    epsilon: float = EPSILON


@dataclass
class BM25Append:
    """Documents appended to an index: their own term-major CSR over the extended vocabulary, and
    the whole corpus's statistics after the append."""
    term_ptr: np.ndarray         # int64 [V_out+1]
    postings: np.ndarray         # uint32 [nnz_add, 2] = (doc id, tf), doc ids >= the old n_docs
    doc_len: np.ndarray          # uint32 [m]
    new_words: List[str]         # vocabulary extension, first-appearance order: ids V, V + 1, ...
    stats: BM25Stats

    @property
    def n_terms(self) -> int:
        return len(self.term_ptr) - 1

    @property
    def nnz(self) -> int:
        return int(self.term_ptr[-1])

    def commit_vocab(self):
        """Extend ``stats.vocab`` in place by the new words."""
        base = len(self.stats.vocab)
        self.stats.vocab.update((w, base + i) for i, w in enumerate(self.new_words))


def csr_append(stats: BM25Stats, token_lists: Sequence[Sequence[str]]) -> BM25Append:
    """The appended documents' CSR and the updated statistics, in O(new tokens + V): no pass over
    the existing postings.  ``stats`` is read, not changed.  A rebuild numbers terms in first
    appearance order over all documents in order; the old documents come first, so it keeps every
    old id and numbers the new terms in first-appearance order over the appended documents -- the
    order used here -- and okapi_idf's sequential mean, hence every idf bit, comes out the same."""
    vocab = stats.vocab
    new: Dict[str, int] = {}
    n_old = len(vocab)
    t_l, d_l, f_l, lens = [], [], [], []
    for d, document in enumerate(token_lists, start=stats.n_docs):
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
    df_out[:n_old] = stats.df
    df_out += count
    first = np.concatenate([stats.first_doc, d[term_ptr[n_old:-1]]])
    n_all = int(stats.n_docs) + len(lens)
    len_all = int(stats.total_len) + sum(lens)
    idf, _ = okapi_idf(df_out, n_all, stats.epsilon)
    return BM25Append(term_ptr, postings, np.asarray(lens, dtype=np.uint32), list(new),
                      BM25Stats(vocab, df_out, first, n_all, len_all, idf, len_all / n_all, stats.k1, stats.b,
                                stats.epsilon))


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


def _ranges(starts: np.ndarray, counts: np.ndarray) -> np.ndarray:
    """Concatenated ``arange(s, s + c)`` for each (s, c)."""
    starts = np.asarray(starts, dtype=np.int64)
    counts = np.asarray(counts, dtype=np.int64)
    excl = np.cumsum(counts) - counts
    return np.repeat(starts - excl, counts) + np.arange(int(counts.sum()), dtype=np.int64)


@dataclass
class BM25Remove:
    """Documents removed from an index: their per-term lists, the surviving terms in the order a
    rebuild numbers them, and the statistics after the removal."""
    removed: np.ndarray          # int64 [m] removed document ids, ascending
    rem_ptr: np.ndarray          # int64 [V+1] per old term, its removed documents ...
    rem_doc: np.ndarray          # uint32 [nnz_rem] ... ascending
    term_map: np.ndarray         # int32 [V] old term id -> new id, -1 = no surviving posting
    term_ptr: np.ndarray         # int64 [V_out+1] the compacted CSR's pointers
    stats: BM25Stats             # after the removal, new term and document ids

    @property
    def n_terms(self) -> int:
        return len(self.term_ptr) - 1

    @property
    def nnz(self) -> int:
        return int(self.term_ptr[-1])

    @property
    def nnz_rem(self) -> int:
        return int(self.rem_ptr[-1])

    def commit_vocab(self):
        """Renumber ``stats.vocab`` in place: the surviving terms, in new id order."""
        words = list(self.stats.vocab)
        live = np.flatnonzero(self.term_map >= 0)
        order = live[np.argsort(self.term_map[live])]
        self.stats.vocab.clear()
        self.stats.vocab.update(zip(map(words.__getitem__, order.tolist()), range(len(order))))


def csr_remove(stats: BM25Stats, ids: Sequence[int], doc_tokens: Callable[[int], Sequence[str]],
               first_postings: Callable[[np.ndarray, np.ndarray], np.ndarray]) -> BM25Remove:
    """The plan of removing documents ``ids`` from an index, equal to what a rebuild over the
    remaining documents computes.  ``stats`` describes the index and is read, not changed;
    ``doc_tokens(d)`` tokenises document d; ``first_postings(terms, counts)`` returns the documents of
    the first ``counts[i]`` postings of each ``terms[i]``, concatenated.

    A rebuild numbers terms in first-appearance order over the remaining documents, i.e. by the key
    (first surviving document, position of the term's first occurrence among that document's
    distinct tokens).  Old ids already follow that key, so a term whose first document survives
    keeps its place relative to the other such terms.  Only an *affected* term (its first document
    removed) moves: its new first document is among its first ``r_t + 1`` postings (r_t = its removed
    count), and the position comes from tokenising that one document.  The affected terms, sorted by
    key, are merged into the others; okapi_idf over the document frequencies in that order gives
    every idf bit of the rebuild.  Work: O(removed tokens + affected terms + tokens of their new first
    documents + V); no pass over the postings, no other document read."""
    vocab, n_docs = stats.vocab, stats.n_docs
    V = len(vocab)
    ids = np.asarray(ids, dtype=np.int64).reshape(-1)
    removed = np.unique(ids)
    if len(removed) != len(ids):
        raise ValueError("duplicate ids")
    if len(removed) and (removed[0] < 0 or removed[-1] >= n_docs):
        raise ValueError(f"ids must lie in [0, {n_docs})")
    n_out = int(n_docs) - len(removed)
    if n_out <= 0:
        raise ValueError("removing every document: the BM25 statistics of an empty corpus are undefined")
    t_l, d_l = [], []
    len_rem = 0
    for d in removed.tolist():
        tokens = doc_tokens(d)
        len_rem += len(tokens)
        for word in dict.fromkeys(tokens):
            t = vocab.get(word)
            if t is None:
                raise ValueError(f"document {d}: token {word!r} is not in the index's vocabulary")
            t_l.append(t); d_l.append(d)
    t = np.asarray(t_l, dtype=np.int64)
    d = np.asarray(d_l, dtype=np.int64)
    order = np.lexsort((d, t))
    t, d = t[order], d[order]
    r = np.bincount(t, minlength=V).astype(np.int64)
    rem_ptr = np.zeros(V + 1, dtype=np.int64)
    np.cumsum(r, out=rem_ptr[1:])
    df_after = stats.df - r
    if (df_after < 0).any():
        raise ValueError("the removed documents' tokens do not match the index's postings")
    alive = df_after > 0
    first = stats.first_doc
    is_removed = lambda a: removed[np.minimum(np.searchsorted(removed, a), len(removed) - 1)] == a
    # affected: alive terms whose first document is removed (only terms with r_t > 0 can be)
    cand = np.nonzero(r)[0]
    aff = cand[alive[cand] & is_removed(first[cand])] if len(removed) else cand[:0]
    first_after = first.copy()
    if len(aff):
        counts = r[aff] + 1
        docs = np.asarray(first_postings(aff, counts), dtype=np.int64)
        idx = np.where(is_removed(docs), len(docs), np.arange(len(docs)))
        pick = np.minimum.reduceat(idx, np.cumsum(counts) - counts)
        if (pick >= len(docs)).any():
            raise ValueError("the removed documents' tokens do not match the index's postings")
        first_after[aff] = docs[pick]
    # within-document positions, from the new first documents of the affected terms
    pos = np.zeros(V, dtype=np.int64)
    for f in np.unique(first_after[aff]).tolist():
        for p, word in enumerate(dict.fromkeys(doc_tokens(f))):
            t = vocab.get(word)
            if t is None:
                raise ValueError(f"document {f}: token {word!r} is not in the index's vocabulary")
            if first_after[t] == f:
                pos[t] = p
    key = (first_after << 17) + pos                     # a document has < 2^16 distinct tokens
    is_aff = np.zeros(V, dtype=bool)
    is_aff[aff] = True
    keep = np.nonzero(alive & ~is_aff)[0]               # already in key order
    a_sorted = aff[np.argsort(key[aff], kind="stable")]
    new_order = np.insert(keep, np.searchsorted(key[keep], key[a_sorted]), a_sorted)
    term_map = np.full(V, -1, dtype=np.int32)
    term_map[new_order] = np.arange(len(new_order), dtype=np.int32)
    df_out = df_after[new_order]
    term_ptr = np.zeros(len(new_order) + 1, dtype=np.int64)
    np.cumsum(df_out, out=term_ptr[1:])
    f_new = first_after[new_order]
    len_out = int(stats.total_len) - len_rem
    idf, _ = okapi_idf(df_out, n_out, stats.epsilon)
    return BM25Remove(removed, rem_ptr, d.astype(np.uint32), term_map, term_ptr,
                      BM25Stats(vocab, df_out, f_new - np.searchsorted(removed, f_new), n_out, len_out, idf,
                                len_out / n_out, stats.k1, stats.b, stats.epsilon))


def remove_csr(term_ptr: np.ndarray, postings: np.ndarray, rem: BM25Remove):
    """Host compaction (the device does the same in lrx_bm25_remove_postings), linear in the postings:
    the postings of the removed documents dropped, the others renumbered and moved to their term's
    new id.  A document map (new id, -1 = removed) renumbers every posting, and kept posting i of term
    t goes to ``rem.term_ptr[term_map[t]] + (i - term_ptr[t]) - k`` with k the removed postings of t
    before it (a running count).  Returns (term_ptr uint64 [V_out+1], postings uint32 [nnz_out, 2])."""
    old_ptr = np.asarray(term_ptr, dtype=np.int64)
    out_ptr = np.asarray(rem.term_ptr, dtype=np.int64)
    n_docs = rem.stats.n_docs + len(rem.removed)
    mark = np.zeros(n_docs, dtype=bool)
    mark[rem.removed] = True
    doc_map = np.arange(n_docs, dtype=np.int64) - np.cumsum(mark)
    doc_map[mark] = -1
    new_doc = doc_map[postings[:, 0]]
    gone = new_doc < 0
    k = np.cumsum(gone)                                  # removed postings up to posting i ...
    before = np.concatenate([[0], k])[old_ptr[:-1]]      # ... and before each term's first posting
    dst = np.arange(len(postings), dtype=np.int64) - k
    dst += np.repeat(out_ptr[np.maximum(rem.term_map, 0)] - old_ptr[:-1] + before, np.diff(old_ptr))
    keep = ~gone
    out = np.empty((int(out_ptr[-1]), 2), dtype=np.uint32)
    assert int(keep.sum()) == len(out), "the removal plan does not describe these postings"
    out[dst[keep], 0] = new_doc[keep]
    out[dst[keep], 1] = postings[keep, 1]
    return out_ptr.astype(np.uint64), out


@dataclass
class BM25Replace:
    """Documents whose text is replaced in place (document ids unchanged): per old term its postings
    of replaced documents (dropped), the terms in the order a rebuild numbers them, per new term its
    inserted entries, and the statistics after the edit."""
    replaced: np.ndarray         # int64 [m] replaced document ids, ascending
    doc_len: np.ndarray          # uint32 [m] their new lengths
    rem_ptr: np.ndarray          # int64 [V+1] per old term, its postings of replaced documents ...
    rem_doc: np.ndarray          # uint32 [nnz_rem] ... ascending (dropped)
    term_map: np.ndarray         # int32 [V] old term id -> new id, -1 = vanished
    new_words: List[str]         # words the old index lacks, in first-appearance order over the new texts ...
    new_map: np.ndarray          # int32 [len(new_words)] ... and their new ids
    ins_ptr: np.ndarray          # int64 [V_out+1] per new term, its inserted entries ...
    ins_postings: np.ndarray     # uint32 [nnz_ins, 2] = (doc, tf), doc ascending per term, every doc replaced
    term_ptr: np.ndarray         # int64 [V_out+1] the new CSR's pointers
    stats: BM25Stats             # after the edit, new term ids

    @property
    def n_terms(self) -> int:
        return len(self.term_ptr) - 1

    @property
    def nnz(self) -> int:
        return int(self.term_ptr[-1])

    @property
    def nnz_rem(self) -> int:
        return int(self.rem_ptr[-1])

    @property
    def nnz_ins(self) -> int:
        return int(self.ins_ptr[-1])

    def commit_vocab(self):
        """Renumber ``stats.vocab`` in place: the old words that remain and the new words, in new id order."""
        words = list(self.stats.vocab) + list(self.new_words)
        ext = np.concatenate([self.term_map, self.new_map]).astype(np.int64)
        live = np.flatnonzero(ext >= 0)
        order = live[np.argsort(ext[live])]
        self.stats.vocab.clear()
        self.stats.vocab.update(zip(map(words.__getitem__, order.tolist()), range(len(order))))


def csr_replace(stats: BM25Stats, ids: Sequence[int], new_token_lists: Sequence[Sequence[str]],
                doc_tokens: Callable[[int], Sequence[str]],
                first_postings: Callable[[np.ndarray, np.ndarray], np.ndarray]) -> BM25Replace:
    """The plan of replacing the text of documents ``ids`` by ``new_token_lists`` (document ids do not
    change), equal to what a rebuild over the edited documents computes.  ``stats`` is read, not
    changed; ``doc_tokens(d)`` tokenises the current text of document d; ``first_postings(terms,
    counts)`` returns the documents of the first ``counts[i]`` postings of each ``terms[i]``.

    A rebuild numbers terms by the key (first document, position of the term's first occurrence
    among that document's distinct tokens).  A term in neither the old nor the new text of a replaced
    document keeps its postings, first document and key.  So does a touched term whose first document
    is unchanged and not replaced.  Every other term that survives is re-keyed: its new first document
    is the smaller of its first posting outside the replaced set (among its first ``r_t + 1`` postings
    when its old first document is replaced) and the first replaced document whose new text holds it;
    the position comes from tokenising that document (its new text if it is replaced).  New words are
    keyed the same way; words left without postings vanish.  The re-keyed terms, sorted by key, are
    merged into the kept ones, and okapi_idf in that order gives every idf bit of the rebuild.  Work:
    O(old and new tokens of the replaced documents + tokens of the new first documents + V)."""
    vocab, n_docs = stats.vocab, int(stats.n_docs)
    V = len(vocab)
    ids = np.asarray(ids, dtype=np.int64).reshape(-1)
    if len(new_token_lists) != len(ids):
        raise ValueError(f"{len(ids)} ids but {len(new_token_lists)} new documents")
    order = np.argsort(ids, kind="stable")
    replaced = ids[order]
    if len(replaced) and (np.diff(replaced) == 0).any():
        raise ValueError("duplicate ids")
    if len(replaced) and (replaced[0] < 0 or replaced[-1] >= n_docs):
        raise ValueError(f"ids must lie in [0, {n_docs})")
    new_lists = [new_token_lists[i] for i in order.tolist()]
    # the dropped entries: every (term, replaced document) of the old texts
    t_l, d_l = [], []
    len_old = 0
    for d in replaced.tolist():
        tokens = doc_tokens(d)
        len_old += len(tokens)
        for word in dict.fromkeys(tokens):
            t = vocab.get(word)
            if t is None:
                raise ValueError(f"document {d}: token {word!r} is not in the index's vocabulary")
            t_l.append(t); d_l.append(d)
    t = np.asarray(t_l, dtype=np.int64)
    d = np.asarray(d_l, dtype=np.int64)
    o = np.lexsort((d, t))
    t, d = t[o], d[o]
    r = np.bincount(t, minlength=V).astype(np.int64)
    rem_ptr = np.zeros(V + 1, dtype=np.int64)
    np.cumsum(r, out=rem_ptr[1:])
    df_kept = stats.df - r
    if (df_kept < 0).any():
        raise ValueError("the replaced documents' tokens do not match the index's postings")
    # the inserted entries: every (term, replaced document, tf) of the new texts; new words get ids
    # V, V + 1, ... in first-appearance order
    new: Dict[str, int] = {}
    it_l, id_l, if_l, lens = [], [], [], []
    for dd, document in zip(replaced.tolist(), new_lists):
        lens.append(len(document))
        freqs: Dict[str, int] = {}
        for word in document:
            freqs[word] = freqs.get(word, 0) + 1
        for word, f in freqs.items():
            tt = vocab.get(word)
            if tt is None:
                tt = new.get(word)
                if tt is None:
                    tt = new[word] = V + len(new)
            it_l.append(tt); id_l.append(dd); if_l.append(f)
    W = V + len(new)
    it = np.asarray(it_l, dtype=np.int64)
    idd = np.asarray(id_l, dtype=np.int64)
    iff = np.asarray(if_l, dtype=np.int64)
    total = int(stats.total_len) - len_old + sum(lens)
    if total <= 0:
        raise ValueError("the edit leaves the corpus without BM25 tokens: avgdl would be 0")
    ins_cnt = np.bincount(it, minlength=W).astype(np.int64)
    df_ext = np.concatenate([df_kept, np.zeros(len(new), dtype=np.int64)]) + ins_cnt
    alive = df_ext > 0
    none = n_docs                                        # "no such document": larger than every id
    is_rep = lambda a: replaced[np.minimum(np.searchsorted(replaced, a), len(replaced) - 1)] == a
    # first replaced document whose new text holds each term (entries are in document order)
    first_ins = np.full(W, none, dtype=np.int64)
    np.minimum.at(first_ins, it, idd)
    # first posting outside the replaced set
    first_old = np.concatenate([stats.first_doc, np.full(len(new), none, dtype=np.int64)])
    first_out = np.where(np.concatenate([df_kept, np.zeros(len(new), dtype=np.int64)]) > 0, first_old, none)
    cand = np.nonzero(r)[0]
    aff = cand[(df_kept[cand] > 0) & is_rep(stats.first_doc[cand])] if len(replaced) else cand[:0]
    if len(aff):
        counts = r[aff] + 1
        docs = np.asarray(first_postings(aff, counts), dtype=np.int64)
        idx = np.where(is_rep(docs), len(docs), np.arange(len(docs)))
        pick = np.minimum.reduceat(idx, np.cumsum(counts) - counts)
        if (pick >= len(docs)).any():
            raise ValueError("the replaced documents' tokens do not match the index's postings")
        first_out[aff] = docs[pick]
    first_after = np.minimum(first_out, first_ins)
    rekey = alive & ((first_after != first_old) | (is_rep(first_after) if len(replaced) else False))
    rk = np.nonzero(rekey)[0]
    # within-document positions of every term whose first document is one of the re-keyed terms'
    pos = np.zeros(W, dtype=np.int64)
    slot = {dd: i for i, dd in enumerate(replaced.tolist())}
    for f in np.unique(first_after[rk]).tolist():
        tokens = new_lists[slot[f]] if f in slot else doc_tokens(f)
        for p, word in enumerate(dict.fromkeys(tokens)):
            tt = vocab.get(word)
            if tt is None:
                tt = new.get(word)
                if tt is None:
                    raise ValueError(f"document {f}: token {word!r} is not in the index's vocabulary")
            if first_after[tt] == f:
                pos[tt] = p
    key = (first_after << 17) + pos                      # a document has < 2^16 distinct tokens
    keep = np.nonzero(alive & ~rekey)[0]                 # old terms with their old keys: in key order
    a_sorted = rk[np.argsort(key[rk], kind="stable")]
    new_order = np.insert(keep, np.searchsorted(key[keep], key[a_sorted]), a_sorted)
    ext_map = np.full(W, -1, dtype=np.int32)
    ext_map[new_order] = np.arange(len(new_order), dtype=np.int32)
    df_out = df_ext[new_order]
    term_ptr = np.zeros(len(new_order) + 1, dtype=np.int64)
    np.cumsum(df_out, out=term_ptr[1:])
    nt = ext_map[it].astype(np.int64)
    o = np.lexsort((idd, nt))
    ins_postings = np.empty((len(o), 2), dtype=np.uint32)
    ins_postings[:, 0] = idd[o]
    ins_postings[:, 1] = iff[o]
    ins_ptr = np.zeros(len(new_order) + 1, dtype=np.int64)
    np.cumsum(np.bincount(nt, minlength=len(new_order)), out=ins_ptr[1:])
    idf, _ = okapi_idf(df_out, n_docs, stats.epsilon)
    return BM25Replace(replaced, np.asarray(lens, dtype=np.uint32), rem_ptr, d.astype(np.uint32), ext_map[:V],
                       list(new), ext_map[V:], ins_ptr, ins_postings, term_ptr,
                       BM25Stats(vocab, df_out, first_after[new_order], n_docs, total, idf, total / n_docs,
                                 stats.k1, stats.b, stats.epsilon))


def replace_csr(term_ptr: np.ndarray, postings: np.ndarray, rep: BM25Replace):
    """Host compaction (the device does the same in lrx_bm25_replace_postings), linear in the postings
    but for one binary search per kept posting into the inserted entries: the postings of the replaced
    documents dropped, the others moved verbatim to their term's new id, each new list merged by
    document with its inserted entries.  Returns (term_ptr uint64 [V_out+1], postings uint32 [nnz_out, 2])."""
    old_ptr = np.asarray(term_ptr, dtype=np.int64)
    out_ptr = np.asarray(rep.term_ptr, dtype=np.int64)
    V, V_out = len(old_ptr) - 1, rep.n_terms
    mark = np.zeros(rep.stats.n_docs, dtype=bool)
    mark[rep.replaced] = True
    term_of = np.repeat(np.arange(V, dtype=np.int64), np.diff(old_ptr))
    keep = ~mark[postings[:, 0]]
    kt = term_of[keep]
    m = rep.term_map[kt].astype(np.int64)
    assert (m >= 0).all(), "the replacement plan does not describe these postings"
    kcount = np.bincount(kt, minlength=V)
    rank = np.arange(len(kt), dtype=np.int64) - np.repeat(np.cumsum(kcount) - kcount, kcount)
    kept = postings[keep]
    ins_ptr = np.asarray(rep.ins_ptr, dtype=np.int64)
    ins_term = np.repeat(np.arange(V_out, dtype=np.int64), np.diff(ins_ptr))
    key_i = (ins_term << 32) | rep.ins_postings[:, 0].astype(np.int64)
    c = np.searchsorted(key_i, (m << 32) | kept[:, 0].astype(np.int64)) - ins_ptr[m]
    dst = out_ptr[m] + rank + c
    out = np.empty((int(out_ptr[-1]), 2), dtype=np.uint32)
    assert len(kept) + rep.nnz_ins == len(out), "the replacement plan does not describe these postings"
    taken = np.zeros(len(out), dtype=bool)
    taken[dst] = True
    assert int(taken.sum()) == len(kept), "the replacement plan does not describe these postings"
    out[dst] = kept
    out[~taken] = rep.ins_postings                       # free slots ascend with (new term, doc)
    return out_ptr.astype(np.uint64), out


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

    def stats(self) -> BM25Stats:
        """The statistics planning reads (csr_append, csr_remove), with a copy of the vocabulary."""
        if self.vocab is None:
            raise ValueError("index has no string vocabulary")
        tp = self.term_ptr.astype(np.int64)
        first = self.postings[np.minimum(tp[:-1], max(self.nnz - 1, 0)), 0].astype(np.int64)
        return BM25Stats(dict(self.vocab), np.diff(tp), first, self.n_docs, int(self.doc_len.astype(np.int64).sum()),
                         self.idf, self.avgdl, self.k1, self.b, self.epsilon)

    # ------------------------------------------------------------------ build
    @classmethod
    def from_stats(cls, stats: BM25Stats, term_ptr, postings, doc_len) -> "BM25Index":
        """The index with these statistics over these postings, with a copy of the vocabulary."""
        return cls(stats.n_docs, doc_len, term_ptr, postings, stats.idf, stats.avgdl, dict(stats.vocab), stats.k1,
                   stats.b, stats.epsilon)

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
        app = csr_append(self.stats(), token_lists)
        app.commit_vocab()
        term_ptr, postings = merge_csr(self.term_ptr, self.postings, app)
        return BM25Index.from_stats(app.stats, term_ptr, postings, np.concatenate([self.doc_len, app.doc_len]))

    # ------------------------------------------------------------------ remove
    def remove(self, ids: Sequence[int], doc_tokens: Callable[[int], Sequence[str]]) -> "BM25Index":
        """This index without documents ``ids`` (the others renumbered by rank): equal, field by field
        and bit for bit, to ``from_token_lists(remaining documents)``, vocabulary order included.
        ``doc_tokens(d)`` tokenises document d; only the removed documents and the new first
        documents of the terms that lose theirs are read (``csr_remove``)."""
        tp = self.term_ptr.astype(np.int64)
        gather = lambda terms, counts: self.postings[_ranges(tp[terms], counts), 0]
        rem = csr_remove(self.stats(), ids, doc_tokens, gather)
        rem.commit_vocab()
        term_ptr, postings = remove_csr(self.term_ptr, self.postings, rem)
        return BM25Index.from_stats(rem.stats, term_ptr, postings, np.delete(self.doc_len, rem.removed))

    # ------------------------------------------------------------------ replace
    def replace(self, ids: Sequence[int], new_token_lists: Sequence[Sequence[str]],
                doc_tokens: Callable[[int], Sequence[str]]) -> "BM25Index":
        """This index with the text of documents ``ids`` replaced by ``new_token_lists`` (ids unchanged):
        equal, field by field and bit for bit, to ``from_token_lists(edited documents)``, vocabulary
        order included.  ``doc_tokens(d)`` tokenises the current document d; only the replaced
        documents and the new first documents of re-keyed terms are read (``csr_replace``)."""
        tp = self.term_ptr.astype(np.int64)
        gather = lambda terms, counts: self.postings[_ranges(tp[terms], counts), 0]
        rep = csr_replace(self.stats(), ids, new_token_lists, doc_tokens, gather)
        rep.commit_vocab()
        term_ptr, postings = replace_csr(self.term_ptr, self.postings, rep)
        doc_len = self.doc_len.copy()
        doc_len[rep.replaced] = rep.doc_len
        return BM25Index.from_stats(rep.stats, term_ptr, postings, doc_len)

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
