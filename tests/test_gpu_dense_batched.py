"""K2b (tensor-core batched top-K, csrc/dense_batched.cu) on corpora shaped like chunk stores.

`create_vector_store.py` writes chunks in document order, so neighbouring rows of a real store are
similar: a query near one chunk of an act has dozens to hundreds of candidates in a few consecutive
256-row tiles.  Every K2b test before this file used isotropic rows with one planted hit.  The
corpora here are seeded and each builder checks, through `k2b_selection` (a CPU restatement of
K2b's candidate bookkeeping), that its corpus reaches the condition it is built for: candidates
crowded into one pass-2 region, a threshold from fewer valid chunks than the depth, ties and
near-ties at the K-th score.  Results must equal the float64 oracle bit for bit with no flag and
no retry, except where more than 1024 rows lie in the band of the K-th score."""
import numpy as np
import pytest
import torch

from oracle import bm25 as obm25
from oracle import flat_ip
from oracle.search import OracleIndex

from legal_rag_engine_b200 import synth
from legal_rag_engine_b200.bm25_index import BM25Index, tokenize

pytestmark = pytest.mark.gpu

SMS = 148                  # B200: the CTA grid, and so the pass-2 region layout
TILE, HALF, CHUNK = 256, 128, 32
CAP = 1024                 # candidates re-scored per query (kDbCap)
SLACK = 2e-5               # 2 * kTcEps


# ------------------------------------------------------------------ CPU restatement
def default_stride(n, K):
    n_tiles = -(-n // TILE)
    return max(1, min(8, n_tiles * 8 // (16 * K)))


def k2b_selection(x, q, K, B, stride=0, sms=SMS):
    """K2b's candidate selection for queries `q` of a batch of B over rows `x`, with fp32 dot products
    standing in for the tensor-core accumulators.  Pass 1: the maximum of every 32-row chunk of tiles
    0, s, 2s, ...; T = K-th largest sampled maximum - slack (chunks past the corpus end count, with
    maximum -inf).  Pass 2: rows with score >= T, region = (tile % CTAs per query tile) * 2 + half.
    Returns per-query candidate counts and largest region fill, and the layout figures."""
    n = len(x)
    n_tiles = -(-n // TILE)
    stride = stride or default_stride(n, K)
    n_samp = -(-n_tiles // stride) * 8
    if n_samp > 16384:
        stride = -(-n_tiles * 8 // 16384)
        n_samp = -(-n_tiles // stride) * 8
    n_mt = -(-B // 128)
    cs = 2 if n_mt >= 2 else 1
    n_mt = -(-n_mt // cs) * cs
    grid = max(n_mt, sms // n_mt * n_mt)
    n_groups = grid // n_mt
    n_regions = 2 * n_groups
    cap = 16
    while cap * n_regions < 2048:
        cap *= 2
    valid = -(-n_tiles // stride) * 8
    if (n_tiles - 1) % stride == 0:
        valid -= 8 - -(-(n - (n_tiles - 1) * TILE) // CHUNK)
    s = q.astype(np.float32) @ x.astype(np.float32).T
    pad = np.full((len(q), n_tiles * TILE), -np.inf, np.float32)
    pad[:, :n] = s
    samp = pad.reshape(len(q), n_tiles, 8, CHUNK).max(-1)[:, ::stride].reshape(len(q), -1)
    thr = -np.sort(-samp, axis=1)[:, K - 1] - SLACK if K <= n_samp else np.full(len(q), -np.inf)
    cand, fill = [], []
    for b in range(len(q)):
        rows = np.nonzero(s[b] >= thr[b])[0]
        region = (rows // TILE % n_groups) * 2 + rows % TILE // HALF
        cand.append(len(rows))
        fill.append(int(np.bincount(region, minlength=n_regions).max()))
    return dict(cand=np.array(cand), fill=np.array(fill), cap=cap, valid=valid, n_samp=n_samp,
                stride=stride)


def region_overflow(sel):
    """Queries whose candidates (at most CAP of them) overfill a pass-2 region."""
    return (sel["fill"] > sel["cap"]) & (sel["cand"] <= CAP)


# ------------------------------------------------------------------ corpora
def _cluster(rng, centre, m, noise):
    v = centre[None, :] + rng.standard_normal((m, len(centre)), dtype=np.float32) * (noise / np.sqrt(len(centre)))
    return (v / np.linalg.norm(v, axis=1, keepdims=True)).astype(np.float16)


def _unit(rng, m):
    v = rng.standard_normal((m, 384), dtype=np.float32)
    return v / np.linalg.norm(v, axis=1, keepdims=True)


N_BLOCKS = 90000
# (first row, length): inside one 128-row half-tile, across a half-tile boundary, across a tile boundary
BLOCKS = [(20 * TILE + 8, 17), (30 * TILE + HALF - 20, 40), (50 * TILE - 150, 300)]


def blocks_corpus():
    """90 000 isotropic rows with three runs of similar rows (an act's consecutive chunks)."""
    rng = np.random.default_rng(11)
    x = synth.host_vectors(N_BLOCKS, seed=12, dup_frac=0.001)
    for (a, m), c in zip(BLOCKS, _unit(rng, len(BLOCKS))):
        x[a:a + m] = _cluster(rng, c, m, 0.6)
    return x


def n_planted(B):
    return min(9, max(1, B // 3))


def block_queries(x, B, seed):
    """B queries: the first n_planted(B) planted on a row of each block in turn, the rest isotropic."""
    q = synth.host_queries(B, seed=seed)
    rows = [a + (7 * j) % m for j, (a, m) in enumerate(BLOCKS * 3)][:n_planted(B)]
    q[:len(rows)] = synth.host_planted_queries(x, rows, seed=seed + 1, noise=0.3)
    return q


def legal_layout_corpus(legal_chunks, noise=1.0):
    """The reference corpus's order: every chunk's vector = its (law, chapter) centre + noise."""
    keys = [(c["metadata"].get("law"), c["metadata"].get("chapter")) for c in legal_chunks]
    group = {k: i for i, k in enumerate(dict.fromkeys(keys))}
    lab = np.array([group[k] for k in keys])
    rng = np.random.default_rng(21)
    cent = _unit(rng, len(group))
    v = cent[lab] + rng.standard_normal((len(keys), 384), dtype=np.float32) * (noise / np.sqrt(384))
    return (v / np.linalg.norm(v, axis=1, keepdims=True)).astype(np.float16)


def legal_queries(x, B, seed):
    rng = np.random.default_rng(seed)
    q = synth.host_queries(B, seed=seed)
    m = max(1, (3 * B) // 4)
    q[:m] = synth.host_planted_queries(x, rng.integers(0, len(x), m), seed=seed + 1, noise=0.8)
    return q


N_DUP = 20000
DUP_RUNS = [(40 * TILE + HALF - 40, 80), (60 * TILE - 45, 90)]   # copies across a half and a tile boundary


def duplicates_corpus():
    x = synth.host_vectors(N_DUP, seed=31, dup_frac=0.0)
    for j, (a, m) in enumerate(DUP_RUNS):
        x[a:a + m] = x[1000 + j]
    return x


def near_tie_corpus():
    """80 consecutive rows across a tile boundary, each a copy of one base row with one coordinate
    moved by one fp16 ulp: their exact scores lie within the 2e-5 slack of one another, several
    exactly equal."""
    x = synth.host_vectors(N_DUP, seed=41, dup_frac=0.0)
    rng = np.random.default_rng(42)
    base = x[500].copy()
    a, m = 70 * TILE - 40, 80
    coords = rng.choice(np.nonzero(np.abs(base) < 2 ** -5)[0], m)   # one ulp <= 2^-15
    coords[::7] = coords[0]                                  # some rows identical: exact ties
    up = rng.random(m) < 0.5
    for i in range(m):
        r = base.copy()
        r[coords[i]] = np.nextafter(r[coords[i]], np.float16(np.inf if up[i] else -np.inf))
        x[a + i] = r
    return x, a, m


SMALL_N = [255, 256, 257, 600, 697, 1100, 2000, 2620, 8193]


# ------------------------------------------------------------------ helpers
@pytest.fixture(scope="module")
def dev():
    from legal_rag_engine_b200.device_index import DeviceIndex
    d = DeviceIndex(0)
    assert torch.cuda.get_device_properties(0).multi_processor_count == SMS
    yield d
    d.close()


def _cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _check_batched(dev, x, q, K, id_base, stride=0, sample=None):
    """K2b against the oracle: every query, or `sample` of them plus all against dense_topk in
    groups of 8 (K2a; widened where its own guard trips, as the search chain does)."""
    E, D, I, flags = dev.dense_topk_batched(_cuda(q), K, stride=stride)
    assert int(flags.sum().item()) == 0, np.nonzero(flags.cpu().numpy())[0]
    E, D, I = E.cpu().numpy(), D.cpu().numpy(), I.cpu().numpy()
    pick = np.arange(len(q)) if sample is None else np.asarray(sample)
    Eo, Do, Io = flat_ip.topk_from_scores(flat_ip.exact_scores(x, q[pick]), K, id_base=id_base)
    np.testing.assert_array_equal(I[pick], Io)
    np.testing.assert_array_equal(E[pick], Eo)
    np.testing.assert_array_equal(D[pick], Do)
    if sample is not None:
        for b0 in range(0, len(q), 8):
            E2, _, I2, f2 = dev.dense_topk(_cuda(q[b0:b0 + 8]), K)
            if int(f2.sum().item()) != 0:
                E2, _, I2, f2 = dev.dense_topk(_cuda(q[b0:b0 + 8]), K, width=512)
            assert int(f2.sum().item()) == 0
            np.testing.assert_array_equal(I[b0:b0 + 8], I2.cpu().numpy())
            np.testing.assert_array_equal(E[b0:b0 + 8], E2.cpu().numpy())
    return E, I


# ------------------------------------------------------------------ 1. K2b at the automatic stride
@pytest.mark.parametrize("B,K,id_base", [(9, 20, 0), (64, 1, 5), (64, 33, 0), (128, 10, 1000), (129, 32, 0),
                                         (256, 64, 7), (257, 20, 0), (1024, 200, 100)])
def test_batched_contiguous_similar_blocks(dev, B, K, id_base):
    x = blocks_corpus()
    q = block_queries(x, B, seed=B + K)
    planted = np.arange(n_planted(B))
    sel = k2b_selection(x, q[planted], K, B)
    # at K = 1 the threshold sits at the top block row: a region fills only at larger depths
    assert K == 1 or region_overflow(sel).any(), sel
    assert (sel["cand"] <= CAP).all()
    sample = None if B <= 129 else np.r_[planted[:6], B // 2, B - 1]
    dev.set_corpus(_cuda(x), id_base=id_base)
    _check_batched(dev, x, q, K, id_base, sample=sample)


@pytest.mark.parametrize("B,K", [(9, 10), (16, 20), (64, 32), (64, 64), (130, 33)])
def test_batched_reference_corpus_layout(dev, legal_chunks, B, K):
    x = legal_layout_corpus(legal_chunks)
    q = legal_queries(x, B, seed=7 * B + K)
    sel = k2b_selection(x, q, K, B)
    if sel["valid"] >= 2 * K:
        assert region_overflow(sel).sum() >= B // 4, sel
    dev.set_corpus(_cuda(x), id_base=3)
    _check_batched(dev, x, q, K, 3)


@pytest.mark.parametrize("B,K", [(9, 20), (64, 32), (257, 10)])
def test_batched_exact_duplicates_order_by_id(dev, B, K):
    x = duplicates_corpus()
    q = synth.host_queries(B, seed=B)
    q[:2] = synth.host_planted_queries(x, [1000, 1001], seed=3, noise=0.2)
    sel = k2b_selection(x, q[:2], K, B)
    assert region_overflow(sel).all(), sel
    dev.set_corpus(_cuda(x), id_base=0)
    E, I = _check_batched(dev, x, q, K, 0)
    for j, (a, m) in enumerate(DUP_RUNS):                   # the source row, then its copies by id
        assert I[j, :K].tolist() == ([1000 + j] + list(range(a, a + m)))[:K]


@pytest.mark.parametrize("B,K", [(9, 32), (33, 64), (129, 20)])
def test_batched_near_ties_at_the_kth_score(dev, B, K):
    x, a, m = near_tie_corpus()
    q = synth.host_queries(B, seed=50 + B)
    q[0] = synth.host_planted_queries(x, [500], seed=5, noise=0.2)[0]
    s = flat_ip.exact_scores(x, q[:1])[0]
    ties = s[a:a + m]
    assert ties.max() - ties.min() < SLACK and len(np.unique(ties)) < m
    kth = np.sort(s)[::-1][K - 1]
    assert ties.min() <= kth <= ties.max()                   # the K-th score falls among them
    assert region_overflow(k2b_selection(x, q[:1], K, B)).all()
    dev.set_corpus(_cuda(x), id_base=11)
    _check_batched(dev, x, q, K, 11)


@pytest.mark.parametrize("n", SMALL_N)
def test_batched_small_corpora_around_the_padding(dev, n):
    """A few tiles: the threshold comes from few chunks, some of them past the corpus end."""
    x = synth.host_vectors(n, seed=n, dup_frac=0.01)
    B = 64
    q = synth.host_queries(B, seed=n + 1)
    q[:8] = synth.host_planted_queries(x, np.arange(8) * (n // 8), seed=2)
    dev.set_corpus(_cuda(x), id_base=n)
    for K in (1, 10, 20, 33, 40, 64, 200, 256):
        sel = k2b_selection(x, q, K, B)
        if (n, K) in ((600, 20), (1100, 40), (2000, 64)):
            assert sel["valid"] < K <= sel["n_samp"]         # T = -FLT_MAX: every row a candidate
        if (n, K) in ((697, 20), (8193, 256)):
            assert K <= sel["valid"] < 2 * K and (sel["fill"] > sel["cap"]).any(), sel
        _check_batched(dev, x, q, K, n)


# ------------------------------------------------------------------ 2. the flag contract
def test_batched_flags_more_than_1024_candidates(dev):
    """1 100 identical rows score the same: every one is within the band of the K-th score, more than
    the 1024 a query's list holds -> flagged (also at stride 1).  The other queries of the batch are
    exact and unflagged."""
    x = synth.host_vectors(50000, seed=61, dup_frac=0.0)
    x[20000:21100] = x[7]
    B, K = 16, 20
    q = synth.host_queries(B, seed=62)
    q[3] = synth.host_planted_queries(x, [7], seed=63, noise=0.2)[0]
    assert k2b_selection(x, q[3:4], K, B)["cand"][0] > CAP
    dev.set_corpus(_cuda(x), id_base=0)
    others = np.r_[0:3, 4:B]
    Eo, _, Io = flat_ip.topk_from_scores(flat_ip.exact_scores(x, q[others]), K)
    for stride in (0, 1):
        E, D, I, flags = dev.dense_topk_batched(_cuda(q), K, stride=stride)
        f = flags.cpu().numpy()
        assert f[3] == 1 and f[others].sum() == 0, f
        np.testing.assert_array_equal(I.cpu().numpy()[others], Io)
        np.testing.assert_array_equal(E.cpu().numpy()[others], Eo)


# ------------------------------------------------------------------ 3. lrx_dense_topk_ex routes B >= 9 to K2b
@pytest.mark.parametrize("B", [9, 33, 64])
def test_dense_topk_batches_on_clustered_rows(dev, B):
    x = blocks_corpus()
    q = block_queries(x, B, seed=300 + B)
    K = 20
    assert region_overflow(k2b_selection(x, q[:n_planted(B)], K, B)).any()
    dev.set_corpus(_cuda(x), id_base=9)
    Eo, Do, Io = flat_ip.topk_from_scores(flat_ip.exact_scores(x, q), K, id_base=9)
    for width in (0, 128):                                  # default (64), and a widened retry's
        E, D, I, flags = dev.dense_topk(_cuda(q), K, width=width)
        assert int(flags.sum().item()) == 0
        np.testing.assert_array_equal(I.cpu().numpy(), Io)
        np.testing.assert_array_equal(E.cpu().numpy(), Eo)
        np.testing.assert_array_equal(D.cpu().numpy(), Do)


# ------------------------------------------------------------------ 4. the search chain
def _assert_results(got, want):
    ids, score, sem, kw = got
    for b, res in enumerate(want):
        assert ids[b, :len(res)].tolist() == [r[0] for r in res]
        assert (ids[b, len(res):] == -1).all()
        for j, r in enumerate(res):
            assert score[b, j] == r[1] and sem[b, j] == r[2] and kw[b, j] == r[3]


def _check_chain(dev, x, csr, q, lists, k, fusion):
    from legal_rag_engine_b200._lib import LrxError
    weights = [0.5 + 0.1 * (b % 2) for b in range(len(q))]
    want = OracleIndex(x, csr).search_batch_vec(q, lists, k, weights, fusion)
    for _ in range(3):                                      # direct, captured, replayed
        try:
            got = dev.search_batch_host(q, lists, k, weights, fusion)
        except LrxError as e:
            pytest.fail(f"search_batch_host raised {e}")
        _assert_results(got, want)


@pytest.mark.parametrize("fusion", ["linear", "rrf"])
@pytest.mark.parametrize("B,k", [(9, 5), (16, 10), (64, 5), (64, 100)])
def test_search_chain_contiguous_similar_blocks(dev, B, k, fusion):
    x = blocks_corpus()
    idx = synth.host_bm25(N_BLOCKS, seed=71, vocab=3000)
    csr = obm25.BM25OkapiCSR.from_postings(idx.n_docs, idx.doc_len, idx.term_ptr.astype(np.int64),
                                           idx.postings[:, 0], idx.postings[:, 1])
    q = block_queries(x, B, seed=400 + B)
    assert region_overflow(k2b_selection(x, q[:n_planted(B)], 2 * k, B, stride=1)).any()
    terms, ptr = synth.host_query_terms(B, 8, seed=401 + B, vocab=3000)
    lists = [terms[ptr[b]:ptr[b + 1]].tolist() for b in range(B)]
    dev.set_corpus(_cuda(x), 0)
    dev.set_postings(idx.term_ptr, idx.postings, idx.doc_len, idx.idf, idx.avgdl, idx.k1, idx.b)
    _check_chain(dev, x, csr, q, lists, k, fusion)


@pytest.mark.parametrize("fusion", ["linear", "rrf"])
@pytest.mark.parametrize("B,k", [(9, 5), (16, 10), (64, 5), (64, 100)])
def test_search_chain_reference_corpus(dev, legal_chunks, legal_texts, reference_queries, B, k, fusion):
    """The reference corpus: its real BM25 postings, stand-in vectors in its (law, chapter) layout."""
    x = legal_layout_corpus(legal_chunks)
    idx = BM25Index.from_texts(legal_texts)
    csr = obm25.BM25OkapiCSR.from_corpus([obm25.tokenize(t) for t in legal_texts])
    q = legal_queries(x, B, seed=500 + B)
    sel = k2b_selection(x, q, 2 * k, B, stride=1)
    if sel["valid"] >= 4 * k:                               # K2b runs (at the parent, already at 2k)
        assert region_overflow(sel).any()
    lists = [idx.term_ids(tokenize(reference_queries[b % len(reference_queries)])) for b in range(B)]
    dev.set_corpus(_cuda(x), 0)
    dev.set_postings(idx.term_ptr, idx.postings, idx.doc_len, idx.idf, idx.avgdl, idx.k1, idx.b)
    _check_chain(dev, x, csr, q, lists, k, fusion)


# ------------------------------------------------------------------ 5. device-pointer chain with its retry
def test_sharded_search_checked_on_clustered_rows(dev):
    from legal_rag_engine_b200.device_index import FUSION
    from legal_rag_engine_b200.sharding import ShardedSearcher
    x = blocks_corpus()
    idx = synth.host_bm25(N_BLOCKS, seed=81, vocab=3000)
    csr = obm25.BM25OkapiCSR.from_postings(idx.n_docs, idx.doc_len, idx.term_ptr.astype(np.int64),
                                           idx.postings[:, 0], idx.postings[:, 1])
    B, k = 24, 10
    q = block_queries(x, B, seed=82)
    assert region_overflow(k2b_selection(x, q[:n_planted(B)], 2 * k, B, stride=1)).any()
    terms, ptr = synth.host_query_terms(B, 8, seed=83, vocab=3000)
    lists = [terms[ptr[b]:ptr[b + 1]].tolist() for b in range(B)]
    weights = [0.5 + 0.1 * (b % 2) for b in range(B)]
    dev.set_corpus(_cuda(x), 0)
    dev.set_postings(idx.term_ptr, idx.postings, idx.doc_len, idx.idf, idx.avgdl, idx.k1, idx.b)
    s = ShardedSearcher(dev)
    for fusion in ("linear", "rrf"):
        outs = s.search_checked(_cuda(q), _cuda(terms), _cuda(ptr), k, FUSION[fusion], _cuda(np.array(weights)))
        ids, score, sem, kw, status = [t.cpu().numpy() for t in outs]
        assert status.sum() == 0
        _assert_results((ids, score, sem, kw), OracleIndex(x, csr).search_batch_vec(q, lists, k, weights, fusion))


# ------------------------------------------------------------------ 6. a coalesced batch through the engine
@pytest.fixture(scope="module")
def seeded_engine(tmp_path_factory, legal_chunks):
    """The reference corpus through create_vector_store with a seeded encoder: real texts in their
    real order, so neighbouring chunks of a chapter embed close to one another."""
    import json
    from legal_rag_engine_b200.engine import RetrievalEngine, create_vector_store
    from legal_rag_engine_b200.tokenizer import HashTokenizer
    d = tmp_path_factory.mktemp("store")
    (d / "chunks.json").write_text(json.dumps(legal_chunks), encoding="utf-8")
    sd = synth.bert_state_dict(42, 0.05, ln_jitter=0.1)
    tok = HashTokenizer(30522)
    create_vector_store(str(d / "chunks.json"), str(d / "vs"), encoder_state_dict=sd, tokenizer=tok)
    eng = RetrievalEngine(str(d / "vs"), encoder_state_dict=sd, tokenizer=tok)
    yield eng
    eng.close()


@pytest.mark.parametrize("fusion", ["linear", "rrf"])
def test_engine_coalesced_batch_answers_as_single_queries(seeded_engine, reference_queries, fusion):
    """A serving front merges concurrent search() calls into one search_batch, which from 9 sub-queries
    scores the batch with K2b.  Each query must get exactly what a search of its own returns."""
    qs = [q for q in reference_queries if q] * 2
    w = [0.5 + 0.1 * (i % 2) for i in range(len(qs))]
    for k in (5, 10):
        got = seeded_engine.search_batch(qs, k=k, hybrid_weights=w, fusion=fusion)
        for q, wi, g in zip(qs, w, got):
            assert g == seeded_engine.search(q, k=k, hybrid_weight=wi, fusion=fusion)
