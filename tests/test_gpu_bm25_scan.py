"""K3, the BM25 scan (csrc/bm25.cu: bm25_bounds_kernel, bm25_scan_kernel, bm25_merge_finalize_kernel;
bm25_score_at in bm25_at.cuh), against the float64 oracle (oracle/bm25.py) on every branch it has.

The scan promises rank_bm25's scores bit for bit, so every comparison here is exact: the maxima, the
scores at candidate ids (-1 and ids outside the shard included), the top-K ids and scores with their
(0.0, -1) padding, and the fused ids / scores / semantic / keyword columns of the search chain.  Ranges
are claimed dynamically and thresholds are shared through atomics, so every call is made twice and
must give the same bits both times.

The CPU tests at the top restate the host-side choices the scan's branches hang on -- bm25_geometry
(per-warp buffer, warps per CTA, grid, token rows), the warp split of bm25_bounds_kernel, the search
chain's list depth and CTAs per SM, the kBigLen choice and the host path's token-row rounding -- and
the GPU cases assert through them, or through the oracle, that they reach the condition they are named
for.  GPU tests carry the gpu mark one by one.
"""
import numpy as np
import pytest
import torch

from oracle import bm25 as obm25
from oracle import flat_ip
from oracle.search import OracleIndex

from legal_rag_engine_b200 import synth
from legal_rag_engine_b200.bm25_index import BM25Index

gpu = pytest.mark.gpu

# csrc/bm25.cu, bm25_at.cuh, merge.cuh, api.cu, include/lrx.h
RANGE = 1024                     # kBmRange: documents per (warp, query) unit
CTAB = 2048                      # kBmCtab: lengths the shared c[len] table covers
TILE_BYTES = (RANGE + 4) * 8     # kBmTileBytes
MAX_WARPS = 8                    # kBmWarps
CTAS_PER_SM = 2                  # kBmCtasPerSm
UNIT_COST = 192.0                # kBmUnitCost
HIST_LO, HIST_HI = 2.0 ** -6, 2.0 ** 10     # the score histogram's range (clamped at both ends)
MERGE_CAP = 4096                 # kMergeCap
K2B_MIN_B = 9                    # kK2bMinB
MAX_QUERY_TERMS = 64             # LRX_MAX_QUERY_TERMS
GRID_Y_MAX = 65535               # CUDA's gridDim.y limit
GLOBAL_ID_LIMIT = 2 ** 32       # lrx_set_corpus: global ids (id_base + local row) stay below it


def far_base(n):
    """The highest shard offset lrx_set_corpus admits for n rows: global ids up to 2^32 - 2, past
    the int32 sign bit, where a 32-bit truncation of an id or an offset would show."""
    return GLOBAL_ID_LIMIT - 1 - n


# ------------------------------------------------------------------ restatements (CPU)
def bm25_geometry(sms, n_local, B, K, ctas_per_sm=0, rows=0):
    """bm25.cu bm25_geometry.  ctas_per_sm: the handle's bm_ctas_per_sm (1: one CTA per SM, else 2);
    rows: bm_rows (0: B * 64)."""
    n_ranges = max(1, -(-n_local // RANGE))
    cap = 64
    while cap < K + 32:
        cap <<= 1
    warps = min(MAX_WARPS, max(2, (94 * 1024 - CTAB * 8) // (TILE_BYTES + cap * 16)))
    grid = -(-(n_ranges * B) // warps)
    grid = min(grid, sms * (1 if ctas_per_sm == 1 else CTAS_PER_SM))
    grid = max(grid, -(-B // warps))
    max_rows = rows if rows > 0 else B * MAX_QUERY_TERMS
    return dict(n_ranges=n_ranges, n_bounds=n_ranges + 1, cap=cap, warps=warps, grid=grid,
                n_warps=grid * warps, max_rows=max_rows, grid_y=min(max_rows, GRID_Y_MAX),
                use_hist=K > 32, bootstrap="lane_maxima" if 0 < K <= 32 else ("bisection" if K > 32 else None))


def query_costs(term_ptr, lists, n_bounds, max_rows):
    """bm25_bounds_kernel: each query's work, float64 in the kernel's order -- a fixed cost per range,
    then the list lengths of its in-vocabulary tokens below the token capacity."""
    tp = np.asarray(term_ptr, dtype=np.int64)
    costs, row = [], 0
    for t_list in lists:
        c = float(n_bounds - 1) * UNIT_COST
        for j, t in enumerate(t_list):
            if row + j >= max_rows:
                break
            if 0 <= t < len(tp) - 1:
                c += float(tp[t + 1] - tp[t])
        costs.append(c)
        row += len(t_list)
    return costs


def warp_split(costs, n_warps):
    """bm25_bounds_kernel's split of the scan's warps: floor shares of n_warps in proportion to the
    costs (at least one warp each), then rounds of one warp per query to the queries with the most
    work per warp (or from those with the least), ranked by counting."""
    B = len(costs)
    total = 0.0
    for c in costs:
        total += c
    share = [max(1, int(float(n_warps) * (c / total))) for c in costs]
    diff = n_warps - sum(share)
    while diff != 0:
        sgn = 1 if diff > 0 else -1
        todo = min(diff * sgn, B)
        can = [sgn > 0 or w > 1 for w in share]
        key = [costs[q] / float(share[q]) * float(sgn) for q in range(B)]
        new = []
        for q in range(B):
            rank = sum(1 for o in range(B) if can[o] and (key[o] > key[q] or (key[o] == key[q] and o < q)))
            new.append(share[q] + sgn if can[q] and rank < todo else share[q])
        moved = sum(new) - sum(share)
        share = new
        if moved == 0:
            break
        diff -= moved
    return share


def chain_choices(B, k, fusion, n_local):
    """api.cu enqueue_search: the BM25 list depth Kb and the handle's bm_ctas_per_sm."""
    Kb = 2 * k if fusion == "rrf" else 0
    one = B < K2B_MIN_B and n_local > 0 and (B <= 4 or n_local >= (4 << 20))
    return Kb, 1 if one else 0


def big_len(max_len):
    """bm25.cu launch_bm25_scan: bm25_scan_kernel<true> when a length falls outside the c[len] table."""
    return max_len + 1 > CTAB


def host_rows(n_tokens):
    """api.cu host_begin_locked: the host path's token capacity, a power of two from 32."""
    rows = 32
    while rows < n_tokens:
        rows *= 2
    return rows


DEPTHS = [1, 32, 33, 96, 97, 224, 225, 256]
BAND = {1: (64, 8), 32: (64, 8), 33: (128, 7), 96: (128, 7), 97: (256, 6), 224: (256, 6), 225: (512, 4),
        256: (512, 4)}


@pytest.mark.parametrize("sms", [148, 132])
@pytest.mark.parametrize("ctas", [0, 1])
@pytest.mark.parametrize("K", [0] + DEPTHS)
def test_geometry_depth_bands(sms, ctas, K):
    g = bm25_geometry(sms, 120_000, 64, K, ctas_per_sm=ctas)
    cap, warps = BAND.get(K, (64, 8))
    assert (g["cap"], g["warps"]) == (cap, warps)
    assert g["cap"] >= K + 32 and g["cap"] & (g["cap"] - 1) == 0
    assert g["use_hist"] == (K > 32)
    assert g["bootstrap"] == (None if K == 0 else ("lane_maxima" if K <= 32 else "bisection"))
    # shared memory per CTA stays under the 94 KB that fits beside a dense-scan CTA
    assert CTAB * 8 + warps * (TILE_BYTES + cap * 16) <= 94 * 1024
    assert g["n_ranges"] == 118 and g["n_bounds"] == 119
    assert g["grid"] <= sms * (1 if ctas == 1 else 2) and g["n_warps"] >= 64
    assert g["max_rows"] == 64 * 64 and g["grid_y"] == 4096


@pytest.mark.parametrize("sms", [148, 132])
def test_geometry_small_shards_and_token_rows(sms):
    g = bm25_geometry(sms, 0, 1, 20)
    assert g["n_ranges"] == 1 and g["grid"] == 1 and g["n_warps"] == 8
    g = bm25_geometry(sms, 1025, 64, 256, ctas_per_sm=1)
    assert g["n_ranges"] == 2 and g["grid"] == 32 and g["n_warps"] == 128
    assert bm25_geometry(sms, 1, 3, 0, rows=1 << 20)["grid_y"] == GRID_Y_MAX
    assert bm25_geometry(sms, 1, 3, 0, rows=65535)["grid_y"] == 65535


def test_warp_split_properties():
    rng = np.random.default_rng(3)
    for trial in range(300):
        B = int(rng.integers(1, 65))
        costs = [float(UNIT_COST * 3 + int(x)) for x in rng.zipf(1.3, size=B) % 10 ** 7]
        n_warps = int(rng.integers(B, 2400))
        share = warp_split(costs, n_warps)
        assert sum(share) == n_warps and min(share) >= 1, (trial, B, n_warps)
    # fewer warps than queries: every query keeps its one warp, the surplus cannot be taken back
    assert warp_split([1.0, 2.0, 3.0], 2) == [1, 1, 1]
    # exact proportions need no rounds
    assert warp_split([1.0, 3.0], 8) == [2, 6]


def test_warp_split_b64_reaches_lane_slot_q_plus_32():
    """The GPU case test_warp_split_b64: one heavy query, an empty and an all-OOV query, light ones."""
    idx = _zipf_index_small()
    lists = _split_lists(idx.n_terms)
    g = bm25_geometry(148, idx.n_docs, 64, 20)
    costs = query_costs(idx.term_ptr, lists, g["n_bounds"], g["max_rows"])
    share = warp_split(costs, g["n_warps"])
    assert sum(share) == g["n_warps"] and all(s >= 1 for s in share[32:])
    assert 1 in share and share[0] == max(share)


def test_chain_choices():
    assert chain_choices(4, 16, "rrf", 3000) == (32, 1)
    assert chain_choices(8, 48, "rrf", 3000) == (96, 0)
    assert chain_choices(8, 112, "rrf", 4 << 20) == (224, 1)
    assert chain_choices(9, 128, "rrf", 4 << 20) == (256, 0)
    assert chain_choices(64, 16, "linear", 300_000) == (0, 0)
    assert chain_choices(1, 10, "linear", 0) == (0, 0)


def test_length_table_and_host_rows():
    assert not big_len(2047) and big_len(2048) and big_len(65535)
    assert host_rows(0) == 32 and host_rows(33) == 64
    assert host_rows(32768) == 32768 and host_rows(32769) == 65536 and host_rows(70_000) == 131072
    # the rows over CUDA's gridDim.y limit: the bounds kernel loops over them
    assert [min(host_rows(n), GRID_Y_MAX) for n in (32768, 32769, 70_000)] == [32768, 65535, 65535]


# ------------------------------------------------------------------ corpora
def _zipf_terms(total, vocab, rng):
    t = np.searchsorted(synth._zipf_cdf(vocab), rng.random(total), side="right")
    return np.minimum(t, vocab - 1).astype(np.int64)


def _index_of_lengths(lens, vocab, seed, extra_docs=(), extra_terms=(), n_terms=None):
    """Documents of the given lengths filled with Zipf terms, plus extra (doc, term) tokens."""
    rng = np.random.default_rng(seed)
    lens = np.asarray(lens, dtype=np.int64)
    docs = np.repeat(np.arange(len(lens), dtype=np.int64), lens)
    terms = _zipf_terms(int(lens.sum()), vocab, rng)
    docs = np.concatenate([docs, np.asarray(extra_docs, dtype=np.int64)])
    terms = np.concatenate([terms, np.asarray(extra_terms, dtype=np.int64)])
    return BM25Index.from_token_arrays(docs, terms, len(lens), n_terms or vocab)


def _zipf_index_small():
    return synth.host_bm25(3000, seed=21, vocab=800)


def _split_lists(n_terms):
    """64 queries: 0 heavy (200 tokens of the densest terms), 1 empty, 2 all out of vocabulary,
    the rest light (3 to 8 tokens)."""
    rng = np.random.default_rng(5)
    lists = [[int(t) for t in rng.integers(0, 4, size=200)], [], [-1, -1, -7]]
    for q in range(3, 64):
        lists.append([int(t) for t in rng.integers(50, n_terms, size=3 + q % 6)])
    return lists


def _longest_index(max_len):
    """20 000 Zipf documents, the longest exactly max_len tokens (doc 10 000), one of max_len - 1."""
    rng = np.random.default_rng(max_len)
    lens = synth.host_doc_lengths(20_000, rng)
    lens[10_000], lens[3] = max_len, max_len - 1
    return _index_of_lengths(lens, 2000, seed=max_len + 1)


LONG_TERM = 3000                 # the term of the document made of one term 65 535 times


def _long_docs_index():
    """100 000 documents, 1 % of them 2 048 to 65 535 tokens long: doc LONG[0] is LONG_TERM 65 535
    times (a posting of tf 65 535), doc LONG[1] 65 535 Zipf tokens, LONG[2] exactly 2 048."""
    n = 100_000
    rng = np.random.default_rng(77)
    lens = synth.host_doc_lengths(n, rng)
    long_ids = np.sort(rng.choice(n, size=n // 100, replace=False))
    long_lens = rng.integers(2048, 6000, size=len(long_ids))
    long_lens[rng.choice(len(long_ids), size=8, replace=False)] = rng.integers(6000, 65536, size=8)
    order = rng.permutation(len(long_ids))
    long_ids = long_ids[order]
    long_lens[:4] = [0, 65535, 2048, 40000]
    lens[long_ids] = long_lens
    extra = np.full(65535, long_ids[0], dtype=np.int64)
    idx = _index_of_lengths(lens, LONG_TERM, seed=78, extra_docs=extra,
                            extra_terms=np.full(65535, LONG_TERM), n_terms=LONG_TERM + 1)
    return idx, long_ids


def _score_range_index(kind):
    """'high': a rare term R in 600 of 50 000 documents three times each, so a query repeating it
    256 times scores above 2^10; 'tiny': 1 000 documents over four terms of document frequency
    499, 499, 501 and 500 -- mean raw idf ~ 0.002, every score below 2^-6, idf(Z) exactly 0;
    'negative': 3 000 documents, five terms in 90 % of them, a rare one in 400 and 30, one in half
    of them -- mean raw idf < 0, so the common terms get a negative floored idf, and idf(Z) is 0."""
    rng = np.random.default_rng({"high": 1, "tiny": 2, "negative": 3}[kind])
    if kind == "high":
        n, vocab = 50_000, 3000
        lens = synth.host_doc_lengths(n, rng)
        R = vocab
        hits = np.repeat(np.sort(rng.choice(n, size=600, replace=False)), 3)
        return _index_of_lengths(lens, vocab, seed=11, extra_docs=hits, extra_terms=np.full(len(hits), R),
                                 n_terms=vocab + 1)
    if kind == "tiny":
        n = 1000
        i = np.arange(n)
        sets = [i[i < 499], i[i >= 501], i[i >= 499], i[i % 2 == 0]]       # A, C (499), B (501), Z (500)
    else:
        n = 3000
        i = np.arange(n)
        sets = [np.sort(rng.choice(n, size=2700, replace=False)) for _ in range(5)]
        sets += [np.sort(rng.choice(n, size=400, replace=False)), np.sort(rng.choice(n, size=30, replace=False)),
                 i[i % 2 == 1]]
    docs, terms = [], []
    for t, s in enumerate(sets):
        tf = rng.integers(1, 4, size=len(s))
        docs.append(np.repeat(s, tf))
        terms.append(np.full(int(tf.sum()), t))
    return BM25Index.from_token_arrays(np.concatenate(docs), np.concatenate(terms), n, len(sets))


def _score_range_lists(kind, n_terms):
    if kind == "high":
        R = n_terms - 1
        return [[R] * 256, [R] * 200 + [5, 9, 17], [3, R, 40], [R]]
    if kind == "tiny":                                   # A 0, C 1, B 2, Z 3
        return [[0], [1], [2, 2], [0, 3, 2], [3], [3, 3, 2]]
    return [[0, 5], [0, 1], [6, 2, 3], [0, 0, 0], [7], [5, 7, 4], [7, 1]]     # commons 0-4, rare 5 6, Z 7


def _csr_of(idx):
    return obm25.BM25OkapiCSR.from_postings(idx.n_docs, idx.doc_len, idx.term_ptr.astype(np.int64),
                                            idx.postings[:, 0], idx.postings[:, 1])


def test_score_range_corpora_reach_their_ranges():
    """The oracle shows each score-range corpus reaches the range it is for (CPU, no device)."""
    idx = _score_range_index("high")
    csr = _csr_of(idx)
    s = csr.get_scores_ids(_score_range_lists("high", idx.n_terms)[0])
    assert (s >= HIST_HI).sum() >= 200                                    # above the histogram's top
    idx = _score_range_index("tiny")
    csr = _csr_of(idx)
    assert 0 < csr.average_idf < 0.01 and csr.idf[3] == 0.0 and csr.idf[2] > 0
    for lst in _score_range_lists("tiny", idx.n_terms):
        s = csr.get_scores_ids(lst)
        assert s.max() < HIST_LO                                          # below the histogram's bottom
    assert (csr.get_scores_ids([0]) > 0).sum() >= 200
    idx = _score_range_index("negative")
    csr = _csr_of(idx)
    assert csr.average_idf < 0 and (csr.idf[:5] < 0).all() and csr.idf[7] == 0.0
    s = csr.get_scores_ids([0, 5])
    assert (s > 0).sum() >= 200 and (s < 0).any()                         # mixed signs
    s = csr.get_scores_ids([0, 1])
    assert s.max() <= 0 and (s < 0).any()                                 # only negative contributions


def test_length_corpora_reach_their_tables():
    for max_len, big in ((2047, False), (2048, True)):
        idx = _longest_index(max_len)
        assert int(idx.doc_len.max()) == max_len and big_len(int(idx.doc_len.max())) == big


# ------------------------------------------------------------------ GPU helpers
@pytest.fixture(scope="module")
def dev():
    from legal_rag_engine_b200.device_index import DeviceIndex
    d = DeviceIndex(0)
    yield d
    d.close()


@pytest.fixture(scope="module")
def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def _load(dev, idx, id_base=0, x=None):
    """Postings resident; the matrix is only needed for its row count unless x is given."""
    if x is None:
        dev.set_corpus(torch.zeros((idx.n_docs, 384), dtype=torch.float16, device="cuda"), id_base,
                       prefilter=False)
    else:
        dev.set_corpus(_cuda(x), id_base)
    dev.set_postings(idx.term_ptr, idx.postings, idx.doc_len, idx.idf, idx.avgdl, idx.k1, idx.b)


def _flat(lists, capacity=0):
    ptr = np.zeros(len(lists) + 1, dtype=np.int32)
    for i, t in enumerate(lists):
        ptr[i + 1] = ptr[i] + len(t)
    terms = np.zeros(max(int(ptr[-1]), capacity, 1), dtype=np.int32)
    terms[:ptr[-1]] = [x for t in lists for x in t]
    return terms, ptr


def _cands(n, id_base, local=(), n_rand=10, seed=0):
    """Candidate ids: -1, the ids just outside the shard, its first and last, `local` ids, random."""
    rng = np.random.default_rng(seed)
    c = [-1, id_base - 1, id_base, id_base + n - 1, id_base + n, id_base + n + 1000]
    c += [id_base + int(i) for i in local]
    c += [id_base + int(i) for i in rng.integers(0, n, size=n_rand)]
    return np.array(c, dtype=np.int64)


def _check_bm25(dev, csr, lists, K, id_base=0, cand=None, scores=None, capacity=0):
    """dev.bm25 twice: the same bits both times, and the oracle's maxima, candidate scores and top-K
    (ties by id, (0.0, -1) padding), bit for bit.  scores: the oracle's rows, when already computed."""
    B, n = len(lists), csr.corpus_size
    cand = _cands(n, id_base) if cand is None else cand
    cands = np.tile(cand, (B, 1))
    terms, ptr = _flat(lists, capacity)
    runs = []
    for _ in range(2):
        cs, mx, ts, ti = dev.bm25(_cuda(terms), _cuda(ptr), _cuda(cands), K)
        runs.append([cs.cpu().numpy(), mx.cpu().numpy(), ts.cpu().numpy(), ti.cpu().numpy()])
    for a, b in zip(runs[0], runs[1]):
        np.testing.assert_array_equal(a.view(np.uint64) if a.dtype == np.float64 else a,
                                      b.view(np.uint64) if b.dtype == np.float64 else b)
    cs, mx, ts, ti = runs[0]
    for q in range(B):
        s = scores[q] if scores is not None else csr.get_scores_ids(lists[q])
        pos = s[s > 0]
        assert _bits(mx[q]) == _bits(pos.max() if len(pos) else 0.0), q
        loc = cands[q] - id_base
        inside = (cands[q] >= 0) & (loc >= 0) & (loc < n)
        want = np.where(inside, s[np.clip(loc, 0, n - 1)], 0.0)
        np.testing.assert_array_equal(_bits(cs[q]), _bits(want), err_msg=f"query {q}")
        so, io = obm25.topk_positive(s, K, id_base)
        np.testing.assert_array_equal(ti[q, :len(io)], io, err_msg=f"query {q}")
        np.testing.assert_array_equal(_bits(ts[q, :len(io)]), _bits(so), err_msg=f"query {q}")
        assert (ti[q, len(io):] == -1).all() and (_bits(ts[q, len(io):]) == 0).all(), q
    return mx


def _search_check(dev, x, csr, lists, ks, fusions=("rrf", "linear"), seed=0):
    """search_batch_host twice per (k, fusion) against OracleIndex: ids, fused score, semantic and
    keyword columns bit for bit, the -1 padding after the oracle's results."""
    B = len(lists)
    rng = np.random.default_rng(seed)
    q = synth.host_queries(B, seed=seed + 1)
    q[0] = synth.host_planted_queries(x, [int(rng.integers(0, len(x)))], seed=seed + 2)[0]
    weights = [0.5 + 0.1 * (b % 2) for b in range(B)]
    oi = OracleIndex(x, csr)
    dense = flat_ip.exact_scores(x, q)
    for fusion in fusions:
        for k in ks:
            want = oi.search_batch_vec(q, lists, k, weights, fusion, dense_scores=dense)
            first = dev.search_batch_host(q, lists, k, weights, fusion)
            again = dev.search_batch_host(q, lists, k, weights, fusion)
            for a, b in zip(first, again):
                np.testing.assert_array_equal(a.view(np.uint64) if a.dtype == np.float64 else a,
                                              b.view(np.uint64) if b.dtype == np.float64 else b)
            ids, score, sem, kw = first
            for b, res in enumerate(want):
                ctx = f"{fusion} k={k} query {b}"
                assert ids[b, :len(res)].tolist() == [r[0] for r in res], ctx
                assert (ids[b, len(res):] == -1).all(), ctx
                for col, arr in ((1, score), (2, sem), (3, kw)):
                    np.testing.assert_array_equal(_bits(arr[b, :len(res)]), _bits([r[col] for r in res]),
                                                  err_msg=ctx)


# ------------------------------------------------------------------ 1. depth bands
@pytest.fixture(scope="module")
def zipf120k():
    idx = synth.host_bm25(120_000, seed=120, vocab=5000)
    return idx, _csr_of(idx)


@gpu
@pytest.mark.parametrize("B", [3, 64])
def test_depth_bands(dev, sms, zipf120k, B):
    """K at both ends of every (buffer, warps per CTA, threshold scheme, bootstrap) band."""
    idx, csr = zipf120k
    _load(dev, idx, id_base=77)
    terms, ptr = synth.host_query_terms(B, 8, seed=B, vocab=5000)
    lists = [terms[ptr[b]:ptr[b + 1]].tolist() for b in range(B)]
    lists[-1] = lists[-1] + [lists[-1][0], -1]                # a repeat and an out-of-vocabulary token
    scores = [csr.get_scores_ids(t) for t in lists]
    warps_seen = set()
    for K in DEPTHS:
        g = bm25_geometry(sms, idx.n_docs, B, K)
        assert (g["cap"], g["warps"]) == BAND[K] and g["use_hist"] == (K > 32)
        warps_seen.add(g["warps"])
        assert min((s > 0).sum() for s in scores) >= K       # every list is full
        _check_bm25(dev, csr, lists, K, id_base=77, scores=scores, cand=_cands(idx.n_docs, 77, seed=K))
    assert warps_seen == {8, 7, 6, 4}


# ------------------------------------------------------------------ 2. length table
@gpu
@pytest.mark.parametrize("max_len", [2047, 2048])
def test_length_table_edge(dev, max_len):
    """Longest document 2 047 tokens: the table's last entry, bm25_scan_kernel<false>; 2 048: the
    first length past it, bm25_scan_kernel<true>."""
    idx = _longest_index(max_len)
    assert big_len(int(idx.doc_len.max())) == (max_len == 2048)
    csr = _csr_of(idx)
    _load(dev, idx)
    top = [int(t) for t in np.argsort(-np.diff(idx.term_ptr.astype(np.int64)))[:40]]
    lists = [top[:8], top[::5], top[10:30] + top[:3], [top[0]] * 40 + [top[39]], [top[1]]]
    for K in (20, 200):
        mx = _check_bm25(dev, csr, lists, K, cand=_cands(idx.n_docs, 0, local=[10_000, 3, 2047, 2048]))
        assert (mx > 0).all()


@gpu
def test_long_documents_and_tf_65535(dev):
    """1 % of 100 000 documents between 2 048 and 65 535 tokens, one of them a single term 65 535
    times; candidates on the long documents."""
    idx, long_ids = _long_docs_index()
    assert int(idx.doc_len.max()) == 65535 and big_len(65535)
    assert int(idx.postings[:, 1].max()) == 65535
    assert ((idx.doc_len >= 2048).sum() >= 1000) and int(idx.doc_len[long_ids[2]]) == 2048
    csr = _csr_of(idx)
    base = far_base(idx.n_docs)
    _load(dev, idx, id_base=base)
    lists = [[LONG_TERM], [LONG_TERM, 0, 1, 2], [0, 1, 2, 3, 4, 5], [7, LONG_TERM, 7, 100, 900],
             list(range(0, 64)), [2999, 1500, 0]]
    cand = _cands(idx.n_docs, base, local=long_ids[:24])
    for K in (20, 200):
        _check_bm25(dev, csr, lists, K, id_base=base, cand=cand)


# ------------------------------------------------------------------ 3. score ranges
@gpu
@pytest.mark.parametrize("kind", ["high", "tiny", "negative"])
def test_score_ranges(dev, kind):
    """Scores above the histogram's top (>= 2^10), all below its bottom (< 2^-6), negative and
    mixed-sign documents with idf floored below 0, and a term of idf exactly 0 -- at K = 20 (lane
    maxima bootstrap, no histogram) and K = 200 (bisection and histogram)."""
    idx = _score_range_index(kind)
    csr = _csr_of(idx)
    lists = _score_range_lists(kind, idx.n_terms)
    scores = [csr.get_scores_ids(t) for t in lists]
    if kind == "high":
        assert (scores[0] >= HIST_HI).sum() >= 200
    elif kind == "tiny":
        assert max(s.max() for s in scores) < HIST_LO and csr.idf[3] == 0.0
        assert scores[4].max() == 0.0                         # the idf-0 term alone scores nothing
    else:
        assert csr.average_idf < 0 and csr.idf[7] == 0.0
        assert (scores[0] > 0).sum() >= 200 and (scores[0] < 0).any()
        assert scores[1].max() <= 0 and scores[3].max() <= 0  # only negative contributions
    _load(dev, idx, id_base=10)
    for K in (20, 200):
        mx = _check_bm25(dev, csr, lists, K, id_base=10, scores=scores,
                         cand=_cands(idx.n_docs, 10, n_rand=40, seed=K))
        if kind == "negative":
            assert mx[1] == 0.0 and mx[3] == 0.0


# ------------------------------------------------------------------ 4. merge overflow
def _tie_index():
    """300 032 documents of two tokens each: term 0 in all of them (floored idf, > 0 because the
    other 50 terms are rare enough), term 1 + i % 50 in document i.  Every score of term 0 ties."""
    n = 300_032
    d = np.repeat(np.arange(n, dtype=np.int64), 2)
    t = np.zeros(2 * n, dtype=np.int64)
    t[1::2] = 1 + np.arange(n) % 50
    return BM25Index.from_token_arrays(d, t, n, 51)


@pytest.fixture(scope="module")
def ties():
    idx = _tie_index()
    return idx, _csr_of(idx)


@gpu
@pytest.mark.parametrize("B", [1, 3])
@pytest.mark.parametrize("K", [20, 256])
def test_merge_overflow_on_ties(dev, sms, ties, B, K):
    """Every document scores the same, so the list is the K lowest ids.  Each warp's list holds the
    first K documents of the first range it claimed (a later range's keys lose the id tie-break).

    K = 256: cap 512, 4 warps per CTA; at B = 1 the grid is min(ceil(293 / 4), 2 SMs) = 74 CTAs,
    296 warps, all resident, each claiming three ranges before its first unit -- so the 293 ranges
    go to at least 98 warps.  The merge's lower bound L is the 256th largest of the heads of the
    first 256 lists: fewer than 256 of them hold keys, so L = 0, or L is the head of the highest
    range among them and the other 255 lie below it.  Every list below L survives whole: at least
    98 x 256 = 25 088 keys, far above kMergeCap = 4 096 -- the retry runs.  B = 3 splits the warps
    three ways (~98 each): L is the 256th largest of three keys per list, so ~85 lists x 256 keys
    survive, again over 4 096.

    K = 20: L is the 20th largest head, near the 20th range; the lists below it hold ~20 x 20 keys,
    a few hundred: the same ties without the retry."""
    idx, csr = ties
    g = bm25_geometry(sms, idx.n_docs, B, K)
    assert g["n_ranges"] == 293
    if K == 256:
        assert g["warps"] == 4 and g["grid"] * g["warps"] >= g["n_ranges"] and g["grid"] <= sms * 2
        assert -(-g["n_ranges"] // 3) * K > MERGE_CAP
    else:
        assert 20 * 20 < MERGE_CAP
    assert csr.idf[0] > 0
    base = far_base(idx.n_docs)
    _load(dev, idx, id_base=base)
    lists = [[0], [0, 0], [0, 5]][:B]
    s0 = csr.get_scores_ids([0])
    assert (s0 == s0[0]).all()                                # one tie over the whole shard
    _, io = obm25.topk_positive(s0, K, base)
    assert io.tolist() == list(range(base, base + K))
    _check_bm25(dev, csr, lists, K, id_base=base,
                cand=_cands(idx.n_docs, base, local=[1023, 1024, 299_999, 300_031]))


# ------------------------------------------------------------------ 5. warp split at B = 64
@gpu
def test_warp_split_b64(dev, sms):
    """One heavy query, an empty and an all-OOV query, 61 light ones: queries 32-63 (lane slot q + 32
    of the split) get warps, some query exactly one."""
    idx = _zipf_index_small()
    csr = _csr_of(idx)
    lists = _split_lists(idx.n_terms)
    for K in (20, 200):
        g = bm25_geometry(sms, idx.n_docs, 64, K)
        share = warp_split(query_costs(idx.term_ptr, lists, g["n_bounds"], g["max_rows"]), g["n_warps"])
        assert all(s >= 1 for s in share[32:]) and 1 in share and sum(share) == g["n_warps"]
        _load(dev, idx, id_base=3)
        mx = _check_bm25(dev, csr, lists, K, id_base=3)
        assert mx[1] == 0.0 and mx[2] == 0.0


@gpu
def test_b64_at_the_default_token_capacity(dev, zipf120k):
    """64 queries x 64 tokens = 4 096 rows, exactly the default capacity B * 64: scored in full, no NaN."""
    idx, csr = zipf120k
    terms, ptr = synth.host_query_terms(64, 64, seed=64, vocab=5000)
    lists = [terms[ptr[b]:ptr[b + 1]].tolist() for b in range(64)]
    assert sum(map(len, lists)) == bm25_geometry(148, idx.n_docs, 64, 20)["max_rows"]
    _load(dev, idx)
    mx = _check_bm25(dev, csr, lists, 20)
    assert not np.isnan(mx).any()


# ------------------------------------------------------------------ 6. long batches
def _long_batch_lists(n_tokens, B, vocab, seed):
    rng = np.random.default_rng(seed)
    cut = np.sort(rng.choice(np.arange(1, n_tokens), size=B - 1, replace=False))
    sizes = np.diff(np.concatenate([[0], cut, [n_tokens]]))
    t = _zipf_terms(n_tokens, vocab, rng)
    t[rng.random(n_tokens) < 0.01] = -1                       # out-of-vocabulary tokens
    out, o = [], 0
    for s in sizes:
        out.append([int(v) for v in t[o:o + s]])
        o += s
    return out


@pytest.fixture(scope="module")
def small_corpus():
    n = 3000
    idx = synth.host_bm25(n, seed=33, vocab=1500)
    return idx, _csr_of(idx), synth.host_vectors(n, seed=34, dup_frac=0.01)


@gpu
@pytest.mark.parametrize("n_tokens", [32768, 32769, 70_000])
def test_long_batch_host_path(dev, small_corpus, n_tokens):
    """More than 32 768 tokens in one host-buffer search: the token capacity rounds up to 65 536
    rows and beyond, more than gridDim.y can hold; the bounds kernel walks the rows in a loop."""
    idx, csr, x = small_corpus
    assert host_rows(n_tokens) > GRID_Y_MAX or n_tokens == 32768
    _load(dev, idx, x=x)
    lists = _long_batch_lists(n_tokens, 8, 1500, seed=n_tokens)
    assert sum(map(len, lists)) == n_tokens
    _search_check(dev, x, csr, lists, ks=(10,), seed=n_tokens)


@gpu
@pytest.mark.parametrize("capacity", [65535, 65536, 70_000])
def test_long_batch_device_path(dev, small_corpus, capacity):
    """lrx_bm25 with a token capacity (lrx_set_query_capacity) of 65 535, 65 536 and 70 000 rows,
    every row live."""
    idx, csr, _ = small_corpus
    lists = _long_batch_lists(capacity, 16, 1500, seed=capacity)
    base = far_base(idx.n_docs)
    _load(dev, idx, id_base=base)
    try:
        g = bm25_geometry(148, idx.n_docs, 16, 20, rows=capacity)
        assert g["max_rows"] == capacity and g["grid_y"] == min(capacity, GRID_Y_MAX)
        mx = _check_bm25(dev, csr, lists, 20, id_base=base, capacity=capacity)
        assert not np.isnan(mx).any()
    finally:
        dev._capacity = 0
        dev._ck(dev.lib.lrx_set_query_capacity(dev.h, 0))


# ------------------------------------------------------------------ 7. range edges, offsets
@gpu
@pytest.mark.parametrize("n", [1023, 1024, 1025])
def test_range_edges_and_far_id_base(dev, n):
    """Shards ending just before, at and just after a 1 024-document range; candidates at local 1 023,
    1 024, n - 1 and n; ids offset so that the shard's last global id is 2^32 - 2.  An offset past
    2^32 is refused: the fused ranking keys hold a 32-bit id."""
    from legal_rag_engine_b200._lib import LrxError
    idx = synth.host_bm25(n, seed=n, vocab=200)
    csr = _csr_of(idx)
    assert bm25_geometry(148, n, 4, 20)["n_ranges"] == (1 if n <= 1024 else 2)
    base = far_base(n)
    assert base > 2 ** 31 and base + n - 1 == GLOBAL_ID_LIMIT - 2
    with pytest.raises(LrxError):
        _load(dev, idx, id_base=5 * GLOBAL_ID_LIMIT + 7)
    with pytest.raises(LrxError):
        _load(dev, idx, id_base=base + 1)
    _load(dev, idx, id_base=base)
    terms, ptr = synth.host_query_terms(4, 8, seed=n + 1, vocab=200)
    lists = [terms[ptr[b]:ptr[b + 1]].tolist() for b in range(4)]
    cand = _cands(n, base, local=[1023, 1024, n - 1, n])
    for K in (20, 256):
        _check_bm25(dev, csr, lists, K, id_base=base, cand=cand)


# ------------------------------------------------------------------ 8. search chain
def _chain_lists(lists, B):
    return [list(lists[b % len(lists)]) for b in range(B)]


CHAIN_CORPORA = ["length_2048", "long_docs", "high", "tiny", "negative", "ties"]


def _chain_case(name):
    if name == "length_2048":
        idx = _longest_index(2048)
        top = [int(t) for t in np.argsort(-np.diff(idx.term_ptr.astype(np.int64)))[:20]]
        lists = [top[:8], top[5:9], [top[0]] * 3]
    elif name == "long_docs":
        idx, _ = _long_docs_index()
        lists = [[LONG_TERM, 0, 1], [2, 3, 4, 5], [LONG_TERM], [10, 500, -1]]
    elif name == "ties":
        idx = _tie_index()
        lists = [[0], [0, 0], [0, 5], [7]]
    else:
        idx = _score_range_index(name)
        lists = _score_range_lists(name, idx.n_terms)
    return idx, lists


@gpu
@pytest.mark.parametrize("name", CHAIN_CORPORA)
def test_search_chain(dev, name):
    """search_batch_host on the corpora above: rrf at k = 16, 48, 112, 128 (BM25 lists of 32, 96, 224,
    256) and linear (no list), at B = 4 (one scan CTA per SM beside K2a), 8 (two), 9 and 64 (K2b).
    The keyword column comes from bm25_score_at inside pack_exchange_kernel."""
    idx, lists = _chain_case(name)
    csr = _csr_of(idx)
    x = synth.host_vectors(idx.n_docs, seed=5, dup_frac=0.01)
    _load(dev, idx, x=x)
    seen = set()
    for B in (4, 8, 9, 64):
        for k in (16, 48, 112, 128):
            seen.add(chain_choices(B, k, "rrf", idx.n_docs))
        _search_check(dev, x, csr, _chain_lists(lists, B), ks=(16, 48, 112, 128), fusions=("rrf",), seed=B)
        _search_check(dev, x, csr, _chain_lists(lists, B), ks=(16,), fusions=("linear",), seed=B)
    assert {c for _, c in seen} == {0, 1} and {kb for kb, _ in seen} == {32, 96, 224, 256}
