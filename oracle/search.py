"""Oracle: ``RetrievalEngine.search`` and the orchestrator fan-out, end to end
(after the encoder), on the fp16 chunk matrix + BM25 postings.

Test infrastructure, see ``oracle/__init__.py``.  Parity unpinned.

Follows ``src/retrieval/retrieval_engine.py:59-96`` and
``src/retrieval/orchestrator.py:38-62``.
"""
from __future__ import annotations

from typing import List, Sequence

import numpy as np

from . import bm25 as obm25
from . import flat_ip, fusion


class OracleIndex:
    def __init__(self, Xh: np.ndarray, bm25: obm25.BM25OkapiCSR):
        assert Xh.dtype == np.float16
        assert Xh.shape[0] == bm25.corpus_size
        self.Xh = Xh
        self.bm25 = bm25

    def search_vec(self, qh: np.ndarray, term_ids: Sequence[int], k: int = 5,
                   hybrid_weight: float = 0.5, fusion_mode: str = "linear", dense_scores=None):
        """One (already encoded) query.  qh: fp16 [384]; term_ids: BM25 term ids
        (-1 = out of vocabulary).  ``dense_scores``: this query's row of
        ``flat_ip.exact_scores`` when the caller has it already (large corpora).
        Returns [(id, score, semantic, keyword)]."""
        scores = (flat_ip.exact_scores(self.Xh, qh[None, :]) if dense_scores is None
                  else np.asarray(dense_scores, dtype=np.float64).reshape(1, -1))
        E, D, I = flat_ip.topk_from_scores(scores, 2 * k)          # :64  index.search(q, k*2)
        bm = self.bm25.get_scores_ids(term_ids)                    # :68
        max_bm25 = obm25.max_or_one(bm)                            # :74
        if fusion_mode == "linear":
            return fusion.linear_fuse(D[0], I[0], bm, max_bm25, k, hybrid_weight)
        if fusion_mode == "rrf":
            dense = [(int(i), float(e), float(bm[i])) for e, i in zip(E[0], I[0]) if i >= 0]
            bs, bi = obm25.topk_positive(bm, 2 * k)
            sparse = [(int(i), float(scores[0, i]), float(s)) for s, i in zip(bs, bi)]
            return fusion.rrf_fuse(dense, sparse, max_bm25, k)
        raise ValueError(fusion_mode)

    def search_batch_vec(self, Qh: np.ndarray, term_id_lists: List[Sequence[int]], k: int,
                         hybrid_weights: Sequence[float], fusion_mode: str = "linear", dense_scores=None):
        """``dense_scores``: ``flat_ip.exact_scores(Xh, Qh)`` computed once for several calls."""
        return [self.search_vec(Qh[i], term_id_lists[i], k, hybrid_weights[i], fusion_mode,
                                None if dense_scores is None else dense_scores[i])
                for i in range(len(term_id_lists))]


def fanout_queries(query: str, user_context: str, key_entities: Sequence[str], category: str):
    """``orchestrator.py:38-56``: the 1 or 4 search strings and their hybrid weights."""
    queries = [query]
    if user_context == "victim_distress":
        offence = next((e for e in key_entities
                        if e.lower() in ["robbery", "assault", "rape", "theft"]), "crime")
        queries.append(f"How to file FIR for {offence} BNSS procedure")
        queries.append(f"Victim compensation rights for {offence} NALSA scheme")
        queries.append("Zero FIR registration procedure BNSS")
    weights = [0.6 if category == "procedure" or "procedure" in q.lower() else 0.5
               for q in queries]
    return queries, weights


def fanout_dedup(result_lists, headers):
    """``orchestrator.py:54-62``: concatenate in query order, keep the first
    occurrence of each truthy ``canonical_header``."""
    out, seen = [], set()
    for results in result_lists:
        for r in results:
            h = headers[r[0]]
            if h and h not in seen:
                out.append(r)
                seen.add(h)
    return out
