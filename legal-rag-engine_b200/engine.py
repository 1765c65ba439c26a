"""Drop-in for the reference's ``src/retrieval/retrieval_engine.py`` and
``create_vector_store.py``: same class, constructor, ``search`` signature, result dicts and
store directory; everything numeric runs in the CUDA library behind include/lrx.h.

    from legal_rag_engine_b200.engine import RetrievalEngine, create_vector_store

Additive surface only: ``search_batch`` (the orchestrator's concept-expansion fan-out in one
launch chain, orchestrator.py:38-62), ``fusion="linear"|"rrf"`` (default "linear" = the
reference's behaviour, retrieval_engine.py:71-96), ``encode``, ``add_chunks`` / ``remove_chunks`` /
``replace_chunks`` / ``save`` (grow, shrink or edit a loaded index without a rebuild; results stay
bit-identical to a rebuild).

There is no CPU fallback: without a CUDA device or the built library the constructor raises.
"""
from __future__ import annotations

import ctypes as C
import json
import logging
import os
import shutil
import tempfile
import threading
from pathlib import Path
from typing import Dict, List, Optional, Sequence

import numpy as np
import torch

from . import store as _store
from ._lib import LRX_MAX_BATCH, LRX_MAX_DEPTH
from .bm25_index import BM25Index, csr_append, csr_remove, csr_replace, tokenize
from .device_index import FUSION, DeviceIndex
from .encoder import SentenceEncoder
from .sharding import shard_range

logger = logging.getLogger("LegalRAG-RetrievalEngine")


def _resolve_model_dir(model_dir: Optional[str]) -> Optional[str]:
    """EMBEDDING_MODEL_DIR, or a snapshot of all-MiniLM-L6-v2 inside the project's
    ``.hf_cache`` (where the reference's build phase caches it, retrieval_engine.py:8-9)."""
    if model_dir:
        return model_dir
    env = os.getenv("EMBEDDING_MODEL_DIR")
    if env:
        return env
    for root in (Path(os.getcwd()) / ".hf_cache", Path(os.getenv("HF_HOME", "")) if os.getenv("HF_HOME") else None):
        if root and root.exists():
            for p in root.rglob("model.safetensors"):
                if "MiniLM-L6" in str(p):
                    return str(p.parent)
    return None


def _chunk_tokens(chunks: Sequence[dict]) -> List[List[str]]:
    """The BM25 tokens of each chunk, after checking it is a dict with a str ``"text"`` of at most
    65 535 tokens (the 8-byte posting stores the document length in 16 bits)."""
    tokens = []
    for i, c in enumerate(chunks):
        if not isinstance(c, dict) or not isinstance(c.get("text"), str):
            raise ValueError(f"chunk {i}: expected a dict with a str 'text'")
        tokens.append(tokenize(c["text"]))
        if len(tokens[-1]) > 65535:
            raise ValueError(f"chunk {i}: {len(tokens[-1])} tokens; a BM25 document holds at most 65535")
    return tokens


def _check_id_types(ids: Sequence) -> None:
    for i in ids:
        if isinstance(i, (bool, np.bool_)) or not isinstance(i, (int, np.integer)):
            raise TypeError(f"chunk ids must be ints, got {i!r}")


def _id_array(ids: Sequence[int], n: int) -> np.ndarray:
    """Chunk ids as int64, after checking they lie in [0, n) and are unique."""
    ids_arr = np.asarray(ids, dtype=np.int64).reshape(-1)
    if len(ids_arr) and (ids_arr.min() < 0 or ids_arr.max() >= n):
        raise ValueError(f"chunk ids must lie in [0, {n})")
    if len(np.unique(ids_arr)) != len(ids_arr):
        raise ValueError("duplicate chunk ids")
    return ids_arr


def _dist_state(group=None):
    """(rank, world) of an initialised torch.distributed job, (0, 1) otherwise."""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(group), dist.get_world_size(group)
    return 0, 1


class RetrievalEngine:
    """``RetrievalEngine(store_dir)`` / ``search(query, k, hybrid_weight)`` exactly as the reference
    (retrieval_engine.py:23-96).

    One process: the whole store on one GPU.  Under ``torchrun`` (torch.distributed initialised,
    one rank per GPU): rank g keeps the contiguous row range ``shard_range(N, g, G)`` of the chunk
    matrix and of the BM25 postings (idf / avgdl stay the whole-corpus statistics), every rank
    encodes the <= 4 query strings redundantly and makes the same ``lrx_search_text_host`` call; the
    candidate exchange runs inside the kernels over NVLink and the fused result is replicated.  The
    server process is rank 0: it calls ``search`` as always (the strings are broadcast to the other
    ranks first); the other ranks sit in ``worker_loop()``.
    """

    def __init__(self, store_dir: str = "data/vector_store", *, device: Optional[int] = None,
                 model_dir: Optional[str] = None, encoder_state_dict: Optional[Dict] = None,
                 tokenizer=None, fusion: str = "linear", group=None, sharded: Optional[bool] = None):
        self.store_dir = Path(store_dir)
        self.fusion = fusion
        self.group = group
        # sharded=None: shard iff torch.distributed is initialised with more than one rank
        self.rank, self.world = _dist_state(group) if sharded in (None, True) else (0, 1)
        if device is None:
            device = int(os.environ.get("LOCAL_RANK", "0")) if self.world > 1 else 0
        self.dev = DeviceIndex(device, self.rank, self.world)
        # 1. model (retrieval_engine.py:27-33)
        if encoder_state_dict is None:
            model_dir = _resolve_model_dir(model_dir)
            if model_dir is None:
                raise FileNotFoundError(
                    "all-MiniLM-L6-v2 weights not found: set EMBEDDING_MODEL_DIR to a directory "
                    "holding model.safetensors and vocab.txt (or pass encoder_state_dict= and tokenizer=)")
        self.model = SentenceEncoder(self.dev, state_dict=encoder_state_dict, model_dir=model_dir,
                                     tokenizer=tokenizer)
        self.model.require_tokenizer()
        # 2-4. index, BM25, metadata (retrieval_engine.py:35-56); a shard keeps its row range
        self.chunks, xh, bm25 = _store.load_store(self.store_dir, mmap=self.world > 1)
        self.n_total = len(self.chunks)
        self.lo, self.hi = shard_range(self.n_total, self.rank, self.world)
        self._lock = threading.RLock()                     # searches see the index before or after a change
        self._stats = bm25.stats()                         # whole-corpus statistics + vocabulary (postings: on the GPU)
        self._sharded_bm25 = bm25 if self.world > 1 else None   # a shard's device holds only its own rows
        local = bm25 if self.world == 1 else bm25.shard(self.lo, self.hi)
        self._x = torch.from_numpy(np.ascontiguousarray(xh[self.lo:self.hi])).to(self.dev.device)
        self.dev.set_corpus(self._x, self.lo)
        self.dev.set_postings(local.term_ptr, local.postings, local.doc_len, bm25.idf, bm25.avgdl,
                              bm25.k1, bm25.b)
        if self.world > 1:
            if not self.dev.exchange_setup(LRX_MAX_BATCH, LRX_MAX_DEPTH // 2, group):
                raise RuntimeError("the GPUs of this box cannot map each other's memory (CUDA IPC / peer "
                                   "access): the sharded engine needs it")
        logger.info("Store resident on GPU %d (shard %d/%d): rows [%d,%d) of %d chunks, %d postings", device,
                    self.rank, self.world, self.lo, self.hi, self.n_total, local.nnz)

    # ------------------------------------------------------------------ API
    def encode(self, texts: Sequence[str]) -> np.ndarray:
        return self.model.encode(texts)

    def search(self, query: str, k: int = 5, hybrid_weight: float = 0.5, fusion: Optional[str] = None):
        return self.search_batch([query], k, [hybrid_weight], fusion)[0]

    def search_batch(self, queries: Sequence[str], k: int = 5,
                     hybrid_weights: Optional[Sequence[float]] = None, fusion: Optional[str] = None):
        """All queries through one encoder pass and one K2 -> K3 -> K4 chain.  Returns one
        result list per query, each exactly what ``search`` returns.  Sharded: called on rank 0
        (the other ranks are in ``worker_loop``)."""
        queries = list(queries)
        if hybrid_weights is None:
            hybrid_weights = [0.5] * len(queries)
        mode = fusion or self.fusion
        FUSION[mode]                                        # KeyError for an unknown fusion
        k = int(k)
        if k > LRX_MAX_DEPTH // 2:
            # the reference honours any k; this library's candidate depth is 2k <= LRX_MAX_DEPTH
            raise ValueError(f"k={k} exceeds the supported result depth {LRX_MAX_DEPTH // 2}")
        if self.world > 1:
            import torch.distributed as dist
            if self.rank != 0:
                raise RuntimeError("search() is called on rank 0; the other ranks run worker_loop()")
            dist.broadcast_object_list([("search", queries, k, list(hybrid_weights), mode)], src=0,
                                       group=self.group)
        return self._search_all(queries, k, list(hybrid_weights), mode)

    def worker_loop(self):
        """Ranks 1..G-1 of a sharded engine: repeat rank 0's calls until it closes."""
        import torch.distributed as dist
        assert self.world > 1 and self.rank != 0
        while True:
            box = [None]
            dist.broadcast_object_list(box, src=0, group=self.group)
            msg = box[0]
            if msg[0] == "stop":
                return
            _, queries, k, weights, mode = msg
            self._search_all(queries, k, weights, mode)

    def _search_all(self, queries, k, weights, mode):
        """Blocks of at most LRX_MAX_BATCH queries.  Queries of at most 64 WordPiece tokens and longer
        ones go in separate blocks: the short ones take the encoder's query path, whose result for a
        query does not depend on what it is batched with (csrc/encoder.cu, small_path), so a query
        returns the same scores however a serving front coalesced it."""
        with self._lock:
            return self._search_all_locked(queries, k, weights, mode)

    def _search_all_locked(self, queries, k, weights, mode):
        tok = self.model.tokenizer
        enc = [tok.encode(q, self.model.MAX_SEQ) for q in queries]
        out: List[Optional[List[dict]]] = [None] * len(queries)
        short = [i for i, e in enumerate(enc) if len(e) <= 64]
        long_ = [i for i, e in enumerate(enc) if len(e) > 64]
        for part in (short, long_):
            for s in range(0, len(part), LRX_MAX_BATCH):
                sel = part[s:s + LRX_MAX_BATCH]
                res = self._search_block([queries[i] for i in sel], [weights[i] for i in sel], k, mode,
                                         [enc[i] for i in sel])
                for i, r in zip(sel, res):
                    out[i] = r
        return out

    def _search_block(self, queries, weights, k, mode, enc):
        B = len(queries)
        if k < 1 or B == 0:
            return [[] for _ in queries]
        S = max(len(e) for e in enc)
        ids = np.zeros((B, S), dtype=np.int32)
        lens = np.empty(B, dtype=np.int32)
        for i, e in enumerate(enc):
            ids[i, :len(e)] = e
            lens[i] = len(e)
        # BM25 side: query.lower().split() -> term ids (retrieval_engine.py:67).  EVERY token is
        # scored, in order, repeats included, as rank_bm25 does; out-of-vocabulary tokens are
        # dropped here because `idf.get(q) or 0` makes them add exactly 0.0.
        term_lists = [[self._stats.vocab[w] for w in tokenize(q) if w in self._stats.vocab] for q in queries]
        o_ids, o_score, o_sem, o_kw = self.dev.search_text_host(ids, lens, term_lists, k, weights, mode)
        results = []
        for b in range(B):
            rows = []
            for j in range(k):
                idx = int(o_ids[b, j])
                if idx < 0:
                    continue
                rows.append({"chunk": self.chunks[idx], "score": float(o_score[b, j]),
                             "semantic": float(o_sem[b, j]), "keyword": float(o_kw[b, j])})
            results.append(rows)
        return results

    # ------------------------------------------------------------------ growth
    @property
    def bm25(self) -> BM25Index:
        """The BM25 index of the whole current corpus, a snapshot that later adds and removals leave as
        it is: on one GPU, the host statistics with the postings read back from the device; on a
        sharded engine (which cannot change), the index it loaded."""
        if self.world > 1:
            return self._sharded_bm25
        with self._lock:
            return BM25Index.from_stats(self._stats, *self.dev.read_postings())

    def add_chunks(self, chunks: Sequence[dict]) -> range:
        """Append chunks to the loaded index; returns their ids (positions in ``self.chunks``).
        Searches afterwards return exactly what an engine over a store rebuilt from all chunks (with
        these rows as their embeddings) returns.  Each chunk is a dict with a str ``"text"``, embedded
        with the encoder ``create_vector_store`` uses and stored as float16.  Input is validated
        before anything changes; a rejected call leaves the engine as it was.  Not supported on a
        sharded engine (world > 1)."""
        if self.world > 1:
            raise NotImplementedError("add_chunks on a sharded engine: rebuild the store instead")
        chunks = list(chunks)
        tokens = _chunk_tokens(chunks)
        with self._lock:
            n = self.n_total
            if n + len(chunks) >= 1 << 32:
                raise ValueError("chunk ids must stay below 2^32")
            if not chunks:
                return range(n, n)
            x16 = self.model.encode([c["text"] for c in chunks]).astype(np.float16)
            app = csr_append(self._stats, tokens)
            # the steps in the order remove_chunks gives them, for the same reason
            staged = self.dev.stage_append(app.term_ptr, app.postings, app.doc_len, app.stats.idf, app.stats.avgdl)
            prefilter = self.dev._prefilter_on
            self.dev.append_rows(torch.from_numpy(x16).to(self.dev.device), prefilter=False)
            self.dev.commit_postings(staged)
            app.commit_vocab()
            self._stats = app.stats
            self.chunks.extend(chunks)
            self.n_total = self.hi = len(self.chunks)
            self._x = self.dev.x
            if prefilter:
                self.dev.build_prefilter()
            return range(n, self.n_total)

    def remove_chunks(self, ids: Sequence[int]) -> np.ndarray:
        """Remove chunks (positions in ``self.chunks``) from the loaded index.  Returns the map from
        old to new ids (int64, -1 for a removed chunk): the remaining chunks keep their order and are
        numbered by rank.  Searches afterwards return exactly what an engine over a store rebuilt
        from the remaining chunks (with their current rows) returns.  Ids must be ints, in range and
        unique, and at least one chunk must remain; a rejected call raises and leaves the engine as
        it was.  To replace a chunk and keep its position, use ``replace_chunks``.  Not supported on a
        sharded engine (world > 1)."""
        if self.world > 1:
            raise NotImplementedError("remove_chunks on a sharded engine: rebuild the store instead")
        ids = list(ids)
        _check_id_types(ids)
        with self._lock:
            n = self.n_total
            ids_arr = _id_array(ids, n)
            if len(ids_arr) >= n:
                raise ValueError("removing every chunk: the BM25 statistics of an empty corpus are undefined")
            ids_map = np.arange(n, dtype=np.int64)
            if not len(ids_arr):
                return ids_map
            rem = csr_remove(self._stats, ids_arr, lambda d: tokenize(self.chunks[d]["text"]), self.dev.posting_docs)
            keep = np.ones(n, dtype=bool)
            keep[rem.removed] = False
            # every step that allocates or checks runs before the handle takes the new postings: the
            # compaction into new buffers (which validates the plan), then the in-place row move
            # through one bounded temporary; the int8 shadow is rebuilt last, over a consistent index
            staged = self.dev.compact_postings(rem)
            prefilter = self.dev._prefilter_on
            self.dev.remove_rows(keep, prefilter=False)
            self.dev.commit_postings(staged)
            rem.commit_vocab()
            self._stats = rem.stats
            self.chunks = [c for c, k in zip(self.chunks, keep.tolist()) if k]
            self.n_total = self.hi = len(self.chunks)
            self._x = self.dev.x
            ids_map[~keep] = -1
            ids_map[keep] = np.arange(self.n_total, dtype=np.int64)
            if prefilter:
                self.dev.build_prefilter()
            return ids_map

    def replace_chunks(self, ids: Sequence[int], chunks: Sequence[dict]) -> None:
        """Replace chunks in place: chunk ``ids[i]`` (its position in ``self.chunks``) becomes
        ``chunks[i]``, and every chunk keeps its position.  Searches afterwards return exactly what an
        engine over a store rebuilt from the edited chunk list (with these rows) returns, BM25
        vocabulary order and idf bits included.  Each new chunk is a dict with a str ``"text"``,
        embedded and stored as ``add_chunks`` does.  Ids must be ints, in range and unique, one per
        chunk, and the edit must leave the corpus some BM25 token; a rejected call raises and leaves
        the engine as it was.  Not supported on a sharded engine (world > 1)."""
        if self.world > 1:
            raise NotImplementedError("replace_chunks on a sharded engine: rebuild the store instead")
        ids, chunks = list(ids), list(chunks)
        _check_id_types(ids)
        if len(ids) != len(chunks):
            raise ValueError(f"{len(ids)} ids but {len(chunks)} chunks")
        tokens = _chunk_tokens(chunks)
        with self._lock:
            ids_arr = _id_array(ids, self.n_total)
            if not len(ids_arr):
                return
            x16 = self.model.encode([c["text"] for c in chunks]).astype(np.float16)
            rep = csr_replace(self._stats, ids_arr, tokens, lambda d: tokenize(self.chunks[d]["text"]),
                              self.dev.posting_docs)
            # the steps in the order remove_chunks gives them, for the same reason: the postings are
            # staged into new buffers (the kernel validates the plan), the rows overwritten in place,
            # then the handle takes the new postings; the int8 shadow is rebuilt last
            doc_len = self.dev.doc_len[:self.n_total].clone()
            doc_len[torch.from_numpy(rep.replaced).to(doc_len.device)] = torch.from_numpy(
                rep.doc_len.astype(np.int32)).to(doc_len.device)
            staged = self.dev.stage_replace(rep, doc_len)
            prefilter = self.dev._prefilter_on
            self.dev.replace_rows(ids_arr, torch.from_numpy(x16).to(self.dev.device), prefilter=False)
            self.dev.commit_postings(staged)
            rep.commit_vocab()
            self._stats = rep.stats
            for i, c in zip(ids_arr.tolist(), chunks):
                self.chunks[i] = c
            if prefilter:
                self.dev.build_prefilter()

    def save(self, store_dir: Optional[str] = None) -> Path:
        """Write the current index (added chunks included) as a store that ``RetrievalEngine`` and
        the reference load: to ``store_dir`` or the directory this engine was loaded from.  The
        files are written into a temporary sibling directory that replaces the target only when
        every file is complete."""
        if self.world > 1:
            raise NotImplementedError("save on a sharded engine: each rank holds only its rows")
        target = Path(store_dir) if store_dir is not None else self.store_dir
        target.parent.mkdir(parents=True, exist_ok=True)
        with self._lock:                                  # re-entrant: self.bm25 below takes it too
            tmp = Path(tempfile.mkdtemp(prefix=f".{target.name}.", dir=target.parent))
            os.chmod(tmp, 0o755)                          # mkdtemp's 0700 would follow the store
            old = None
            try:
                x = self._x.cpu().numpy().astype(np.float32)
                _store.save_store(tmp, self.chunks, x, self.bm25)
                if target.exists():
                    old = Path(tempfile.mkdtemp(prefix=f".{target.name}.old.", dir=target.parent))
                    os.rename(target, old / target.name)
                os.rename(tmp, target)
            except BaseException:
                if old is not None and (old / target.name).exists() and not target.exists():
                    os.rename(old / target.name, target)  # put the previous store back
                shutil.rmtree(tmp, ignore_errors=True)
                raise
            if old is not None:
                shutil.rmtree(old, ignore_errors=True)
        return target

    def close(self):
        if getattr(self, "world", 1) > 1 and self.rank == 0 and self.dev.h:
            import torch.distributed as dist
            dist.broadcast_object_list([("stop",)], src=0, group=self.group)
        if getattr(self, "world", 1) > 1 and self.dev.h:
            import torch.distributed as dist
            dist.barrier(group=self.group)                  # nobody unmaps while a peer may store
        self.dev.close()


def fanout_queries(query: str, user_context: str, key_entities: Sequence[str], category: str):
    """The orchestrator's concept expansion (orchestrator.py:38-56) as data: the search
    strings and their hybrid weights, ready for ``search_batch``."""
    queries = [query]
    if user_context == "victim_distress":
        offence = next((e for e in key_entities if e.lower() in ["robbery", "assault", "rape", "theft"]),
                       "crime")
        queries += [f"How to file FIR for {offence} BNSS procedure",
                    f"Victim compensation rights for {offence} NALSA scheme",
                    "Zero FIR registration procedure BNSS"]
    weights = [0.6 if category == "procedure" or "procedure" in q.lower() else 0.5 for q in queries]
    return queries, weights


def merge_fanout(result_lists: Sequence[List[dict]]) -> List[dict]:
    """orchestrator.py:54-62: concatenate in query order, first occurrence of each truthy
    ``canonical_header`` wins."""
    out, seen = [], set()
    for results in result_lists:
        for r in results:
            cid = r["chunk"].get("canonical_header")
            if cid and cid not in seen:
                out.append(r)
                seen.add(cid)
    return out


def create_vector_store(chunks_path: str = "legal_chunks.json", save_dir: str = "data/vector_store",
                        *, device: Optional[int] = None, model_dir: Optional[str] = None,
                        encoder_state_dict: Optional[Dict] = None, tokenizer=None,
                        batch_size: int = 1024, group=None):
    """Index build (create_vector_store.py:14-83): embed every chunk text on the GPU, build the
    BM25 statistics/postings, write the store.  Under ``torchrun`` the encode loop
    (create_vector_store.py:41-46) is data-parallel: rank g embeds the chunk range
    ``shard_range(N, g, G)``, the rows are gathered over NCCL and rank 0 writes the store."""
    chunks_path = Path(chunks_path)
    if not chunks_path.exists():
        print(f"Error: {chunks_path} not found. Run ingest_legal_docs.py first.")
        return
    with open(chunks_path, "r", encoding="utf-8") as f:
        chunks = json.load(f)
    if not chunks:
        print("No chunks to process.")
        return
    if encoder_state_dict is None:
        model_dir = _resolve_model_dir(model_dir)
        if model_dir is None:
            raise FileNotFoundError("all-MiniLM-L6-v2 weights not found: set EMBEDDING_MODEL_DIR")
    rank, world = _dist_state(group)
    if device is None:
        device = int(os.environ.get("LOCAL_RANK", "0")) if world > 1 else 0
    dev = DeviceIndex(device)
    try:
        enc = SentenceEncoder(dev, state_dict=encoder_state_dict, model_dir=model_dir, tokenizer=tokenizer)
        enc.require_tokenizer()
        texts = [c["text"] for c in chunks]
        lo, hi = shard_range(len(texts), rank, world)
        x = enc.encode(texts[lo:hi], batch_size=batch_size)   # unit float32 rows of this rank's range
        if world > 1:
            import torch.distributed as dist
            per = -(-len(texts) // world)
            mine = torch.zeros((per, x.shape[1]), dtype=torch.float32, device=dev.device)
            mine[:hi - lo] = torch.from_numpy(x).to(dev.device)
            every = torch.empty((world * per, x.shape[1]), dtype=torch.float32, device=dev.device)
            dist.all_gather_into_tensor(every, mine, group=group)
            x = every[:len(texts)].cpu().numpy()
        if rank == 0:
            bm25 = BM25Index.from_texts(texts)                 # text.lower().split()
            _store.save_store(save_dir, chunks, x, bm25)
        if world > 1:
            import torch.distributed as dist
            dist.barrier(group=group)
    finally:
        dev.close()
    if rank == 0:
        print(f"Vector store created: {save_dir}  ({len(chunks)} chunks, dim {x.shape[1]})")
    return save_dir
