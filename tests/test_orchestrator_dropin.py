"""The drop-in boundary, end to end on the host side: the shim ``src/retrieval/retrieval_engine.py``
and this package's ``RetrievalEngine``, called as the reference's ``src/retrieval/orchestrator.py``
calls them (``RetrievalEngine(store_dir)``, ``engine.search(q, k=k, hybrid_weight=w)``,
``engine.chunks``).  With ``LRX_REFERENCE_DIR`` pointing at a checkout of the reference project, its
UNMODIFIED ``orchestrator.py`` also runs over the shim (that file is not part of this repository, so
the test is skipped without it).

No GPU here, so the device boundary is replaced by an oracle-backed double (test infrastructure):
``DeviceIndex`` -> the CPU oracle of K2..K4, ``lrx_encode_host`` -> the fp32 oracle encoder.
Everything above it is the product's host code: the checkpoint loader (a synthetic
``model.safetensors`` + ``vocab.txt`` written here, found through EMBEDDING_MODEL_DIR), the
WordPiece tokenizer, the store reader, ``query.lower().split()`` -> term ids, the result dicts.
The results are compared with the oracle path restated call by call
(oracle/search.py fan-out + oracle/postprocess.py)."""
import copy
import importlib
import json
import os
import shutil
import sys
from collections import Counter
from pathlib import Path

import numpy as np
import pytest
import torch

from conftest import ROOT

REF_ORCH = (Path(os.environ["LRX_REFERENCE_DIR"]) / "src" / "retrieval" / "orchestrator.py"
            if os.environ.get("LRX_REFERENCE_DIR") else None)

STUB_CLASSIFIER = '''
from typing import List, Optional
from pydantic import BaseModel, Field

class QueryIntent(BaseModel):
    category: str
    sub_intent: Optional[str] = None
    key_entities: List[str] = Field(default_factory=list)
    user_context: str
    confidence: float

CANNED = {}

class QueryClassifier:
    def classify(self, query: str) -> QueryIntent:
        return QueryIntent(**CANNED[query])
'''

INTENTS = {
    "I was robbed at knife point, what should I do?":
        dict(category="procedure", sub_intent="report FIR", key_entities=["robbery", "BNSS"],
             user_context="victim_distress", confidence=0.9),
    "What is the punishment for murder?":
        dict(category="punishment", sub_intent=None, key_entities=["BNS"], user_context="informational",
             confidence=0.8),
    "Compensation for victims of acid attack":
        # (sub_intent must be a string here: with None the reference's own orchestrator.py:85 raises)
        dict(category="compensation", sub_intent="victim compensation claim", key_entities=["assault"],
             user_context="victim_distress", confidence=0.7),
}


class OracleDevice:
    """Stands where DeviceIndex stands; answers with the CPU oracle."""

    def __init__(self, device=0, rank=0, world=1):
        self.device = torch.device("cpu")
        self.rank, self.world, self.h = rank, world, True
        self.sd = None

    def set_corpus(self, x, id_base=0):
        self.x = x.numpy()
        assert id_base == 0

    def set_postings(self, term_ptr, postings, doc_len, idf, avgdl, k1=1.5, b=0.75):
        from oracle import bm25 as obm25
        self.csr = obm25.BM25OkapiCSR.from_postings(len(doc_len), doc_len, np.asarray(term_ptr).astype(np.int64),
                                                    postings[:, 0], postings[:, 1])
        np.testing.assert_array_equal(self.csr.idf, idf)
        assert self.csr.avgdl == avgdl
        self.postings = (np.asarray(term_ptr, dtype=np.uint64), np.asarray(postings, dtype=np.uint32),
                         np.asarray(doc_len, dtype=np.uint32))

    def read_postings(self):
        return self.postings

    def search_text_host(self, tok_ids, tok_lens, term_lists, k, weights, fusion):
        from oracle import encoder as oenc
        from oracle.search import OracleIndex
        q = oenc.encode_ids(self.sd, np.asarray(tok_ids), np.asarray(tok_lens)).astype(np.float16)
        res = OracleIndex(self.x, self.csr).search_batch_vec(q, term_lists, k, weights, fusion)
        B = len(term_lists)
        ids = np.full((B, k), -1, dtype=np.int64)
        out = [np.zeros((B, k)) for _ in range(3)]
        for b, rows in enumerate(res):
            for j, (i, s, sem, kw) in enumerate(rows):
                ids[b, j] = i
                out[0][b, j], out[1][b, j], out[2][b, j] = s, sem, kw
        return ids, out[0], out[1], out[2]

    def close(self):
        self.h = None


@pytest.fixture(scope="module")
def store_deployment(tmp_path_factory, legal_chunks):
    """A checkpoint directory and a vector store built from the reference's corpus."""
    from safetensors.numpy import save_file
    from legal_rag_engine_b200 import synth, store
    from legal_rag_engine_b200.bm25_index import BM25Index
    from legal_rag_engine_b200.tokenizer import WordPieceTokenizer, basic_tokenize
    from oracle import encoder as oenc
    root = tmp_path_factory.mktemp("deploy")
    chunks = [c for c in legal_chunks if len(c["text"]) < 700][:160] + \
             [c for c in legal_chunks if "FIR" in c["text"] and len(c["text"]) < 1500][:60]
    seen, uniq = set(), []
    for c in chunks:                                   # keep list order, drop repeats of the same object
        if id(c) not in seen:
            seen.add(id(c))
            uniq.append(c)
    chunks = uniq
    texts = [c["text"] for c in chunks]
    # ---- a checkpoint directory as sentence-transformers lays it out: model.safetensors + vocab.txt
    cnt = Counter(t for x in texts for t in basic_tokenize(x))
    vocab = ["[PAD]"] + [f"[unused{i}]" for i in range(99)] + ["[UNK]", "[CLS]", "[SEP]", "[MASK]"]
    chars = sorted({ch for w in cnt for ch in w})
    vocab += chars + ["##" + c for c in chars] + [w for w, _ in cnt.most_common(1500) if len(w) > 1]
    vocab = list(dict.fromkeys(vocab))
    model_dir = root / "model"
    model_dir.mkdir()
    (model_dir / "vocab.txt").write_text("\n".join(vocab) + "\n", encoding="utf-8")
    sd = synth.bert_state_dict(7, 0.05, vocab=len(vocab), ln_jitter=0.1)
    save_file({k: np.ascontiguousarray(v) for k, v in sd.items()}, str(model_dir / "model.safetensors"))
    # ---- the store, as create_vector_store writes it (embeddings from the fp32 oracle encoder)
    tok = WordPieceTokenizer.from_file(model_dir / "vocab.txt")
    enc = [tok.encode(t, 256) for t in texts]
    x = np.zeros((len(texts), 384), dtype=np.float32)
    for s in range(0, len(texts), 16):
        idx = list(range(s, min(len(texts), s + 16)))
        S = max(len(enc[i]) for i in idx)
        ids = np.zeros((len(idx), S), dtype=np.int32)
        lens = np.array([len(enc[i]) for i in idx], dtype=np.int32)
        for r, i in enumerate(idx):
            ids[r, :len(enc[i])] = enc[i]
        x[idx] = oenc.encode_ids(sd, ids, lens)
    vs = root / "data" / "vector_store"
    store.save_store(vs, chunks, x, BM25Index.from_texts(texts))
    return root, vs, model_dir, sd, chunks


@pytest.fixture(scope="module")
def deployment(store_deployment):
    """`store_deployment` + the reference tree's package with ONE file replaced."""
    if REF_ORCH is None or not REF_ORCH.exists():
        pytest.skip("set LRX_REFERENCE_DIR to a checkout of the reference project")
    root, vs, model_dir, sd, chunks = store_deployment
    pkg = root / "src" / "retrieval"
    pkg.mkdir(parents=True)
    (root / "src" / "__init__.py").write_text("")
    (pkg / "__init__.py").write_text("")
    shutil.copy(REF_ORCH, pkg / "orchestrator.py")                                   # unmodified
    shutil.copy(ROOT / "src" / "retrieval" / "retrieval_engine.py", pkg / "retrieval_engine.py")
    (pkg / "classifier.py").write_text(STUB_CLASSIFIER)
    return root, vs, model_dir, sd, chunks


def _oracle_device(monkeypatch, model_dir):
    """The device boundary -> the oracle double; the checkpoint is found through EMBEDDING_MODEL_DIR."""
    from legal_rag_engine_b200 import encoder as lenc
    from legal_rag_engine_b200 import engine as leng
    from oracle import encoder as oenc

    def fake_upload(dev, state_dict):
        dev.sd = {k: np.asarray(v) for k, v in lenc._strip(state_dict).items()}
        dev.vocab_size = int(dev.sd["embeddings.word_embeddings.weight"].shape[0])
    monkeypatch.setattr(leng, "DeviceIndex", OracleDevice)
    monkeypatch.setattr(lenc, "upload_weights", fake_upload)
    monkeypatch.setattr(lenc.SentenceEncoder, "encode_ids",
                        lambda self, ids, lens: oenc.encode_ids(self.dev.sd, np.asarray(ids), np.asarray(lens)))
    monkeypatch.setenv("EMBEDDING_MODEL_DIR", str(model_dir))


def test_shim_engine_answers_the_orchestrator_calls_as_the_oracle(store_deployment, monkeypatch):
    """What orchestrator.py:10,57 asks of the engine, through the shim: ``RetrievalEngine(store_dir)``
    (positional), then ``search(q, k=5, hybrid_weight=w)`` for every fan-out string; the result
    dicts carry the engine's own ``chunks`` objects and the oracle's scores."""
    root, vs, model_dir, sd, chunks = store_deployment
    from oracle import search as osearch
    _oracle_device(monkeypatch, model_dir)
    shim = importlib.import_module("src.retrieval.retrieval_engine")
    assert Path(shim.__file__).resolve() == ROOT / "src" / "retrieval" / "retrieval_engine.py"
    eng = shim.RetrievalEngine(str(vs))
    try:
        assert type(eng).__module__ == "legal_rag_engine_b200.engine" and len(eng.chunks) == len(chunks)
        assert type(eng.model.tokenizer).__name__ == "WordPieceTokenizer"     # the checkpoint's vocab.txt
        np.testing.assert_array_equal(
            eng.dev.sd["encoder.layer.3.output.dense.weight"], sd["encoder.layer.3.output.dense.weight"])
        csr, x = eng.dev.csr, eng.dev.x
        csr.vocab = eng.bm25.vocab
        oidx = osearch.OracleIndex(x, csr)
        n_sub = 0
        for query, intent in INTENTS.items():
            qs, ws = osearch.fanout_queries(query, intent["user_context"], intent["key_entities"],
                                            intent["category"])
            for q, w in zip(qs, ws):
                got = eng.search(q, k=5, hybrid_weight=w)
                qh = eng.encode([q]).astype(np.float16)[0]
                want = oidx.search_vec(qh, csr.term_ids(q.lower().split()), 5, w, "linear")
                assert 1 <= len(got) <= 5 and len(got) == len(want), q
                for r, (i, s, sem, kw) in zip(got, want):
                    assert r["chunk"] is eng.chunks[i], q
                    assert (r["score"], r["semantic"], r["keyword"]) == (s, sem, kw), q
                n_sub += 1
        assert n_sub == 9                                 # two fan-outs of 4 strings and one single query
    finally:
        eng.close()


def test_reference_orchestrator_runs_unchanged_over_the_engine(deployment, monkeypatch):
    root, vs, model_dir, sd, chunks = deployment
    from oracle import postprocess as opost
    from oracle import search as osearch
    _oracle_device(monkeypatch, model_dir)
    saved = {k: v for k, v in sys.modules.items() if k == "src" or k.startswith("src.")}
    for k in saved:
        del sys.modules[k]
    monkeypatch.syspath_prepend(str(root))
    try:
        orch_mod = importlib.import_module("src.retrieval.orchestrator")
        assert Path(orch_mod.__file__).read_bytes() == REF_ORCH.read_bytes()
        importlib.import_module("src.retrieval.classifier").CANNED.update(INTENTS)
        orch = orch_mod.LegalOrchestrator(str(vs))                 # RetrievalEngine(store_dir), positional
        eng = orch.engine
        assert type(eng).__module__ == "legal_rag_engine_b200.engine" and len(eng.chunks) == len(chunks)
        assert type(eng.model.tokenizer).__name__ == "WordPieceTokenizer"     # the checkpoint's vocab.txt
        np.testing.assert_array_equal(
            eng.dev.sd["encoder.layer.3.output.dense.weight"], sd["encoder.layer.3.output.dense.weight"])
        # ---- expected: the oracle path, call by call
        csr, x = eng.dev.csr, eng.dev.x
        csr.vocab = eng.bm25.vocab
        oidx = osearch.OracleIndex(x, csr)
        lookup = opost.section_lookup(chunks)
        for query, intent in INTENTS.items():
            got = orch.orchestrate(query, k=5)
            assert got["intent"]["category"] == intent["category"]
            qs, ws = osearch.fanout_queries(query, intent["user_context"], intent["key_entities"],
                                            intent["category"])
            assert len(qs) == (4 if intent["user_context"] == "victim_distress" else 1)
            lists = []
            for q, w in zip(qs, ws):
                qh = eng.encode([q]).astype(np.float16)[0]
                rows = oidx.search_vec(qh, csr.term_ids(q.lower().split()), 5, w, "linear")
                lists.append([{"chunk": copy.deepcopy(chunks[i]), "score": s, "semantic": sem, "keyword": kw}
                              for i, s, sem, kw in rows])
            flat, seen = [], set()
            for rs in lists:                                        # orchestrator.py:54-62
                for r in rs:
                    cid = r["chunk"].get("canonical_header")
                    if cid and cid not in seen:
                        flat.append(r)
                        seen.add(cid)
            want = opost.expand_results(opost.prioritize_results(flat, dict(intent))[:5], lookup)
            key = lambda rs: [(r["chunk"]["canonical_header"], r["score"], r["semantic"], r["keyword"],
                               r.get("parent_context")) for r in rs]
            assert key(got["results"]) == key(want)
            assert 1 <= len(got["results"]) <= 5
            assert all(r["chunk"] is eng.chunks[eng.chunks.index(r["chunk"])] for r in got["results"])
    finally:
        for k in [k for k in sys.modules if k == "src" or k.startswith("src.")]:
            del sys.modules[k]
        sys.modules.update(saved)


def test_checkpoint_without_vocab_is_an_error(tmp_path):
    """A model directory with weights but no vocab.txt must not fall back to the hash tokenizer."""
    from legal_rag_engine_b200.tokenizer import load_tokenizer
    (tmp_path / "model.safetensors").write_bytes(b"")
    with pytest.raises(FileNotFoundError, match="vocab.txt"):
        load_tokenizer(str(tmp_path))
    with pytest.raises(FileNotFoundError):
        load_tokenizer(None)
    (tmp_path / "0_Transformer").mkdir()
    (tmp_path / "0_Transformer" / "vocab.txt").write_text("[PAD]\n[UNK]\n[CLS]\n[SEP]\nzero\n", encoding="utf-8")
    tok = load_tokenizer(str(tmp_path))
    assert tok.encode("zero xyz") == [2, 4, 1, 3]
