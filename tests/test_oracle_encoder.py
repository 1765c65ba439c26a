"""The encoder oracle (oracle/encoder.py) is pinned against HuggingFace BertModel outputs
(tests/golden/encoder_golden.npz, made by tests/golden/make_encoder_golden.py)."""
import numpy as np
import pytest

from legal_rag_engine_b200 import synth
from legal_rag_engine_b200.tokenizer import HashTokenizer, WordPieceTokenizer, basic_tokenize
from oracle import encoder as oenc

from conftest import GOLDEN


@pytest.mark.parametrize("case", [0, 1])
def test_bert_restatement_matches_huggingface_golden(case):
    g = np.load(GOLDEN / "encoder_golden.npz")
    wseed, std, jit, b, s, tseed = g[f"case_{case}"]
    sd = synth.bert_state_dict(int(wseed), float(std), ln_jitter=float(jit))
    ids, lens = synth.token_batch(int(b), int(s), int(tseed))
    mask = (np.arange(int(s))[None] < lens[:, None]).astype(np.int64)
    hid = oenc.bert_hidden(sd, ids, mask).numpy()
    want = g[f"hidden_{case}"]
    valid = mask.astype(bool)
    # padded positions are unspecified (HF computes them, nobody reads them)
    np.testing.assert_allclose(hid[valid], want[valid], rtol=0, atol=2e-5)


def test_pool_normalize_unit_and_masked():
    rng = np.random.default_rng(0)
    import torch
    h = torch.from_numpy(rng.standard_normal((3, 9, 384)).astype(np.float32))
    lens = np.array([9, 4, 2])
    mask = (np.arange(9)[None] < lens[:, None]).astype(np.int64)
    e = oenc.pool_normalize(h, mask)
    np.testing.assert_allclose(np.linalg.norm(e, axis=1), 1.0, atol=1e-6)
    h2 = h.clone()
    h2[1, 4:] = 1e6                       # padded positions must not matter
    np.testing.assert_array_equal(oenc.pool_normalize(h2, mask)[1], e[1])
    want = h[2, :2].mean(0).numpy()
    np.testing.assert_allclose(e[2], want / np.linalg.norm(want), atol=1e-6)


@pytest.mark.parametrize("case", [0, 1])
def test_float64_oracle_agrees_with_float32_on_golden_inputs(case):
    """The float64 restatement (the reference of the encoder kernel tests) is the same function as
    the float32 one the golden file pins: embeddings within float32 rounding of each other, unit
    norm to double precision, and the len = 0 row stays the zero vector in both."""
    import torch
    g = np.load(GOLDEN / "encoder_golden.npz")
    wseed, std, jit, b, s, tseed = g[f"case_{case}"]
    sd = synth.bert_state_dict(int(wseed), float(std), ln_jitter=float(jit))
    ids, lens = synth.token_batch(int(b), int(s), int(tseed))
    ids = np.concatenate([ids, ids[:1]])
    lens = np.concatenate([lens, [0]])                     # a fully masked row
    e32 = oenc.encode_ids(sd, ids, lens)
    e64 = oenc.encode_ids(sd, ids, lens, dtype=torch.float64)
    assert e32.dtype == np.float32 and e64.dtype == np.float64
    np.testing.assert_allclose(e64[:-1], e32[:-1].astype(np.float64), rtol=0, atol=1e-5)
    np.testing.assert_allclose(np.linalg.norm(e64[:-1], axis=1), 1.0, rtol=0, atol=1e-12)
    assert not e32[-1].any() and not e64[-1].any()
    mask = (np.arange(int(s))[None] < lens[:, None]).astype(np.int64)
    h64 = oenc.bert_hidden(sd, ids, mask, dtype=torch.float64)
    assert h64.dtype == torch.float64
    valid = mask.astype(bool)
    np.testing.assert_allclose(h64.numpy()[valid], g[f"hidden_{case}"][valid[:-1]], rtol=0, atol=2e-5)


def test_tokenizers():
    assert basic_tokenize("What is the procedure for Zero FIR?") == \
        ["what", "is", "the", "procedure", "for", "zero", "fir", "?"]
    assert basic_tokenize("Café  naïve\tBNSS-173(1)") == ["cafe", "naive", "bnss", "-", "173", "(", "1", ")"]
    vocab = {w: i for i, w in enumerate(["[PAD]", "[UNK]", "[CLS]", "[SEP]", "zero", "fir", "?", "un",
                                         "##aff", "##able", "what"])}
    tok = WordPieceTokenizer(vocab)
    assert tok.encode("What zero FIR? unaffable xyz") == [2, 10, 4, 5, 6, 7, 8, 9, 1, 3]
    assert len(tok.encode("zero " * 500, 256)) == 256
    h = HashTokenizer(30522)
    ids = h.encode("Zero FIR registration procedure BNSS")
    assert ids[0] == 101 and ids[-1] == 102 and len(ids) == 7
    assert all(1000 <= i < 30522 for i in ids[1:-1])
    assert ids == h.encode("zero fir   registration procedure bnss")


def test_wordpiece_pinned_to_hf_tokenizers_on_reference_corpus(legal_texts, reference_queries):
    """The reference tokenises with the BertTokenizer of all-MiniLM-L6-v2 (HF `tokenizers`
    underneath).  Without its vocab.txt the pin is on the ALGORITHM: over a WordPiece vocabulary
    built from the reference's own corpus, WordPieceTokenizer must give the ids of
    tokenizers.BertWordPieceTokenizer(lowercase=True) for every chunk and query."""
    tokenizers = pytest.importorskip("tokenizers")
    from collections import Counter
    cnt = Counter(t for x in legal_texts for t in basic_tokenize(x))
    vocab = ["[PAD]"] + [f"[unused{i}]" for i in range(99)] + ["[UNK]", "[CLS]", "[SEP]", "[MASK]"]
    chars = sorted({ch for w in cnt for ch in w})
    vocab += chars + ["##" + c for c in chars]
    vocab += [w for w, _ in cnt.most_common(4000) if len(w) > 1]
    vocab += ["##" + w[2:] for w, _ in cnt.most_common(600) if len(w) > 4]      # some real suffix pieces
    v = {w: i for i, w in enumerate(dict.fromkeys(vocab))}
    tok = WordPieceTokenizer(v)
    hf = tokenizers.BertWordPieceTokenizer(dict(v), lowercase=True)
    hf.enable_truncation(256)
    texts = list(legal_texts) + list(reference_queries) + ["Caf\u00e9 na\u00efve \u2014 \u00a7 173(1) \u201cZero FIR\u201d \u4e2d\u6587"]
    want = [e.ids for e in hf.encode_batch(texts)]
    got = [tok.encode(t, 256) for t in texts]
    assert got == want
    assert tok.encode_batch(texts, 256) == want               # the batch path is the library itself
