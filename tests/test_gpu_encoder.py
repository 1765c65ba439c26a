"""K1 on the GPU: the tcgen05 GEMM stage against torch float64 on the same fp16 operands, and
the whole encoder (lrx_encode / lrx_encode_host through the C ABI) against the float32 oracle
(oracle/encoder.py, pinned to HuggingFace BertModel).  Tolerance from BASELINE.json north_star:
embeddings cosine >= 0.9999 of fp32."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

COS_MIN = 0.9999


@pytest.fixture(scope="module")
def dev():
    from legal_rag_engine_b200.device_index import DeviceIndex
    d = DeviceIndex(0)
    yield d
    d.close()


def _rand16(shape, seed, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(shape, generator=g) * scale).to(torch.float16).cuda()


@pytest.mark.parametrize("M,N,K", [(1, 128, 64), (100, 128, 384), (128, 384, 384), (300, 1152, 384),
                                   (257, 384, 1536), (1000, 1536, 384)])
def test_gemm_raw_accumulators(dev, M, N, K):
    a, w = _rand16((M, K), 1), _rand16((N, K), 2, 0.1)
    got = dev.gemm_f16(a, w, epi=3)
    want = a.double() @ w.double().T
    # fp16 x fp16 products are exact in fp32; the error is the fp32 accumulation order
    tol = 4e-6 * float((a.double().abs() @ w.double().abs().T).max())
    assert float((got.double() - want).abs().max()) <= tol


@pytest.mark.parametrize("M", [5, 129, 700])
def test_gemm_bias_and_gelu(dev, M):
    a, w = _rand16((M, 384), 3), _rand16((1536, 384), 4, 0.1)
    bias = torch.randn(1536, generator=torch.Generator().manual_seed(5)).cuda()
    ref = a.float() @ w.float().T + bias
    got0 = dev.gemm_f16(a, w, epi=0, bias=bias)
    got1 = dev.gemm_f16(a, w, epi=1, bias=bias)
    torch.testing.assert_close(got0.float(), ref, rtol=2e-3, atol=2e-3)
    torch.testing.assert_close(got1.float(), torch.nn.functional.gelu(ref), rtol=2e-3, atol=2e-3)


@pytest.mark.parametrize("M,K", [(7, 384), (128, 384), (333, 1536)])
def test_gemm_residual_layernorm(dev, M, K):
    a, w = _rand16((M, K), 6), _rand16((384, K), 7, 0.1)
    g = torch.Generator().manual_seed(8)
    bias, gamma, beta = (torch.randn(384, generator=g).cuda() for _ in range(3))
    res = _rand16((M, 384), 9)
    got = dev.gemm_f16(a, w, epi=2, bias=bias, residual=res, gamma=gamma, beta=beta, eps=1e-12)
    pre = a.float() @ w.float().T + bias + res.float()
    want = torch.nn.functional.layer_norm(pre, (384,), gamma, beta, 1e-12)
    torch.testing.assert_close(got.float(), want, rtol=3e-3, atol=3e-3)


def _cos(a, b):
    return (a * b).sum(1) / (np.linalg.norm(a, axis=1) * np.linalg.norm(b, axis=1))


@pytest.mark.parametrize("wseed,std,jit,B,S,full", [
    (42, 0.02, 0.0, 3, 24, False), (43, 0.06, 0.2, 4, 40, False), (44, 0.05, 0.1, 2, 128, True),
    (45, 0.05, 0.1, 5, 256, False), (46, 0.04, 0.1, 70, 128, False), (47, 0.05, 0.1, 1, 7, True),
    # query-sized batches (<= 128 tokens, S <= 64): the single-launch cluster kernel
    (48, 0.05, 0.1, 4, 32, False), (49, 0.05, 0.1, 2, 64, True), (50, 0.06, 0.2, 8, 16, False),
    (51, 0.05, 0.1, 1, 64, False), (52, 0.05, 0.1, 5, 25, False), (53, 0.05, 0.1, 16, 8, True)])
def test_encoder_matches_fp32_oracle(dev, wseed, std, jit, B, S, full):
    from legal_rag_engine_b200 import synth
    from legal_rag_engine_b200.encoder import SentenceEncoder
    from oracle import encoder as oenc
    sd = synth.bert_state_dict(wseed, std, ln_jitter=jit)
    enc = SentenceEncoder(dev, state_dict=sd)
    ids, lens = synth.token_batch(B, S, seed=wseed + 100, full=full)
    want = oenc.encode_ids(sd, ids, lens)
    got = enc.encode_ids(ids, lens)                       # host form (lrx_encode_host)
    cos = _cos(got.astype(np.float64), want.astype(np.float64))
    assert cos.min() >= COS_MIN, cos
    np.testing.assert_allclose(np.linalg.norm(got, axis=1), 1.0, atol=1e-5)
    # device form: same numbers, plus the fp16 copy that feeds the dense scan
    o32, o16 = enc.encode_ids_device(torch.from_numpy(ids).cuda(), torch.from_numpy(lens).cuda())
    np.testing.assert_array_equal(o32.cpu().numpy(), got)
    np.testing.assert_array_equal(o16.cpu().numpy(), got.astype(np.float16))


def test_encoder_padding_is_inert(dev):
    """Content of the padded positions and the padded width S must not change a row."""
    from legal_rag_engine_b200 import synth
    from legal_rag_engine_b200.encoder import SentenceEncoder
    sd = synth.bert_state_dict(50, 0.05, ln_jitter=0.1)
    enc = SentenceEncoder(dev, state_dict=sd)
    ids, lens = synth.token_batch(6, 48, seed=3)
    a = enc.encode_ids(ids, lens)
    ids2 = ids.copy()
    for i, n in enumerate(lens):
        ids2[i, n:] = 4242
    np.testing.assert_array_equal(enc.encode_ids(ids2, lens), a)
    wide = np.zeros((6, 80), dtype=np.int32)
    wide[:, :48] = ids
    b = enc.encode_ids(wide, lens)
    assert _cos(a.astype(np.float64), b.astype(np.float64)).min() > 0.999999


def test_small_batch_kernel_agrees_with_the_gemm_chain(dev):
    """The same query batch through the one-launch cluster kernel and, padded to 80 tokens (S > 64),
    through the tcgen05 GEMM chain: same embeddings to fp16 rounding noise; padding inert on the
    small path."""
    from legal_rag_engine_b200 import synth
    from legal_rag_engine_b200.encoder import SentenceEncoder
    sd = synth.bert_state_dict(54, 0.05, ln_jitter=0.1)
    enc = SentenceEncoder(dev, state_dict=sd)
    ids, lens = synth.token_batch(4, 30, seed=9)
    small = enc.encode_ids(ids, lens)
    wide80 = np.zeros((4, 80), dtype=np.int32)
    wide80[:, :30] = ids
    chain = enc.encode_ids(wide80, lens)
    assert _cos(small.astype(np.float64), chain.astype(np.float64)).min() > 0.99999
    ids2 = ids.copy()
    for i, n in enumerate(lens):
        ids2[i, n:] = 777
    np.testing.assert_array_equal(enc.encode_ids(ids2, lens), small)
    wide = np.zeros((2, 64), dtype=np.int32)
    wide[:, :30] = ids[:2]
    assert _cos(enc.encode_ids(wide, lens[:2]).astype(np.float64), small[:2].astype(np.float64)).min() > 0.999999


def test_query_encoder_is_batch_invariant(dev):
    """A query's embedding must not depend on what it was batched with, nor on the padded length of
    the batch (the serving front coalesces concurrent requests): bit-equal alone, inside a batch
    of 32, and padded to 48 tokens (the kernel's 64-row variant instead of the 32-row one)."""
    from legal_rag_engine_b200 import synth
    from legal_rag_engine_b200.encoder import SentenceEncoder
    sd = synth.bert_state_dict(55, 0.05, ln_jitter=0.1)
    enc = SentenceEncoder(dev, state_dict=sd)
    ids, lens = synth.token_batch(32, 30, seed=11)
    full = enc.encode_ids(ids, lens)                 # 32 sequences: 64-row groups, two per group
    for i in (0, 5, 31):
        np.testing.assert_array_equal(enc.encode_ids(ids[i:i + 1], lens[i:i + 1])[0], full[i])
    np.testing.assert_array_equal(enc.encode_ids(ids[3:11], lens[3:11]), full[3:11])
    wide = np.zeros((32, 48), dtype=np.int32)
    wide[:, :30] = ids
    np.testing.assert_array_equal(enc.encode_ids(wide, lens), full)
    tight = ids[:, :int(lens.max())]
    np.testing.assert_array_equal(enc.encode_ids(np.ascontiguousarray(tight), lens), full)


def test_encode_texts_batches_and_order(dev):
    from legal_rag_engine_b200 import synth
    from legal_rag_engine_b200.encoder import SentenceEncoder
    sd = synth.bert_state_dict(51, 0.05)
    from legal_rag_engine_b200.tokenizer import HashTokenizer
    enc = SentenceEncoder(dev, state_dict=sd, tokenizer=HashTokenizer(30522))
    texts = ["zero fir registration procedure bnss", "what is the punishment for murder?",
             "a", "compensation for victims of acid attack " * 40]
    all_at_once = enc.encode(texts)
    one_by_one = np.concatenate([enc.encode([t]) for t in texts])
    assert _cos(all_at_once.astype(np.float64), one_by_one.astype(np.float64)).min() > 0.99999
    assert all_at_once.shape == (4, 384)
