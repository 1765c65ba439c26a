"""K1 on the index-build path, against float64.

* GEMM launch plans at build sizes (lrx_gemm_f16): every production shape at row counts that reach
  the clustered / A-resident plans, padded cluster row blocks and a second persistent round, with
  error bounds derived per epilogue; rows bit-identical whatever tile they land in; no byte written
  outside the output.
* The attention kernel alone (lrx_debug_attention) at every length class up to 512, against float64
  softmax(Q K^T / sqrt(32) + mask) V, with poisoned padding and large logits.
* The whole encoder at long, multi-chunk batches and over the full reference-corpus build, against
  the float64 oracle (oracle/encoder.py with dtype=torch.float64 on the GPU).
* Batch invariance of the GEMM chain: a sequence's embedding is bit-identical alone, in any batch,
  at any padded width, through both entry points, and after the workspace has grown.

The CPU tests at the top restate the launch-plan choices (tc_gemm.cu gemm_plan / gemm_box_rows_w,
encoder.cu small_path) and check that every GPU case below reaches the plan it is named for; they
run without a GPU.  GPU tests carry the gpu mark one by one and derive every plan threshold from the
device's SM count.
"""
import ctypes as C
import json
import math

import numpy as np
import pytest
import torch

gpu = pytest.mark.gpu

COS_MIN = 0.9999                 # BASELINE.json north star
U32 = 2.0 ** -24                 # unit roundoff of float32
KCHUNK_TOKENS = 148 * 128        # encoder.cu kChunkTokens: tokens per activation chunk (a constant, not the SM count)


# ------------------------------------------------------------------ plan restatements (CPU)
def gemm_plan(sms, M, N, K, epi):
    """tc_gemm.cu gemm_plan: (bn, ares, cs)."""
    bn = 384 if epi == 2 else (192 if N % 192 == 0 else (256 if N % 256 == 0 else 128))
    m_tiles = (M + 127) // 128
    big = m_tiles >= sms // 2
    ares = K == 384 and (big or N // bn == 1)
    cs = 2 if big and (ares or N // bn == 1) else 1
    return bn, ares, cs


def gemm_box_rows_w(sms, M, N, K, epi):
    bn, _, cs = gemm_plan(sms, M, N, K, epi)
    return bn // cs if cs > 1 else (128 if bn > 256 else bn)


def gemm_geometry(sms, M, N, K, epi):
    """tc_gemm.cu launch_cfg: (row blocks after cluster padding, work units, grid, persistent rounds)."""
    bn, ares, cs = gemm_plan(sms, M, N, K, epi)
    m_tiles = (M + 127) // 128
    if cs > 1:
        m_tiles = (m_tiles + cs - 1) // cs * cs
    units = m_tiles if ares else m_tiles * (N // bn)
    grid = min(units, sms)
    if cs > 1:
        grid = grid // cs * cs
    return m_tiles, units, grid, -(-units // grid)


def small_path(B, S):
    """encoder.cu small_path: 0 GEMM chain, 2 / 4 cluster kernel with 32- / 64-row groups."""
    if S > 64:
        return 0
    if S <= 32 and -(-B // (32 // S)) <= 14:
        return 2
    return 4 if -(-B // (64 // S)) <= 64 else 0


SHAPES = [(1152, 384, 0), (1536, 384, 1), (384, 384, 2), (384, 1536, 2),   # QKV, FFN up, out proj, FFN down
          (1152, 384, 3), (1536, 1536, 3)]
PRODUCTION = SHAPES[:4]
SMALL_PLAN = {(1152, 384, 0): (192, False, 1), (1536, 384, 1): (192, False, 1), (384, 384, 2): (384, True, 1),
              (384, 1536, 2): (384, False, 1), (1152, 384, 3): (192, False, 1), (1536, 1536, 3): (192, False, 1)}
BIG_PLAN = {(1152, 384, 0): (192, True, 2), (1536, 384, 1): (192, True, 2), (384, 384, 2): (384, True, 2),
            (384, 1536, 2): (384, False, 2), (1152, 384, 3): (192, True, 2),
            (1536, 1536, 3): (192, False, 1)}     # the big plan without clusters: 8 n-blocks, K = 1536
ROW_NAMES = ["m1", "m127", "m129", "below_big", "at_big", "odd_tiles", "one_wave", "second_round", "three_waves"]


def row_count(name, sms):
    half = sms // 2
    odd = half + 1 if (half + 1) % 2 else half + 2          # smallest odd tile count past the threshold
    return {"m1": 1, "m127": 127, "m129": 129,
            "below_big": (half - 1) * 128,                   # half - 1 row tiles
            "at_big": (half - 1) * 128 + 1,                  # half row tiles, the last with one row
            "odd_tiles": (odd - 1) * 128 + 37,               # odd tile count: clusters pad a row block
            "one_wave": sms * 128,
            "second_round": sms * 128 + 1,                   # one tile (padded pair) past the first wave
            "three_waves": 3 * sms * 128 + 77}[name]


def expected_plan(shape, name):
    return SMALL_PLAN[shape] if name in ("m1", "m127", "m129", "below_big") else BIG_PLAN[shape]


@pytest.mark.parametrize("sms", [148, 132])
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "n%d_k%d_epi%d" % s)
@pytest.mark.parametrize("name", ROW_NAMES)
def test_gemm_case_reaches_its_plan(sms, shape, name):
    N, K, epi = shape
    M = row_count(name, sms)
    plan = gemm_plan(sms, M, N, K, epi)
    assert plan == expected_plan(shape, name), (M, plan)
    m_tiles, units, grid, rounds = gemm_geometry(sms, M, N, K, epi)
    real_tiles = (M + 127) // 128
    if name == "below_big":
        assert real_tiles == sms // 2 - 1
    if name == "at_big":
        assert real_tiles == sms // 2
    if plan[2] == 2:
        assert m_tiles % 2 == 0 and grid % 2 == 0
        if name in ("odd_tiles", "second_round", "three_waves"):
            assert real_tiles % 2 == 1 and m_tiles == real_tiles + 1        # a padded row block
    if name == "one_wave" and plan[1]:
        assert units == sms and rounds == 1
    if name in ("second_round", "three_waves"):
        assert rounds >= 2                                                   # persistent loop goes round
    if name == "three_waves":
        assert rounds >= 3 and units % grid != 0                             # ragged last round
    # the W tensor map the caller builds has the box the launcher's plan expects
    box = gemm_box_rows_w(sms, M, N, K, epi)
    assert box == (plan[0] // 2 if plan[2] == 2 else (128 if plan[0] > 256 else plan[0]))


@pytest.mark.parametrize("sms", [148, 132])
def test_encoder_w_map_set_matches_the_plan_of_every_chunk(sms):
    """encoder.cu builds two W tensor-map sets (at 128 rows and at kChunkTokens rows) and picks one
    per chunk by its row-tile count; each must give the box the launcher's plan uses for that chunk."""
    for T in list(range(1, 40 * 128, 7)) + list(range(sms * 64 - 300, KCHUNK_TOKENS + 1, 13)):
        pl = ((T + 127) // 128) >= sms // 2
        Mp = KCHUNK_TOKENS if pl else 128
        for N, K, epi in PRODUCTION:
            assert gemm_box_rows_w(sms, Mp, N, K, epi) == gemm_box_rows_w(sms, T, N, K, epi), (T, N, K, epi)


SMALL_PATH_CASES = [(32, 14, 2), (32, 15, 4), (64, 64, 4), (64, 65, 0)]


@pytest.mark.parametrize("S,B,path", SMALL_PATH_CASES)
def test_small_path_boundaries(S, B, path):
    assert small_path(B, S) == path


def _long_batch(S, sms):
    """B so that the call spans more than one activation chunk, the first chunk on the big GEMM plans
    and the last below the big threshold (both W map sets in one call)."""
    spc = KCHUNK_TOKENS // S
    B = spc + max(1, spc // 12)
    last = B - spc * (B // spc)
    return B, spc, last


LONG_S = [65, 100, 257, 300, 384, 511, 512]


@pytest.mark.parametrize("sms", [148, 132])
@pytest.mark.parametrize("S", LONG_S)
def test_long_batches_use_both_plan_sets(sms, S):
    B, spc, last = _long_batch(S, sms)
    assert small_path(B, S) == 0 and B > spc and last > 0
    assert (spc * S + 127) // 128 >= sms // 2            # full chunks: clustered plans
    assert (last * S + 127) // 128 < sms // 2            # tail chunk: the small-M plans


# ------------------------------------------------------------------------- GPU fixtures
@pytest.fixture(scope="module")
def dev():
    from legal_rag_engine_b200.device_index import DeviceIndex
    d = DeviceIndex(0)
    yield d
    d.close()


@pytest.fixture(scope="module")
def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _rand16(shape, seed, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(shape, generator=g) * scale).to(torch.float16).cuda()


def _randf(n, seed, scale=1.0, shift=0.0):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(n, generator=g) * scale + shift).cuda()


def _gemm_into(dev, a, w, epi, out, bias=None, residual=None, gamma=None, beta=None, eps=1e-12):
    M, K = a.shape
    N = w.shape[0]
    dev._ck(dev.lib.lrx_gemm_f16(dev.h, _p(a), _p(w), M, N, K, epi, _p(bias), _p(residual), _p(gamma),
                                 _p(beta), float(eps), _p(out)))
    torch.cuda.synchronize()


def _same_bits(a, b):
    assert a.shape == b.shape and a.dtype == b.dtype
    it = torch.int16 if a.element_size() == 2 else torch.int32
    return torch.equal(a.contiguous().view(it), b.contiguous().view(it))


def half_ulp16(x):
    """Half an fp16 ulp at magnitude x (float64 tensor, x >= 0): 2^(e - 11) for x in [2^e, 2^(e+1)),
    2^-25 in the subnormal range."""
    e = torch.floor(torch.log2(torch.clamp(x, min=2.0 ** -14)))
    return torch.exp2(e - 11)


# ------------------------------------------------------------------------------ §2 GEMM
# Operands: A ~ N(0, 1), W ~ N(0, 0.1^2) in fp16, bias / residual / gamma / beta ~ N(0, 1) (float32).
# The reference is float64 on the same fp16 operands.
#
# Accumulation term (every epilogue): fp16 x fp16 products are exact in fp32; only the fp32
# accumulation order differs from float64.  The bound of the existing raw-accumulator test is kept:
#     acc = 4e-6 * max_ij (|A| |W|^T)_ij.
# epi 3 (raw fp32):   |out - ref| <= acc.
# epi 0 (+bias, fp16):  x = acc32 + bias is one more fp32 rounding (2^-24 |x|); the store rounds to
#     nearest fp16: half an fp16 ulp at |ref| + err.
# epi 1 (+bias, GELU, fp16):  the kernel evaluates 0.5 x (1 + tanh(u(x))) with u fitted to the erf form
#     (<= 2.6e-5 with an exact tanh, tools/gelu_fit.py) and tanh on tanh.approx.f16x2: the argument
#     is rounded to fp16 (relative 2^-11; |d tanh/du| |u| <= 0.45) and the approximation's absolute
#     error is 2^-10.987, so |delta tanh| <= 1.46 * 2^-11 and 0.5 |x| |delta tanh| <= 2^-11 |x|.  An
#     error e in x moves GELU by at most max|GELU'| e = 1.13 e; the polynomial and the final FMA are a
#     few fp32 roundings (8 * 2^-24 |x|).  Then the fp16 store.
# epi 2 (+bias +residual, LayerNorm, fp16):  the pre-norm row carries D = acc + 2 * 2^-24 |pre| (two
#     fp32 adds).  LayerNorm y = gamma z + beta with z = (pre - mean) / sigma; a perturbation d of the
#     row moves z_j by (d_j - mean(d) - z_j mean(z d)) / sigma, at most (2 + |z_j|) D / sigma (mean
#     |z| <= 1).  The fp32 statistics (two 192-term partial sums per row, a square root, two
#     products) add at most 256 * 2^-24 (|gamma z| + |beta|).  Then the fp16 store.
ACC_REL = 4e-6


def _gemm_operands(M, N, K, epi, seed):
    a, w = _rand16((M, K), seed), _rand16((N, K), seed + 1, 0.1)
    bias = _randf(N, seed + 2) if epi != 3 else None
    res = gamma = beta = None
    if epi == 2:
        res = _rand16((M, N), seed + 3)
        gamma, beta = _randf(N, seed + 4), _randf(N, seed + 5)
    return a, w, bias, res, gamma, beta


def _gemm_bound_check(a, w, got, epi, bias, res, gamma, beta):
    """max(|got - ref| / bound) for the epilogue's derived bound (see above); asserts it is <= 1."""
    ad, wd = a.double(), w.double()
    mm = ad @ wd.T
    acc = ACC_REL * float((ad.abs() @ wd.abs().T).max())
    g = got.double()
    if epi == 3:
        err, bound = (g - mm).abs(), torch.full_like(mm, acc)
    elif epi == 0:
        ref = mm + bias.double()
        e = acc + U32 * ref.abs()
        err, bound = (g - ref).abs(), e + half_ulp16(ref.abs() + e)
    elif epi == 1:
        x = mm + bias.double()
        ref = 0.5 * x * (1.0 + torch.erf(x / math.sqrt(2.0)))
        e = 1.13 * (acc + U32 * x.abs()) + 2.6e-5 + 2.0 ** -11 * x.abs() + 8 * U32 * x.abs()
        err, bound = (g - ref).abs(), e + half_ulp16(ref.abs() + e)
    else:
        pre = mm + bias.double() + res.double()
        mean = pre.mean(1, keepdim=True)
        sigma = torch.sqrt(((pre - mean) ** 2).mean(1, keepdim=True) + 1e-12)
        z = (pre - mean) / sigma
        gd, bd = gamma.double(), beta.double()
        ref = gd * z + bd
        D = acc + 2 * U32 * pre.abs().max(1, keepdim=True).values
        e = gd.abs() * (2.0 + z.abs()) * D / sigma + 256 * U32 * ((gd * z).abs() + bd.abs())
        err, bound = (g - ref).abs(), e + half_ulp16(ref.abs() + e)
    assert torch.isfinite(g).all()
    ratio = float((err / bound).max())
    return ratio


@gpu
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "n%d_k%d_epi%d" % s)
@pytest.mark.parametrize("name", ROW_NAMES)
def test_gemm_build_sizes_against_float64(dev, sms, shape, name):
    N, K, epi = shape
    M = row_count(name, sms)
    assert gemm_plan(sms, M, N, K, epi) == expected_plan(shape, name)
    a, w, bias, res, gamma, beta = _gemm_operands(M, N, K, epi, seed=1000 + 17 * ROW_NAMES.index(name) + epi)
    got = dev.gemm_f16(a, w, epi=epi, bias=bias, residual=res, gamma=gamma, beta=beta, eps=1e-12)
    ratio = _gemm_bound_check(a, w, got, epi, bias, res, gamma, beta)
    print(f"MEASURE gemm epi={epi} N={N} K={K} M={M} plan={gemm_plan(sms, M, N, K, epi)} err/bound={ratio:.4f}")
    assert ratio <= 1.0


def _placed_rows(sms):
    """Row positions of a big call (sms + 1 row tiles: the last one is a second-round tile and, with
    clusters, the real half of a padded pair): first tile, cluster rank 1's tile, last tile."""
    M_big = sms * 128 + 61
    pos = [0, 1, 77, 128, 255, sms * 128, M_big - 1]
    return M_big, pos


@gpu
@pytest.mark.parametrize("shape", PRODUCTION, ids=lambda s: "n%d_k%d_epi%d" % s)
def test_gemm_rows_are_bit_identical_in_any_tile(dev, sms, shape):
    N, K, epi = shape
    M_big, pos = _placed_rows(sms)
    assert gemm_plan(sms, M_big, N, K, epi) == BIG_PLAN[shape]
    assert gemm_plan(sms, len(pos), N, K, epi) == SMALL_PLAN[shape]
    a, w, bias, res, gamma, beta = _gemm_operands(M_big, N, K, epi, seed=77 + epi)
    big = dev.gemm_f16(a, w, epi=epi, bias=bias, residual=res, gamma=gamma, beta=beta, eps=1e-12)
    idx = torch.tensor(pos, device="cuda")
    a_s = a[idx].contiguous()
    r_s = res[idx].contiguous() if res is not None else None
    small = dev.gemm_f16(a_s, w, epi=epi, bias=bias, residual=r_s, gamma=gamma, beta=beta, eps=1e-12)
    assert _same_bits(small, big[idx])
    # and one row alone (M = 1)
    one = dev.gemm_f16(a[-1:].contiguous(), w, epi=epi, bias=bias,
                       residual=res[-1:].contiguous() if res is not None else None, gamma=gamma, beta=beta,
                       eps=1e-12)
    assert _same_bits(one[0], big[-1])


@gpu
@pytest.mark.parametrize("shape", PRODUCTION + [(1536, 1536, 3)], ids=lambda s: "n%d_k%d_epi%d" % s)
@pytest.mark.parametrize("name", ["m129", "odd_tiles", "second_round"])
def test_gemm_writes_nothing_outside_its_output(dev, sms, shape, name):
    """out (and the LayerNorm residual) as 16-byte aligned views inside larger sentinel-filled buffers:
    ragged M, padded cluster row blocks; the bytes around the view stay as they were."""
    N, K, epi = shape
    M = row_count(name, sms) + (50 if name == "second_round" else 0)     # every case ends in a ragged tile
    a, w, bias, res, gamma, beta = _gemm_operands(M, N, K, epi, seed=5 + epi)
    want = dev.gemm_f16(a, w, epi=epi, bias=bias, residual=res, gamma=gamma, beta=beta, eps=1e-12)
    pad = 8 * 1024                                        # elements on each side (16-byte multiples)
    if epi == 3:
        buf = torch.full((pad + M * N + pad,), 0x5A5A5A5A, dtype=torch.int32, device="cuda")
        out = buf[pad:pad + M * N].view(torch.float32)
    else:
        buf = torch.full((pad + M * N + pad,), 0x5A5A, dtype=torch.int16, device="cuda")
        out = buf[pad:pad + M * N].view(torch.float16)
    before = buf.clone()
    rv = None
    if res is not None:
        rbuf = torch.full((pad + M * N + pad,), float("nan"), dtype=torch.float16, device="cuda")
        rbuf[pad:pad + M * N] = res.reshape(-1)
        rv = rbuf[pad:pad + M * N]
    _gemm_into(dev, a, w, epi, out, bias, rv, gamma, beta)
    assert torch.equal(buf[:pad], before[:pad]) and torch.equal(buf[pad + M * N:], before[pad + M * N:])
    assert _same_bits(out.view(M, N), want)


# -------------------------------------------------------------------------- §3 attention
HD, NH = 32, 12
ATT_S = [1, 2, 15, 16, 17, 63, 64, 65, 127, 128, 129, 200, 255, 256, 257, 320, 511, 512]


def _att_lens(S):
    """Per-sequence lens: 1, S, len mod 64 in {0, 1, 63}, one past S (clamps to S), 0, negative."""
    cand = {1, S, max(1, S - 1)}
    for k in range(1, 9):
        cand |= {64 * k - 1, 64 * k, 64 * k + 1}
    lens = sorted(c for c in cand if 1 <= c <= S)
    return lens + [S + 9, 0, -5]


def _att_clean(S, L, mode, g):
    """Clean [S, 1152] q | k | v rows for one sequence of effective length L (rows >= L are what an
    added key would read)."""
    q = torch.randn(S, NH, HD, generator=g, dtype=torch.float64)
    k = torch.randn(S, NH, HD, generator=g, dtype=torch.float64)
    v = torch.randn(S, NH, HD, generator=g, dtype=torch.float64)
    if mode != "unit":
        # logit(r, j) = q_r . k_j / sqrt(32) ~ sqrt(32) * 2 * b_j = 11.3 b_j: up to ~40
        q = 2.0 + 0.1 * q
        jj = torch.arange(S, dtype=torch.float64)
        if mode == "rising":                # the running maximum rises in every 64-key block
            b = 3.5 * jj / max(L - 1, 1)
        else:                               # the maximum sits in key 0 (first block); the edge keys
            b = 0.5 * torch.rand(S, generator=g, dtype=torch.float64) - 0.25     # stay within e^-2 of it
            b[0] = 3.5
            b[max(L - 1, 0):] = 3.35
        k = b[:, None, None] + 0.1 * k
    return torch.cat([q.reshape(S, -1), k.reshape(S, -1), v.reshape(S, -1)], 1).to(torch.float16)


def _att_ref(qkv, L, nk=None):
    """float64 attention of one sequence's first L query rows over its first nk (default L) keys ->
    ([L, 384] out, [L, 384] P|V|, A, Lmax, sum|V|)."""
    nk = L if nk is None else nk
    x = qkv.double()
    q = x[:L, :384].reshape(L, NH, HD).permute(1, 0, 2)
    k = x[:nk, 384:768].reshape(nk, NH, HD).permute(1, 0, 2)
    v = x[:nk, 768:].reshape(nk, NH, HD).permute(1, 0, 2)
    s = q @ k.transpose(1, 2) / math.sqrt(HD)
    P = torch.softmax(s, -1)
    out = (P @ v).permute(1, 0, 2).reshape(L, 384)
    pv = (P @ v.abs()).permute(1, 0, 2).reshape(L, 384)
    A = ((q.abs() @ k.abs().transpose(1, 2)).amax(-1) / math.sqrt(HD))          # [NH, L]
    Lmax = s.abs().amax(-1)                                                      # [NH, L]
    vsum = v.abs().sum(1)                                                        # [NH, HD]
    per_row = lambda t: t.permute(1, 0)[:, :, None].expand(L, NH, HD).reshape(L, 384)
    return out, pv, per_row(A), per_row(Lmax), vsum.reshape(1, 384).expand(L, 384)


def _att_bound(ref, pv, A, Lmax, vsum, L):
    """|o - ref| <= 2^-11 (P|V|) + 2^-11 |ref| + c.
    2^-11 (P|V|): P is rounded to fp16 (relative 2^-11) before P V.  2^-11 |ref|: the fp16 store.
    c: each p carries a relative error eps_p = 34 u A (fp32 Q K^T of 32 exact products) + 6 u Lmax (the
    scale constant, the running-maximum product and the FMA feeding ex2, in natural-log units) +
    2^-21 (ex2.approx.ftz.f32), which moves o by at most 2 eps_p (P|V|) (numerator and normaliser);
    the fp32 P V accumulation (Sk/16 MMA steps + 16 inside one) and the normaliser's sums (Sk/8 + 20
    roundings) add (Sk/16 + 16) 2^-23 + (Sk/8 + 20) u of (P|V|); p below 2^-14 is an fp16 subnormal
    (absolute 2^-25 each, normaliser >= 1): 2^-25 sum|V|; a subnormal output rounds by 2^-25.  The
    rounding of the error itself is covered by another 2^-11 of the non-store terms."""
    Sk = (L + 63) // 64 * 64
    eps_p = 34 * U32 * A + 6 * U32 * Lmax + 2.0 ** -21
    c = (2 * eps_p + (Sk / 16 + 16) * 2.0 ** -23 + (Sk / 8 + 20) * U32) * pv + 2.0 ** -25 * vsum + 2.0 ** -25
    t = 2.0 ** -11 * pv + c
    return t + 2.0 ** -11 * ref.abs() + 2.0 ** -11 * t


def _attention(dev, qkv, lens, B, S):
    ctx = torch.full((B * S, 384), float("nan"), dtype=torch.float16, device="cuda")
    dev._ck(dev.lib.lrx_debug_attention(dev.h, _p(qkv), _p(lens), B, S, _p(ctx)))
    return ctx


@gpu
@pytest.mark.parametrize("mode", ["unit", "rising", "first_block"])
@pytest.mark.parametrize("S", ATT_S)
def test_attention_against_float64(dev, S, mode):
    lens = _att_lens(S)
    B = len(lens)
    g = torch.Generator().manual_seed(S * 7 + len(mode))
    buf = torch.empty((B * S, 1152), dtype=torch.float16)
    refs, sens = [], []
    for b, ln in enumerate(lens):
        L = min(max(ln, 0), S)
        clean = _att_clean(S, max(L, 1), mode, g)
        if L > 0:
            ref = _att_ref(clean.cuda(), L)
            bound = _att_bound(*ref, L)
            refs.append((b, L, ref[0], bound))
            # sensitivity: one key dropped / added at the mask edge must move the reference past the bound
            # (all L query rows; with its only key dropped a row would be empty: zeros)
            alts = [_att_ref(clean.cuda(), L, L - 1)[0] if L > 1 else torch.zeros_like(ref[0])]
            if L < S:
                alts.append(_att_ref(clean.cuda(), L, L + 1)[0])
            for alt in alts:
                sens.append(bool(((alt - ref[0]).abs() > bound).any()))
        poisoned = clean.clone()
        if L < S:
            if b % 2:
                poisoned[L:] = float("nan")
            else:
                poisoned[L:] = torch.where(torch.arange(1152) % 2 == 0, 65504.0, -65504.0).to(torch.float16)
        buf[b * S:(b + 1) * S] = poisoned
    assert all(sens), sens
    lens_t = torch.tensor(lens, dtype=torch.int32, device="cuda")
    ctx = _attention(dev, buf.cuda(), lens_t, B, S).view(B, S, 384)
    worst = 0.0
    for b, L, ref, bound in refs:
        o = ctx[b, :L].double()
        assert torch.isfinite(o).all(), (b, L)
        worst = max(worst, float(((o - ref).abs() / bound).max()))
    print(f"MEASURE attention S={S} mode={mode} err/bound={worst:.4f}")
    assert worst <= 1.0
    # rows >= len (and every row of len <= 0): exactly +0
    for b, ln in enumerate(lens):
        L = min(max(ln, 0), S)
        assert (ctx[b, L:].view(torch.int16) == 0).all(), (b, ln)


@gpu
def test_attention_entry_rejects_bad_arguments(dev):
    from legal_rag_engine_b200._lib import LrxError
    qkv = torch.zeros((513 * 2, 1152), dtype=torch.float16, device="cuda")
    ctx = torch.zeros((513 * 2, 384), dtype=torch.float16, device="cuda")
    lens = torch.ones(2, dtype=torch.int32, device="cuda")
    for B, S in ((0, 8), (2, 0), (2, 513)):
        with pytest.raises(LrxError):
            dev._ck(dev.lib.lrx_debug_attention(dev.h, _p(qkv), _p(lens), B, S, _p(ctx)))
    with pytest.raises(LrxError):
        dev._ck(dev.lib.lrx_debug_attention(dev.h, C.c_void_p(0), _p(lens), 2, 8, _p(ctx)))


# ------------------------------------------------------------------- §4 the whole encoder
def _cos(a, b):
    return (a * b).sum(1) / (np.linalg.norm(a, axis=1) * np.linalg.norm(b, axis=1))


def _ref64(sd, ids, lens, chunk=128):
    from oracle import encoder as oenc
    return np.concatenate([oenc.encode_ids(sd, ids[s:s + chunk], lens[s:s + chunk], dtype=torch.float64,
                                           device="cuda") for s in range(0, len(ids), chunk)])


@pytest.fixture(scope="module")
def sd():
    from legal_rag_engine_b200 import synth
    return synth.bert_state_dict(42, 0.05, ln_jitter=0.1)


@pytest.fixture(scope="module")
def enc(dev, sd):
    from legal_rag_engine_b200.encoder import SentenceEncoder
    return SentenceEncoder(dev, state_dict=sd)


@gpu
@pytest.mark.parametrize("full", [True, False], ids=["full", "ragged"])
@pytest.mark.parametrize("S", LONG_S)
def test_long_chunked_batches_against_float64(enc, sd, sms, S, full):
    from legal_rag_engine_b200 import synth
    B, spc, last = _long_batch(S, sms)
    assert (spc * S + 127) // 128 >= sms // 2 and (last * S + 127) // 128 < sms // 2
    ids, lens = synth.token_batch(B, S, seed=300 + S, full=full)
    got = enc.encode_ids(ids, lens)                                  # lrx_encode_host
    want = _ref64(sd, ids, lens)
    cos = _cos(got.astype(np.float64), want)
    print(f"MEASURE encoder S={S} B={B} full={full} min_cos={cos.min():.7f}")
    assert cos.min() >= COS_MIN, (cos.argmin(), cos.min())
    np.testing.assert_allclose(np.linalg.norm(got.astype(np.float64), axis=1), 1.0, rtol=0, atol=1e-5)
    o32, o16 = enc.encode_ids_device(torch.from_numpy(ids).cuda(), torch.from_numpy(lens).cuda())
    torch.cuda.synchronize()
    np.testing.assert_array_equal(o32.cpu().numpy(), got)            # lrx_encode == lrx_encode_host
    assert torch.equal(o16, o32.to(torch.float16))                   # fp16 copy = fp32 rounded


@pytest.fixture(scope="module")
def corpus_store(tmp_path_factory, legal_chunks, sd):
    """The full reference corpus (2 620 chunks) built with create_vector_store, as in test_gpu_engine."""
    from legal_rag_engine_b200.engine import create_vector_store
    from legal_rag_engine_b200.tokenizer import HashTokenizer
    d = tmp_path_factory.mktemp("bulk_store")
    src = d / "legal_chunks.json"
    src.write_text(json.dumps(legal_chunks), encoding="utf-8")
    tok = HashTokenizer(30522)
    create_vector_store(str(src), str(d / "vs"), encoder_state_dict=sd, tokenizer=tok)
    return d / "vs", tok


@gpu
def test_reference_corpus_build_every_row_against_float64(corpus_store, sd, legal_texts):
    vs, tok = corpus_store
    xh = np.load(vs / "vectors.f16.npy")
    assert xh.shape == (len(legal_texts), 384)
    enc_ids = [tok.encode(t, 256) for t in legal_texts]
    order = sorted(range(len(enc_ids)), key=lambda i: len(enc_ids[i]))
    want = np.empty((len(enc_ids), 384))
    for s in range(0, len(order), 128):
        sel = order[s:s + 128]
        S = max(len(enc_ids[i]) for i in sel)
        ids = np.zeros((len(sel), S), dtype=np.int32)
        lens = np.array([len(enc_ids[i]) for i in sel], dtype=np.int32)
        for r, i in enumerate(sel):
            ids[r, :lens[r]] = enc_ids[i]
        want[sel] = _ref64(sd, ids, lens)
    cos = _cos(xh.astype(np.float64), want)
    print(f"MEASURE corpus rows={len(cos)} min_cos={cos.min():.7f} at row {int(cos.argmin())}")
    assert cos.min() >= COS_MIN, (int(cos.argmin()), float(cos.min()))


@gpu
@pytest.mark.parametrize("B,S", [(3, 40), (5, 150)], ids=["cluster_kernel", "chain"])
def test_out_of_range_ids_embed_as_id_zero(enc, sd, B, S):
    from legal_rag_engine_b200 import synth
    vocab = sd["embeddings.word_embeddings.weight"].shape[0]
    ids, lens = synth.token_batch(B, S, seed=900 + S)
    bad = ids.copy()
    rng = np.random.default_rng(S)
    for b in range(B):
        pos = rng.choice(np.arange(1, max(lens[b] - 1, 2)), size=min(4, max(lens[b] - 2, 1)), replace=False)
        bad[b, pos] = rng.choice([vocab, vocab + 12345, -1, -(2 ** 31)], size=len(pos))
    zero = np.where((bad < 0) | (bad >= vocab), 0, bad).astype(np.int32)
    assert (zero != ids).any()
    np.testing.assert_array_equal(enc.encode_ids(bad, lens), enc.encode_ids(zero, lens))


@gpu
@pytest.mark.parametrize("S,B,path", SMALL_PATH_CASES)
def test_small_path_boundaries_against_float64(enc, sd, S, B, path):
    from legal_rag_engine_b200 import synth
    assert small_path(B, S) == path
    ids, lens = synth.token_batch(B, S, seed=600 + B + S)
    got = enc.encode_ids(ids, lens)
    cos = _cos(got.astype(np.float64), _ref64(sd, ids, lens))
    print(f"MEASURE small_path S={S} B={B} path={path} min_cos={cos.min():.7f}")
    assert cos.min() >= COS_MIN


# ---------------------------------------------------------- §5 invariance of the GEMM chain
def _widen(ids, S):
    out = np.zeros((ids.shape[0], S), dtype=np.int32)
    out[:, :ids.shape[1]] = ids
    return out


@gpu
def test_chain_embeddings_are_bit_identical_in_any_batch(dev, sd, sms):
    """S > 64: every call takes the tcgen05 chain.  A sequence's embedding alone is the one it gets in
    batches of 2, 70 and 200 (first and last sequence of a chunk, a tail chunk on the small-M plans),
    padded to 128 and 512 tokens, through lrx_encode and lrx_encode_host, and after the activation
    workspace has grown (fresh handle: small call, large call, small call)."""
    from legal_rag_engine_b200 import synth
    from legal_rag_engine_b200.device_index import DeviceIndex
    from legal_rag_engine_b200.encoder import SentenceEncoder
    d = DeviceIndex(0)
    try:
        enc = SentenceEncoder(d, state_dict=sd)
        ids, lens = synth.token_batch(200, 65, seed=4242)
        lens[:4] = [65, 64, 1, 2]
        for i in range(4):
            ids[i, lens[i]:] = 0
            ids[i, lens[i] - 1] = 102
        probe = [0, 1, 2, 3, 38, 69, 70, 147, 148, 199]
        alone = {i: enc.encode_ids(ids[i:i + 1], lens[i:i + 1])[0] for i in probe}
        first_small = enc.encode_ids(ids[:2], lens[:2])
        # the workspace grows: 37 sequences of 512 tokens per chunk
        wide = enc.encode_ids(_widen(ids[:40], 512), lens[:40])
        assert small_path(40, 512) == 0
        np.testing.assert_array_equal(enc.encode_ids(ids[:2], lens[:2]), first_small)
        for i in probe:
            if i < 40:
                np.testing.assert_array_equal(wide[i], alone[i], err_msg=f"S=512 batch row {i}")
            np.testing.assert_array_equal(enc.encode_ids(_widen(ids[i:i + 1], 128), lens[i:i + 1])[0],
                                          alone[i], err_msg=f"alone at S=128 row {i}")
        np.testing.assert_array_equal(first_small, np.stack([alone[0], alone[1]]))
        b70 = enc.encode_ids(ids[:70], lens[:70])
        for i in (0, 1, 2, 3, 69):
            np.testing.assert_array_equal(b70[i], alone[i], err_msg=f"B=70 row {i}")
        # B = 200 at S = 65: one chunk on the big plans; at S = 128: a full chunk of 148 sequences plus
        # a tail chunk of 52 on the small-M plans
        assert (200 * 65 + 127) // 128 >= sms // 2
        assert KCHUNK_TOKENS // 128 == 148 and 52 * 128 // 128 < sms // 2
        for S in (65, 128):
            x = ids if S == 65 else _widen(ids, S)
            host = enc.encode_ids(x, lens)
            o32, _ = enc.encode_ids_device(torch.from_numpy(x).cuda(), torch.from_numpy(lens).cuda())
            torch.cuda.synchronize()
            np.testing.assert_array_equal(o32.cpu().numpy(), host)
            for i in probe:
                np.testing.assert_array_equal(host[i], alone[i], err_msg=f"B=200 S={S} row {i}")
    finally:
        d.close()


@gpu
@pytest.mark.parametrize("fusion", ["linear", "rrf"])
def test_long_queries_coalesced_equal_alone(corpus_store, sd, legal_texts, fusion):
    """search_batch puts queries of more than 64 tokens in blocks of their own (the GEMM chain),
    padded to the block's longest: each must return bit for bit what it returns alone."""
    from legal_rag_engine_b200.engine import RetrievalEngine
    vs, tok = corpus_store
    eng = RetrievalEngine(str(vs), encoder_state_dict=sd, tokenizer=tok)
    try:
        words = " ".join(legal_texts).split()
        qs = [" ".join(words[o:o + n]) for o, n in ((0, 70), (500, 95), (900, 140), (1500, 230), (2100, 66))]
        assert all(len(tok.encode(q, 256)) > 64 for q in qs)
        assert len({len(tok.encode(q, 256)) for q in qs}) == len(qs)
        ws = [0.5, 0.3, 0.7, 0.5, 0.6]
        strip = lambda rs: [(id(r["chunk"]), r["score"], r["semantic"], r["keyword"]) for r in rs]
        batch = eng.search_batch(qs, k=10, hybrid_weights=ws, fusion=fusion)
        for q, w, got in zip(qs, ws, batch):
            assert strip(got) == strip(eng.search(q, k=10, hybrid_weight=w, fusion=fusion))
    finally:
        eng.close()
