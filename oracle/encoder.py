"""Oracle: the all-MiniLM-L6-v2 sentence encoder as the reference calls it,
``SentenceTransformer(...).encode([text], convert_to_numpy=True)`` followed by
``faiss.normalize_L2`` (``src/retrieval/retrieval_engine.py:28,61-62``;
``create_vector_store.py:33-34,45,51``), restated in float32.

Test infrastructure, see ``oracle/__init__.py``.  The arithmetic lives in two PyPI
wheels that are absent from /root/reference (sentence-transformers >= 2.2.0 driving a
HuggingFace ``BertModel``, ``requirements.txt:6``); the restatement follows their
published modules:

  BertEmbeddings     word[id] + position[arange(S)] + token_type[0] -> LayerNorm(eps 1e-12)
  BertSelfAttention  softmax(Q K^T / sqrt(32) + (1 - mask) * finfo.min) V, 12 heads x 32
  BertSelfOutput     LayerNorm(dense(ctx) + x)
  BertIntermediate   gelu(dense(x)), exact erf form
  BertOutput         LayerNorm(dense(h) + x)
  Pooling (mean)     sum(h * mask) / clamp(sum(mask), min=1e-9)
  Normalize          F.normalize(p=2, dim=1)  = x / max(||x||, 1e-12)
  faiss.normalize_L2 x *= 1 / sqrt(sum x^2)   (rows with zero norm untouched)

``dtype`` / ``device`` (keywords of the three entry points): the defaults, float32 on the CPU, are
the restatement the golden file pins; ``dtype=torch.float64, device="cuda"`` runs the same
arithmetic in double precision on a GPU -- the reference the kernel tests measure error against
when thousands of rows are needed (the faiss step is then float64 as well).

PINNED against HuggingFace ``transformers.BertModel`` (installed in the build
container) by ``tests/golden/make_encoder_golden.py``: the golden file holds BertModel's
own outputs for seeded weights; ``tests/test_oracle_encoder.py`` checks this restatement
against them.  (The sentence-transformers / faiss wrappers themselves are not
installable here: their three post-processing steps are restated from their docs.)
"""
from __future__ import annotations

from typing import Dict

import numpy as np
import torch

HIDDEN, HEADS, HEAD_DIM, FFN, LAYERS = 384, 12, 32, 1536, 6
LN_EPS = 1e-12


def _t(a, dtype=torch.float32, device="cpu") -> torch.Tensor:
    if isinstance(a, torch.Tensor):
        return a.detach().to(device=device, dtype=dtype)
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(device=device, dtype=dtype)


def _layer_norm(x, g, b):
    mean = x.mean(-1, keepdim=True)
    var = ((x - mean) ** 2).mean(-1, keepdim=True)
    return (x - mean) / torch.sqrt(var + LN_EPS) * g + b


def bert_hidden(sd: Dict[str, np.ndarray], ids: np.ndarray, mask: np.ndarray, *,
                dtype=torch.float32, device="cpu") -> torch.Tensor:
    """Last hidden state [B,S,384] (``dtype``, on ``device``) of the 6-layer BertModel without
    pooler.  ``sd``: HuggingFace state_dict names -> arrays; ``ids``/``mask``: int [B,S]."""
    w = {k: _t(v, dtype, device) for k, v in sd.items()}
    ids_t = torch.from_numpy(np.asarray(ids, dtype=np.int64)).to(device)
    mask_t = torch.from_numpy(np.asarray(mask, dtype=np.int64)).to(device)
    B, S = ids_t.shape
    x = (w["embeddings.word_embeddings.weight"][ids_t]
         + w["embeddings.position_embeddings.weight"][torch.arange(S, device=device)][None]
         + w["embeddings.token_type_embeddings.weight"][0][None, None])
    x = _layer_norm(x, w["embeddings.LayerNorm.weight"], w["embeddings.LayerNorm.bias"])
    ext = (1.0 - mask_t[:, None, None, :].to(dtype)) * torch.finfo(dtype).min
    for l in range(LAYERS):
        p = f"encoder.layer.{l}."
        lin = lambda t, name: t @ w[p + name + ".weight"].T + w[p + name + ".bias"]
        split = lambda t: t.view(B, S, HEADS, HEAD_DIM).permute(0, 2, 1, 3)
        q = split(lin(x, "attention.self.query"))
        k = split(lin(x, "attention.self.key"))
        v = split(lin(x, "attention.self.value"))
        scores = q @ k.transpose(-1, -2) / np.sqrt(HEAD_DIM) + ext
        ctx = torch.softmax(scores, dim=-1) @ v
        ctx = ctx.permute(0, 2, 1, 3).reshape(B, S, HIDDEN)
        x = _layer_norm(lin(ctx, "attention.output.dense") + x,
                        w[p + "attention.output.LayerNorm.weight"],
                        w[p + "attention.output.LayerNorm.bias"])
        h = lin(x, "intermediate.dense")
        h = h * 0.5 * (1.0 + torch.erf(h / np.sqrt(2.0)))
        x = _layer_norm(lin(h, "output.dense") + x, w[p + "output.LayerNorm.weight"],
                        w[p + "output.LayerNorm.bias"])
    return x


def pool_normalize(hidden: torch.Tensor, mask: np.ndarray, *, dtype=torch.float32) -> np.ndarray:
    """sentence-transformers Pooling(mean) + Normalize, then faiss.normalize_L2; ``dtype`` [B,384]
    numpy rows (faiss's own step is float32; with ``dtype=torch.float64`` it is float64 too)."""
    m = torch.from_numpy(np.asarray(mask, dtype=np.int64)).to(device=hidden.device, dtype=dtype)[:, :, None]
    hidden = hidden.to(dtype)
    emb = (hidden * m).sum(1) / torch.clamp(m.sum(1), min=1e-9)
    emb = emb / torch.clamp(emb.norm(dim=1, keepdim=True), min=1e-12)
    npt = np.float64 if dtype == torch.float64 else np.float32
    out = emb.cpu().numpy().astype(npt)
    n2 = (out ** 2).sum(axis=1, dtype=npt)                                 # fvec_norm_L2sqr
    nz = n2 > 0
    out[nz] *= (npt(1.0) / np.sqrt(n2[nz]))[:, None]
    return out


def encode_ids(sd, ids: np.ndarray, lens: np.ndarray, *, dtype=torch.float32, device="cpu") -> np.ndarray:
    """[B,384] unit embeddings (float32, or float64 with ``dtype=torch.float64``) for 0-padded id
    rows with prefix masks of length ``lens``."""
    ids = np.asarray(ids)
    mask = (np.arange(ids.shape[1])[None, :] < np.asarray(lens)[:, None]).astype(np.int64)
    return pool_normalize(bert_hidden(sd, ids, mask, dtype=dtype, device=device), mask, dtype=dtype)
