"""ctypes binding of include/lrx.h.

There is no CPU fallback: if the CUDA library has not been built, or exports
fewer symbols than the header declares, importing fails loudly.
"""
from __future__ import annotations

import ctypes as C
import re
from pathlib import Path

import os

HERE = Path(__file__).resolve().parent
# LRX_LIB: another build of the same library (kernel A/B runs); default = the in-tree build
LIB_PATH = Path(os.environ["LRX_LIB"]) if os.environ.get("LRX_LIB") else HERE / "csrc" / "liblrx.so"
HEADER = HERE.parent / "include" / "lrx.h"

LRX_DIM = 384
LRX_MAX_BATCH = 64
LRX_MAX_DEPTH = 256
LRX_MAX_QUERY_TERMS = 64
LRX_IPC_HANDLE_BYTES = 64
LRX_FUSE_LINEAR, LRX_FUSE_RRF = 0, 1
LRX_E_AMBIGUOUS = -5
LRX_E_PEER = -7


class LrxError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"lrx error {code}: {msg}")
        self.code = code


class lrx_config(C.Structure):
    _fields_ = [("device", C.c_int32), ("dim", C.c_int32), ("rank", C.c_int32),
                ("world", C.c_int32)]


_fp = C.c_void_p   # device pointers to float32 tensors


class lrx_bert_layer(C.Structure):
    _fields_ = [(n, _fp) for n in ("wq", "bq", "wk", "bk", "wv", "bv", "wo", "bo", "ln1_g", "ln1_b",
                                   "w1", "b1", "w2", "b2", "ln2_g", "ln2_b")]


class lrx_bert_weights(C.Structure):
    _fields_ = [("vocab_size", C.c_int32), ("max_positions", C.c_int32),
                ("word_emb", _fp), ("pos_emb", _fp), ("type_emb", _fp),
                ("emb_ln_g", _fp), ("emb_ln_b", _fp), ("layers", lrx_bert_layer * 6)]


def declared_symbols():
    """Every function include/lrx.h declares (used by the symbol-coverage test)."""
    text = HEADER.read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(lrx_[a-z0-9_]+)\s*\(", text)))


_vp, _i32, _i64, _f64 = C.c_void_p, C.c_int32, C.c_int64, C.c_double

_SIGNATURES = {
    "lrx_open": (C.c_int, [C.POINTER(lrx_config), C.POINTER(_vp)]),
    "lrx_close": (C.c_int, [_vp]),
    "lrx_last_error": (C.c_char_p, [_vp]),
    "lrx_set_stream": (C.c_int, [_vp, _vp]),
    "lrx_version": (C.c_char_p, []),
    "lrx_set_corpus": (C.c_int, [_vp, _vp, _i64, _i64, _i32]),
    "lrx_dense_prefilter_bytes": (_i64, [_i64]),
    "lrx_build_dense_prefilter": (C.c_int, [_vp, _vp, _i64, C.POINTER(C.c_double)]),
    "lrx_set_dense_prefilter": (C.c_int, [_vp, _vp, _i64, C.POINTER(C.c_double)]),
    "lrx_set_postings": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _i64, _f64, _f64, _f64, _i32]),
    "lrx_bm25_build_postings": (C.c_int, [_vp, _vp, _i64, _vp, _vp]),
    "lrx_bm25_append_postings": (C.c_int, [_vp, _vp, _vp, _i64, _i64, _i64, _vp, _vp, _i64, _i64, _vp,
                                           _i64, _vp, _vp]),
    "lrx_bm25_remove_postings": (C.c_int, [_vp, _vp, _vp, _i64, _i64, _i64, _vp, _i64, _vp, _vp, _vp, _vp,
                                           _i64, _vp]),
    "lrx_bm25_replace_postings": (C.c_int, [_vp, _vp, _vp, _i64, _i64, _i64, _vp, _i64, _vp, _vp, _vp, _vp, _vp,
                                            _i64, _vp, _vp, _i64, _vp]),
    "lrx_set_encoder_weights": (C.c_int, [_vp, C.POINTER(lrx_bert_weights)]),
    "lrx_encode": (C.c_int, [_vp, _vp, _vp, _i32, _i32, _vp, _vp]),
    "lrx_encode_host": (C.c_int, [_vp, _vp, _vp, _i32, _i32, _vp]),
    "lrx_gemm_f16": (C.c_int, [_vp, _vp, _vp, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _vp, C.c_float,
                               _vp]),
    "lrx_dense_topk": (C.c_int, [_vp, _vp, _i32, _i32, _vp, _vp, _vp, _vp]),
    "lrx_dense_topk_ex": (C.c_int, [_vp, _vp, _i32, _i32, _i32, _vp, _vp, _vp, _vp]),
    "lrx_dense_topk_batched": (C.c_int, [_vp, _vp, _i32, _i32, _i32, _vp, _vp, _vp, _vp]),
    "lrx_dense_at": (C.c_int, [_vp, _vp, _i32, _vp, _i32, _vp]),
    "lrx_bm25": (C.c_int, [_vp, _vp, _vp, _i32, _vp, _i32, _vp, _vp, _i32, _vp, _vp]),
    "lrx_exchange_export": (C.c_int, [_vp, _i32, _i32, _vp]),
    "lrx_exchange_import": (C.c_int, [_vp, _vp]),
    "lrx_search_sharded": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _vp,
                                     _vp]),
    "lrx_set_query_capacity": (C.c_int, [_vp, _i32]),
    "lrx_set_exchange_timeout": (C.c_int, [_vp, _i32]),
    "lrx_search_host_begin": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32]),
    "lrx_search_text_host_begin": (C.c_int, [_vp, _vp, _vp, _i32, _vp, _vp, _vp, _i32, _i32, _i32]),
    "lrx_search_host_end": (C.c_int, [_vp, _vp, _vp, _vp, _vp]),
    "lrx_search_batch_host": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _vp, _vp, _vp,
                                        _vp]),
    "lrx_search_text_host": (C.c_int, [_vp, _vp, _vp, _i32, _vp, _vp, _vp, _i32, _i32, _i32, _vp, _vp,
                                       _vp, _vp]),
    "lrx_debug_bm25_divcheck": (C.c_int, [_vp, _f64, _f64, _f64, _i32, _i32, C.POINTER(C.c_uint64)]),
    "lrx_debug_attention": (C.c_int, [_vp, _vp, _vp, _i32, _i32, _vp]),
    "lrx_launch_count": (_i64, [_vp]),
    "lrx_profile_enable": (C.c_int, [_vp, _i32]),
    "lrx_profile_read": (C.c_int, [_vp, _i32, C.POINTER(C.c_double), C.POINTER(C.c_int64)]),
}

_lib = None


def load():
    """Load liblrx.so (building is the job of __graft_entry__.build / build.py)."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; "
            f"g.build()'` (nvcc, sm_100a). This engine has no CPU fallback.")
    lib = C.CDLL(str(LIB_PATH))
    for name, (res, args) in _SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as e:
            raise ImportError(f"{LIB_PATH} does not export {name}; rebuild it") from e
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int, handle=None):
    if rc != 0:
        lib = load()
        msg = lib.lrx_last_error(handle)
        raise LrxError(rc, msg.decode() if msg else "?")
