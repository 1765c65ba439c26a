"""One GPU shard of the hybrid index: torch owns the device memory, the C ABI
(include/lrx.h) runs the kernels.  Thin, typed wrappers; no arithmetic here."""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence

import numpy as np
import torch

from . import _lib
from ._lib import LRX_DIM, LRX_FUSE_LINEAR, LRX_FUSE_RRF

FUSION = {"linear": LRX_FUSE_LINEAR, "rrf": LRX_FUSE_RRF}


def _ptr(t: Optional[torch.Tensor]):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _to(a, dt: torch.dtype, device) -> torch.Tensor:
    """A tensor, or a numpy array uploaded (unsigned integers as the signed type of their width),
    on `device` as `dt`."""
    if isinstance(a, np.ndarray):
        if a.dtype == np.uint64:
            a = a.view(np.int64)
        elif a.dtype == np.uint32:
            a = a.view(np.int32)
        a = torch.from_numpy(np.ascontiguousarray(a))
    return a.to(device, dtype=dt).contiguous()


class DeviceIndex:
    def __init__(self, device: int = 0, rank: int = 0, world: int = 1):
        if not torch.cuda.is_available():
            raise RuntimeError("DeviceIndex needs a CUDA device: this engine has no CPU fallback")
        self.lib = _lib.load()
        self.device = torch.device("cuda", device)
        self.rank, self.world = rank, world
        cfg = _lib.lrx_config(device, LRX_DIM, rank, world)
        h = C.c_void_p()
        _lib.check(self.lib.lrx_open(C.byref(cfg), C.byref(h)))
        self.h = h
        self.x = None
        self._xbuf = None
        self._q8 = None
        self._prefilter_on = False
        self.n_local = 0
        self.id_base = 0
        self._post = None
        self._capacity = 0
        self._pending = None
        self.use_current_stream()

    def close(self):
        if getattr(self, "h", None) is not None and self.h:
            self.lib.lrx_close(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        _lib.check(rc, self.h)

    def use_current_stream(self):
        """Bind the library to torch's current stream on this device."""
        s = torch.cuda.current_stream(self.device).cuda_stream
        self._ck(self.lib.lrx_set_stream(self.h, C.c_void_p(s)))

    # ------------------------------------------------------------- residency
    def set_corpus(self, x: torch.Tensor, id_base: int = 0, prefilter: bool = True):
        """Make the fp16 chunk matrix resident.  `prefilter`: also build the int8 shadow K2a scans
        for up to 4 queries at a time (388 B/row instead of 768; results unchanged, see
        include/lrx.h)."""
        assert x.dtype == torch.float16 and x.is_cuda and x.is_contiguous()
        assert x.dim() == 2 and x.shape[1] == LRX_DIM
        self.x, self.n_local, self.id_base = x, int(x.shape[0]), int(id_base)
        self._xbuf = x                                      # the rows append_rows can fill: x is its prefix
        self._ck(self.lib.lrx_set_corpus(self.h, _ptr(x), self.n_local, self.id_base, LRX_DIM))
        self._q8 = None
        self._prefilter_on = False
        if prefilter and self.n_local > 0:
            self.build_prefilter()

    def append_rows(self, x_new: torch.Tensor, prefilter: Optional[bool] = None):
        """Append fp16 rows (local ids n_local, n_local + 1, ...).  The matrix is the prefix of a
        capacity buffer; a buffer too small is replaced by one 1/16 larger than needed (the old rows
        are copied on the device, the old buffer freed) before the handle takes the new matrix.
        `prefilter` (default: as before) rebuilds the int8 shadow (its row scales sit after the
        padded rows, so it cannot grow in place)."""
        assert x_new.dtype == torch.float16 and x_new.is_cuda and x_new.dim() == 2
        assert x_new.shape[1] == LRX_DIM
        n, m = self.n_local, int(x_new.shape[0])
        if m == 0:
            return
        buf = self._xbuf
        if buf is None or buf.shape[0] < n + m:
            grown = torch.empty((n + m + (n + m) // 16, LRX_DIM), dtype=torch.float16, device=self.device)
            if n:
                grown[:n].copy_(self.x)
            buf = grown
        buf[n:n + m].copy_(x_new)
        if prefilter is None:
            prefilter = self._prefilter_on
        self._q8 = None                                     # the shadow of the old matrix
        self.set_corpus(buf[:n + m], self.id_base, prefilter=prefilter)
        self._xbuf = buf

    @property
    def capacity(self) -> int:
        """Rows the matrix buffer holds before append_rows has to grow it."""
        return int(self._xbuf.shape[0]) if self._xbuf is not None else 0

    def build_prefilter(self):
        nbytes = int(self.lib.lrx_dense_prefilter_bytes(self.n_local))
        buf = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
        bounds = (C.c_double * 2)()
        self._ck(self.lib.lrx_build_dense_prefilter(self.h, _ptr(buf), nbytes, bounds))
        self._q8 = (buf, nbytes, (float(bounds[0]), float(bounds[1])))
        self._prefilter_on = True

    def set_prefilter(self, on: bool):
        """Switch the int8 pre-filter of an index that has a shadow (A/B runs, tests)."""
        if on:
            if self._q8 is None:
                self.build_prefilter()
                return
            buf, nbytes, b = self._q8
            self._ck(self.lib.lrx_set_dense_prefilter(self.h, _ptr(buf), nbytes, (C.c_double * 2)(*b)))
        else:
            self._ck(self.lib.lrx_set_dense_prefilter(self.h, C.c_void_p(0), 0, None))
        self._prefilter_on = bool(on)

    @property
    def prefilter_bounds(self):
        """(max row error norm, max row norm) of the int8 shadow, or None."""
        return self._q8[2] if self._q8 is not None else None

    def set_postings(self, term_ptr, postings, doc_len, idf, avgdl: float, k1: float = 1.5,
                     b: float = 0.75):
        """Make the BM25 postings resident.  term_ptr int64/uint64 [V+1]; postings
        int32/uint32 [nnz,2] = (local doc, tf); doc_len int32/uint32 [n]; idf float64 [V]
        (GLOBAL statistics) -- torch CUDA tensors or numpy arrays (uploaded).  The 8-byte
        scoring layout {doc, u16 tf, u16 len} is built on the device (index-build step)."""
        tp = _to(term_ptr, torch.int64, self.device)
        po = _to(postings, torch.int32, self.device)
        dl = _to(doc_len, torch.int32, self.device)
        idf_t = _to(idf, torch.float64, self.device)
        nnz = int(tp[-1].item())
        assert po.shape[0] == nnz, (po.shape, nnz)
        dl1 = dl if dl.numel() else torch.zeros(1, dtype=torch.int32, device=self.device)   # no documents: one 0
        p8 = torch.zeros((nnz + 2, 2), dtype=torch.int32, device=self.device)   # 8 B / posting, padded
        self._ck(self.lib.lrx_bm25_build_postings(self.h, _ptr(po), nnz, _ptr(dl1), _ptr(p8)))
        del po
        self._install(tp, p8, idf_t, dl, avgdl, k1, b, int(dl1.max().item()))

    def _install(self, tp, p8, idf_t, doc_len, avgdl: float, k1: float, b: float, max_len: int):
        """Hand the handle these postings (lrx_set_postings): the one place that does, and the one
        writer of the fields that describe them.  Buffers it replaces are dropped only after the
        handle has taken the new ones, so a failure leaves the index as it was."""
        n_terms, nnz = int(tp.numel()) - 1, int(p8.shape[0]) - 2
        self._ck(self.lib.lrx_set_postings(self.h, _ptr(tp), _ptr(p8), _ptr(idf_t), n_terms, nnz, float(avgdl),
                                           float(k1), float(b), max_len))
        self._post = (tp, p8, idf_t)
        self._post_args = (nnz, float(avgdl), float(k1), float(b), max_len)
        self.doc_len, self.n_terms, self.n_docs = doc_len, n_terms, int(doc_len.numel())

    def stage_append(self, add_ptr, add_postings, add_doc_len, idf, avgdl: float):
        """Documents n_docs, n_docs + 1, ... merged on the device (lrx_bm25_append_postings) into new
        buffers: a staged index for `commit_postings`; the handle is not changed.  Their own CSR (add_ptr
        int64 [V_out+1], add_postings uint32 [nnz_add, 2] = (local doc, tf)), lengths, and the whole
        corpus's new idf float64 [V_out] / avgdl."""
        tp, p8, _ = self._post
        nnz, max_len = self._post_args[0], self._post_args[4]
        add_len = np.asarray(add_doc_len, dtype=np.uint32)
        ap = _to(add_ptr, torch.int64, self.device)
        ad = _to(np.asarray(add_postings, dtype=np.uint32).reshape(-1, 2), torch.int32, self.device)
        dl = torch.cat([self.doc_len[:self.n_docs], _to(add_len, torch.int32, self.device)])
        n_terms_out, nnz_add = len(add_ptr) - 1, int(add_ptr[-1])
        tp_out = torch.empty(n_terms_out + 1, dtype=torch.int64, device=self.device)
        p8_out = torch.empty((nnz + nnz_add + 2, 2), dtype=torch.int32, device=self.device)
        self._ck(self.lib.lrx_bm25_append_postings(
            self.h, _ptr(tp), _ptr(p8), self.n_terms, nnz, self.n_docs, _ptr(ap), _ptr(ad), n_terms_out, nnz_add,
            _ptr(dl), int(dl.numel()), _ptr(tp_out), _ptr(p8_out)))
        max_len = max(max_len, int(add_len.max()) if len(add_len) else 0)
        return tp_out, p8_out, _to(idf, torch.float64, self.device), dl, float(avgdl), max_len

    def append_postings(self, add_ptr, add_postings, add_doc_len, idf, avgdl: float):
        """stage_append + commit_postings: a failure leaves the index as it was."""
        self.commit_postings(self.stage_append(add_ptr, add_postings, add_doc_len, idf, avgdl))

    def remove_rows(self, keep, prefilter: Optional[bool] = None, chunk: int = 1 << 20):
        """Keep only the rows `keep` (ascending local ids, or a bool mask over n_local), moved to the
        front of the capacity buffer in order.  The kept ids ascend, so every row moves toward the
        front: the move runs in place, `chunk` rows at a time through one temporary allocated before
        the first row moves.  `prefilter` (default: as before) rebuilds the int8 shadow."""
        keep = keep.to(self.device) if isinstance(keep, torch.Tensor) else torch.as_tensor(np.asarray(keep),
                                                                                          device=self.device)
        idx = torch.nonzero(keep).flatten() if keep.dtype == torch.bool else keep.to(torch.int64)
        n, buf = int(idx.numel()), self._xbuf
        tmp = torch.empty((min(n, chunk), LRX_DIM), dtype=torch.float16, device=self.device)
        for a in range(0, n, chunk):                        # sources of later chunks lie past a + chunk
            c = min(chunk, n - a)
            torch.index_select(self.x, 0, idx[a:a + c], out=tmp[:c])
            buf[a:a + c].copy_(tmp[:c])
        del tmp
        if prefilter is None:
            prefilter = self._prefilter_on
        self._q8 = None                                     # the shadow of the old matrix
        self.set_corpus(buf[:n], self.id_base, prefilter=prefilter)
        self._xbuf = buf

    def posting_docs(self, terms: np.ndarray, counts: np.ndarray) -> np.ndarray:
        """Documents of the first counts[i] resident postings of each terms[i], concatenated."""
        tp, p8, _ = self._post
        t = torch.from_numpy(np.ascontiguousarray(terms, dtype=np.int64)).to(self.device)
        c = torch.from_numpy(np.ascontiguousarray(counts, dtype=np.int64)).to(self.device)
        excl = torch.cumsum(c, 0) - c
        idx = torch.repeat_interleave(tp[t] - excl, c) + torch.arange(int(counts.sum()), device=self.device)
        return (p8[idx, 0].to(torch.int64) & 0xFFFFFFFF).cpu().numpy()

    def compact_postings(self, rem):
        """The resident postings without the documents of a removal plan (bm25_index.BM25Remove),
        compacted on the device into new buffers (lrx_bm25_remove_postings), with the compacted
        doc_len: a staged index for `commit_postings`.  The handle is not changed; a plan that does
        not describe the postings raises LrxError (LRX_E_ARG)."""
        tp, p8, _ = self._post
        nnz = self._post_args[0]
        removed = _to(np.asarray(rem.removed).astype(np.uint32), torch.int32, self.device)
        rem_ptr = _to(np.asarray(rem.rem_ptr, dtype=np.int64), torch.int64, self.device)
        rem_doc = _to(np.asarray(rem.rem_doc, dtype=np.uint32), torch.int32, self.device)
        term_map = _to(np.asarray(rem.term_map, dtype=np.int32), torch.int32, self.device)
        tp_out = _to(np.asarray(rem.term_ptr, dtype=np.int64), torch.int64, self.device)
        p8_out = torch.empty((rem.nnz + 2, 2), dtype=torch.int32, device=self.device)
        self._ck(self.lib.lrx_bm25_remove_postings(
            self.h, _ptr(tp), _ptr(p8), self.n_terms, nnz, self.n_docs, _ptr(removed), len(rem.removed),
            _ptr(rem_ptr), _ptr(rem_doc), _ptr(term_map), _ptr(tp_out), rem.n_terms, _ptr(p8_out)))
        keep = torch.ones(self.n_docs, dtype=torch.bool, device=self.device)
        keep[removed.to(torch.int64)] = False
        dl = self.doc_len[:self.n_docs][keep]
        idf_t = _to(rem.stats.idf, torch.float64, self.device)
        return tp_out, p8_out, idf_t, dl, float(rem.stats.avgdl), int(dl.max().item())

    def stage_replace(self, rep, doc_len_new):
        """The resident postings with the text of a replacement plan's documents (bm25_index.BM25Replace)
        replaced, merged on the device into new buffers (lrx_bm25_replace_postings): a staged index for
        `commit_postings`.  `doc_len_new` [n_docs]: every document's length after the edit (torch or
        numpy).  The handle is not changed; a plan that does not describe the postings raises LrxError
        (LRX_E_ARG)."""
        tp, p8, _ = self._post
        nnz = self._post_args[0]
        replaced = _to(np.asarray(rep.replaced).astype(np.uint32), torch.int32, self.device)
        rem_ptr = _to(np.asarray(rep.rem_ptr, dtype=np.int64), torch.int64, self.device)
        rem_doc = _to(np.asarray(rep.rem_doc, dtype=np.uint32), torch.int32, self.device)
        term_map = _to(np.asarray(rep.term_map, dtype=np.int32), torch.int32, self.device)
        ins_ptr = _to(np.asarray(rep.ins_ptr, dtype=np.int64), torch.int64, self.device)
        ins = _to(np.asarray(rep.ins_postings, dtype=np.uint32).reshape(-1, 2), torch.int32, self.device)
        dl = _to(np.asarray(doc_len_new, dtype=np.uint32) if not isinstance(doc_len_new, torch.Tensor)
                 else doc_len_new, torch.int32, self.device)
        assert dl.numel() == self.n_docs, (dl.numel(), self.n_docs)
        tp_out = _to(np.asarray(rep.term_ptr, dtype=np.int64), torch.int64, self.device)
        p8_out = torch.empty((rep.nnz + 2, 2), dtype=torch.int32, device=self.device)
        self._ck(self.lib.lrx_bm25_replace_postings(
            self.h, _ptr(tp), _ptr(p8), self.n_terms, nnz, self.n_docs, _ptr(replaced), len(rep.replaced),
            _ptr(rem_ptr), _ptr(rem_doc), _ptr(term_map), _ptr(ins_ptr), _ptr(ins), rep.nnz_ins, _ptr(dl),
            _ptr(tp_out), rep.n_terms, _ptr(p8_out)))
        idf_t = _to(rep.stats.idf, torch.float64, self.device)
        return tp_out, p8_out, idf_t, dl, float(rep.stats.avgdl), int(dl.max().item())

    def replace_rows(self, ids, x_new: torch.Tensor, prefilter: Optional[bool] = None):
        """Overwrite the fp16 rows `ids` (local ids, a sequence or a tensor) in place with `x_new`.  The int8 shadow of the old
        rows is dropped from the handle first; `prefilter` (default: as before) rebuilds it."""
        assert x_new.dtype == torch.float16 and x_new.is_cuda and x_new.dim() == 2
        idx = (ids.to(self.device, torch.int64) if isinstance(ids, torch.Tensor)
               else torch.as_tensor(np.asarray(ids, dtype=np.int64), device=self.device))
        assert x_new.shape == (idx.numel(), LRX_DIM)
        if prefilter is None:
            prefilter = self._prefilter_on
        if self._prefilter_on:
            self.set_prefilter(False)
        self._q8 = None                                     # the shadow of the old rows
        self.x.index_copy_(0, idx, x_new)
        if prefilter:
            self.build_prefilter()

    def commit_postings(self, staged):
        """Make a staged index of `stage_append`, `compact_postings` or `stage_replace` resident."""
        tp_out, p8_out, idf_t, dl, avgdl, max_len = staged
        _, _, k1, b, _ = self._post_args
        self._install(tp_out, p8_out, idf_t, dl, avgdl, k1, b, max_len)

    def remove_postings(self, rem):
        """compact_postings + commit_postings: a failure leaves the index as it was."""
        self.commit_postings(self.compact_postings(rem))

    def read_postings(self):
        """The resident postings on the host as an index build holds them: (term_ptr uint64 [V+1],
        postings uint32 [nnz, 2] = (doc, tf), doc_len uint32 [n_docs]).  The 8-byte entries
        {u32 doc, u16 tf, u16 len} are copied as they are and the tf split off on the host, so the
        device needs no temporary the size of the postings."""
        tp, p8, _ = self._post
        postings = p8[:self._post_args[0]].cpu().numpy().view(np.uint32)
        postings[:, 1] &= 0xFFFF
        return (tp.cpu().numpy().view(np.uint64), postings,
                self.doc_len[:self.n_docs].cpu().numpy().view(np.uint32))

    def clone_view(self) -> "DeviceIndex":
        """A second handle (own stream binding, workspaces, exchange region) over the SAME resident
        matrix and postings -- no copies: lets two query batches be in flight on two streams, one
        batch's merges and fusion running under the other's scans."""
        other = DeviceIndex(self.device.index, self.rank, self.world)
        if self.x is not None:
            other.set_corpus(self.x, self.id_base, prefilter=False)
            if self._q8 is not None:                        # the same shadow, no second copy
                other._q8 = self._q8
                other.set_prefilter(True)
        if self._post is not None:
            other._install(*self._post, self.doc_len, *self._post_args[1:])
        return other

    def _cap(self, q_terms: Optional[torch.Tensor], B: int):
        """Device-pointer calls: the library sizes its per-token tables from a capacity it cannot
        read off the device; the tensor's length is an upper bound of the batch's token count."""
        n = int(q_terms.numel()) if q_terms is not None else 0
        want = n if n > B * _lib.LRX_MAX_QUERY_TERMS else 0          # 0 = the default B * 64
        if want != self._capacity:
            self._ck(self.lib.lrx_set_query_capacity(self.h, want))
            self._capacity = want

    def set_exchange_timeout(self, milliseconds: int):
        self._ck(self.lib.lrx_set_exchange_timeout(self.h, int(milliseconds)))

    # ---------------------------------------------------------------- stages
    def dense_topk(self, q: torch.Tensor, K: int, width: int = 0):
        assert q.dtype == torch.float16 and q.is_cuda and q.is_contiguous()
        B = int(q.shape[0])
        exact = torch.empty((B, K), dtype=torch.float64, device=self.device)
        D = torch.empty((B, K), dtype=torch.float32, device=self.device)
        I = torch.empty((B, K), dtype=torch.int64, device=self.device)
        flags = torch.empty(B, dtype=torch.int32, device=self.device)
        self._ck(self.lib.lrx_dense_topk_ex(self.h, _ptr(q), B, K, width, _ptr(exact), _ptr(D),
                                            _ptr(I), _ptr(flags)))
        return exact, D, I, flags

    def dense_topk_batched(self, q: torch.Tensor, K: int, stride: int = 0):
        """K2b: tensor-core path for large batches (B up to 4096).  Same outputs as dense_topk."""
        assert q.dtype == torch.float16 and q.is_cuda and q.is_contiguous()
        B = int(q.shape[0])
        exact = torch.empty((B, K), dtype=torch.float64, device=self.device)
        D = torch.empty((B, K), dtype=torch.float32, device=self.device)
        I = torch.empty((B, K), dtype=torch.int64, device=self.device)
        flags = torch.empty(B, dtype=torch.int32, device=self.device)
        self._ck(self.lib.lrx_dense_topk_batched(self.h, _ptr(q), B, K, stride, _ptr(exact), _ptr(D),
                                                 _ptr(I), _ptr(flags)))
        return exact, D, I, flags

    def dense_at(self, q: torch.Tensor, ids: torch.Tensor):
        B, n = int(ids.shape[0]), int(ids.shape[1])
        out = torch.empty((B, n), dtype=torch.float64, device=self.device)
        self._ck(self.lib.lrx_dense_at(self.h, _ptr(q), B, _ptr(ids.contiguous()), n, _ptr(out)))
        return out

    def bm25(self, q_terms: torch.Tensor, q_ptr: torch.Tensor, cand_ids: Optional[torch.Tensor] = None,
             K: int = 0):
        """Returns (cand_scores [B,n] or None, max [B], top_scores [B,K], top_ids [B,K])."""
        B = int(q_ptr.numel() - 1)
        n = int(cand_ids.shape[1]) if cand_ids is not None else 0
        cs = torch.empty((B, n), dtype=torch.float64, device=self.device) if n else None
        mx = torch.empty(B, dtype=torch.float64, device=self.device)
        ts = torch.empty((B, max(K, 1)), dtype=torch.float64, device=self.device)
        ti = torch.empty((B, max(K, 1)), dtype=torch.int64, device=self.device)
        if q_terms.numel() == 0:
            q_terms = torch.zeros(1, dtype=torch.int32, device=self.device)
        self._cap(q_terms, B)
        self._ck(self.lib.lrx_bm25(self.h, _ptr(q_terms), _ptr(q_ptr), B,
                                   _ptr(cand_ids.contiguous() if n else None), n, _ptr(cs), _ptr(mx),
                                   K, _ptr(ts), _ptr(ti)))
        return cs, mx, ts[:, :K], ti[:, :K]

    # ------------------------------------ peer-memory exchange (world > 1, one box)
    def exchange_setup(self, B_max: int, k_max: int, group=None) -> bool:
        """Allocate this rank's exchange region, swap IPC handles with the other ranks (one
        all-gather of 64 bytes at start-up) and open theirs: afterwards `search_sharded` needs no
        collective call per query batch.  Returns False -- on EVERY rank, the outcome is agreed by
        an all-reduce -- when some rank could not export or map a region (e.g. no peer access
        between the GPUs): a sharded search cannot run on that box."""
        import torch.distributed as dist
        from ._lib import LRX_IPC_HANDLE_BYTES, LrxError
        ok = 1
        mine = (C.c_ubyte * LRX_IPC_HANDLE_BYTES)()
        try:
            self._ck(self.lib.lrx_exchange_export(self.h, B_max, k_max, C.cast(mine, C.c_void_p)))
        except LrxError:
            ok = 0
        world = dist.get_world_size(group)
        t = torch.tensor(list(mine), dtype=torch.uint8, device=self.device)
        every = torch.empty(world * LRX_IPC_HANDLE_BYTES, dtype=torch.uint8, device=self.device)
        dist.all_gather_into_tensor(every, t, group=group)
        flag = torch.tensor([ok], dtype=torch.int32, device=self.device)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=group)      # did everybody export?
        if int(flag.item()) == 1:
            host = every.cpu().numpy().tobytes()
            buf = (C.c_ubyte * len(host)).from_buffer_copy(host)
            try:
                self._ck(self.lib.lrx_exchange_import(self.h, C.cast(buf, C.c_void_p)))
            except LrxError:
                ok = 0
        else:
            ok = 0
        flag = torch.tensor([ok], dtype=torch.int32, device=self.device)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=group)      # ... and map every region?
        return int(flag.item()) == 1       # the all-reduce also orders "mapped" before the first store

    def search_sharded(self, q, q_terms, q_ptr, k: int, mode: int, weights, outs, width: int = 0):
        """K2 + K3 on this shard, block stored into every peer's region (world > 1), K4: the
        replicated result.  One captured launch chain per (shape, buffers), replayed per call."""
        B = int(q.shape[0])
        ids, score, sem, kw, status = outs
        if q_terms.numel() == 0:
            q_terms = torch.zeros(1, dtype=torch.int32, device=self.device)
        self._cap(q_terms, B)
        self._ck(self.lib.lrx_search_sharded(self.h, _ptr(q), _ptr(q_terms), _ptr(q_ptr), _ptr(weights),
                                             B, k, mode, width, _ptr(ids), _ptr(score), _ptr(sem),
                                             _ptr(kw), _ptr(status)))
        return outs

    def alloc_outputs(self, B: int, k: int):
        return (torch.empty((B, k), dtype=torch.int64, device=self.device),
                torch.empty((B, k), dtype=torch.float64, device=self.device),
                torch.empty((B, k), dtype=torch.float64, device=self.device),
                torch.empty((B, k), dtype=torch.float64, device=self.device),
                torch.empty(B, dtype=torch.int32, device=self.device))

    # ----------------------------------------------------- whole search, host
    @staticmethod
    def _host_args(q_fp16, term_lists, weights):
        q_fp16 = np.ascontiguousarray(q_fp16, dtype=np.float16)
        B = q_fp16.shape[0]
        ptr = np.zeros(B + 1, dtype=np.int32)
        for i, t in enumerate(term_lists):
            ptr[i + 1] = ptr[i] + len(t)
        terms = np.fromiter((int(x) for t in term_lists for x in t), dtype=np.int32, count=int(ptr[-1]))
        if terms.size == 0:
            terms = np.zeros(1, dtype=np.int32)
        return q_fp16, B, terms, ptr, np.ascontiguousarray(weights, dtype=np.float64)

    def search_batch_host(self, q_fp16: np.ndarray, term_lists: Sequence[Sequence[int]], k: int,
                          weights: Sequence[float], fusion: str = "linear"):
        """Host buffers in, host buffers out (H2D + kernels + D2H inside the call); on a shard
        (world > 1) every rank makes the same call and gets the replicated result.
        Returns (ids int64 [B,k], score, semantic, keyword float64 [B,k])."""
        self.search_host_begin(q_fp16, term_lists, k, weights, fusion)
        return self.search_host_end()

    def search_host_begin(self, q_fp16: np.ndarray, term_lists: Sequence[Sequence[int]], k: int,
                          weights: Sequence[float], fusion: str = "linear"):
        """Stage + enqueue (H2D, chain, D2H) and return at once; `search_host_end` collects.  With
        two handles over one index (`clone_view`) two batches are in flight."""
        q_fp16, B, terms, ptr, w = self._host_args(q_fp16, term_lists, weights)
        vp = lambda a: a.ctypes.data_as(C.c_void_p)
        self._ck(self.lib.lrx_search_host_begin(self.h, vp(q_fp16), vp(terms), vp(ptr), vp(w), B, k,
                                                FUSION[fusion]))
        self._pending = (B, k)

    def search_host_end(self):
        B, k = self._pending
        self._pending = None
        ids = np.empty((B, k), dtype=np.int64)
        score = np.empty((B, k), dtype=np.float64)
        sem = np.empty((B, k), dtype=np.float64)
        kw = np.empty((B, k), dtype=np.float64)
        vp = lambda a: a.ctypes.data_as(C.c_void_p)
        self._ck(self.lib.lrx_search_host_end(self.h, vp(ids), vp(score), vp(sem), vp(kw)))
        return ids, score, sem, kw

    def search_text_host_begin(self, tok_ids: np.ndarray, tok_lens: np.ndarray, term_lists, k: int,
                               weights: Sequence[float], fusion: str = "linear"):
        """`search_text_host` split in two: stage + enqueue (H2D, encoder, chain, D2H) and return at
        once; `search_host_end` collects.  Several handles over one index keep several batches in
        flight, the encoder of one under the scans of another."""
        tok_ids = np.ascontiguousarray(tok_ids, dtype=np.int32)
        tok_lens = np.ascontiguousarray(tok_lens, dtype=np.int32)
        B, S = tok_ids.shape
        _, _, terms, ptr, w = self._host_args(np.zeros((B, LRX_DIM), np.float16), term_lists, weights)
        vp = lambda a: a.ctypes.data_as(C.c_void_p)
        self._ck(self.lib.lrx_search_text_host_begin(self.h, vp(tok_ids), vp(tok_lens), S, vp(terms), vp(ptr),
                                                     vp(w), B, k, FUSION[fusion]))
        self._pending = (B, k)

    def search_text_host(self, tok_ids: np.ndarray, tok_lens: np.ndarray, term_lists, k: int,
                         weights: Sequence[float], fusion: str = "linear"):
        """The whole of RetrievalEngine.search for tokenised strings: WordPiece ids [B,S] + lens [B]
        and BM25 term-id lists in, fused results out (K1 -> K2 || K3 -> K4 in one call)."""
        tok_ids = np.ascontiguousarray(tok_ids, dtype=np.int32)
        tok_lens = np.ascontiguousarray(tok_lens, dtype=np.int32)
        B, S = tok_ids.shape
        _, _, terms, ptr, w = self._host_args(np.zeros((B, LRX_DIM), np.float16), term_lists, weights)
        ids = np.empty((B, k), dtype=np.int64)
        score, sem, kw = (np.empty((B, k), dtype=np.float64) for _ in range(3))
        vp = lambda a: a.ctypes.data_as(C.c_void_p)
        self._ck(self.lib.lrx_search_text_host(self.h, vp(tok_ids), vp(tok_lens), S, vp(terms), vp(ptr),
                                               vp(w), B, k, FUSION[fusion], vp(ids), vp(score), vp(sem),
                                               vp(kw)))
        return ids, score, sem, kw

    # ------------------------------------------------------ K1 stage: GEMM
    def gemm_f16(self, a: torch.Tensor, w: torch.Tensor, epi: int = 3, bias=None, residual=None,
                 gamma=None, beta=None, eps: float = 1e-12):
        """out[M,N] = epi(a[M,K] @ w[N,K]^T) on the tensor cores (lrx_gemm_f16)."""
        assert a.dtype == torch.float16 and w.dtype == torch.float16
        assert a.is_contiguous() and w.is_contiguous()
        M, K = a.shape
        N = w.shape[0]
        out = torch.empty((M, N), dtype=torch.float32 if epi == 3 else torch.float16,
                          device=self.device)
        self._ck(self.lib.lrx_gemm_f16(self.h, _ptr(a), _ptr(w), M, N, K, epi, _ptr(bias),
                                       _ptr(residual), _ptr(gamma), _ptr(beta), float(eps), _ptr(out)))
        return out

    def profile(self, on: bool):
        self._ck(self.lib.lrx_profile_enable(self.h, 1 if on else 0))

    def profile_read(self, which: int):
        """(summed device ms, launches) of kernel `which` (0 dense scan, 1 BM25 scan)."""
        ms, n = C.c_double(), C.c_int64()
        self._ck(self.lib.lrx_profile_read(self.h, which, C.byref(ms), C.byref(n)))
        return ms.value, n.value

    @property
    def launches(self) -> int:
        return int(self.lib.lrx_launch_count(self.h))
