#!/usr/bin/env python
"""Headline benchmark: hybrid top-10 queries/s over 10 M x 384 chunks (BASELINE.json
config C4: fp16 chunk matrix + BM25 postings over a 50 k-term Zipf vocabulary, one user
query = 4 fan-out sub-queries, RRF fusion), strong-scaled over 1/2/4/8 B200.

    python bench.py --gpus N --steps K --warmup W            # our CUDA path
    python bench.py --impl reference --gpus N ...            # the reference's CPU path
    torchrun ... bench.py --gpus N ...                       # N > 1, one rank per GPU

One JSON line on stdout (rank 0).  A "step" is one user query: K2 (dense scan + top-k)
|| K3 (BM25) -> candidate exchange between the shards (N > 1, inside the kernels) -> K4
(fusion), one captured launch chain.  `value` is measured with the queries already resident
in HBM; `e2e` goes through the host-buffer C-ABI calls (lrx_search_host_begin / _end) with the
H2D / D2H copies of every step inside the timed region.  Both keep `in_flight` query batches in
flight (one handle + stream each), the same number at every N.  Before the timed region a
sample of the pool queries is checked against an on-device float64 brute force (`parity`).
"""
from __future__ import annotations

import argparse
import json
import math
import os
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

K_TOP = 10
N_SUB = 4                      # fan-out sub-queries per user query (orchestrator.py:39-48)
N_TERMS = 8                    # BM25 tokens per sub-query
WEIGHTS = [0.5, 0.6, 0.5, 0.6]  # orchestrator.py:56
POOL = 16                      # distinct user queries cycled through the timed steps
RRF_K0 = 60.0


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200,
                    help="timed steps of the headline region (one user query each); the e2e and the "
                         "two-users regions time as many steps")
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--rows", type=int, default=10_000_000)
    ap.add_argument("--fusion", default="rrf", choices=["rrf", "linear"])
    ap.add_argument("--in-flight", type=int, default=3,
                    help="query batches in flight (one handle + stream each), the same at every N: one "
                         "batch's merges / exchange / fusion run under the next one's scans")
    ap.add_argument("--k", type=int, default=10,
                    help="result depth (10 = the headline metric; 100 with --rows 100000000 --gpus 8 = config C5)")
    ap.add_argument("--parity-queries", type=int, default=8,
                    help="pool queries checked against the on-device float64 brute force (0 = skip)")
    ap.add_argument("--kernel-events", default="on", choices=["on", "off"],
                    help="CUDA event nodes around the two streaming kernels inside the captured chains of the "
                         "timed region (the roofline figure); off = A/B runs of the chain without them")
    ap.add_argument("--prefilter", default="on", choices=["on", "off"],
                    help="int8 shadow of the matrix for the dense scan (388 B/row instead of 768; results "
                         "unchanged).  off: the plain fp16 scan")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-stages", action="store_true", help="skip the K1 / K2a / K2b stage measurements")
    ap.add_argument("--cpu-sample-rows", type=int, default=1_000_000)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed region, write the results of its last step (ids, score, semantic, "
                         "keyword, status of every sub-query, as float64) to DIR/<name>.npy, so that two "
                         "builds can be compared output for output on the same seeded inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the results of the CUDA path (--impl ours)")
    return args


# ------------------------------------------------------------------ clocks
class ClockSampler:
    """Samples SM clock / throttle reasons of one GPU while the timed region runs."""

    def __init__(self, index: int):
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._t = None
        self._nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nvml = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self._nvml = None

    def _loop(self):
        nv = self._nvml
        names = {}
        for n in dir(nv):
            if n.startswith("nvmlClocksThrottleReason") or n.startswith("nvmlClocksEventReason"):
                v = getattr(nv, n)
                if isinstance(v, int) and v not in (0,):
                    names[v] = n.replace("nvmlClocksThrottleReason", "").replace("nvmlClocksEventReason", "")
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM))
                mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
                for bit, name in names.items():
                    if mask & bit and bit & (bit - 1) == 0:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.02)

    def start(self):
        if self._nvml is not None:
            self._t = threading.Thread(target=self._loop, daemon=True)
            self._t.start()

    def stop(self):
        self._stop.set()
        if self._t is not None:
            self._t.join()
        reasons = sorted(r for r in self.reasons if r not in ("GpuIdle", "None", "ApplicationsClocksSetting"))
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None,
                "sm_max_mhz": self.max_mhz, "reasons": reasons, "samples": len(self.samples)}


# ------------------------------------------------------------- query pool
def make_query_pool(seed=999):
    from legal_rag_engine_b200 import synth
    q = synth.host_queries(POOL * N_SUB, seed=4321).reshape(POOL, N_SUB, 384)
    terms, _ = synth.host_query_terms(POOL * N_SUB, N_TERMS, seed=seed)
    terms = terms.reshape(POOL, N_SUB * N_TERMS)
    ptr = (np.arange(N_SUB + 1) * N_TERMS).astype(np.int32)
    return q, terms, ptr


# ------------------------------------------------------- fusion, restated for the parity check
def fuse_expected(dense, sparse, maxbm, k, w, mode):
    """retrieval_engine.py:71-96 (linear) / the build definition of RRF (SURVEY.md 8 A11) on the
    brute-force lists.  dense / sparse: [(id, dense_f64, bm25_f64)] best first."""
    mx = maxbm if maxbm > 0 else 1.0
    if mode == "linear":
        rows = []
        for i, de, bm in dense:
            sem = float(np.float32(de))
            kw = bm / mx
            rows.append((i, sem * (1 - w) + kw * w, sem, kw))
        rows.sort(key=lambda r: r[1], reverse=True)          # stable
        return rows[:k]
    acc, info = {}, {}
    for r, (i, de, bm) in enumerate(dense, start=1):
        acc[i] = 0.0 + 1.0 / (RRF_K0 + r)
        info[i] = (de, bm)
    for r, (i, de, bm) in enumerate(sparse, start=1):
        acc[i] = acc.get(i, 0.0) + 1.0 / (RRF_K0 + r)
        info[i] = (de, bm)
    items = sorted(acc.items(), key=lambda kv: (-kv[1], kv[0]))[:k]
    return [(i, s, float(np.float32(info[i][0])), info[i][1] / mx) for i, s in items]


def parity_check(dev, lo, n_local, avgdl, qh, th, pool_ids, k, mode, searcher, ptr_dev, w_dev, world, rank):
    """Untimed result check at the benchmark's own size: for the pool queries `pool_ids`, every
    rank computes on its shard, with torch float64 on the device buffers the kernels read,
      * exact inner products of all rows (fp16 x fp16 products and their sums are exact in float64
        in any order) -> local top-2k by (score desc, id asc),
      * BM25Okapi scores of all local documents, token by token in rank_bm25's operation order
        -> local max and local top-2k positive scores;
    the lists are all-gathered, merged, fused by `fuse_expected` and compared BIT FOR BIT with what
    the engine returns (ids, fused score, semantic, keyword).  Returns (queries checked, mismatches)."""
    import torch
    import torch.distributed as dist
    device = dev.device
    K = 2 * k
    PAD = 32
    tp, p8, idf_t = dev._post
    x = dev.x
    nq = len(pool_ids) * N_SUB
    Q = torch.from_numpy(np.concatenate([qh[p] for p in pool_ids], 0)).to(device)      # [nq,384] fp16
    Qd = Q.double()
    # ---- dense: exact scores chunk by chunk, running top-(K+PAD)
    best_s = torch.full((nq, 0), 0.0, dtype=torch.float64, device=device)
    best_i = torch.zeros((nq, 0), dtype=torch.int64, device=device)
    chunk = 1 << 20
    for r0 in range(0, n_local, chunk):
        r1 = min(n_local, r0 + chunk)
        s = Qd @ x[r0:r1].double().T                                   # [nq, rows]
        kk = min(K + PAD, r1 - r0)
        v, i = torch.topk(s, kk, dim=1)
        best_s = torch.cat([best_s, v], 1)
        best_i = torch.cat([best_i, i + (lo + r0)], 1)
        if best_s.shape[1] > 4 * (K + PAD):
            v, j = torch.topk(best_s, K + PAD, dim=1)
            best_s, best_i = v, torch.gather(best_i, 1, j)
        del s
    kk = min(K + PAD, best_s.shape[1])
    v, j = torch.topk(best_s, kk, dim=1)
    d_s = torch.full((nq, K + PAD), -float("inf"), dtype=torch.float64, device=device)
    d_i = torch.full((nq, K + PAD), -1, dtype=torch.int64, device=device)
    d_s[:, :kk], d_i[:, :kk] = v, torch.gather(best_i, 1, j)
    # ---- BM25: all local documents
    k1, b = 1.5, 0.75
    avg_t = torch.tensor(avgdl, dtype=torch.float64, device=device)   # a TENSOR divisor: torch turns a
    #                                  division by a Python scalar into a multiplication by its reciprocal
    b_s = torch.zeros((nq, K + PAD), dtype=torch.float64, device=device)
    b_i = torch.full((nq, K + PAD), -1, dtype=torch.int64, device=device)
    b_max = torch.zeros(nq, dtype=torch.float64, device=device)
    bm_full = []
    for n, p in enumerate(pool_ids):
        for sq in range(N_SUB):
            score = torch.zeros(n_local, dtype=torch.float64, device=device)
            for t in th[p][sq * N_TERMS:(sq + 1) * N_TERMS]:
                t = int(t)
                if t < 0:
                    continue
                w = float(idf_t[t].item())
                if w == 0.0:
                    continue
                s0, s1 = int(tp[t].item()), int(tp[t + 1].item())
                if s1 == s0:
                    continue
                doc = p8[s0:s1, 0].long()
                w1 = p8[s0:s1, 1].long()
                tf = (w1 & 0xffff).double()
                dl = ((w1 >> 16) & 0xffff).double()
                den = tf + k1 * (1 - b + b * dl / avg_t)
                score[doc] += w * (tf * (k1 + 1) / den)                  # doc ids unique within a term
            qi = n * N_SUB + sq
            bm_full.append(score)
            pos = torch.where(score > 0, score, torch.zeros_like(score))
            b_max[qi] = pos.max() if n_local else 0.0
            kk = min(K + PAD, n_local)
            v, i = torch.topk(pos, kk)
            b_s[qi, :kk] = v
            b_i[qi, :kk] = torch.where(v > 0, i + lo, torch.full_like(i, -1))
    # ---- gather the shards' lists
    def gather(t):
        if world == 1:
            return t.unsqueeze(0)
        out = torch.empty((world,) + tuple(t.shape), dtype=t.dtype, device=device)
        dist.all_gather_into_tensor(out, t.contiguous())
        return out
    gd_s, gd_i, gb_s, gb_i = (gather(t).cpu().numpy() for t in (d_s, d_i, b_s, b_i))
    if world > 1:
        dist.all_reduce(b_max, op=dist.ReduceOp.MAX)
    maxbm = b_max.cpu().numpy()

    def merged(sc, ids, qi, positive):
        s = sc[:, qi, :].reshape(-1)
        i = ids[:, qi, :].reshape(-1)
        keep = (i >= 0) & ((s > 0) if positive else np.isfinite(s))
        s, i = s[keep], i[keep]
        order = np.lexsort((i, -s))[:K]
        return s[order], i[order]
    dense_lists = [merged(gd_s, gd_i, qi, False) for qi in range(nq)]
    sparse_lists = [merged(gb_s, gb_i, qi, True) for qi in range(nq)]
    # ---- the other score of every listed document (owned by exactly one shard)
    need_b = torch.zeros((nq, K), dtype=torch.float64, device=device)     # bm25 at dense hits
    need_d = torch.zeros((nq, K), dtype=torch.float64, device=device)     # dense at bm25 hits
    for qi in range(nq):
        di = torch.from_numpy(dense_lists[qi][1]).to(device)
        own = (di >= lo) & (di < lo + n_local)
        if own.any():
            need_b[qi, :len(di)][own] = bm_full[qi][di[own] - lo]
        si = torch.from_numpy(sparse_lists[qi][1]).to(device)
        own = (si >= lo) & (si < lo + n_local)
        if own.any():
            need_d[qi, :len(si)][own] = x[si[own] - lo].double() @ Qd[qi]
    if world > 1:
        dist.all_reduce(need_b)
        dist.all_reduce(need_d)
    need_b, need_d = need_b.cpu().numpy(), need_d.cpu().numpy()
    # ---- the engine's answers for the same queries
    bad = 0
    detail = []
    for n, p in enumerate(pool_ids):
        q_dev = torch.from_numpy(qh[p]).to(device)
        t_dev = torch.from_numpy(th[p]).to(device)
        outs = searcher.search_checked(q_dev, t_dev, ptr_dev, k, {"linear": 0, "rrf": 1}[mode], w_dev)
        ids, score, sem, kw, _ = [o.cpu().numpy() for o in outs]
        ok = True
        for sq in range(N_SUB):
            qi = n * N_SUB + sq
            ds, di = dense_lists[qi]
            ss, si = sparse_lists[qi]
            dense = [(int(i), float(s), float(need_b[qi, j])) for j, (s, i) in enumerate(zip(ds, di))]
            sparse = [(int(i), float(need_d[qi, j]), float(s)) for j, (s, i) in enumerate(zip(ss, si))]
            want = fuse_expected(dense, sparse, float(maxbm[qi]), k, WEIGHTS[sq], mode)
            got = [(int(ids[sq, j]), float(score[sq, j]), float(sem[sq, j]), float(kw[sq, j]))
                   for j in range(k) if ids[sq, j] >= 0]
            if got != want:
                ok = False
                if len(detail) < 3:
                    detail.append({"pool": int(p), "sub": sq, "got": got[:3], "want": want[:3]})
        bad += 0 if ok else 1
    return len(pool_ids), bad, detail


# ------------------------------------------------------------ CPU baseline
class CpuReference:
    """The reference's CPU path for one user query on bounded samples (both stages are O(N) scans,
    scaled linearly in the number of chunks afterwards):
      dense : FAISS-style fp32 sequential scan + heap, one core per sub-query
              (oracle/c/flat_ip_scan.c, the published nq < 20 algorithm), on `sample_rows` rows;
      BM25  : rank_bm25's dict-per-document list-comprehension, literally
              (oracle.bm25.BM25OkapiLiteral), on a `bm_docs`-document sample;
      fusion: the two max() sweeps (:74) + RRF over the two top-2k lists."""

    def __init__(self, sample_rows: int, threads: int, bm_docs: int = 20_000):
        from legal_rag_engine_b200 import synth
        from oracle import bm25 as obm25
        self.sample_rows, self.bm_docs, self.threads = sample_rows, bm_docs, threads
        rng = np.random.default_rng(5)
        xs = rng.standard_normal((sample_rows, 384), dtype=np.float32)
        xs /= np.linalg.norm(xs, axis=1, keepdims=True)
        self.xs = xs
        self.q, self.terms, _ = make_query_pool()
        idx = synth.host_bm25(bm_docs, seed=777)
        term_of = np.repeat(np.arange(idx.n_terms), np.diff(idx.term_ptr.astype(np.int64)))
        order = np.argsort(idx.postings[:, 0], kind="stable")
        docs = [[] for _ in range(bm_docs)]
        for t, d, f in zip(term_of[order], idx.postings[order, 0], idx.postings[order, 1]):
            docs[d].extend([str(t)] * int(f))
        self.lit = obm25.BM25OkapiLiteral(docs)

    def step(self, s: int):
        """-> (dense seconds, bm25 + max + fusion seconds) of one user query on the samples."""
        from oracle import cbaseline, fusion
        from oracle import bm25 as obm25
        qs = self.q[s % POOL].astype(np.float32)
        t0 = time.perf_counter()
        D, I = cbaseline.flat_ip_search_f32(self.xs, qs, 2 * K_TOP, self.threads)
        t1 = time.perf_counter()
        for b in range(N_SUB):
            toks = [str(t) for t in self.terms[s % POOL][b * N_TERMS:(b + 1) * N_TERMS]]
            bm = self.lit.get_scores(toks)
            mx = max(bm) if max(bm) > 0 else 1.0       # the two Python max() sweeps (:74)
            Ib = np.minimum(I[b], self.bm_docs - 1)
            dense = [(int(i), float(d), float(bm[i])) for d, i in zip(D[b], Ib)]
            bs, bi = obm25.topk_positive(bm, 2 * K_TOP)
            sparse = [(int(i), 0.0, float(sc)) for sc, i in zip(bs, bi)]
            fusion.rrf_fuse(dense, sparse, mx, K_TOP)
        t2 = time.perf_counter()
        return t1 - t0, t2 - t1

    def run(self, steps: int, warmup: int, rows_total: int):
        for s in range(warmup):
            self.step(s)
        td = tb = 0.0
        for s in range(steps):
            a, b = self.step(warmup + s)
            td += a
            tb += b
        td /= steps
        tb /= steps
        full = td * rows_total / self.sample_rows + tb * rows_total / self.bm_docs
        return {"measured_ms_per_step_on_samples": (td + tb) * 1e3,
                "measured_dense_ms": td * 1e3, "measured_bm25_fusion_ms": tb * 1e3,
                "dense_sample_rows": self.sample_rows, "bm25_sample_docs": self.bm_docs,
                "dense_scale": rows_total / self.sample_rows, "bm25_scale": rows_total / self.bm_docs,
                "extrapolated_ms_per_step": full * 1e3,
                "extrapolated_split_s": {"dense": td * rows_total / self.sample_rows,
                                         "bm25_max_fusion": tb * rows_total / self.bm_docs}}

    def describe(self):
        return (f"dense: fp32 seq scan+heap on {self.sample_rows} rows x {N_SUB} sub-queries "
                f"({min(self.threads, N_SUB)} threads, one per sub-query as FAISS nq<20); BM25: literal "
                f"rank_bm25 dict loop on {self.bm_docs} docs x {N_SUB}x{N_TERMS} tokens (1 thread, pure "
                f"Python as the reference) + max() + RRF; both scaled linearly to the full corpus")


def run_reference(args):
    """Reference arm: the oracle port of the reference's CPU path, `--warmup` + `--steps` steps on
    bounded samples.  `value` is an ESTIMATE at the full configuration (linear in the rows), marked
    so; the measured per-step time on the samples is printed beside it."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    steps, warmup = max(1, args.steps), max(0, args.warmup)
    ref = CpuReference(args.cpu_sample_rows, threads)
    m = ref.run(steps, warmup, args.rows)
    qps = 1e3 / m["extrapolated_ms_per_step"]
    line = {
        "impl": "reference", "metric": metric_name(args),
        "value": qps, "unit": "queries/s", "n_gpus": args.gpus, "steps": steps,
        "warmup": warmup, "ms_per_step": m["extrapolated_ms_per_step"], "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32/f64", "data": "synthetic",
        "estimated": True,
        "estimate": m,
        "config": workload_config(args),
        "cpu_baseline": {"value": qps, "unit": "queries/s", "cores": threads, "kind": "port",
                         "sample": ref.describe()},
        "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def metric_name(args):
    if args.k == 10 and args.rows == 10_000_000:
        return "hybrid top-10 queries/sec @10Mx384 chunks"          # BASELINE.json's metric
    return f"hybrid top-{args.k} queries/sec @{args.rows}x384 chunks (not the headline config)"


def workload_config(args):
    return {"workload": f"{'C4' if args.k == 10 else 'C5-like'}: {args.rows} x 384 fp16 chunks + BM25 postings (50k-term Zipf vocab), "
                        f"{N_SUB} fan-out sub-queries x {N_TERMS} tokens per user query, top-{K_TOP}, "
                        f"fusion={args.fusion}",
            "rows": args.rows, "sub_queries": N_SUB, "k": K_TOP, "fusion": args.fusion,
            "encoder": "excluded (queries enter as fp16 vectors + term ids)",
            "l2": "inputs larger than L2 (>= 0.96 GB matrix shard per GPU streamed every step)"}


# ------------------------------------------------ CPU legs of BASELINE.md section 4 (N = 1, rank 0)
def cpu_legs(dev, n_local, avgdl, th, threads):
    """Measured on the box's host cores, bounded to a few seconds each:
      bm25_csr_full : the "fair CPU" BM25 -- CSR gather in C (oracle/c, float64, rank_bm25's operation
                      order) over the FULL corpus: the posting lists of the query's terms are copied
                      from the GPU index as they are, the score vector has one float64 per document;
      dense_blas    : torch.mm fp32 + topk, B = 1024 over 1 M rows (FAISS's BLAS regime, nq >= 20);
      encoder_hf    : transformers.BertModel fp32 on CPU, B = 32, S = 128 (random-init MiniLM-L6)."""
    import ctypes as C
    import torch
    from oracle import cbaseline
    out = {"cores": threads}
    # ---- fair-CPU BM25 at full size
    try:
        tp, p8, idf_t = dev._post
        terms = sorted({int(t) for t in th[0] if t >= 0})
        tph = tp.cpu().numpy()
        remap = {t: i for i, t in enumerate(terms)}
        ptr = np.zeros(len(terms) + 1, dtype=np.int64)
        docs, tfs = [], []
        for i, t in enumerate(terms):
            seg = p8[int(tph[t]):int(tph[t + 1])].cpu().numpy()
            docs.append(seg[:, 0].astype(np.int64))
            tfs.append((seg[:, 1] & 0xffff).astype(np.int64))
            ptr[i + 1] = ptr[i] + len(seg)
        post_doc, post_tf = np.concatenate(docs), np.concatenate(tfs)
        idf = idf_t.cpu().numpy()[terms].copy()
        dl = dev.doc_len.cpu().numpy().astype(np.float64)
        doc_norm = 1.5 * (1 - 0.75 + 0.75 * dl / avgdl)
        lib = cbaseline.load()
        t0 = time.perf_counter()
        n_post = 0
        for b in range(N_SUB):
            qt = np.array([remap[int(t)] for t in th[0][b * N_TERMS:(b + 1) * N_TERMS] if t >= 0], dtype=np.int32)
            score = np.zeros(n_local, dtype=np.float64)
            lib.oracle_bm25_scores(ptr.ctypes.data, post_doc.ctypes.data, post_tf.ctypes.data, idf.ctypes.data,
                                   doc_norm.ctypes.data, C.c_double(1.5), qt.ctypes.data, len(qt),
                                   score.ctypes.data)
            mx = score.max()
            n_post += int(sum(ptr[i + 1] - ptr[i] for i in qt))
        dt = time.perf_counter() - t0
        out["bm25_csr_full"] = {"docs": n_local, "postings_scored": n_post, "s_per_user_query": dt,
                                "threads": 1, "note": "C CSR gather + max over the full corpus, 4 sub-queries"}
        del post_doc, post_tf, docs, tfs
    except Exception as e:
        out["bm25_csr_full"] = {"error": repr(e)}
    # ---- dense, BLAS regime
    try:
        rows, Bq = 1_000_000, 1024
        rng = np.random.default_rng(7)
        xs = torch.from_numpy(rng.standard_normal((rows, 384), dtype=np.float32))
        qs = torch.from_numpy(rng.standard_normal((Bq, 384), dtype=np.float32))
        torch.set_num_threads(threads)
        torch.topk(qs @ xs.T, 20, dim=1)
        t0 = time.perf_counter()
        torch.topk(qs @ xs.T, 20, dim=1)
        dt = time.perf_counter() - t0
        out["dense_blas"] = {"rows": rows, "batch": Bq, "s_per_call": dt, "queries_per_s": Bq / dt,
                             "threads": threads}
        del xs, qs
    except Exception as e:
        out["dense_blas"] = {"error": repr(e)}
    # ---- encoder
    try:
        from transformers import BertConfig, BertModel
        cfg = BertConfig(vocab_size=30522, hidden_size=384, num_hidden_layers=6, num_attention_heads=12,
                         intermediate_size=1536, max_position_embeddings=512)
        model = BertModel(cfg, add_pooling_layer=False).eval()
        ids = torch.randint(1000, 30522, (32, 128))
        with torch.no_grad():
            model(input_ids=ids)
            t0 = time.perf_counter()
            model(input_ids=ids)
            dt = time.perf_counter() - t0
        out["encoder_hf"] = {"batch": 32, "seq_len": 128, "s_per_call": dt, "seq_per_s": 32 / dt,
                             "threads": threads}
    except Exception as e:
        out["encoder_hf"] = {"error": repr(e)}
    return out


# --------------------------------------------------- stage measurements (K1, K2a, K2b)
def measure_tokenisation():
    """SURVEY 8f N3: the host step in front of the path, on the reference's real corpus
    (tests/golden/legal_chunks.json.gz: 2 620 chunks) with a WordPiece vocabulary built from it
    (the checkpoint's vocab.txt is not on disk): queries/s of the per-query WordPiece + BM25
    whitespace tokenisation (retrieval_engine.py:61,67) and chunks/s of the index build's batch
    encode (create_vector_store.py:45,60)."""
    import gzip
    from collections import Counter
    from legal_rag_engine_b200.bm25_index import tokenize
    from legal_rag_engine_b200.tokenizer import WordPieceTokenizer, basic_tokenize
    chunks = json.loads(gzip.open(ROOT / "tests" / "golden" / "legal_chunks.json.gz", "rt", encoding="utf-8").read())
    texts = [c["text"] for c in chunks]
    cnt = Counter(w for t in texts for w in basic_tokenize(t))
    chars = sorted({ch for w in cnt for ch in w})
    vocab = ["[PAD]"] + [f"[unused{i}]" for i in range(99)] + ["[UNK]", "[CLS]", "[SEP]", "[MASK]"]
    vocab += chars + ["##" + c for c in chars] + [w for w, _ in cnt.most_common(8000) if len(w) > 1]
    tok = WordPieceTokenizer({w: i for i, w in enumerate(dict.fromkeys(vocab))})
    queries = ["What is the procedure for Zero FIR?", "Compensation for victims of acid attack",
               "Definition of a public servant under BNS", "Procedure after arrest of a suspect in rape case",
               "How to file FIR for robbery BNSS procedure", "What is the punishment for murder?"] * 200
    t0 = time.perf_counter()
    n_tok = sum(len(tok.encode(q, 256)) for q in queries)
    t_wp = time.perf_counter() - t0
    t0 = time.perf_counter()
    n_ws = sum(len(tokenize(q)) for q in queries)
    t_ws = time.perf_counter() - t0
    tok.encode_batch(texts[:200], 256)                                # builds the fast tokenizer once
    t0 = time.perf_counter()
    enc = tok.encode_batch(texts * 4, 256)[:len(texts)]
    t_b = (time.perf_counter() - t0) / 4
    t0 = time.perf_counter()
    n_ct = sum(len(tokenize(t)) for t in texts)
    t_c = time.perf_counter() - t0
    return {"query_wordpiece_per_s": len(queries) / t_wp, "query_whitespace_per_s": len(queries) / t_ws,
            "query_tokens": n_tok // len(queries), "build_wordpiece_chunks_per_s": len(texts) / t_b,
            "build_whitespace_chunks_per_s": len(texts) / t_c, "chunks": len(texts),
            "wordpiece_tokens": int(sum(len(e) for e in enc)), "whitespace_tokens": n_ct,
            "note": "host side, one process; the batch encode uses the multi-threaded `tokenizers` library when present"}



def measure_stages(dev, n_local, peaks, hbm_peak, th=None, ptr_h=None, fusion="rrf"):
    """Stages beside the headline (rank 0, N = 1).  Tensor-bound ones against the measured bf16 peak,
    HBM-bound ones against the measured copy bandwidth:
      encoder_sweep  config C2: K1 at B in {1..4096} x S in {128, 256} (seeded random weights);
      c3_*           config C3: dense top-10 over 1 M rows at batch 1, 4 (K2a, HBM) and 1024 (K2b);
      dense_batched  K2b at B = 1024 over the whole resident shard;
      search_text_host  the whole search with the encoder in the call."""
    import torch
    from legal_rag_engine_b200 import synth
    from legal_rag_engine_b200.device_index import DeviceIndex
    from legal_rag_engine_b200.encoder import SentenceEncoder
    peak_tf = float(peaks.get("bf16_tflops", 1590.0))
    peak_sus = float(peaks.get("bf16_tflops_sustained", peak_tf))
    out = {"peak_tflops": peak_tf, "peak_tflops_sustained": peak_sus,
           "peak_source": "measured (MEASURED_PEAKS.json bf16_tflops = burst, the denominator of `frac`; "
                          "bf16_tflops_sustained = back-to-back for 4 s, the denominator of `frac_sustained`)"
                          if "bf16_tflops" in peaks else "fallback 1590"}
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(fn, n_it, warm=2):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        ev0.record()
        for _ in range(n_it):
            fn()
        ev1.record()
        torch.cuda.synchronize()
        return ev0.elapsed_time(ev1) / n_it

    sd = synth.bert_state_dict(42, 0.02)
    enc = SentenceEncoder(dev, state_dict=sd)
    sweep = []
    for S in (128, 256):
        for B in (1, 4, 16, 64, 256, 1024, 4096):
            ids, lens = synth.token_batch(B, S, seed=1, full=True)
            d_ids, d_lens = torch.from_numpy(ids).to(dev.device), torch.from_numpy(lens).to(dev.device)
            ms = timed(lambda: enc.encode_ids_device(d_ids, d_lens), 5 if B >= 1024 else 20)
            flop = B * S * (6 * (2 * 384 * 1152 + 2 * 384 * 384 + 2 * 2 * 384 * 1536) + 6 * 4 * S * 384)
            rec = {"batch": B, "seq_len": S, "ms": ms, "seq_per_s": B / ms * 1e3, "tflops": flop / ms / 1e9,
                   "frac": flop / ms / 1e9 / peak_tf, "frac_sustained": flop / ms / 1e9 / peak_sus, "bound": "tensor"}
            sweep.append(rec)
            if B == 1024:
                out[f"encoder_S{S}"] = dict(rec, flop_per_seq=flop / B)
    out["encoder_sweep"] = sweep

    # ---- the whole of RetrievalEngine.search for one fan-out, encoder included: WordPiece ids and
    #      BM25 term ids in host memory -> K1 -> K2 || K3 -> K4 -> fused results in host memory
    if th is not None:
        S = 32
        ids, lens = synth.token_batch(N_SUB, S, seed=5, full=True)
        lists = [[th[p][b * N_TERMS:(b + 1) * N_TERMS].tolist() for b in range(N_SUB)] for p in range(POOL)]
        state = {"i": 0}

        def text_step():
            state["i"] += 1
            dev.search_text_host(ids, lens, lists[state["i"] % POOL], K_TOP, WEIGHTS, fusion)
        ms = timed(text_step, 30, warm=4)
        out["search_text_host"] = {"queries_per_s": 1e3 / ms, "ms": ms, "sub_queries": N_SUB, "seq_len": S,
                                   "note": "encoder (K1) + dense + BM25 + fusion in one call, host buffers "
                                           "in and out; random-init MiniLM-L6 weights"}
        d_ids, d_lens = torch.from_numpy(ids).to(dev.device), torch.from_numpy(lens).to(dev.device)
        ms = timed(lambda: enc.encode_ids_device(d_ids, d_lens), 30)
        out["encoder_query_batch"] = {"batch": N_SUB, "seq_len": S, "ms": ms}
        # the same call split in begin / end on three handles over the one index: three batches in
        # flight, one batch's encoder and small kernels under another's scans
        try:
            views = [dev.clone_view() for _ in range(2)]
            hs = [dev] + views
            encs = [SentenceEncoder(v, state_dict=sd) for v in views]
            sts = [torch.cuda.Stream(device=dev.device) for _ in hs]
            for d_, s_ in zip(hs, sts):
                with torch.cuda.stream(s_):
                    d_.use_current_stream()

            def run_pipe(n):
                for i in range(n):
                    d_ = hs[i % 3]
                    if i >= 3:
                        d_.search_host_end()
                    d_.search_text_host_begin(ids, lens, lists[i % POOL], K_TOP, WEIGHTS, fusion)
                for i in range(max(0, n - 3), n):
                    hs[i % 3].search_host_end()
            run_pipe(9)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            run_pipe(90)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            out["search_text_host_pipelined"] = {"queries_per_s": 90 / dt, "ms": dt / 90 * 1e3, "in_flight": 3,
                                                 "call": "lrx_search_text_host_begin / lrx_search_host_end"}
            del encs
            for v in views:
                v.close()
            dev.use_current_stream()
        except Exception as e:                                        # a reported extra, never fatal
            out["search_text_host_pipelined"] = {"error": repr(e)}
    try:
        out["host_tokenisation"] = measure_tokenisation()
    except Exception as e:                                            # a reported extra, never fatal
        out["host_tokenisation"] = {"error": repr(e)}

    def k2b(d, rows, label):
        B, K = 1024, 2 * K_TOP
        q = torch.from_numpy(synth.host_queries(B, seed=4321)).to(d.device)
        for _ in range(2):
            res = d.dense_topk_batched(q, K)
        torch.cuda.synchronize()
        overflow = int(res[3].sum().item())
        d.profile(True)
        d.profile_read(0)
        ms = timed(lambda: d.dense_topk_batched(q, K), 3, warm=0)
        kms, kn = d.profile_read(0)
        d.profile(False)
        flop = 2.0 * B * 384 * rows                                   # algorithmic: one pass of Q . X^T
        return {"batch": B, "rows": rows, "K": K, "queries_per_s": B / ms * 1e3, "ms": ms,
                "gemm_ms": kms / 3, "tflops_call": flop / ms / 1e9, "frac_call": flop / ms / 1e9 / peak_tf,
                "frac_call_sustained": flop / ms / 1e9 / peak_sus,
                "tflops_gemm_kernels": flop / (kms / 3) / 1e9, "frac": flop / (kms / 3) / 1e9 / peak_tf,
                "bound": "tensor", "flops": "algorithmic 2*B*384*rows (the sampled first pass is NOT counted)",
                "candidate_overflow_queries": overflow, "config": label}

    out["dense_batched"] = k2b(dev, n_local, "resident shard")

    # ---- config C3: 1 M rows
    rows = min(1_000_000, n_local)
    d3 = DeviceIndex(dev.device.index)
    try:
        d3.set_corpus(dev.x[:rows], 0)
        for B in (1, 4):
            q = torch.from_numpy(synth.host_queries(B, seed=77)).to(dev.device)
            d3.dense_topk(q, 2 * K_TOP)
            d3.profile(True)
            d3.profile_read(0)
            ms = timed(lambda: d3.dense_topk(q, 2 * K_TOP), 20, warm=0)
            kms, kn = d3.profile_read(0)
            d3.profile(False)
            kern, row_bytes, sbytes = scan_kernel_of(d3, rows, 2 * K_TOP)
            gbs = sbytes / (kms / kn * 1e-3) / 1e9
            out[f"c3_dense_b{B}"] = {"rows": rows, "batch": B, "call_ms": ms, "queries_per_s": B / ms * 1e3,
                                     "kernel": kern, "bytes_per_row": row_bytes,
                                     "scan_ms": kms / kn, "achieved_GBps": gbs, "frac": gbs / hbm_peak,
                                     "frac_of_8TBs_nominal": gbs / 8000.0, "bound": "hbm"}
        out["c3_dense_b1024"] = k2b(d3, rows, "C3: 1 M rows")
    finally:
        d3.close()
    return out


def scan_kernel_of(dev, n_local, K):
    """(kernel name, algorithmic bytes per row, algorithmic bytes per launch) of the dense scan a
    search of depth K runs on this index: with the int8 shadow resident (lrx_build_dense_prefilter)
    the scan streams 384 B of int8 + a 4-byte scale per row of the shadow (padded to 128-row
    tiles) instead of the 768-byte fp16 row."""
    if dev.prefilter_bounds is not None and (K <= 64 or (K <= 224 and n_local >= 32768)):
        n_pad = (n_local + 127) // 128 * 128
        return "dense_scan_q8_kernel", 388, n_pad * 388
    return "dense_scan_kernel<4>", 768, n_local * 768


def scan_traffic_from_profile(n_local, kernel="dense_scan_kernel"):
    """dram bytes of the dense scan kernel from the committed ncu --set full capture (profiles/),
    scaled per row: the kernel reads each row exactly once, so bytes/row is size independent."""
    kernel = kernel.split("<")[0]
    for name in ("r2_scan_q8_full.json", "r2_scan_kernels_final_full.json", "r2_scan_kernels_full.json",
                 "r1_scan_kernels_v3_full.json"):
        try:
            prof = json.loads((ROOT / "profiles" / name).read_text())
            for l in prof["launches"]:
                if l["kernel"].split("<")[0].split("(")[0].endswith(kernel) and "traffic_bytes_per_launch" in l:
                    rows = prof.get("rows", 10_000_000)
                    return l["traffic_bytes_per_launch"] / rows * n_local, name
        except Exception:
            continue
    return None, None


# ------------------------------------------------------------------- ours
def run_ours(args):
    import torch
    import torch.distributed as dist
    from legal_rag_engine_b200 import synth
    from legal_rag_engine_b200.bm25_index import okapi_idf
    from legal_rag_engine_b200.device_index import DeviceIndex, FUSION

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torchrun for --gpus > 1")
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        # keep stdout to the one JSON line: NCCL prints its version banner there at VERSION level
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=device)

    # ---- this rank's shard: contiguous global id range (SURVEY 8e)
    per = -(-args.rows // world)
    lo, hi = rank * per, min(args.rows, (rank + 1) * per)
    n_local = hi - lo
    t_build = time.time()
    x = synth.device_vectors(n_local, device, seed=1234 + rank)
    bm = synth.device_bm25(n_local, device, seed=777 + rank)
    df = bm["df"].clone()
    tot_len = torch.tensor([int(bm["doc_len"].sum().item())], dtype=torch.int64, device=device)
    if world > 1:
        dist.all_reduce(df)
        dist.all_reduce(tot_len)
    idf, _ = okapi_idf(df.cpu().numpy(), args.rows)
    avgdl = int(tot_len.item()) / args.rows
    dev = DeviceIndex(local, rank, world)
    dev.set_corpus(x, lo, prefilter=(args.prefilter == "on"))
    dev.set_postings(bm["term_ptr"], bm["postings"], bm["doc_len"], idf, avgdl)
    nnz_local = bm["nnz"]
    df_local = bm["df"].cpu().numpy()
    del bm
    torch.cuda.synchronize()
    t_build = time.time() - t_build

    mode = FUSION[args.fusion]
    qh, th, ptr_h = make_query_pool()
    q_dev = torch.from_numpy(qh).to(device)
    t_dev = torch.from_numpy(th).to(device)
    ptr_dev = torch.from_numpy(ptr_h).to(device)
    w_dev = torch.tensor(WEIGHTS, dtype=torch.float64, device=device)
    from legal_rag_engine_b200.sharding import ShardedSearcher
    # `in_flight` query batches at a time, each on its own handle (same resident matrix and
    # postings, own workspaces / exchange region) and stream, so that one batch's merges,
    # exchange and fusion run under the next batch's scans.
    n_fly = max(1, args.in_flight)
    devs = [dev] + [dev.clone_view() for _ in range(n_fly - 1)]
    streams = [torch.cuda.Stream(device) for _ in range(n_fly)]
    for d, st in zip(devs, streams):
        with torch.cuda.stream(st):
            d.use_current_stream()
    searchers = [ShardedSearcher(d) for d in devs]     # K2+K3 local -> exchange -> K4
    searcher = searchers[0]
    all_outs = [sr.buffers(N_SUB, K_TOP)[2] for sr in searchers]

    def step(i):
        p, j = i % POOL, i % n_fly
        with torch.cuda.stream(streams[j]):
            searchers[j].search(q_dev[p], t_dev[p], ptr_dev, K_TOP, mode, w_dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # Every (handle, query buffer) pair needs a direct call and a capturing call before it replays.
    warm = max(args.warmup, 3, 2 * POOL * n_fly // math.gcd(POOL, n_fly) + n_fly)
    for i in range(warm):
        step(i)
    barrier()
    for o in all_outs:
        assert int(o[4].sum().item()) == 0, "status words set on the benchmark queries"

    # ---- parity at the benchmark's own size (untimed)
    parity = None
    if args.parity_queries > 0:
        with torch.cuda.stream(streams[0]):
            pool_ids = list(range(0, POOL, max(1, POOL // args.parity_queries)))[:args.parity_queries]
            t0 = time.time()
            n_checked, n_bad, detail = parity_check(dev, lo, n_local, avgdl, qh, th, pool_ids, K_TOP,
                                                    args.fusion, searcher, ptr_dev, w_dev, world, rank)
            parity = {"queries": n_checked, "sub_queries": n_checked * N_SUB, "mismatches": n_bad,
                      "against": "on-device float64 brute force of every shard (exact inner products of all "
                                 "rows; BM25Okapi of all documents in rank_bm25's operation order), lists "
                                 "all-gathered, merged (score desc, id asc), fused; ids, fused score, "
                                 "semantic and keyword compared bit for bit",
                      "seconds": round(time.time() - t0, 1)}
            if n_bad:
                parity["detail"] = detail
        barrier()
        if n_bad:
            if rank == 0:
                print(json.dumps({"error": "parity check failed", "parity": parity}), flush=True)
            raise SystemExit(3)

    # ---- timed region: device-resident queries
    clocks = ClockSampler(local)
    launches0 = sum(d.launches for d in devs)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed_block(n_steps, i0):
        barrier()
        ev0.record()
        for st in streams:
            st.wait_event(ev0)
        t_h = time.perf_counter()
        for i in range(n_steps):
            step(i0 + i)
        t_h = time.perf_counter() - t_h
        for st in streams:
            torch.cuda.current_stream().wait_stream(st)
        ev1.record()
        barrier()
        t = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), t_h

    clocks.start()
    ms, t_host = timed_block(args.steps, warm)
    timed_steps = args.steps
    clk = clocks.stop()
    launches = sum(d.launches for d in devs) - launches0
    for o in all_outs:
        assert int(o[4].sum().item()) == 0, "status words set in the timed region"
    if args.dump_outputs and rank == 0:
        # the last timed step ran on handle (warm + steps - 1) % n_fly; the results are replicated
        # on every rank.  Copied now: the passes below reuse the handles' output buffers.
        last_outs = all_outs[(warm + args.steps - 1) % n_fly]
        out_dir = Path(args.dump_outputs)
        out_dir.mkdir(parents=True, exist_ok=True)
        for name, t in zip(("ids", "score", "semantic", "keyword", "status"), last_outs):
            np.save(out_dir / f"{name}.npy", t.cpu().numpy().astype(np.float64))

    # ---- roofline pass: the same chain, the same queries, ONE batch in flight, with CUDA event
    #      nodes around the two streaming kernels inside the captured chains.  With two batches in
    #      flight an event pair would also time the wait for the other batch's CTAs to leave the SMs
    #      (two dense-scan CTAs do not fit one SM), not the kernel; the step time above is what two
    #      in flight buy, the kernel time below is what the kernel does while BM25 runs beside it.
    scan_ms = scan_n = bm_ms = bm_n = 0
    roof_steps = 0
    if args.kernel_events == "on":
        dev.profile(True)
        for i in range(2 * POOL):                               # direct call + capture with the event nodes
            with torch.cuda.stream(streams[0]):
                searchers[0].search(q_dev[i % POOL], t_dev[i % POOL], ptr_dev, K_TOP, mode, w_dev)
        barrier()
        dev.profile_read(0); dev.profile_read(1)
        roof_steps = max(args.steps, POOL)
        ev0.record()
        streams[0].wait_event(ev0)
        for i in range(roof_steps):
            with torch.cuda.stream(streams[0]):
                searchers[0].search(q_dev[i % POOL], t_dev[i % POOL], ptr_dev, K_TOP, mode, w_dev)
        torch.cuda.current_stream().wait_stream(streams[0])
        ev1.record()
        barrier()
        roof_step_ms = ev0.elapsed_time(ev1) / roof_steps
        scan_ms, scan_n = dev.profile_read(0)
        bm_ms, bm_n = dev.profile_read(1)
        dev.profile(False)

    # ---- end to end: host buffers through the C ABI (lrx_search_host_begin / _end), the H2D copy of
    #      every step's inputs and the D2H copy of its results inside the timed region, the same
    #      number of batches in flight
    h2d = N_SUB * 384 * 2 + N_SUB * N_TERMS * 4 + (N_SUB + 1) * 4 + N_SUB * 8
    d2h = N_SUB * K_TOP * (8 * 4) + N_SUB * 4
    lists = [[th[p][b * N_TERMS:(b + 1) * N_TERMS].tolist() for b in range(N_SUB)] for p in range(POOL)]

    def e2e_run(n):
        res = None
        for i in range(n):
            d = devs[i % n_fly]
            if i >= n_fly:
                res = d.search_host_end()
            d.search_host_begin(qh[i % POOL], lists[i % POOL], K_TOP, WEIGHTS, args.fusion)
        for i in range(max(0, n - n_fly), n):
            res = devs[i % n_fly].search_host_end()
        return res

    e2e_run(max(6, 3 * n_fly))
    barrier()
    e2e_steps = args.steps
    ev0.record()
    last = e2e_run(e2e_steps)
    ev1.record()
    barrier()
    e2e_ms = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(e2e_ms, op=dist.ReduceOp.MAX)
    e2e_ms = float(e2e_ms.item())
    assert last is not None and (last[0][:, 0] >= 0).all()

    # ---- two user queries per launch chain (8 sub-queries): ONE pass of the matrix serves both --
    #      the dense scan's MMA tile has 8 query columns either way (SURVEY 8(d): "matrix read once
    #      regardless of B <= 16") -- which is what a serving front does with concurrent requests
    #      (serving.MicroBatchingEngine).  Same host-buffer calls, same batches in flight; NOT the
    #      headline (a step of `value` / `e2e` is one user query), reported beside it.
    batched = None
    try:
        q2 = [np.ascontiguousarray(np.concatenate([qh[p], qh[(p + 1) % POOL]], 0)) for p in range(POOL)]
        l2 = [lists[p] + lists[(p + 1) % POOL] for p in range(POOL)]

        def two_run(n):
            for i in range(n):
                d = devs[i % n_fly]
                if i >= n_fly:
                    d.search_host_end()
                d.search_host_begin(q2[i % POOL], l2[i % POOL], K_TOP, WEIGHTS * 2, args.fusion)
            for i in range(max(0, n - n_fly), n):
                devs[i % n_fly].search_host_end()
        two_run(max(6, 3 * n_fly))
        barrier()
        two_steps = args.steps
        ev0.record()
        two_run(two_steps)
        ev1.record()
        barrier()
        two_ms = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(two_ms, op=dist.ReduceOp.MAX)
        two_ms = float(two_ms.item())
        batched = {"users_per_step": 2, "sub_queries_per_step": 2 * N_SUB,
                   "value": 2 * two_steps / (two_ms * 1e-3), "unit": "queries/s",
                   "ms_per_step": two_ms / two_steps, "steps": two_steps, "in_flight": n_fly,
                   "call": "lrx_search_host_begin / lrx_search_host_end (host buffers in and out)",
                   "note": "two user queries share one matrix pass; not the headline"}
    except Exception as e:                                            # a reported extra, never fatal
        batched = {"error": repr(e)}

    # ---- the dominant kernel ALONE (no BM25 scan beside it): the same launches through
    #      lrx_dense_topk, events inside the library -- what the kernel does with the HBM to itself
    dev.use_current_stream()           # handle 0 back on torch's default stream for what follows
    dev.profile(True); dev.profile_read(0); dev.profile_read(1)
    for i in range(20):
        dev.dense_topk(q_dev[i % POOL], 2 * K_TOP)
    torch.cuda.synchronize()
    alone_ms, alone_n = dev.profile_read(0)
    for i in range(20):
        dev.bm25(t_dev[i % POOL], ptr_dev, None, 2 * K_TOP if args.fusion == "rrf" else 0)
    torch.cuda.synchronize()
    bm_alone_ms, bm_alone_n = dev.profile_read(1)
    dev.profile(False)

    # ---- roofline of the dominant kernel (dense_scan_kernel), algorithmic bytes / event time
    peaks = {}
    try:
        peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
    scan_kernel, scan_row_bytes, scan_bytes = scan_kernel_of(dev, n_local, 2 * K_TOP)
    scan_gbs = scan_bytes / (scan_ms / max(scan_n, 1) * 1e-3) / 1e9 if scan_ms > 0 else 0.0
    # BM25 kernel: sum over query tokens of df_local * 8 B ({u32 doc, u16 tf, u16 len}),
    # averaged over the pool
    bm_bytes = float(np.mean([df_local[th[p]].sum() * 8 for p in range(POOL)]))
    bm_gbs = bm_bytes / (bm_ms / max(bm_n, 1) * 1e-3) / 1e9 if bm_ms > 0 else 0.0
    bm_alone_gbs = bm_bytes / (bm_alone_ms / max(bm_alone_n, 1) * 1e-3) / 1e9 if bm_alone_ms > 0 else 0.0
    traffic, traffic_src = scan_traffic_from_profile(n_local, scan_kernel)
    q8 = scan_row_bytes != 768

    if rank == 0:
        qps = timed_steps / (ms * 1e-3)
        step_ms = ms / timed_steps
        line = {
            "metric": metric_name(args),
            "value": qps, "unit": "queries/s", "n_gpus": world, "steps": args.steps,
            "warmup": warm, "ms_per_step": step_ms,
            "timed_steps": timed_steps, "timed_region_ms": ms,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": ("f16 matrix + its int8 shadow: s8 x s8 -> s32 scan of the shadow, exact f64 re-score "
                      "of the fp16 rows; f64 BM25" if q8 else
                      "f16 matrix, f32 scan + exact f64 re-score; f64 BM25"), "data": "synthetic",
            "config": dict(workload_config(args), parallelism=f"row-shard x{world}",
                           exchange=(searcher.exchange if world > 1 else "none"),
                           in_flight=n_fly, launch="one captured CUDA graph per batch",
                           rows_per_gpu=n_local, nnz_per_gpu=nnz_local, build_s=round(t_build, 1),
                           dense_prefilter=("int8 shadow, bounds (max row error, max row norm) = "
                                            f"{dev.prefilter_bounds}" if q8 else "off")),
            "parity": parity,
            "e2e": {"value": e2e_steps / (e2e_ms * 1e-3), "unit": "queries/s",
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": e2e_ms / e2e_steps, "steps": e2e_steps, "in_flight": n_fly,
                    "call": "lrx_search_host_begin / lrx_search_host_end (host buffers in and out)"},
            "two_users_per_step": batched,
            "gpu_launches": int(launches),
            "host_enqueue_ms_per_step": t_host * 1e3 / timed_steps,
            "clocks": clk,
            "roofline": {"bound": "hbm", "kernel": scan_kernel, "achieved": scan_gbs,
                         "peak": peak, "unit": "GB/s", "frac": scan_gbs / peak, "peak_source": peak_src,
                         "peak_note": "the measured peak is a COPY (reads + writes); a read-only stream can "
                                      "exceed it, so frac may pass 1 -- see frac_of_8TBs_nominal",
                         "frac_of_8TBs_nominal": scan_gbs / 8000.0, "traffic": traffic,
                         "traffic_source": f"ncu --set full dram__bytes_read+write per launch "
                                           f"(profiles/{traffic_src}), scaled by rows",
                         "bytes_per_launch": scan_bytes, "bytes_per_row": scan_row_bytes,
                         "bytes_note": ("algorithmic bytes of THIS kernel: 384 int8 + one fp32 scale per row of "
                                        "the shadow; the fp16 matrix (768 B/row, SURVEY 8d) is only read at the "
                                        "256 merged candidates per sub-query" if q8 else
                                        "768 B per fp16 row (SURVEY 8d)"),
                         "fp16_matrix_equivalent_GBps": (n_local * 768 / (scan_ms / max(scan_n, 1) * 1e-3) / 1e9
                                                         if scan_ms > 0 else 0.0),
                         "ms_per_launch": scan_ms / max(scan_n, 1),
                         "launches_timed": int(scan_n),
                         "timing": "CUDA event nodes around the kernel inside the captured chains; a pass of "
                                   f"{roof_steps} steps with ONE batch in flight right after the timed region "
                                   "(with two in flight an event pair also times the wait for the other "
                                   "batch's CTAs to leave the SMs); last replay of every chain",
                         "pass_ms_per_step": roof_step_ms if roof_steps else None,
                         "share_of_step": (scan_ms / max(scan_n, 1)) / roof_step_ms if roof_steps else None,
                         "alone": {"note": "the same kernel with the GPU to itself (20 launches of "
                                           "lrx_dense_topk after the timed region, same events)",
                                   "ms_per_launch": alone_ms / max(alone_n, 1),
                                   "achieved": scan_bytes / (alone_ms / max(alone_n, 1) * 1e-3) / 1e9
                                   if alone_ms > 0 else 0.0,
                                   "frac": scan_bytes / (alone_ms / max(alone_n, 1) * 1e-3) / 1e9 / peak
                                   if alone_ms > 0 else 0.0},
                         "concurrent": {"note": "bm25_scan_kernel runs on the same SMs at the same time "
                                                "(side stream) and, with two batches in flight, so do the "
                                                "other batch's kernels: they share the HBM bandwidth",
                                        "bytes_per_step": scan_bytes + bm_bytes,
                                        "step_achieved": (scan_bytes + bm_bytes) / (step_ms * 1e-3) / 1e9,
                                        "step_frac": (scan_bytes + bm_bytes) / (step_ms * 1e-3) / 1e9 / peak}},
            "bm25_kernel": {"kernel": "bm25_scan_kernel", "bound": "hbm",
                            "in_step": {"achieved": bm_gbs, "frac": bm_gbs / peak,
                                        "ms_per_launch": bm_ms / max(bm_n, 1),
                                        "note": "sharing the SMs and the HBM with the dense scan"},
                            "alone": {"achieved": bm_alone_gbs, "frac": bm_alone_gbs / peak,
                                      "ms_per_launch": bm_alone_ms / max(bm_alone_n, 1)},
                            "unit": "GB/s", "bytes_per_launch": bm_bytes},
        }
        if world == 1 and not args.no_stages:
            try:
                line["stages"] = measure_stages(dev, n_local, peaks, peak, th, ptr_h, args.fusion)
            except Exception as e:                      # a stage problem must not void the headline
                line["stages"] = {"error": repr(e)}
        if world == 1 and not args.no_cpu_baseline:
            threads = os.cpu_count() or 1
            ref = CpuReference(args.cpu_sample_rows, threads)
            m = ref.run(2, 1, args.rows)
            line["cpu_baseline"] = {"value": 1e3 / m["extrapolated_ms_per_step"], "unit": "queries/s",
                                    "cores": threads, "kind": "port", "estimated": True,
                                    "sample": ref.describe(), "estimate": m}
            del ref
            try:
                line["cpu_legs"] = cpu_legs(dev, n_local, avgdl, th, threads)
            except Exception as e:
                line["cpu_legs"] = {"error": repr(e)}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()                 # nobody unmaps its exchange region while a peer may store
    for d in devs[1:]:
        d.close()
    dev.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    global K_TOP
    args = parse()
    K_TOP = args.k
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
