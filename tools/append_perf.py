#!/usr/bin/env python
"""Index append at scale: a 10 M-row synthetic index (synth.device_vectors / device_bm25) grown by
m = 1 000, 10 000, 100 000 rows in turn.  Per append: ms of each phase (matrix append, int8 shadow
rebuild, postings merge, lrx_set_postings), the merge's algorithmic bytes over its time beside a
cudaMemcpyAsync D2D moving the same bytes, and search queries/s on the grown index against an index
built from scratch over the same rows.  Also the host rebuild the append replaces (BM25Index.from_texts
on a sample, and the lrx_set_postings upload of the whole index).

    python tools/append_perf.py [--rows 10000000] [--out profiles/append_perf_b200.json]
"""
import argparse
import ctypes as C
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
from legal_rag_engine_b200 import synth                                  # noqa: E402
from legal_rag_engine_b200.bm25_index import BM25Index, okapi_idf       # noqa: E402
from legal_rag_engine_b200.device_index import DeviceIndex, _ptr        # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--rows", type=int, default=10_000_000)
ap.add_argument("--adds", default="1000,10000,100000")
ap.add_argument("--reps", type=int, default=5, help="timed repeats of the merge and of the copy")
ap.add_argument("--search-iters", type=int, default=100)
ap.add_argument("--host-docs", type=int, default=100_000, help="documents of the host rebuild sample")
ap.add_argument("--out", default=None)
a = ap.parse_args()


def power_limit():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    r = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1), r


def qps(d, q, lists, k=5, iters=100):
    w = [0.5] * len(lists)
    for _ in range(3):
        d.search_batch_host(q, lists, k, w)
    torch.cuda.synchronize()
    t = time.perf_counter()
    for _ in range(iters):
        out = d.search_batch_host(q, lists, k, w)
    return len(lists) * iters / (time.perf_counter() - t), out


dev = DeviceIndex(0)
gpu = torch.cuda.get_device_name(0)
res = {"gpu": gpu, "power_limit": power_limit(), "rows": a.rows, "appends": []}
x = synth.device_vectors(a.rows, dev.device, seed=1234)
bm = synth.device_bm25(a.rows, dev.device, seed=777)
dev.set_corpus(x, 0, prefilter=True)
dev.set_postings(bm["term_ptr"], bm["postings"], bm["doc_len"], bm["idf"], bm["avgdl"])
df = bm["df"].cpu().numpy().astype(np.int64)
total_len = int(bm["doc_len"].sum().item())
del x, bm
torch.cuda.empty_cache()
B = 4
q = synth.host_queries(B, seed=4321)
terms, ptr = synth.host_query_terms(B, 8, seed=999)
lists = [terms[ptr[b]:ptr[b + 1]].tolist() for b in range(B)]

for i, m in enumerate(int(s) for s in a.adds.split(",")):
    n = dev.n_local
    xa = synth.device_vectors(m, dev.device, seed=5000 + i)
    ba = synth.device_bm25(m, dev.device, seed=6000 + i)
    add_ptr = ba["term_ptr"]
    add_post = ba["postings"].clone()
    add_post[:, 0] += n
    add_len = ba["doc_len"]
    df = df + ba["df"].cpu().numpy()
    total_len += int(add_len.sum().item())
    idf, _ = okapi_idf(df, n + m)
    avgdl = total_len / (n + m)
    row = {"n_before": n, "m": m}

    # postings merge: the kernels alone, into buffers of their own, repeated
    tp, p8, _ = dev._post
    nnz = dev._post_args[0]
    nnz_add = int(add_ptr[-1].item())
    V_out = int(add_ptr.numel() - 1)
    dl = torch.cat([dev.doc_len[:dev.n_docs], add_len])
    tp_out = torch.empty(V_out + 1, dtype=torch.int64, device=dev.device)
    p8_out = torch.empty((nnz + nnz_add + 2, 2), dtype=torch.int32, device=dev.device)
    merge = lambda: dev._ck(dev.lib.lrx_bm25_append_postings(
        dev.h, _ptr(tp), _ptr(p8), dev.n_terms, nnz, dev.n_docs, _ptr(add_ptr), _ptr(add_post), V_out, nnz_add,
        _ptr(dl), n + m, _ptr(tp_out), _ptr(p8_out)))
    merge()
    ms = sorted(timed(merge)[0] for _ in range(a.reps))
    # bytes the merge must move: old postings read + written, appended pairs read + postings written,
    # the three pointer tables
    nbytes = 16 * nnz + 16 * nnz_add + 8 * (dev.n_terms + 1) + 16 * (V_out + 1)
    src = torch.empty(nbytes // 2, dtype=torch.uint8, device=dev.device)
    dst = torch.empty_like(src)
    dst.copy_(src)
    cp = sorted(timed(lambda: dst.copy_(src))[0] for _ in range(a.reps))
    del src, dst
    row.update(merge_ms=ms[len(ms) // 2], merge_bytes=nbytes, merge_GBps=nbytes / ms[len(ms) // 2] / 1e6,
               memcpy_same_bytes_ms=cp[len(cp) // 2], memcpy_GBps=nbytes / cp[len(cp) // 2] / 1e6,
               merge_over_memcpy_rate=cp[len(cp) // 2] / ms[len(ms) // 2])
    del tp_out, p8_out, dl
    # the engine's path, phase by phase: postings (merge + set_postings), matrix, shadow
    row["append_postings_ms"], _ = timed(lambda: dev.append_postings(add_ptr.cpu().numpy(),
                                                                     add_post.cpu().numpy(),
                                                                     add_len.cpu().numpy(), idf, avgdl))
    tp, p8, idf_t = dev._post
    row["set_postings_ms"], _ = timed(lambda: dev._ck(dev.lib.lrx_set_postings(
        dev.h, _ptr(tp), _ptr(p8), _ptr(idf_t), dev.n_terms, dev._post_args[0], *dev._post_args[1:])))
    cap = dev.capacity
    dev._prefilter_on = False                         # matrix alone; the shadow is timed next
    row["matrix_append_ms"], _ = timed(lambda: dev.append_rows(xa))
    row["matrix_grew"] = dev.capacity != cap
    row["shadow_rebuild_ms"], _ = timed(dev.build_prefilter)
    # search on the grown index vs an index built from scratch over the same rows and postings
    row["qps_grown"], got = qps(dev, q, lists, iters=a.search_iters)
    ref = DeviceIndex(0)
    tp_h, pairs, dl_h = dev.read_postings()
    ref.set_corpus(dev.x.clone(), 0, prefilter=True)
    ref.set_postings(tp_h, pairs, dl_h, idf, avgdl)
    del tp_h, pairs, dl_h
    row["qps_scratch"], want = qps(ref, q, lists, iters=a.search_iters)
    row["qps_grown_again"], _ = qps(dev, q, lists, iters=a.search_iters)
    row["results_equal"] = all(np.array_equal(u, v) for u, v in zip(got, want))
    ref.close()
    del ref, xa, ba, add_post
    torch.cuda.empty_cache()
    res["appends"].append(row)
    print(json.dumps(row), flush=True)

# the host rebuild the append replaces: BM25Index.from_texts over a sample of synthetic documents
# (measured), and the lrx_set_postings upload of the whole index (measured at full size)
rng = np.random.default_rng(7)
vocab = np.array([f"w{i}" for i in range(synth.VOCAB)])
lens = synth.host_doc_lengths(a.host_docs, rng)
cdf = synth._zipf_cdf(synth.VOCAB)
toks = vocab[np.minimum(np.searchsorted(cdf, rng.random(int(lens.sum())), side="right"), synth.VOCAB - 1)]
texts = [" ".join(t) for t in np.split(toks, np.cumsum(lens)[:-1])]
t = time.perf_counter()
BM25Index.from_texts(texts)
host_s = time.perf_counter() - t
tp_h, pairs, dl_h = dev.read_postings()
idf_h = dev._post[2].cpu().numpy()
up = DeviceIndex(0)
torch.cuda.synchronize()
t = time.perf_counter()
up.set_postings(tp_h, pairs, dl_h, idf_h, dev._post_args[1])
torch.cuda.synchronize()
res["host_rebuild"] = {"from_texts_docs": a.host_docs, "from_texts_s": host_s,
                       "from_texts_s_per_million_docs": host_s / a.host_docs * 1e6,
                       "set_postings_upload_s": time.perf_counter() - t, "upload_docs": dev.n_docs}
up.close()
print(json.dumps({"gpu": gpu, "power_limit": res["power_limit"], "host_rebuild": res["host_rebuild"]}), flush=True)
if a.out:
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text(json.dumps(res, indent=1) + "\n")
dev.close()
