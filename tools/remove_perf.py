#!/usr/bin/env python
"""Index removal at scale: a 10 M-row synthetic index (synth.device_vectors / device_bm25) shrunk by
m = 1 000, 10 000, 100 000 scattered rows and one contiguous block of 100 000, in turn.  Per removal:
the postings compaction (lrx_bm25_remove_postings, median of --reps calls, CUDA events) with its
bytes and rate beside a cudaMemcpyAsync D2D moving the same bytes, lrx_set_postings, the matrix
compaction and the int8 shadow rebuild, and search queries/s on the shrunk index against an index
built from scratch over the same rows and postings.  Also the host plan (bm25_index.csr_remove) on
the reference corpus and on a synthetic text corpus, beside the host rebuild it replaces.

    python tools/remove_perf.py [--rows 10000000] [--out profiles/remove_perf_b200.json]
"""
import argparse
import gzip
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
from legal_rag_engine_b200.bm25_index import (BM25Index, BM25Remove, BM25Stats, _ranges,  # noqa: E402
                                              csr_remove, okapi_idf, tokenize)
from legal_rag_engine_b200.device_index import DeviceIndex, _ptr        # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--rows", type=int, default=10_000_000)
ap.add_argument("--removals", default="1000,10000,100000,block100000")
ap.add_argument("--reps", type=int, default=5, help="timed repeats of the compaction and of the copy")
ap.add_argument("--search-iters", type=int, default=100)
ap.add_argument("--host-docs", type=int, default=100_000, help="documents of the synthetic text corpus")
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


def device_plan(dev, removed, df, total_len):
    """The removal plan of a synthetic index (no string vocabulary: the surviving terms keep their
    relative order), from the resident postings."""
    tp, p8, _ = dev._post
    nnz = dev._post_args[0]
    V = dev.n_terms
    doc = p8[:nnz, 0]
    gone = torch.isin(doc, removed.to(torch.int32))
    term_of = torch.repeat_interleave(torch.arange(V, device=dev.device), tp[1:] - tp[:-1])
    t_gone = term_of[gone]
    del term_of
    r = torch.bincount(t_gone, minlength=V).cpu().numpy().astype(np.int64)
    rem_doc = doc[gone].cpu().numpy().view(np.uint32)
    del gone, t_gone
    rem_ptr = np.zeros(V + 1, dtype=np.int64)
    np.cumsum(r, out=rem_ptr[1:])
    df_out = df - r
    alive = np.nonzero(df_out > 0)[0]
    term_map = np.full(V, -1, dtype=np.int32)
    term_map[alive] = np.arange(len(alive), dtype=np.int32)
    df_out = df_out[alive]
    term_ptr = np.zeros(len(alive) + 1, dtype=np.int64)
    np.cumsum(df_out, out=term_ptr[1:])
    rem_h = removed.cpu().numpy()
    n_out = dev.n_docs - len(rem_h)
    len_out = total_len - int(dev.doc_len[removed].to(torch.int64).sum().item())
    idf, _ = okapi_idf(df_out, n_out)
    return BM25Remove(rem_h, rem_ptr, rem_doc, term_map, term_ptr,
                      BM25Stats({}, df_out, np.zeros(0, np.int64), n_out, len_out, idf, len_out / n_out)), df_out


dev = DeviceIndex(0)
gpu = torch.cuda.get_device_name(0)
res = {"gpu": gpu, "power_limit": power_limit(), "rows": a.rows, "removals": []}
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
lists0 = [terms[ptr[b]:ptr[b + 1]].tolist() for b in range(B)]
term_map_all = np.arange(len(df), dtype=np.int64)             # original term id -> current id

g = torch.Generator(device=dev.device)
g.manual_seed(99)
for spec in a.removals.split(","):
    n = dev.n_local
    if spec.startswith("block"):
        m = int(spec[5:])
        lo = n // 3
        removed = torch.arange(lo, lo + m, device=dev.device)
    else:
        m = int(spec)
        removed = torch.sort(torch.randperm(n, generator=g, device=dev.device)[:m]).values
    row = {"n_before": n, "m": m, "pattern": "block" if spec.startswith("block") else "scattered"}
    rem, df_new = device_plan(dev, removed, df, total_len)
    row["terms_emptied"] = int((rem.term_map == -1).sum())
    # tiles of the copy kernel whose term span exceeds its shared-memory cache (kRmTile + 1 = 2 049
    # terms) and which read the per-term tables from global memory instead
    tp_d = dev._post[0]
    starts = torch.clamp(torch.arange(0, dev._post_args[0] + 2048, 2048, device=dev.device), max=dev._post_args[0] - 1)
    t0 = torch.searchsorted(tp_d, starts, right=True) - 1
    row["tiles"] = int(starts.numel() - 1)
    row["tiles_over_cache"] = int(((t0[1:] - t0[:-1] + 1) > 2049).sum().item())

    # the compaction kernel alone, into buffers of its own, repeated
    tp, p8, _ = dev._post
    nnz = dev._post_args[0]
    up = lambda arr, dt, v: torch.from_numpy(np.ascontiguousarray(arr, dtype=dt).view(v)).to(dev.device)
    rm_d = up(rem.removed, np.uint32, np.int32)
    rp_d, rd_d = up(rem.rem_ptr, np.int64, np.int64), up(rem.rem_doc, np.uint32, np.int32)
    tm_d, to_d = up(rem.term_map, np.int32, np.int32), up(rem.term_ptr, np.int64, np.int64)
    p8_out = torch.empty((rem.nnz + 2, 2), dtype=torch.int32, device=dev.device)
    compact = lambda: dev._ck(dev.lib.lrx_bm25_remove_postings(
        dev.h, _ptr(tp), _ptr(p8), dev.n_terms, nnz, dev.n_docs, _ptr(rm_d), m, _ptr(rp_d), _ptr(rd_d),
        _ptr(tm_d), _ptr(to_d), rem.n_terms, _ptr(p8_out)))
    compact()
    ms = sorted(timed(compact)[0] for _ in range(a.reps))
    # bytes the compaction must move: postings read + kept ones written, the document map (written,
    # then read once per posting at most: counted once), the per-term tables and removed lists
    V = dev.n_terms
    nbytes = (8 * nnz + 8 * rem.nnz + 4 * dev.n_docs + 8 * (V + 1) * 2 + 4 * V + 8 * (rem.n_terms + 1)
              + 4 * rem.nnz_rem + 4 * m)
    src = torch.empty(nbytes // 2, dtype=torch.uint8, device=dev.device)
    dst = torch.empty_like(src)
    dst.copy_(src)
    cp = sorted(timed(lambda: dst.copy_(src))[0] for _ in range(a.reps))
    del src, dst, p8_out
    med, cmed = ms[len(ms) // 2], cp[len(cp) // 2]
    row.update(kernel_ms=med, kernel_ms_all=ms, kernel_bytes=nbytes, kernel_TBps=nbytes / med / 1e9,
               memcpy_same_bytes_ms=cmed, memcpy_TBps=nbytes / cmed / 1e9, kernel_over_memcpy_rate=cmed / med,
               nnz_before=nnz, nnz_after=rem.nnz, nnz_removed=rem.nnz_rem)
    # the engine's path, phase by phase: postings (compaction + set_postings), matrix, shadow
    row["remove_postings_ms"], _ = timed(lambda: dev.remove_postings(rem))
    tp, p8, idf_t = dev._post
    row["set_postings_ms"], _ = timed(lambda: dev._ck(dev.lib.lrx_set_postings(
        dev.h, _ptr(tp), _ptr(p8), _ptr(idf_t), dev.n_terms, dev._post_args[0], *dev._post_args[1:])))
    keep = torch.ones(n, dtype=torch.bool, device=dev.device)
    keep[removed] = False
    row["matrix_compaction_ms"], _ = timed(lambda: dev.remove_rows(keep, prefilter=False))   # the shadow: next
    row["shadow_rebuild_ms"], _ = timed(dev.build_prefilter)
    df, total_len = df_new, rem.stats.total_len
    term_map_all = np.where(term_map_all >= 0, rem.term_map[np.maximum(term_map_all, 0)], -1)
    lists = [[int(term_map_all[t]) for t in l if term_map_all[t] >= 0] for l in lists0]
    # search on the shrunk index vs an index built from scratch over the same rows and postings
    row["qps_after_removal"], got = qps(dev, q, lists, iters=a.search_iters)
    ref = DeviceIndex(0)
    tp_h, pairs, dl_h = dev.read_postings()
    ref.set_corpus(dev.x.clone(), 0, prefilter=True)
    ref.set_postings(tp_h, pairs, dl_h, rem.stats.idf, rem.stats.avgdl)
    del tp_h, pairs, dl_h
    row["qps_scratch"], want = qps(ref, q, lists, iters=a.search_iters)
    row["qps_after_removal_again"], _ = qps(dev, q, lists, iters=a.search_iters)
    row["results_equal"] = all(np.array_equal(u, v) for u, v in zip(got, want))
    ref.close()
    del ref, rm_d, rp_d, rd_d, tm_d, to_d, keep
    torch.cuda.empty_cache()
    res["removals"].append(row)
    print(json.dumps(row), flush=True)
dev.close()


# the host plan: the reference corpus, then a synthetic text corpus, beside the host rebuild
def host_plan(docs, removed, label):
    full = BM25Index.from_token_lists(docs)
    tp = full.term_ptr.astype(np.int64)
    stats = full.stats()
    calls = []
    tok = lambda d: calls.append(d) or docs[d]
    gather = lambda t, c: full.postings[_ranges(tp[t], c), 0]
    t = time.perf_counter()
    rem = csr_remove(stats, removed, tok, gather)
    plan_s = time.perf_counter() - t
    gone = set(removed)
    t = time.perf_counter()
    want = BM25Index.from_token_lists([d for i, d in enumerate(docs) if i not in gone])
    rebuild_s = time.perf_counter() - t
    rem.commit_vocab()
    assert list(rem.stats.vocab) == list(want.vocab)
    assert np.array_equal(rem.stats.idf.view(np.uint64), want.idf.view(np.uint64))
    return {"corpus": label, "docs": len(docs), "removed": len(removed), "plan_s": plan_s,
            "documents_read": len(calls), "host_rebuild_s": rebuild_s}


with gzip.open(ROOT / "tests" / "golden" / "legal_chunks.json.gz", "rt", encoding="utf-8") as f:
    ref_docs = [tokenize(c["text"]) for c in json.load(f)]
rng = np.random.default_rng(7)
res["host_plan"] = [host_plan(ref_docs, sorted(rng.choice(len(ref_docs), 262, replace=False).tolist()),
                              "reference (legal_chunks.json)")]
vocab = np.array([f"w{i}" for i in range(synth.VOCAB)])
lens = synth.host_doc_lengths(a.host_docs, rng)
cdf = synth._zipf_cdf(synth.VOCAB)
toks = vocab[np.minimum(np.searchsorted(cdf, rng.random(int(lens.sum())), side="right"), synth.VOCAB - 1)]
syn_docs = [t.tolist() for t in np.split(toks, np.cumsum(lens)[:-1])]
for m in (100, 1000):
    res["host_plan"].append(host_plan(syn_docs, sorted(rng.choice(a.host_docs, m, replace=False).tolist()),
                                      "synthetic Zipf text"))
print(json.dumps({"gpu": gpu, "power_limit": res["power_limit"], "host_plan": res["host_plan"]}), flush=True)
if a.out:
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text(json.dumps(res, indent=1) + "\n")
