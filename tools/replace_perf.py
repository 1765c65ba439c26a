#!/usr/bin/env python
"""Index replacement at scale: in a 10 M-row synthetic index (synth.device_vectors / device_bm25), the
text of m = 1 000, 10 000, 100 000 documents is replaced, scattered and as one contiguous block, in
turn.  A replaced document takes the postings and length of the document n / 2 ids away, so the new
text follows the corpus's Zipf law.  Per replacement: the postings merge (lrx_bm25_replace_postings,
median of --reps calls, CUDA events) with its bytes and rate beside a cudaMemcpyAsync D2D moving the
same bytes, the staged path with lrx_set_postings, the in-place row overwrite and the int8 shadow
rebuild, and search queries/s on the edited index against an index built from scratch over the same
rows and postings (results asserted identical).  Also the host plan (bm25_index.csr_replace) on the
reference corpus and on a synthetic text corpus, beside the host rebuild it replaces.

    python tools/replace_perf.py [--rows 10000000] [--out profiles/replace_perf_b200.json]
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
from legal_rag_engine_b200.bm25_index import (BM25Index, BM25Replace, BM25Stats, _ranges,  # noqa: E402
                                              csr_replace, okapi_idf, tokenize)
from legal_rag_engine_b200.device_index import DeviceIndex, _ptr        # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--rows", type=int, default=10_000_000)
ap.add_argument("--replacements", default="1000,10000,100000,block1000,block10000,block100000")
ap.add_argument("--reps", type=int, default=5, help="timed repeats of the merge and of the copy")
ap.add_argument("--search-iters", type=int, default=100)
ap.add_argument("--host-docs", type=int, default=100_000, help="documents of the synthetic text corpus")
ap.add_argument("--out", default=None)
a = ap.parse_args()


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
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


def device_plan(dev, replaced, df, total_len):
    """The replacement plan of a synthetic index (no string vocabulary: the surviving terms keep their
    relative order), from the resident postings.  Replaced document d takes the postings and length of
    document (d + n / 2) mod n.  Returns (plan, new doc_len tensor, new df)."""
    tp, p8, _ = dev._post
    nnz, V, n = dev._post_args[0], dev.n_terms, dev.n_docs
    doc = p8[:nnz, 0]
    term_of = torch.repeat_interleave(torch.arange(V, device=dev.device), tp[1:] - tp[:-1])
    gone = torch.isin(doc, replaced.to(torch.int32))
    r = torch.bincount(term_of[gone], minlength=V).cpu().numpy().astype(np.int64)
    rem_doc = doc[gone].cpu().numpy().view(np.uint32)
    del gone
    src = (replaced + n // 2) % n
    to_dst = torch.full((n,), -1, dtype=torch.int64, device=dev.device)
    to_dst[src] = replaced
    sel = torch.isin(doc, src.to(torch.int32))
    it = term_of[sel]
    idd = to_dst[doc[sel].to(torch.int64)]
    itf = p8[:nnz, 1][sel] & 0xFFFF
    del term_of, sel, to_dst
    ins_cnt = torch.bincount(it, minlength=V).cpu().numpy().astype(np.int64)
    df_new = df - r + ins_cnt
    alive = np.nonzero(df_new > 0)[0]
    term_map = np.full(V, -1, dtype=np.int32)
    term_map[alive] = np.arange(len(alive), dtype=np.int32)
    nt = torch.from_numpy(term_map).to(dev.device)[it].to(torch.int64)
    order = torch.argsort(nt * n + idd)
    ins = torch.stack([idd[order], itf[order].to(torch.int64)], 1).cpu().numpy().astype(np.uint32)
    ins_ptr = np.zeros(len(alive) + 1, dtype=np.int64)
    np.cumsum(ins_cnt[alive], out=ins_ptr[1:])
    rem_ptr = np.zeros(V + 1, dtype=np.int64)
    np.cumsum(r, out=rem_ptr[1:])
    term_ptr = np.zeros(len(alive) + 1, dtype=np.int64)
    np.cumsum(df_new[alive], out=term_ptr[1:])
    doc_len = dev.doc_len[:n].clone()
    doc_len[replaced] = dev.doc_len[src]
    len_out = int(doc_len.to(torch.int64).sum().item())
    idf, _ = okapi_idf(df_new[alive], n)
    rep = BM25Replace(replaced.cpu().numpy(), doc_len[replaced].cpu().numpy().astype(np.uint32), rem_ptr, rem_doc,
                      term_map, [], np.zeros(0, np.int32), ins_ptr, ins, term_ptr,
                      BM25Stats({}, df_new[alive], np.zeros(0, np.int64), n, len_out, idf, len_out / n))
    return rep, doc_len, df_new[alive]


dev = DeviceIndex(0)
gpu = torch.cuda.get_device_name(0)
res = {"gpu": gpu, "card": card(), "rows": a.rows, "replacements": []}
print(json.dumps({"gpu": gpu, "card": res["card"]}), flush=True)
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
for spec in a.replacements.split(","):
    n = dev.n_local
    block = spec.startswith("block")
    m = int(spec[5:] if block else spec)
    if block:
        replaced = torch.arange(n // 3, n // 3 + m, device=dev.device)
    else:
        replaced = torch.sort(torch.randperm(n, generator=g, device=dev.device)[:m]).values
    row = {"n": n, "m": m, "pattern": "block" if block else "scattered"}
    rep, doc_len, df_new = device_plan(dev, replaced, df, total_len)
    row["terms_vanished"] = int((rep.term_map == -1).sum())

    # the merge kernel alone, into buffers of its own, repeated
    tp, p8, _ = dev._post
    nnz = dev._post_args[0]
    up = lambda arr, dt, v: torch.from_numpy(np.ascontiguousarray(arr, dtype=dt).view(v)).to(dev.device)
    rp_d = up(rep.replaced, np.uint32, np.int32)
    rmp_d, rmd_d = up(rep.rem_ptr, np.int64, np.int64), up(rep.rem_doc, np.uint32, np.int32)
    tm_d, ip_d = up(rep.term_map, np.int32, np.int32), up(rep.ins_ptr, np.int64, np.int64)
    in_d, to_d = up(rep.ins_postings, np.uint32, np.int32), up(rep.term_ptr, np.int64, np.int64)
    dl_d = doc_len.to(torch.int32).contiguous()
    p8_out = torch.empty((rep.nnz + 2, 2), dtype=torch.int32, device=dev.device)
    merge = lambda: dev._ck(dev.lib.lrx_bm25_replace_postings(
        dev.h, _ptr(tp), _ptr(p8), dev.n_terms, nnz, dev.n_docs, _ptr(rp_d), m, _ptr(rmp_d), _ptr(rmd_d),
        _ptr(tm_d), _ptr(ip_d), _ptr(in_d), rep.nnz_ins, _ptr(dl_d), _ptr(to_d), rep.n_terms, _ptr(p8_out)))
    merge()
    ms = sorted(timed(merge)[0] for _ in range(a.reps))
    # bytes the merge must move: postings read + written, the replaced-document bits, the per-term
    # tables, the dropped and inserted lists and the replaced documents' lengths
    V = dev.n_terms
    nbytes = (8 * nnz + 8 * rep.nnz + (n + 7) // 8 + 8 * (V + 1) * 2 + 4 * V + 8 * (rep.n_terms + 1) * 2
              + 4 * rep.nnz_rem + 8 * rep.nnz_ins + 4 * m + 4 * m)
    src = torch.empty(nbytes // 2, dtype=torch.uint8, device=dev.device)
    dst = torch.empty_like(src)
    dst.copy_(src)
    cp = sorted(timed(lambda: dst.copy_(src))[0] for _ in range(a.reps))
    del src, dst, p8_out
    med, cmed = ms[len(ms) // 2], cp[len(cp) // 2]
    row.update(kernel_ms=med, kernel_ms_all=ms, kernel_bytes=nbytes, kernel_TBps=nbytes / med / 1e9,
               memcpy_same_bytes_ms=cmed, memcpy_TBps=nbytes / cmed / 1e9, kernel_over_memcpy_rate=cmed / med,
               nnz_before=nnz, nnz_after=rep.nnz, nnz_dropped=rep.nnz_rem, nnz_inserted=rep.nnz_ins)
    # the engine's path, phase by phase: postings (stage + set_postings), rows, shadow
    row["stage_and_commit_ms"], _ = timed(lambda: dev.commit_postings(dev.stage_replace(rep, doc_len)))
    x_new = synth.device_vectors(m, dev.device, seed=m + 5)
    row["row_overwrite_ms"], _ = timed(lambda: dev.replace_rows(replaced, x_new, prefilter=False))
    row["shadow_rebuild_ms"], _ = timed(dev.build_prefilter)
    del x_new
    df, total_len = df_new, rep.stats.total_len
    term_map_all = np.where(term_map_all >= 0, rep.term_map[np.maximum(term_map_all, 0)], -1)
    lists = [[int(term_map_all[t]) for t in l if term_map_all[t] >= 0] for l in lists0]
    # search on the edited index vs an index built from scratch over the same rows and postings
    row["qps_after_replace"], got = qps(dev, q, lists, iters=a.search_iters)
    ref = DeviceIndex(0)
    tp_h, pairs, dl_h = dev.read_postings()
    ref.set_corpus(dev.x.clone(), 0, prefilter=True)
    ref.set_postings(tp_h, pairs, dl_h, rep.stats.idf, rep.stats.avgdl)
    del tp_h, pairs, dl_h
    row["qps_scratch"], want = qps(ref, q, lists, iters=a.search_iters)
    row["qps_after_replace_again"], _ = qps(dev, q, lists, iters=a.search_iters)
    row["results_equal"] = all(np.array_equal(u, v) for u, v in zip(got, want))
    assert row["results_equal"], row
    ref.close()
    del ref, rp_d, rmp_d, rmd_d, tm_d, ip_d, in_d, to_d, dl_d
    torch.cuda.empty_cache()
    res["replacements"].append(row)
    print(json.dumps(row), flush=True)
dev.close()


# the host plan: the reference corpus, then a synthetic text corpus, beside the host rebuild
def host_plan(docs, ids, new, label):
    full = BM25Index.from_token_lists(docs)
    tp = full.term_ptr.astype(np.int64)
    stats = full.stats()
    calls = []
    tok = lambda d: calls.append(d) or docs[d]
    gather = lambda t, c: full.postings[_ranges(tp[t], c), 0]
    t = time.perf_counter()
    rep = csr_replace(stats, ids, new, tok, gather)
    plan_s = time.perf_counter() - t
    edited = list(docs)
    for i, d in zip(ids, new):
        edited[i] = d
    t = time.perf_counter()
    want = BM25Index.from_token_lists(edited)
    rebuild_s = time.perf_counter() - t
    rep.commit_vocab()
    assert list(rep.stats.vocab) == list(want.vocab)
    assert np.array_equal(rep.stats.idf.view(np.uint64), want.idf.view(np.uint64))
    return {"corpus": label, "docs": len(docs), "replaced": len(ids), "plan_s": plan_s,
            "documents_read": len(calls), "host_rebuild_s": rebuild_s}


with gzip.open(ROOT / "tests" / "golden" / "legal_chunks.json.gz", "rt", encoding="utf-8") as f:
    ref_docs = [tokenize(c["text"]) for c in json.load(f)]
rng = np.random.default_rng(7)
ids = sorted(rng.choice(len(ref_docs), 262, replace=False).tolist())
res["host_plan"] = [host_plan(ref_docs, ids, [ref_docs[i][::-1] for i in ids], "reference (legal_chunks.json)")]
vocab = np.array([f"w{i}" for i in range(synth.VOCAB)])
lens = synth.host_doc_lengths(a.host_docs, rng)
cdf = synth._zipf_cdf(synth.VOCAB)
toks = vocab[np.minimum(np.searchsorted(cdf, rng.random(int(lens.sum())), side="right"), synth.VOCAB - 1)]
syn_docs = [t.tolist() for t in np.split(toks, np.cumsum(lens)[:-1])]
for m in (100, 1000):
    ids = sorted(rng.choice(a.host_docs, m, replace=False).tolist())
    res["host_plan"].append(host_plan(syn_docs, ids, [syn_docs[(i + a.host_docs // 2) % a.host_docs] for i in ids],
                                      "synthetic Zipf text"))
print(json.dumps({"gpu": gpu, "card": res["card"], "host_plan": res["host_plan"]}), flush=True)
if a.out:
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text(json.dumps(res, indent=1) + "\n")
