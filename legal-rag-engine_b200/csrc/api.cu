// The C ABI of include/lrx.h: argument checking, error strings, workspace
// management and the K5 launch sequence (all sub-queries of a fan-out batched
// through one K2 -> K3 -> K4 chain).  No CPU fallback anywhere.
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>

#include "common.cuh"
#include "handle.h"

namespace lrx {

cudaError_t ensure_ws(lrx_handle* h, void** p, size_t* have, size_t need) {
    if (*have >= need && *p != nullptr) return cudaSuccess;
    // a captured launch chain holds the old pointers: never move a workspace while capturing, and
    // retire every instantiated plan when one moves
    if (h->capturing) return cudaErrorStreamCaptureUnsupported;
    h->ws_epoch++;
    if (*p != nullptr) {
        cudaError_t e = cudaFree(*p);   // synchronises: safe against in-flight users
        *p = nullptr;
        *have = 0;
        if (e != cudaSuccess) return e;
    }
    size_t sz = need + need / 4 + 256;
    cudaError_t e = cudaMalloc(p, sz);
    if (e == cudaSuccess) *have = sz;
    return e;
}

void prof_begin(lrx_handle* h, int which, cudaStream_t st) {
    if (!h->prof) return;
    cudaEvent_t e;
    if (cudaEventCreate(&e) != cudaSuccess) return;
    if (h->capturing && h->cap_plan != nullptr) {
        // inside a captured chain: an external event-record node, re-recorded by every replay of
        // the plan (lrx_profile_read takes each plan's last replay)
        cudaEventRecordWithFlags(e, st ? st : h->stream, cudaEventRecordExternal);
        h->cap_plan->prof_ev[which].push_back(e);
    } else {
        cudaEventRecord(e, st ? st : h->stream);
        h->prof_ev[which].push_back(e);
    }
}
void prof_end(lrx_handle* h, int which, cudaStream_t st) { prof_begin(h, which, st); }

std::recursive_mutex& attr_mutex() {
    static std::recursive_mutex m;
    return m;
}

static std::string g_err;   // failures before a handle exists
static std::mutex g_err_mu;

static int fail(lrx_handle* h, int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (h != nullptr) {
        h->err = buf;
    } else {
        std::lock_guard<std::mutex> g(g_err_mu);
        g_err = buf;
    }
    return code;
}

#define LRX_CUDA(h, expr)                                                                   \
    do {                                                                                    \
        cudaError_t _e = (expr);                                                            \
        if (_e != cudaSuccess)                                                              \
            return fail((h), LRX_E_CUDA, "%s: %s (%s:%d)", #expr, cudaGetErrorString(_e),   \
                        __FILE__, __LINE__);                                                \
    } while (0)

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

static void drop_plans(lrx_handle* h) {
    for (lrx_plan* pl : h->plans) {
        if (pl->exec != nullptr) cudaGraphExecDestroy(pl->exec);
        for (int w = 0; w < 2; ++w)
            for (cudaEvent_t e : pl->prof_ev[w]) cudaEventDestroy(e);
        delete pl;
    }
    h->plans.clear();
}

}  // namespace lrx

using namespace lrx;

extern "C" {

const char* lrx_version(void) { return "lrx 0.3 sm_100a"; }

const char* lrx_last_error(const lrx_handle* h) {
    if (h != nullptr) return h->err.c_str();
    return g_err.c_str();
}

int lrx_open(const lrx_config* cfg, lrx_handle** out) {
    if (cfg == nullptr || out == nullptr) return fail(nullptr, LRX_E_ARG, "lrx_open: null argument");
    if (cfg->dim != LRX_DIM) return fail(nullptr, LRX_E_ARG, "lrx_open: dim must be %d", LRX_DIM);
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev <= 0)
        return fail(nullptr, LRX_E_DEVICE, "lrx_open: no CUDA device (%s); there is no CPU fallback",
                    cudaGetErrorString(e));
    if (cfg->device < 0 || cfg->device >= ndev)
        return fail(nullptr, LRX_E_DEVICE, "lrx_open: device %d out of range (%d devices)",
                    cfg->device, ndev);
    cudaDeviceProp prop;
    e = cudaGetDeviceProperties(&prop, cfg->device);
    if (e != cudaSuccess)
        return fail(nullptr, LRX_E_DEVICE, "lrx_open: cudaGetDeviceProperties: %s",
                    cudaGetErrorString(e));
    if (prop.major != 10)
        return fail(nullptr, LRX_E_DEVICE,
                    "lrx_open: device %d is sm_%d%d; this library is built for sm_100a only",
                    cfg->device, prop.major, prop.minor);
    e = cudaSetDevice(cfg->device);
    if (e != cudaSuccess)
        return fail(nullptr, LRX_E_DEVICE, "lrx_open: cudaSetDevice: %s", cudaGetErrorString(e));
    lrx_handle* h = new (std::nothrow) lrx_handle();
    if (h == nullptr) return fail(nullptr, LRX_E_NOMEM, "lrx_open: out of memory");
    h->device = cfg->device;
    h->num_sms = prop.multiProcessorCount;
    h->rank = cfg->rank;
    h->world = cfg->world > 0 ? cfg->world : 1;
    // The side stream carries the BM25 chain (bounds -> scan -> merge), the longer of the two chains of
    // a batch since the int8 dense scan: it gets the high stream priority, so that its CTAs are placed
    // first when SM slots free up (profiles/r2_runs/ab_aux_stream_priority.txt: two users per chain + 4 %,
    // latency of one batch at 10 M rows 0.86 -> 0.80 ms).
    int prio_lo = 0, prio_hi = 0;
    cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
    if (cudaStreamCreateWithPriority(&h->aux, cudaStreamNonBlocking, prio_hi) != cudaSuccess ||
        cudaStreamCreateWithFlags(&h->cap, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming) != cudaSuccess ||
        cudaMalloc((void**)&h->pack_done, 256) != cudaSuccess ||
        cudaMemset(h->pack_done, 0, 256) != cudaSuccess) {
        delete h;
        return fail(nullptr, LRX_E_CUDA, "lrx_open: cannot create side stream / events");
    }
    *out = h;
    return LRX_OK;
}

int lrx_close(lrx_handle* h) {
    if (h == nullptr) return LRX_OK;
    cudaSetDevice(h->device);
    cudaDeviceSynchronize();
    drop_plans(h);
    for (int w = 0; w < 2; ++w)
        for (cudaEvent_t e : h->prof_ev[w]) cudaEventDestroy(e);
    if (h->cap) cudaStreamDestroy(h->cap);
    if (h->pack_done) cudaFree(h->pack_done);
    void* ws[] = {h->ws_dense_part, h->ws_bm_part, h->ws_bm_max, h->ws_misc, h->ws_io, h->ws_rm};
    for (void* p : ws)
        if (p != nullptr) cudaFree(p);
    encoder_free(h);
    for (int w = 0; w < LRX_MAX_WORLD; ++w)
        if (h->xchg_peer[w] != nullptr && w != h->rank) cudaIpcCloseMemHandle(h->xchg_peer[w]);
    if (h->bm_ctab != nullptr) cudaFree(h->bm_ctab);
    if (h->xchg != nullptr) cudaFree(h->xchg);
    if (h->xchg_peer_dev != nullptr) cudaFree(h->xchg_peer_dev);
    if (h->ws_host != nullptr) cudaFreeHost(h->ws_host);
    if (h->aux) cudaStreamDestroy(h->aux);
    if (h->ev_fork) cudaEventDestroy(h->ev_fork);
    if (h->ev_join) cudaEventDestroy(h->ev_join);
    delete h;
    return LRX_OK;
}

int lrx_set_stream(lrx_handle* h, void* cuda_stream) {
    if (h == nullptr) return fail(nullptr, LRX_E_ARG, "lrx_set_stream: null handle");
    std::lock_guard<std::mutex> g(h->mu);
    h->stream = (cudaStream_t)cuda_stream;
    return LRX_OK;
}

int lrx_debug_bm25_divcheck(lrx_handle* h, double avgdl, double k1, double b, int32_t n_tf,
                            int32_t n_len, uint64_t* host_mismatches) {
    if (h == nullptr) return fail(nullptr, LRX_E_ARG, "lrx_debug_bm25_divcheck: null handle");
    if (host_mismatches == nullptr || n_tf <= 0 || n_len <= 0 || !(avgdl > 0.0))
        return fail(h, LRX_E_ARG, "lrx_debug_bm25_divcheck: bad argument");
    std::lock_guard<std::mutex> g(h->mu);
    LRX_CUDA(h, cudaSetDevice(h->device));
    unsigned long long bad = 0;
    LRX_CUDA(h, launch_bm25_divcheck(h, avgdl, k1, b, n_tf, n_len, &bad));
    *host_mismatches = bad;
    return LRX_OK;
}

int lrx_debug_attention(lrx_handle* h, const void* dev_qkv_fp16, const int32_t* dev_lens, int32_t B,
                        int32_t S, void* dev_ctx_fp16) {
    if (h == nullptr) return fail(nullptr, LRX_E_ARG, "lrx_debug_attention: null handle");
    if (B < 1 || B > (1 << 20)) return fail(h, LRX_E_ARG, "lrx_debug_attention: B must be in [1, 2^20]");
    if (S < 1 || S > 512) return fail(h, LRX_E_ARG, "lrx_debug_attention: S must be in [1,512]");
    if (dev_qkv_fp16 == nullptr || dev_lens == nullptr || dev_ctx_fp16 == nullptr)
        return fail(h, LRX_E_ARG, "lrx_debug_attention: null pointer");
    if ((((uintptr_t)dev_qkv_fp16 | (uintptr_t)dev_ctx_fp16) & 15) != 0 || ((uintptr_t)dev_lens & 3) != 0)
        return fail(h, LRX_E_ARG, "lrx_debug_attention: misaligned pointer");
    std::lock_guard<std::mutex> g(h->mu);
    LRX_CUDA(h, cudaSetDevice(h->device));
    LRX_CUDA(h, encoder_debug_attention(h, dev_qkv_fp16, dev_lens, B, S, dev_ctx_fp16));
    return LRX_OK;
}

int64_t lrx_launch_count(const lrx_handle* h) { return h ? h->launches : 0; }

int lrx_profile_enable(lrx_handle* h, int32_t on) {
    if (h == nullptr) return fail(nullptr, LRX_E_ARG, "lrx_profile_enable: null handle");
    std::lock_guard<std::mutex> g(h->mu);
    h->prof = (on != 0);
    return LRX_OK;
}

int lrx_profile_read(lrx_handle* h, int32_t which, double* total_ms, int64_t* n_launches) {
    if (h == nullptr) return fail(nullptr, LRX_E_ARG, "lrx_profile_read: null handle");
    std::lock_guard<std::mutex> g(h->mu);
    if (which < 0 || which > 1 || total_ms == nullptr || n_launches == nullptr)
        return fail(h, LRX_E_ARG, "lrx_profile_read: bad argument");
    LRX_CUDA(h, cudaSetDevice(h->device));
    LRX_CUDA(h, cudaStreamSynchronize(h->stream));
    std::vector<cudaEvent_t>& ev = h->prof_ev[which];
    double ms = 0.0;
    int64_t n = 0;
    auto add = [&](const std::vector<cudaEvent_t>& v) {
        for (size_t i = 0; i + 1 < v.size(); i += 2) {
            float t = 0.f;
            if (cudaEventElapsedTime(&t, v[i], v[i + 1]) == cudaSuccess) {
                ms += t;
                ++n;
            }
        }
    };
    add(ev);
    for (cudaEvent_t e : ev) cudaEventDestroy(e);
    ev.clear();
    // captured chains: the event nodes hold the times of each plan's LAST replay
    for (lrx_plan* pl : h->plans)
        if (pl->replayed) add(pl->prof_ev[which]);
    if (which == 1)
        for (lrx_plan* pl : h->plans) pl->replayed = false;
    *total_ms = ms;
    *n_launches = n;
    return LRX_OK;
}

int lrx_set_corpus(lrx_handle* h, const void* dev_x_fp16, int64_t n_local, int64_t id_base,
                   int32_t dim) {
    if (h == nullptr) return fail(nullptr, LRX_E_ARG, "lrx_set_corpus: null handle");
    std::lock_guard<std::mutex> g(h->mu);
    if (dim != LRX_DIM) return fail(h, LRX_E_ARG, "lrx_set_corpus: dim must be %d", LRX_DIM);
    if (n_local < 0 || n_local >= (1ll << 32))
        return fail(h, LRX_E_ARG, "lrx_set_corpus: n_local %lld out of range", (long long)n_local);
    if (id_base < 0 || id_base + n_local >= (1ll << 32))
        return fail(h, LRX_E_ARG, "lrx_set_corpus: global ids must stay below 2^32");
    if (n_local > 0 && (dev_x_fp16 == nullptr || ((uintptr_t)dev_x_fp16 & 15) != 0))
        return fail(h, LRX_E_ARG, "lrx_set_corpus: matrix pointer must be non-null, 16-byte aligned");
    h->x = dev_x_fp16;
    h->n_local = n_local;
    h->id_base = id_base;
    h->q8 = nullptr;                      // a shadow belongs to the matrix it was built from
    h->q8_err = h->q8_norm = 0.0;
    h->ws_epoch++;                        // captured chains hold the old matrix
    return LRX_OK;
}

int64_t lrx_dense_prefilter_bytes(int64_t n_local) {
    if (n_local < 0 || n_local >= (1ll << 32)) return 0;
    return dense_q8_bytes(n_local);
}

int lrx_build_dense_prefilter(lrx_handle* h, void* dev_buf, int64_t bytes, double* host_bounds_out) {
    if (h == nullptr) return fail(nullptr, LRX_E_ARG, "lrx_build_dense_prefilter: null handle");
    std::lock_guard<std::mutex> g(h->mu);
    if (h->x == nullptr && h->n_local > 0) return fail(h, LRX_E_STATE, "lrx_build_dense_prefilter: corpus not set");
    if (host_bounds_out == nullptr || (h->n_local > 0 && dev_buf == nullptr) || ((uintptr_t)dev_buf & 15) != 0)
        return fail(h, LRX_E_ARG, "lrx_build_dense_prefilter: null or misaligned pointer");
    if (bytes < dense_q8_bytes(h->n_local))
        return fail(h, LRX_E_ARG, "lrx_build_dense_prefilter: buffer smaller than lrx_dense_prefilter_bytes(%lld)",
                    (long long)h->n_local);
    LRX_CUDA(h, cudaSetDevice(h->device));
    LRX_CUDA(h, launch_dense_q8_build(h, dev_buf, host_bounds_out));
    h->q8 = (h->n_local > 0) ? dev_buf : nullptr;
    h->q8_err = host_bounds_out[0];
    h->q8_norm = host_bounds_out[1];
    h->ws_epoch++;                        // captured chains were built without the shadow
    return LRX_OK;
}

int lrx_set_dense_prefilter(lrx_handle* h, const void* dev_buf, int64_t bytes, const double* host_bounds) {
    if (h == nullptr) return fail(nullptr, LRX_E_ARG, "lrx_set_dense_prefilter: null handle");
    std::lock_guard<std::mutex> g(h->mu);
    if (dev_buf != nullptr) {
        if (host_bounds == nullptr || ((uintptr_t)dev_buf & 15) != 0)
            return fail(h, LRX_E_ARG, "lrx_set_dense_prefilter: null bounds or misaligned buffer");
        if (bytes < dense_q8_bytes(h->n_local))
            return fail(h, LRX_E_ARG, "lrx_set_dense_prefilter: buffer smaller than lrx_dense_prefilter_bytes(%lld)",
                        (long long)h->n_local);
        if (!(host_bounds[0] >= 0.0) || !(host_bounds[1] >= 0.0))
            return fail(h, LRX_E_ARG, "lrx_set_dense_prefilter: bounds must be >= 0");
    }
    h->q8 = (h->n_local > 0) ? dev_buf : nullptr;
    h->q8_err = dev_buf ? host_bounds[0] : 0.0;
    h->q8_norm = dev_buf ? host_bounds[1] : 0.0;
    h->ws_epoch++;
    return LRX_OK;
}

int lrx_set_postings(lrx_handle* h, const uint64_t* dev_term_ptr, const void* dev_postings,
                     const double* dev_idf, int64_t n_terms, int64_t nnz, double avgdl, double k1,
                     double b, int32_t max_doc_len) {
    if (h == nullptr) return fail(nullptr, LRX_E_ARG, "lrx_set_postings: null handle");
    std::lock_guard<std::mutex> g(h->mu);
    if (n_terms < 0 || nnz < 0) return fail(h, LRX_E_ARG, "lrx_set_postings: negative size");
    if (dev_term_ptr == nullptr || dev_idf == nullptr || (nnz > 0 && dev_postings == nullptr))
        return fail(h, LRX_E_ARG, "lrx_set_postings: null pointer");
    if (((uintptr_t)dev_postings & 15) != 0)
        return fail(h, LRX_E_ARG, "lrx_set_postings: postings must be 16-byte aligned");
    if (!(avgdl > 0.0)) return fail(h, LRX_E_ARG, "lrx_set_postings: avgdl must be > 0");
    if (max_doc_len < 0 || max_doc_len > 65535)
        return fail(h, LRX_E_ARG, "lrx_set_postings: max_doc_len must be in [0,65535] "
                                  "(the 8-byte posting stores the document length in 16 bits)");
    LRX_CUDA(h, cudaSetDevice(h->device));
    LRX_CUDA(h, launch_bm25_lut(h, avgdl, k1, b, max_doc_len));
    h->term_ptr = dev_term_ptr;
    h->postings = dev_postings;
    h->idf = dev_idf;
    h->n_terms = n_terms;
    h->nnz = nnz;
    h->ws_epoch++;                        // captured chains hold the old postings
    return LRX_OK;
}

int lrx_bm25_build_postings(lrx_handle* h, const uint32_t* dev_doc_tf, int64_t nnz,
                            const uint32_t* dev_doc_len, void* dev_postings_out) {
    if (h == nullptr) return fail(nullptr, LRX_E_ARG, "lrx_bm25_build_postings: null handle");
    std::lock_guard<std::mutex> g(h->mu);
    if (nnz < 0 || (nnz > 0 && (dev_doc_tf == nullptr || dev_doc_len == nullptr ||
                                dev_postings_out == nullptr)))
        return fail(h, LRX_E_ARG, "lrx_bm25_build_postings: bad argument");
    if ((((uintptr_t)dev_postings_out | (uintptr_t)dev_doc_tf) & 7) != 0)
        return fail(h, LRX_E_ARG, "lrx_bm25_build_postings: buffers must be 8-byte aligned");
    LRX_CUDA(h, cudaSetDevice(h->device));
    int overflow = 0;
    LRX_CUDA(h, launch_bm25_pack(h, dev_doc_tf, nnz, dev_doc_len, dev_postings_out, &overflow));
    if (overflow)
        return fail(h, LRX_E_ARG, "lrx_bm25_build_postings: a term frequency or document length "
                                  "exceeds 65535 (16-bit posting fields)");
    return LRX_OK;
}

int lrx_bm25_append_postings(lrx_handle* h, const uint64_t* dev_term_ptr, const void* dev_postings,
                             int64_t n_terms, int64_t nnz, int64_t n_docs_old,
                             const uint64_t* dev_add_ptr, const uint32_t* dev_add_doc_tf,
                             int64_t n_terms_out, int64_t nnz_add, const uint32_t* dev_doc_len,
                             int64_t n_docs_out, uint64_t* dev_term_ptr_out, void* dev_postings_out) {
    if (h == nullptr) return fail(nullptr, LRX_E_ARG, "lrx_bm25_append_postings: null handle");
    std::lock_guard<std::mutex> g(h->mu);
    if (n_terms < 0 || nnz < 0 || n_docs_old < 0 || nnz_add < 0 || n_terms_out < n_terms ||
        n_docs_out < n_docs_old || n_docs_out >= (1ll << 32))
        return fail(h, LRX_E_ARG, "lrx_bm25_append_postings: bad size");
    if (dev_term_ptr == nullptr || dev_add_ptr == nullptr || dev_term_ptr_out == nullptr ||
        (nnz > 0 && dev_postings == nullptr) ||
        (nnz_add > 0 && (dev_add_doc_tf == nullptr || dev_doc_len == nullptr)) ||
        (nnz + nnz_add > 0 && dev_postings_out == nullptr))
        return fail(h, LRX_E_ARG, "lrx_bm25_append_postings: null pointer");
    if ((((uintptr_t)dev_postings | (uintptr_t)dev_postings_out) & 15) != 0 ||
        (((uintptr_t)dev_add_doc_tf | (uintptr_t)dev_term_ptr | (uintptr_t)dev_add_ptr |
          (uintptr_t)dev_term_ptr_out) & 7) != 0)
        return fail(h, LRX_E_ARG, "lrx_bm25_append_postings: postings must be 16-byte aligned, "
                                  "pointer tables and (doc, tf) pairs 8-byte aligned");
    LRX_CUDA(h, cudaSetDevice(h->device));
    int bad = 0;
    LRX_CUDA(h, launch_bm25_append(h, dev_term_ptr, dev_postings, n_terms, nnz, n_docs_old, dev_add_ptr,
                                   dev_add_doc_tf, n_terms_out, nnz_add, dev_doc_len, n_docs_out,
                                   dev_term_ptr_out, dev_postings_out, &bad));
    if (bad == 2)
        return fail(h, LRX_E_ARG, "lrx_bm25_append_postings: term_ptr[n_terms] != nnz or "
                                  "add_ptr[n_terms_out] != nnz_add");
    if (bad)
        return fail(h, LRX_E_ARG, "lrx_bm25_append_postings: a term frequency or document length "
                                  "exceeds 65535, or an appended doc id is outside [n_docs_old, n_docs_out)");
    return LRX_OK;
}

int lrx_bm25_remove_postings(lrx_handle* h, const uint64_t* dev_term_ptr, const void* dev_postings,
                             int64_t n_terms, int64_t nnz, int64_t n_docs_old,
                             const uint32_t* dev_removed_docs, int64_t n_removed,
                             const uint64_t* dev_rem_ptr, const uint32_t* dev_rem_doc,
                             const int32_t* dev_term_map, const uint64_t* dev_term_ptr_out,
                             int64_t n_terms_out, void* dev_postings_out) {
    if (h == nullptr) return fail(nullptr, LRX_E_ARG, "lrx_bm25_remove_postings: null handle");
    std::lock_guard<std::mutex> g(h->mu);
    if (n_terms < 0 || nnz < 0 || n_docs_old < 0 || n_docs_old >= (1ll << 32) || n_removed < 0 ||
        n_removed > n_docs_old || n_terms_out < 0 || n_terms_out > n_terms)
        return fail(h, LRX_E_ARG, "lrx_bm25_remove_postings: bad size");
    if (dev_term_ptr == nullptr || dev_rem_ptr == nullptr || dev_term_ptr_out == nullptr ||
        (n_terms > 0 && dev_term_map == nullptr) || (n_removed > 0 && dev_removed_docs == nullptr) ||
        (nnz > 0 && (dev_postings == nullptr || dev_postings_out == nullptr)))
        return fail(h, LRX_E_ARG, "lrx_bm25_remove_postings: null pointer");
    if ((((uintptr_t)dev_postings | (uintptr_t)dev_postings_out) & 15) != 0 ||
        (((uintptr_t)dev_term_ptr | (uintptr_t)dev_rem_ptr | (uintptr_t)dev_term_ptr_out) & 7) != 0 ||
        (((uintptr_t)dev_removed_docs | (uintptr_t)dev_rem_doc | (uintptr_t)dev_term_map) & 3) != 0)
        return fail(h, LRX_E_ARG, "lrx_bm25_remove_postings: postings must be 16-byte aligned, pointer "
                                  "tables 8-byte aligned, id arrays 4-byte aligned");
    LRX_CUDA(h, cudaSetDevice(h->device));
    int bad = 0;
    LRX_CUDA(h, launch_bm25_remove(h, dev_term_ptr, dev_postings, n_terms, nnz, n_docs_old, dev_removed_docs,
                                   n_removed, dev_rem_ptr, dev_rem_doc, dev_term_map, dev_term_ptr_out,
                                   n_terms_out, dev_postings_out, &bad));
    if (bad == 2)
        return fail(h, LRX_E_ARG, "lrx_bm25_remove_postings: term_ptr[n_terms] != nnz, term_ptr_out[0] != 0 "
                                  "or term_ptr_out[n_terms_out] != nnz - rem_ptr[n_terms]");
    if (bad)
        return fail(h, LRX_E_ARG, "lrx_bm25_remove_postings: the removal does not describe the index (removed "
                                  "ids unsorted or out of range, a removed list unsorted or not the term's "
                                  "removed postings, term_map not a bijection onto the surviving terms, or an "
                                  "output range of the wrong length)");
    return LRX_OK;
}

int lrx_bm25_replace_postings(lrx_handle* h, const uint64_t* dev_term_ptr, const void* dev_postings,
                              int64_t n_terms, int64_t nnz, int64_t n_docs,
                              const uint32_t* dev_replaced_docs, int64_t n_replaced,
                              const uint64_t* dev_rem_ptr, const uint32_t* dev_rem_doc,
                              const int32_t* dev_term_map, const uint64_t* dev_ins_ptr,
                              const uint32_t* dev_ins_doc_tf, int64_t nnz_ins, const uint32_t* dev_doc_len,
                              const uint64_t* dev_term_ptr_out, int64_t n_terms_out, void* dev_postings_out) {
    if (h == nullptr) return fail(nullptr, LRX_E_ARG, "lrx_bm25_replace_postings: null handle");
    std::lock_guard<std::mutex> g(h->mu);
    if (n_terms < 0 || nnz < 0 || n_docs < 0 || n_docs >= (1ll << 32) || n_replaced < 0 || n_replaced > n_docs ||
        nnz_ins < 0 || n_terms_out < 0 || n_terms_out > INT32_MAX)
        return fail(h, LRX_E_ARG, "lrx_bm25_replace_postings: bad size");
    if (dev_term_ptr == nullptr || dev_rem_ptr == nullptr || dev_ins_ptr == nullptr || dev_term_ptr_out == nullptr ||
        (n_terms > 0 && dev_term_map == nullptr) || (n_replaced > 0 && dev_replaced_docs == nullptr) ||
        (nnz_ins > 0 && (dev_ins_doc_tf == nullptr || dev_doc_len == nullptr)) ||
        (nnz > 0 && dev_postings == nullptr) || (nnz + nnz_ins > 0 && dev_postings_out == nullptr))
        return fail(h, LRX_E_ARG, "lrx_bm25_replace_postings: null pointer");
    if ((((uintptr_t)dev_postings | (uintptr_t)dev_postings_out) & 15) != 0 ||
        (((uintptr_t)dev_term_ptr | (uintptr_t)dev_rem_ptr | (uintptr_t)dev_ins_ptr | (uintptr_t)dev_ins_doc_tf |
          (uintptr_t)dev_term_ptr_out) & 7) != 0 ||
        (((uintptr_t)dev_replaced_docs | (uintptr_t)dev_rem_doc | (uintptr_t)dev_term_map |
          (uintptr_t)dev_doc_len) & 3) != 0)
        return fail(h, LRX_E_ARG, "lrx_bm25_replace_postings: postings must be 16-byte aligned, pointer "
                                  "tables and (doc, tf) pairs 8-byte aligned, id arrays 4-byte aligned");
    LRX_CUDA(h, cudaSetDevice(h->device));
    int bad = 0;
    LRX_CUDA(h, launch_bm25_replace(h, dev_term_ptr, dev_postings, n_terms, nnz, n_docs, dev_replaced_docs,
                                    n_replaced, dev_rem_ptr, dev_rem_doc, dev_term_map, dev_ins_ptr, dev_ins_doc_tf,
                                    nnz_ins, dev_doc_len, dev_term_ptr_out, n_terms_out, dev_postings_out, &bad));
    if (bad == 2)
        return fail(h, LRX_E_ARG, "lrx_bm25_replace_postings: term_ptr[n_terms] != nnz, ins_ptr[0] != 0, "
                                  "ins_ptr[n_terms_out] != nnz_ins, term_ptr_out[0] != 0 or term_ptr_out[n_terms_out] "
                                  "!= nnz - rem_ptr[n_terms] + nnz_ins");
    if (bad)
        return fail(h, LRX_E_ARG, "lrx_bm25_replace_postings: the replacement does not describe the index "
                                  "(replaced ids unsorted or out of range, a dropped list unsorted or not the "
                                  "term's postings of replaced documents, an inserted list unsorted or holding a "
                                  "document that is not replaced, a tf or length over 65535, term_map not "
                                  "injective, or an output range of the wrong length)");
    return LRX_OK;
}

int lrx_set_encoder_weights(lrx_handle* h, const lrx_bert_weights* w) {
    if (h == nullptr) return fail(nullptr, LRX_E_ARG, "lrx_set_encoder_weights: null handle");
    std::lock_guard<std::mutex> g(h->mu);
    if (w == nullptr) return fail(h, LRX_E_ARG, "lrx_set_encoder_weights: null weights");
    if (w->vocab_size < 1 || w->max_positions < 1)
        return fail(h, LRX_E_ARG, "lrx_set_encoder_weights: bad vocab_size / max_positions");
    const float* top[] = {w->word_emb, w->pos_emb, w->type_emb, w->emb_ln_g, w->emb_ln_b};
    for (const float* p : top)
        if (p == nullptr) return fail(h, LRX_E_ARG, "lrx_set_encoder_weights: null embedding tensor");
    for (int l = 0; l < LRX_BERT_LAYERS; ++l) {
        const lrx_bert_layer& s = w->layers[l];
        const float* ps[] = {s.wq, s.bq, s.wk, s.bk, s.wv, s.bv, s.wo, s.bo, s.ln1_g, s.ln1_b,
                             s.w1, s.b1, s.w2, s.b2, s.ln2_g, s.ln2_b};
        for (const float* p : ps)
            if (p == nullptr)
                return fail(h, LRX_E_ARG, "lrx_set_encoder_weights: null tensor in layer %d", l);
    }
    LRX_CUDA(h, cudaSetDevice(h->device));
    LRX_CUDA(h, encoder_set_weights(h, w));
    return LRX_OK;
}

static int check_encode(lrx_handle* h, const char* fn, int B, int S) {
    if (h->encoder == nullptr) return fail(h, LRX_E_STATE, "%s: encoder weights not set", fn);
    if (B < 1 || B > (1 << 20)) return fail(h, LRX_E_ARG, "%s: B must be in [1, 2^20]", fn);
    if (S < 1 || S > 512) return fail(h, LRX_E_ARG, "%s: S must be in [1,512]", fn);
    return LRX_OK;
}

int lrx_encode(lrx_handle* h, const int32_t* dev_ids, const int32_t* dev_lens, int32_t B, int32_t S,
               float* dev_out_f32, void* dev_out_f16) {
    if (h == nullptr) return fail(nullptr, LRX_E_ARG, "lrx_encode: null handle");
    std::lock_guard<std::mutex> g(h->mu);
    int rc = check_encode(h, "lrx_encode", B, S);
    if (rc != LRX_OK) return rc;
    if (dev_ids == nullptr || dev_lens == nullptr || (dev_out_f32 == nullptr && dev_out_f16 == nullptr))
        return fail(h, LRX_E_ARG, "lrx_encode: null pointer");
    LRX_CUDA(h, cudaSetDevice(h->device));
    LRX_CUDA(h, encoder_forward(h, dev_ids, dev_lens, B, S, dev_out_f32, dev_out_f16));
    return LRX_OK;
}

int lrx_encode_host(lrx_handle* h, const int32_t* host_ids, const int32_t* host_lens, int32_t B,
                    int32_t S, float* host_out_f32) {
    if (h == nullptr) return fail(nullptr, LRX_E_ARG, "lrx_encode_host: null handle");
    std::lock_guard<std::mutex> g(h->mu);
    int rc = check_encode(h, "lrx_encode_host", B, S);
    if (rc != LRX_OK) return rc;
    if (host_ids == nullptr || host_lens == nullptr || host_out_f32 == nullptr)
        return fail(h, LRX_E_ARG, "lrx_encode_host: null pointer");
    LRX_CUDA(h, cudaSetDevice(h->device));
    LRX_CUDA(h, encoder_forward_host(h, host_ids, host_lens, B, S, host_out_f32));
    return LRX_OK;
}

int lrx_gemm_f16(lrx_handle* h, const void* dev_a, const void* dev_w, int32_t M, int32_t N, int32_t K,
                 int32_t epi, const float* dev_bias, const void* dev_residual,
                 const float* dev_gamma, const float* dev_beta, float eps, void* dev_out) {
    if (h == nullptr) return fail(nullptr, LRX_E_ARG, "lrx_gemm_f16: null handle");
    std::lock_guard<std::mutex> g(h->mu);
    if (M < 1 || N < 128 || N % 128 != 0 || K < 64 || K % 64 != 0)
        return fail(h, LRX_E_ARG, "lrx_gemm_f16: need M >= 1, N %% 128 == 0, K %% 64 == 0");
    if (epi < 0 || epi > 3 || (epi == 2 && N != 384) || (epi != 3 && N > 1536))
        return fail(h, LRX_E_ARG, "lrx_gemm_f16: bad epilogue (LayerNorm needs N == 384; epi 0-2 need N <= 1536)");
    if (dev_a == nullptr || dev_w == nullptr || dev_out == nullptr ||
        (epi != 3 && dev_bias == nullptr) ||
        (epi == 2 && (dev_residual == nullptr || dev_gamma == nullptr || dev_beta == nullptr)))
        return fail(h, LRX_E_ARG, "lrx_gemm_f16: null pointer");
    if ((((uintptr_t)dev_a | (uintptr_t)dev_w | (uintptr_t)dev_out) & 15) != 0)
        return fail(h, LRX_E_ARG, "lrx_gemm_f16: operands must be 16-byte aligned");
    LRX_CUDA(h, cudaSetDevice(h->device));
    LRX_CUDA(h, gemm_f16_adhoc(h, dev_a, dev_w, M, N, K, epi, dev_bias, dev_residual, dev_gamma,
                               dev_beta, eps, dev_out));
    return LRX_OK;
}

// K2 by batch size (SURVEY.md 8b: "K2a/K2b chosen by B"): up to 8 queries share ONE streaming pass
// of the matrix (K2a, HBM-bound: the 8 columns of its MMA tile are all queries then); from 9 queries
// on the tensor-core kernel scores the whole batch in one pass (K2b) where K2a would need
// ceil(B / 8) -- measured at 10 M rows: B = 64 1.32 ms against 18.1 ms (tools/k2_crossover.py); both
// emit the same exact lists.  A widened retry (exactness guard / candidate overflow) runs K2a at
// that width: width is K2a's parameter, and K2b flags only a query with more than 1024 rows near its
// K-th score, which K2b at any stride would flag again.
constexpr int kK2bMinB = 9;
static cudaError_t launch_dense_auto(lrx_handle* h, const void* q, int B, int K, int width, double* exact,
                                     float* D, int64_t* I, int32_t* flags) {
    if (B >= kK2bMinB && h->n_local > 0 && ((uintptr_t)q & 15) == 0 && width <= dense_default_width(K))
        return launch_dense_topk_batched(h, q, B, K, 0, exact, D, I, flags);
    return launch_dense_topk(h, q, B, K, width, exact, D, I, flags);
}

static int check_dense(lrx_handle* h, const char* fn, int B, int K) {
    if (h->x == nullptr && h->n_local > 0) return fail(h, LRX_E_STATE, "%s: corpus not set", fn);
    if (B < 1 || B > LRX_MAX_BATCH) return fail(h, LRX_E_ARG, "%s: B must be in [1,%d]", fn, LRX_MAX_BATCH);
    if (K < 1 || K > LRX_MAX_DEPTH) return fail(h, LRX_E_ARG, "%s: K must be in [1,%d]", fn, LRX_MAX_DEPTH);
    return LRX_OK;
}

int lrx_dense_topk_ex(lrx_handle* h, const void* dev_q_fp16, int32_t B, int32_t K, int32_t width,
                      double* dev_exact, float* dev_D, int64_t* dev_I, int32_t* dev_flags) {
    if (h == nullptr) return fail(nullptr, LRX_E_ARG, "lrx_dense_topk: null handle");
    std::lock_guard<std::mutex> g(h->mu);
    int rc = check_dense(h, "lrx_dense_topk", B, K);
    if (rc != LRX_OK) return rc;
    if (dev_q_fp16 == nullptr || dev_exact == nullptr || dev_D == nullptr || dev_I == nullptr ||
        dev_flags == nullptr)
        return fail(h, LRX_E_ARG, "lrx_dense_topk: null pointer");
    if (width <= 0) width = dense_default_width(K);
    if (width < K || width > 512 || (width & (width - 1)) != 0)
        return fail(h, LRX_E_ARG, "lrx_dense_topk: width must be a power of two in [K,512]");
    LRX_CUDA(h, cudaSetDevice(h->device));
    LRX_CUDA(h, launch_dense_auto(h, dev_q_fp16, B, K, width, dev_exact, dev_D, dev_I, dev_flags));
    return LRX_OK;
}

int lrx_dense_topk(lrx_handle* h, const void* dev_q_fp16, int32_t B, int32_t K, double* dev_exact,
                   float* dev_D, int64_t* dev_I, int32_t* dev_flags) {
    return lrx_dense_topk_ex(h, dev_q_fp16, B, K, 0, dev_exact, dev_D, dev_I, dev_flags);
}

int lrx_dense_topk_batched(lrx_handle* h, const void* dev_q_fp16, int32_t B, int32_t K, int32_t stride,
                           double* dev_exact, float* dev_D, int64_t* dev_I, int32_t* dev_flags) {
    if (h == nullptr) return fail(nullptr, LRX_E_ARG, "lrx_dense_topk_batched: null handle");
    std::lock_guard<std::mutex> g(h->mu);
    if (h->x == nullptr || h->n_local < 1) return fail(h, LRX_E_STATE, "lrx_dense_topk_batched: corpus not set");
    if (B < 1 || B > 4096) return fail(h, LRX_E_ARG, "lrx_dense_topk_batched: B must be in [1,4096]");
    if (K < 1 || K > LRX_MAX_DEPTH) return fail(h, LRX_E_ARG, "lrx_dense_topk_batched: K must be in [1,%d]", LRX_MAX_DEPTH);
    if (stride < 0) return fail(h, LRX_E_ARG, "lrx_dense_topk_batched: stride < 0");
    if (dev_q_fp16 == nullptr || dev_exact == nullptr || dev_D == nullptr || dev_I == nullptr ||
        dev_flags == nullptr || ((uintptr_t)dev_q_fp16 & 15) != 0)
        return fail(h, LRX_E_ARG, "lrx_dense_topk_batched: null or misaligned pointer");
    LRX_CUDA(h, cudaSetDevice(h->device));
    LRX_CUDA(h, launch_dense_topk_batched(h, dev_q_fp16, B, K, stride, dev_exact, dev_D, dev_I, dev_flags));
    return LRX_OK;
}

int lrx_dense_at(lrx_handle* h, const void* dev_q_fp16, int32_t B, const int64_t* dev_ids,
                 int32_t n, double* dev_out) {
    if (h == nullptr) return fail(nullptr, LRX_E_ARG, "lrx_dense_at: null handle");
    std::lock_guard<std::mutex> g(h->mu);
    if (h->x == nullptr && h->n_local > 0) return fail(h, LRX_E_STATE, "lrx_dense_at: corpus not set");
    if (B < 1 || B > LRX_MAX_BATCH || n < 0) return fail(h, LRX_E_ARG, "lrx_dense_at: bad B/n");
    if (dev_q_fp16 == nullptr || (n > 0 && (dev_ids == nullptr || dev_out == nullptr)))
        return fail(h, LRX_E_ARG, "lrx_dense_at: null pointer");
    LRX_CUDA(h, cudaSetDevice(h->device));
    LRX_CUDA(h, launch_dense_at(h, dev_q_fp16, B, dev_ids, n, dev_out));
    return LRX_OK;
}

int lrx_bm25(lrx_handle* h, const int32_t* dev_q_terms, const int32_t* dev_q_ptr, int32_t B,
             const int64_t* dev_cand_ids, int32_t n_cand, double* dev_cand_scores, double* dev_max,
             int32_t K, double* dev_top_scores, int64_t* dev_top_ids) {
    if (h == nullptr) return fail(nullptr, LRX_E_ARG, "lrx_bm25: null handle");
    std::lock_guard<std::mutex> g(h->mu);
    if (h->term_ptr == nullptr) return fail(h, LRX_E_STATE, "lrx_bm25: postings not set");
    if (B < 1 || B > LRX_MAX_BATCH) return fail(h, LRX_E_ARG, "lrx_bm25: B must be in [1,%d]", LRX_MAX_BATCH);
    if (K < 0 || K > LRX_MAX_DEPTH) return fail(h, LRX_E_ARG, "lrx_bm25: K must be in [0,%d]", LRX_MAX_DEPTH);
    if (n_cand < 0) return fail(h, LRX_E_ARG, "lrx_bm25: n_cand < 0");
    if (dev_q_ptr == nullptr || dev_max == nullptr ||
        (n_cand > 0 && (dev_cand_ids == nullptr || dev_cand_scores == nullptr)) ||
        (K > 0 && (dev_top_scores == nullptr || dev_top_ids == nullptr)))
        return fail(h, LRX_E_ARG, "lrx_bm25: null pointer");
    LRX_CUDA(h, cudaSetDevice(h->device));
    h->bm_rows = h->bm_rows_cfg;
    h->bm_list_k = K;
    h->bm_ctas_per_sm = 0;
    LRX_CUDA(h, launch_bm25(h, dev_q_terms, dev_q_ptr, B, dev_cand_ids, n_cand, dev_cand_scores,
                            dev_max, K, dev_top_scores, dev_top_ids));
    return LRX_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------
// K5: the launch chain of one query batch.
//
// Two chains side by side.  Main stream: dense scan -> merge + exact re-score.  Side stream: BM25
// range bounds -> BM25 scan -> merge + max.  Neither needs the other's result (the BM25 scores AT
// the dense candidates are looked up afterwards, inside the packing kernel), and the two scans
// are built to share an SM -- the dense scan is bound by HBM and leaves the issue slots idle, the
// BM25 scan is bound by issue/FP64 latency and leaves HBM idle; one CTA of each fits the registers
// and the shared memory of an SM.  The dense scan is launched first so that its 148 CTAs are
// placed before the BM25 CTAs fill the rest.  After the join: pack (+ peer exchange) -> fusion.
//
// The whole chain is captured once per (shape, pointers) into a CUDA graph and replayed with a
// single cudaGraphLaunch (run_planned): 8 launches + 4 event operations from the host per batch
// become one, which is what the small shards of an 8-GPU box need (0.18 ms of GPU work per batch).

// ---- packed block: [B][2][2k] records | [B] double | [B] int32, 16-byte padded
static void packed_layout(int B, int k, size_t* o_max, size_t* o_flags, size_t* total) {
    const size_t rec = (size_t)B * 2 * (2 * k) * sizeof(lrx_record);
    *o_max = rec;
    *o_flags = rec + (size_t)B * sizeof(double);
    *total = align_up(*o_flags + (size_t)B * sizeof(int32_t), 16);
}

// scratch carved out of ws_misc for one local chain
struct LocalScratch {
    double* dense_exact;
    float* dense_D;
    int64_t* dense_I;
    double* bm_scores;
    int64_t* bm_ids;
    double* maxbm;
    int32_t* flags;
    unsigned char* block;       // packed block of this shard (world == 1)
};

static int carve_scratch(lrx_handle* h, int B, int k, LocalScratch* s) {
    const int K = 2 * k;
    const size_t n = (size_t)B * K;
    size_t o_max, o_flags, total;
    packed_layout(B, k, &o_max, &o_flags, &total);
    const size_t need = n * (2 * sizeof(double) + 2 * sizeof(int64_t) + sizeof(float)) +
                        (size_t)B * (sizeof(double) + sizeof(int32_t)) + total + 2048;
    LRX_CUDA(h, ensure_ws(h, &h->ws_misc, &h->ws_misc_bytes, need));
    char* p = (char*)h->ws_misc;
    s->dense_exact = (double*)p; p += n * sizeof(double);
    s->bm_scores = (double*)p;   p += n * sizeof(double);
    s->dense_I = (int64_t*)p;    p += n * sizeof(int64_t);
    s->bm_ids = (int64_t*)p;     p += n * sizeof(int64_t);
    s->maxbm = (double*)p;       p += align_up((size_t)B * sizeof(double), 16);
    s->block = (unsigned char*)p; p += align_up(total, 256);
    s->dense_D = (float*)p;      p += align_up(n * sizeof(float), 16);
    s->flags = (int32_t*)p;
    return LRX_OK;
}

static int check_search_args(lrx_handle* h, const char* fn, int B, int k, int mode, int* width) {
    const int K = 2 * k;   // index.search(query_vector, k * 2)  (retrieval_engine.py:64)
    if (k < 1) return fail(h, LRX_E_ARG, "%s: k must be >= 1", fn);
    int rc = check_dense(h, fn, B, K);
    if (rc != LRX_OK) return rc;
    if (h->term_ptr == nullptr) return fail(h, LRX_E_STATE, "%s: postings not set", fn);
    if (mode != LRX_FUSE_LINEAR && mode != LRX_FUSE_RRF)
        return fail(h, LRX_E_ARG, "%s: unknown fusion mode %d", fn, mode);
    if (*width <= 0) *width = dense_default_width(K);
    if (*width < K || *width > 512 || (*width & (*width - 1)) != 0)
        return fail(h, LRX_E_ARG, "%s: width must be a power of two in [2k,512]", fn);
    if (h->world * K > 2048) return fail(h, LRX_E_ARG, "%s: world*2k must be <= 2048", fn);
    return LRX_OK;
}

// K2 + K3 on this shard -> packed block -> K4.  world == 1: the block stays in the scratch
// (s.block); world > 1: it is stored into every shard's exchange region, and K4 reads all the
// shards' blocks from this rank's region.  Arguments are checked by the callers.
static int enqueue_search(lrx_handle* h, const LocalScratch& s, const void* q, const int32_t* q_terms,
                          const int32_t* q_ptr, const double* weights, int B, int k, int mode, int width,
                          int64_t* ids, double* score, double* sem, double* kw, int32_t* status) {
    const int K = 2 * k;
    size_t o_max, o_flags, total;
    packed_layout(B, k, &o_max, &o_flags, &total);
    const bool peers = h->world > 1;
    const int Kb = (mode == LRX_FUSE_RRF) ? K : 0;
    h->bm_list_k = Kb;
    // K2a's CTA shares the SM (profiles/r2_runs/ab_bm25_chain_ctas.txt; 5..8 queries on a small shard keep
    // the second wave: there the BM25 scan outlasts the dense scan by far and the wave does real work)
    h->bm_ctas_per_sm = (B < kK2bMinB && h->n_local > 0 && (B <= 4 || h->n_local >= (4ll << 20))) ? 1 : 0;
    LRX_CUDA(h, cudaEventRecord(h->ev_fork, h->stream));
    LRX_CUDA(h, cudaStreamWaitEvent(h->aux, h->ev_fork, 0));
    LRX_CUDA(h, launch_dense_auto(h, q, B, K, width, s.dense_exact, s.dense_D, s.dense_I, s.flags));
    LRX_CUDA(h, launch_bm25_bounds(h, q_terms, q_ptr, B, h->aux));
    LRX_CUDA(h, launch_bm25_scan(h, q_terms, q_ptr, B, s.maxbm, Kb, s.bm_scores, s.bm_ids, h->aux));
    LRX_CUDA(h, cudaEventRecord(h->ev_join, h->aux));
    LRX_CUDA(h, cudaStreamWaitEvent(h->stream, h->ev_join, 0));   // join
    LRX_CUDA(h, launch_pack_exchange(h, q_terms, q_ptr, B, K, mode, s.dense_exact, s.dense_I, s.bm_scores,
                                     s.bm_ids, s.maxbm, s.flags, q, s.block, peers, o_max, o_flags));
    LRX_CUDA(h, launch_fuse(h, peers ? h->xchg : s.block, peers ? h->xchg_slot : total, o_max, o_flags, peers,
                            h->world, B, K, k, mode, weights, ids, score, sem, kw, status));
    return LRX_OK;
}

// ---- captured chains
static bool key_in(const std::vector<std::vector<uint64_t>>& set, const std::vector<uint64_t>& key) {
    for (const auto& k : set)
        if (k == key) return true;
    return false;
}

// Runs `enqueue` (a callable that launches a chain on h->stream / h->aux) either directly or as a
// replay of its captured graph.  First call with a key: direct (it also grows the workspaces and
// sets the function attributes, neither of which may happen while capturing).  Second call:
// capture + instantiate + replay.  Later calls: one cudaGraphLaunch.  A chain that cannot be
// captured stays on the direct path.
template <typename F>
static int run_planned(lrx_handle* h, std::vector<uint64_t> key, F&& enqueue) {
    key.push_back(h->prof ? 1u : 0u);
    for (size_t i = 0; i < h->plans.size(); ++i) {
        lrx_plan* pl = h->plans[i];
        if (pl->key != key) continue;
        if (pl->epoch == h->ws_epoch) {
            LRX_CUDA(h, cudaGraphLaunch(pl->exec, h->stream));
            h->launches += pl->kernels;
            pl->stamp = ++h->plan_clock;
            pl->replayed = true;
            return LRX_OK;
        }
        cudaGraphExecDestroy(pl->exec);                      // stale: a workspace or the index moved
        for (int w = 0; w < 2; ++w)
            for (cudaEvent_t e : pl->prof_ev[w]) cudaEventDestroy(e);
        delete pl;
        h->plans.erase(h->plans.begin() + (long)i);
        break;
    }
    if (key_in(h->eager_keys, key)) return enqueue();
    if (!key_in(h->seen_keys, key)) {
        if (h->seen_keys.size() >= 256) h->seen_keys.clear();
        h->seen_keys.push_back(key);
        return enqueue();
    }
    // ---- capture on the handle's own stream (the user's may be the legacy default stream)
    lrx_plan* pl = new (std::nothrow) lrx_plan();
    if (pl == nullptr) return enqueue();
    cudaStream_t user = h->stream;
    const int64_t l0 = h->launches;
    cudaGraph_t graph = nullptr;
    cudaError_t ce = cudaStreamBeginCapture(h->cap, cudaStreamCaptureModeRelaxed);
    int rc = LRX_E_CUDA;
    if (ce == cudaSuccess) {
        h->capturing = true; h->cap_plan = pl; h->stream = h->cap;
        rc = enqueue();
        h->stream = user; h->capturing = false; h->cap_plan = nullptr;
        ce = cudaStreamEndCapture(h->cap, &graph);
    }
    pl->kernels = h->launches - l0;
    h->launches = l0;
    if (rc == LRX_OK && ce == cudaSuccess && graph != nullptr)
        ce = cudaGraphInstantiate(&pl->exec, graph, 0);
    if (graph != nullptr) cudaGraphDestroy(graph);
    if (rc != LRX_OK || ce != cudaSuccess || pl->exec == nullptr) {
        cudaGetLastError();                                  // clear the capture error
        for (int w = 0; w < 2; ++w)
            for (cudaEvent_t e : pl->prof_ev[w]) cudaEventDestroy(e);
        if (pl->exec != nullptr) cudaGraphExecDestroy(pl->exec);
        delete pl;
        if (h->eager_keys.size() >= 256) h->eager_keys.clear();
        h->eager_keys.push_back(key);
        return enqueue();
    }
    pl->key = key;
    pl->epoch = h->ws_epoch;
    if (h->plans.size() >= 96) {                             // evict the least recently used plan
        size_t lru = 0;
        for (size_t i = 1; i < h->plans.size(); ++i)
            if (h->plans[i]->stamp < h->plans[lru]->stamp) lru = i;
        lrx_plan* old = h->plans[lru];
        cudaGraphExecDestroy(old->exec);
        for (int w = 0; w < 2; ++w)
            for (cudaEvent_t e : old->prof_ev[w]) cudaEventDestroy(e);
        delete old;
        h->plans.erase(h->plans.begin() + (long)lru);
    }
    h->plans.push_back(pl);
    LRX_CUDA(h, cudaGraphLaunch(pl->exec, h->stream));
    h->launches += pl->kernels;
    pl->stamp = ++h->plan_clock;
    pl->replayed = true;
    return LRX_OK;
}

static uint64_t pk(const void* p) { return (uint64_t)(uintptr_t)p; }

extern "C" {

int lrx_set_query_capacity(lrx_handle* h, int32_t max_total_terms) {
    if (h == nullptr) return fail(nullptr, LRX_E_ARG, "lrx_set_query_capacity: null handle");
    std::lock_guard<std::mutex> g(h->mu);
    if (max_total_terms < 0 || max_total_terms > (1 << 20))
        return fail(h, LRX_E_ARG, "lrx_set_query_capacity: capacity must be in [0, 2^20]");
    h->bm_rows_cfg = max_total_terms;
    return LRX_OK;
}

int lrx_set_exchange_timeout(lrx_handle* h, int32_t milliseconds) {
    if (h == nullptr) return fail(nullptr, LRX_E_ARG, "lrx_set_exchange_timeout: null handle");
    std::lock_guard<std::mutex> g(h->mu);
    if (milliseconds < 1) return fail(h, LRX_E_ARG, "lrx_set_exchange_timeout: must be >= 1 ms");
    h->xchg_timeout_ms = milliseconds;
    h->ws_epoch++;                        // the bound is a kernel argument of the captured chains
    return LRX_OK;
}

// ---- peer exchange: region = data [2 parities][world][slot] | flags u64 [2][world] | ctr u64
static_assert(sizeof(cudaIpcMemHandle_t) == LRX_IPC_HANDLE_BYTES, "IPC handle size");

int lrx_exchange_export(lrx_handle* h, int32_t B_max, int32_t k_max, void* host_handle_out) {
    if (h == nullptr) return fail(nullptr, LRX_E_ARG, "lrx_exchange_export: null handle");
    std::lock_guard<std::mutex> g(h->mu);
    if (host_handle_out == nullptr || B_max < 1 || B_max > LRX_MAX_BATCH || k_max < 1 ||
        2 * k_max > LRX_MAX_DEPTH)
        return fail(h, LRX_E_ARG, "lrx_exchange_export: bad argument");
    if (h->world < 2 || h->world > LRX_MAX_WORLD)
        return fail(h, LRX_E_STATE, "lrx_exchange_export: world must be in [2,%d]", LRX_MAX_WORLD);
    if (h->xchg != nullptr) return fail(h, LRX_E_STATE, "lrx_exchange_export: already exported");
    LRX_CUDA(h, cudaSetDevice(h->device));
    size_t o_max, o_flags, total;
    packed_layout(B_max, k_max, &o_max, &o_flags, &total);
    h->xchg_slot = align_up(total, 256);
    h->xchg_bytes = 2 * (size_t)h->world * h->xchg_slot +
                    (2 * (size_t)h->world + 2) * sizeof(unsigned long long);
    LRX_CUDA(h, cudaMalloc(&h->xchg, h->xchg_bytes));
    LRX_CUDA(h, cudaMemset(h->xchg, 0, h->xchg_bytes));
    LRX_CUDA(h, cudaDeviceSynchronize());
    cudaIpcMemHandle_t ipc;
    LRX_CUDA(h, cudaIpcGetMemHandle(&ipc, h->xchg));
    memcpy(host_handle_out, &ipc, sizeof(ipc));
    return LRX_OK;
}

int lrx_exchange_import(lrx_handle* h, const void* host_handles_all) {
    if (h == nullptr) return fail(nullptr, LRX_E_ARG, "lrx_exchange_import: null handle");
    std::lock_guard<std::mutex> g(h->mu);
    if (host_handles_all == nullptr) return fail(h, LRX_E_ARG, "lrx_exchange_import: null pointer");
    if (h->xchg == nullptr) return fail(h, LRX_E_STATE, "lrx_exchange_import: export first");
    if (h->xchg_ready) return fail(h, LRX_E_STATE, "lrx_exchange_import: already imported");
    LRX_CUDA(h, cudaSetDevice(h->device));
    for (int w = 0; w < h->world; ++w) {
        if (w == h->rank) { h->xchg_peer[w] = h->xchg; continue; }
        cudaIpcMemHandle_t ipc;
        memcpy(&ipc, (const char*)host_handles_all + (size_t)w * sizeof(ipc), sizeof(ipc));
        LRX_CUDA(h, cudaIpcOpenMemHandle(&h->xchg_peer[w], ipc, cudaIpcMemLazyEnablePeerAccess));
    }
    LRX_CUDA(h, cudaMalloc((void**)&h->xchg_peer_dev, LRX_MAX_WORLD * sizeof(void*)));
    LRX_CUDA(h, cudaMemcpy(h->xchg_peer_dev, h->xchg_peer, LRX_MAX_WORLD * sizeof(void*),
                           cudaMemcpyHostToDevice));
    h->xchg_ready = true;
    return LRX_OK;
}

// K2 + K3 on this shard -> packed block (world == 1: handle workspace; world > 1: every shard's
// exchange region) -> K4.  Every argument is checked BEFORE anything is enqueued: the call's
// sequence number lives on the device and only advances when the packing kernel runs, so a call
// that is refused here leaves this rank in step with its peers.
static int search_device_locked(lrx_handle* h, const char* fn, const void* q, const int32_t* q_terms,
                                const int32_t* q_ptr, const double* weights, int B, int k, int mode,
                                int width, int64_t* ids, double* score, double* sem, double* kw,
                                int32_t* status) {
    int rc = check_search_args(h, fn, B, k, mode, &width);
    if (rc != LRX_OK) return rc;
    const bool peers = h->world > 1;
    if (peers && !h->xchg_ready) return fail(h, LRX_E_STATE, "%s: exchange not set up", fn);
    size_t o_max, o_flags, total;
    packed_layout(B, k, &o_max, &o_flags, &total);
    if (peers && total > h->xchg_slot)
        return fail(h, LRX_E_ARG, "%s: batch larger than the exported exchange slots", fn);
    LocalScratch s;
    rc = carve_scratch(h, B, k, &s);
    if (rc != LRX_OK) return rc;
    return run_planned(
        h, {2u, pk(q), pk(q_terms), pk(q_ptr), pk(weights), pk(ids), pk(score), pk(sem), pk(kw), pk(status),
            (uint64_t)B, (uint64_t)k, (uint64_t)mode, (uint64_t)width, (uint64_t)h->bm_rows},
        [&]() -> int {
            return enqueue_search(h, s, q, q_terms, q_ptr, weights, B, k, mode, width, ids, score, sem, kw,
                                  status);
        });
}

int lrx_search_sharded(lrx_handle* h, const void* dev_q_fp16, const int32_t* dev_q_terms,
                       const int32_t* dev_q_ptr, const double* dev_weights, int32_t B, int32_t k,
                       int32_t mode, int32_t width, int64_t* dev_ids, double* dev_score,
                       double* dev_sem, double* dev_kw, int32_t* dev_status) {
    if (h == nullptr) return fail(nullptr, LRX_E_ARG, "lrx_search_sharded: null handle");
    std::lock_guard<std::mutex> g(h->mu);
    if (dev_q_fp16 == nullptr || dev_q_ptr == nullptr || dev_ids == nullptr || dev_score == nullptr ||
        dev_sem == nullptr || dev_kw == nullptr || dev_status == nullptr ||
        (mode == LRX_FUSE_LINEAR && dev_weights == nullptr))
        return fail(h, LRX_E_ARG, "lrx_search_sharded: null pointer");
    LRX_CUDA(h, cudaSetDevice(h->device));
    h->bm_rows = h->bm_rows_cfg;
    return search_device_locked(h, "lrx_search_sharded", dev_q_fp16, dev_q_terms, dev_q_ptr, dev_weights,
                                B, k, mode, width, dev_ids, dev_score, dev_sem, dev_kw, dev_status);
}

// ---- host-buffer searches: staging layout (same offsets in pinned host memory and on the device)
struct HostLayout {
    size_t o_q, o_w, o_ptr, o_terms, o_tok, o_len, in_bytes;
    size_t o_ids, o_score, o_sem, o_kw, o_status, out_bytes, total;
};

static HostLayout host_layout(int B, int k, int rows, bool encode, int S) {
    HostLayout L;
    size_t off = 0;
    L.o_q = off;       off = align_up(off + (size_t)B * kRowBytes, 256);
    L.o_w = off;       off = align_up(off + (size_t)B * sizeof(double), 256);
    L.o_ptr = off;     off = align_up(off + (size_t)(B + 1) * sizeof(int32_t), 256);
    L.o_terms = off;   off = align_up(off + (size_t)rows * sizeof(int32_t), 256);
    L.o_tok = off;     off = align_up(off + (encode ? (size_t)B * S * sizeof(int32_t) : 0), 256);
    L.o_len = off;     off = align_up(off + (encode ? (size_t)B * sizeof(int32_t) : 0), 256);
    L.in_bytes = off;
    L.o_ids = off;     off = align_up(off + (size_t)B * k * sizeof(int64_t), 256);
    L.o_score = off;   off = align_up(off + (size_t)B * k * sizeof(double), 256);
    L.o_sem = off;     off = align_up(off + (size_t)B * k * sizeof(double), 256);
    L.o_kw = off;      off = align_up(off + (size_t)B * k * sizeof(double), 256);
    L.o_status = off;  off = align_up(off + (size_t)B * sizeof(int32_t), 256);
    L.out_bytes = off - L.in_bytes;
    L.total = off;
    return L;
}

// H2D of the staged inputs, (K1,) K2..K4, D2H of the results -- one captured chain per shape.
static int enqueue_host_chain(lrx_handle* h, const lrx_pending& p) {
    const HostLayout L = host_layout(p.B, p.k, p.rows, p.encode, p.S);
    char* hp = (char*)h->ws_host;
    char* dp = (char*)h->ws_io;
    h->bm_rows = p.rows;
    return run_planned(
        h, {3u, (uint64_t)p.B, (uint64_t)p.k, (uint64_t)p.mode, (uint64_t)p.width, (uint64_t)p.rows,
            (uint64_t)p.encode, (uint64_t)p.S, pk(hp), pk(dp)},
        [&]() -> int {
            LRX_CUDA(h, cudaMemcpyAsync(dp, hp, L.in_bytes, cudaMemcpyHostToDevice, h->stream));
            // K1: token ids -> fp16 unit query vectors, straight into the K2 operand slot.  (Measured:
            // the BM25 chain cannot usefully run UNDER the encoder -- its persistent CTAs take every SM
            // and the encoder's GEMM CTAs, which need a whole SM's shared memory, wait for them -- so
            // K1 runs first and the two scans share the SMs afterwards.)
            if (p.encode)
                LRX_CUDA(h, encoder_forward(h, (const int32_t*)(dp + L.o_tok), (const int32_t*)(dp + L.o_len),
                                            p.B, p.S, nullptr, dp + L.o_q));
            LocalScratch s;
            int rc = carve_scratch(h, p.B, p.k, &s);
            if (rc != LRX_OK) return rc;
            rc = enqueue_search(h, s, dp + L.o_q, (const int32_t*)(dp + L.o_terms), (const int32_t*)(dp + L.o_ptr),
                                (const double*)(dp + L.o_w), p.B, p.k, p.mode, p.width, (int64_t*)(dp + L.o_ids),
                                (double*)(dp + L.o_score), (double*)(dp + L.o_sem), (double*)(dp + L.o_kw),
                                (int32_t*)(dp + L.o_status));
            if (rc != LRX_OK) return rc;
            LRX_CUDA(h, cudaMemcpyAsync(hp + L.in_bytes, dp + L.in_bytes, L.out_bytes, cudaMemcpyDeviceToHost,
                                        h->stream));
            return LRX_OK;
        });
}

// Stage the inputs of a host-buffer search and enqueue its chain; the results are collected by
// host_end_locked.  host_q_fp16 == NULL: the query vectors come from the encoder (token ids).
static int host_begin_locked(lrx_handle* h, const char* fn, const void* host_q_fp16,
                             const int32_t* host_tok, const int32_t* host_lens, int S,
                             const int32_t* host_q_terms, const int32_t* host_q_ptr,
                             const double* host_weights, int32_t B, int32_t k, int32_t mode) {
    if (h->pend.active)
        return fail(h, LRX_E_STATE, "%s: a host search is already in flight on this handle "
                                    "(call lrx_search_host_end first)", fn);
    const bool encode = (host_q_fp16 == nullptr);
    int width = 0;
    int rc = check_search_args(h, fn, B, k, mode, &width);
    if (rc != LRX_OK) return rc;
    if (h->world > 1 && !h->xchg_ready) return fail(h, LRX_E_STATE, "%s: exchange not set up", fn);
    const int nt = host_q_ptr[B];
    if (nt < 0 || host_q_ptr[0] != 0 || nt > (1 << 20)) return fail(h, LRX_E_ARG, "%s: bad q_ptr", fn);
    if (nt > 0 && host_q_terms == nullptr) return fail(h, LRX_E_ARG, "%s: null terms", fn);
    for (int b = 0; b < B; ++b)
        if (host_q_ptr[b + 1] < host_q_ptr[b]) return fail(h, LRX_E_ARG, "%s: q_ptr must not decrease", fn);
    if (h->world > 1) {
        size_t o_max, o_flags, total;
        packed_layout(B, k, &o_max, &o_flags, &total);
        if (total > h->xchg_slot)
            return fail(h, LRX_E_ARG, "%s: batch larger than the exported exchange slots", fn);
    }
    LRX_CUDA(h, cudaSetDevice(h->device));
    // token capacity of the batch: every token is scored (retrieval_engine.py:67-68 has no limit);
    // rounded up so that batches of similar size share a captured chain
    int rows = 32;
    while (rows < nt) rows *= 2;
    lrx_pending p;
    p.active = true; p.encode = encode; p.B = B; p.k = k; p.mode = mode; p.width = width; p.rows = rows;
    p.S = encode ? S : 0;
    const HostLayout L = host_layout(B, k, rows, encode, p.S);
    if (h->ws_host_bytes < L.total) {
        if (h->ws_host != nullptr) cudaFreeHost(h->ws_host);
        h->ws_host = nullptr;
        h->ws_host_bytes = 0;
        h->ws_epoch++;
        LRX_CUDA(h, cudaMallocHost(&h->ws_host, L.total * 2));
        h->ws_host_bytes = L.total * 2;
    }
    LRX_CUDA(h, ensure_ws(h, &h->ws_io, &h->ws_io_bytes, L.total));
    char* hp = (char*)h->ws_host;
    if (!encode) memcpy(hp + L.o_q, host_q_fp16, (size_t)B * kRowBytes);
    memcpy(hp + L.o_w, host_weights, (size_t)B * sizeof(double));
    memcpy(hp + L.o_ptr, host_q_ptr, (size_t)(B + 1) * sizeof(int32_t));
    if (nt > 0) memcpy(hp + L.o_terms, host_q_terms, (size_t)nt * sizeof(int32_t));
    if (encode) {
        memcpy(hp + L.o_tok, host_tok, (size_t)B * S * sizeof(int32_t));
        memcpy(hp + L.o_len, host_lens, (size_t)B * sizeof(int32_t));
    }
    rc = enqueue_host_chain(h, p);
    if (rc != LRX_OK) return rc;
    h->pend = p;
    return LRX_OK;
}

static int host_end_locked(lrx_handle* h, const char* fn, int64_t* host_ids_out, double* host_score,
                           double* host_sem, double* host_kw) {
    if (!h->pend.active) return fail(h, LRX_E_STATE, "%s: no host search in flight", fn);
    lrx_pending p = h->pend;
    h->pend.active = false;
    LRX_CUDA(h, cudaSetDevice(h->device));
    char* hp = (char*)h->ws_host;
    for (;;) {
        const HostLayout L = host_layout(p.B, p.k, p.rows, p.encode, p.S);
        LRX_CUDA(h, cudaStreamSynchronize(h->stream));
        int st = 0;
        const int32_t* sp = (const int32_t*)(hp + L.o_status);
        for (int b = 0; b < p.B; ++b) {
            if (sp[b] < 0) return fail(h, LRX_E_PEER, "%s: a peer shard did not publish its candidates within "
                                                      "%d ms (lrx_set_exchange_timeout)", fn, h->xchg_timeout_ms);
            st |= sp[b];
        }
        if (st & 2) return fail(h, LRX_E_ARG, "%s: a shard saw more query tokens than its capacity", fn);
        if (st == 0) {
            memcpy(host_ids_out, hp + L.o_ids, (size_t)p.B * p.k * sizeof(int64_t));
            memcpy(host_score, hp + L.o_score, (size_t)p.B * p.k * sizeof(double));
            memcpy(host_sem, hp + L.o_sem, (size_t)p.B * p.k * sizeof(double));
            memcpy(host_kw, hp + L.o_kw, (size_t)p.B * p.k * sizeof(double));
            return LRX_OK;
        }
        // the exactness guard of the dense scan tripped on some shard (the status is the OR over all
        // shards, so every rank takes this branch together): widen the candidate lists and rerun on
        // the inputs still staged on the device
        if (p.width >= 512)
            return fail(h, LRX_E_AMBIGUOUS,
                        "dense candidates are not separable at width 512 (more than ~500 rows "
                        "within the fp32 error band of the 2k-th score)");
        p.width *= 2;
        int rc = enqueue_host_chain(h, p);
        if (rc != LRX_OK) return rc;
    }
}

int lrx_search_host_begin(lrx_handle* h, const void* host_q_fp16, const int32_t* host_q_terms,
                          const int32_t* host_q_ptr, const double* host_weights, int32_t B, int32_t k,
                          int32_t mode) {
    if (h == nullptr) return fail(nullptr, LRX_E_ARG, "lrx_search_host_begin: null handle");
    std::lock_guard<std::mutex> g(h->mu);
    if (host_q_fp16 == nullptr || host_q_ptr == nullptr || host_weights == nullptr)
        return fail(h, LRX_E_ARG, "lrx_search_host_begin: null pointer");
    return host_begin_locked(h, "lrx_search_host_begin", host_q_fp16, nullptr, nullptr, 0, host_q_terms,
                             host_q_ptr, host_weights, B, k, mode);
}

int lrx_search_text_host_begin(lrx_handle* h, const int32_t* host_tok_ids, const int32_t* host_tok_lens,
                               int32_t S, const int32_t* host_q_terms, const int32_t* host_q_ptr,
                               const double* host_weights, int32_t B, int32_t k, int32_t mode) {
    if (h == nullptr) return fail(nullptr, LRX_E_ARG, "lrx_search_text_host_begin: null handle");
    std::lock_guard<std::mutex> g(h->mu);
    if (host_tok_ids == nullptr || host_tok_lens == nullptr || host_q_ptr == nullptr || host_weights == nullptr)
        return fail(h, LRX_E_ARG, "lrx_search_text_host_begin: null pointer");
    if (h->encoder == nullptr) return fail(h, LRX_E_STATE, "lrx_search_text_host_begin: encoder weights not set");
    if (S < 1 || S > 512) return fail(h, LRX_E_ARG, "lrx_search_text_host_begin: S must be in [1,512]");
    return host_begin_locked(h, "lrx_search_text_host_begin", nullptr, host_tok_ids, host_tok_lens, S,
                             host_q_terms, host_q_ptr, host_weights, B, k, mode);
}

int lrx_search_host_end(lrx_handle* h, int64_t* host_ids, double* host_score, double* host_sem,
                        double* host_kw) {
    if (h == nullptr) return fail(nullptr, LRX_E_ARG, "lrx_search_host_end: null handle");
    std::lock_guard<std::mutex> g(h->mu);
    if (host_ids == nullptr || host_score == nullptr || host_sem == nullptr || host_kw == nullptr)
        return fail(h, LRX_E_ARG, "lrx_search_host_end: null pointer");
    return host_end_locked(h, "lrx_search_host_end", host_ids, host_score, host_sem, host_kw);
}

int lrx_search_batch_host(lrx_handle* h, const void* host_q_fp16, const int32_t* host_q_terms,
                          const int32_t* host_q_ptr, const double* host_weights, int32_t B,
                          int32_t k, int32_t mode, int64_t* host_ids, double* host_score,
                          double* host_sem, double* host_kw) {
    if (h == nullptr) return fail(nullptr, LRX_E_ARG, "lrx_search_batch_host: null handle");
    std::lock_guard<std::mutex> g(h->mu);
    if (host_q_fp16 == nullptr || host_q_ptr == nullptr || host_weights == nullptr ||
        host_ids == nullptr || host_score == nullptr || host_sem == nullptr || host_kw == nullptr)
        return fail(h, LRX_E_ARG, "lrx_search_batch_host: null pointer");
    int rc = host_begin_locked(h, "lrx_search_batch_host", host_q_fp16, nullptr, nullptr, 0, host_q_terms,
                               host_q_ptr, host_weights, B, k, mode);
    if (rc != LRX_OK) return rc;
    return host_end_locked(h, "lrx_search_batch_host", host_ids, host_score, host_sem, host_kw);
}

int lrx_search_text_host(lrx_handle* h, const int32_t* host_tok_ids, const int32_t* host_tok_lens,
                         int32_t S, const int32_t* host_q_terms, const int32_t* host_q_ptr,
                         const double* host_weights, int32_t B, int32_t k, int32_t mode,
                         int64_t* host_ids, double* host_score, double* host_sem, double* host_kw) {
    if (h == nullptr) return fail(nullptr, LRX_E_ARG, "lrx_search_text_host: null handle");
    std::lock_guard<std::mutex> g(h->mu);
    if (host_tok_ids == nullptr || host_tok_lens == nullptr || host_q_ptr == nullptr ||
        host_weights == nullptr || host_ids == nullptr || host_score == nullptr ||
        host_sem == nullptr || host_kw == nullptr)
        return fail(h, LRX_E_ARG, "lrx_search_text_host: null pointer");
    if (h->encoder == nullptr) return fail(h, LRX_E_STATE, "lrx_search_text_host: encoder weights not set");
    if (S < 1 || S > 512) return fail(h, LRX_E_ARG, "lrx_search_text_host: S must be in [1,512]");
    int rc = host_begin_locked(h, "lrx_search_text_host", nullptr, host_tok_ids, host_tok_lens, S,
                               host_q_terms, host_q_ptr, host_weights, B, k, mode);
    if (rc != LRX_OK) return rc;
    return host_end_locked(h, "lrx_search_text_host", host_ids, host_score, host_sem, host_kw);
}

}  // extern "C"
