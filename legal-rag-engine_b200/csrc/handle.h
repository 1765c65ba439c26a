// Internal: the handle behind include/lrx.h and the host-side launchers each
// .cu file exports to api.cu.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <mutex>
#include <string>
#include <vector>

#include "../../include/lrx.h"

// One candidate of one sub-query on one shard: the unit of the packed block the shards exchange
// (SURVEY.md section 8e).  24 bytes.
struct lrx_record {
    int64_t id;            // global chunk id, -1 = empty slot
    double dense;          // exact inner product (see oracle/flat_ip.py)
    double bm25;           // exact BM25Okapi score of that chunk
};

// One captured launch chain (CUDA graph) of a search entry point, keyed on everything the
// launches depend on (shapes, mode, pointers); replayed with one cudaGraphLaunch.
struct lrx_plan {
    std::vector<uint64_t> key;
    cudaGraphExec_t exec = nullptr;
    uint64_t epoch = 0;                    // handle->ws_epoch at capture: a moved workspace retires it
    int64_t kernels = 0;                   // kernel launches inside (lrx_launch_count)
    uint64_t stamp = 0;                    // last use (LRU eviction)
    bool replayed = false;                 // since the last lrx_profile_read
    std::vector<cudaEvent_t> prof_ev[2];   // external event nodes around the two streaming kernels
};

// A host-buffer search between lrx_search_host_begin and lrx_search_host_end.
struct lrx_pending {
    bool active = false;
    bool encode = false;
    int B = 0, k = 0, mode = 0, width = 0, rows = 0, S = 0;
};

struct lrx_handle {
    int device = 0;
    int num_sms = 0;
    int rank = 0, world = 1;
    cudaStream_t stream = 0;
    // side stream + fork/join events: the BM25 bounds kernel (query-only) runs in the
    // shadow of the dense scan
    cudaStream_t aux = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    std::mutex mu;
    std::string err;
    int64_t launches = 0;

    // optional per-kernel timing (bench.py's roofline figure): CUDA event pairs
    // recorded on the launch stream around the two streaming kernels
    bool prof = false;
    std::vector<cudaEvent_t> prof_ev[2];   // [0] dense_scan_kernel, [1] bm25_scan_kernel

    // corpus (caller-owned)
    const void* x = nullptr;      // fp16 [n_local, 384]
    int64_t n_local = 0, id_base = 0;

    // int8 shadow of the corpus for the K2a pre-filter (caller-owned, lrx_build_dense_prefilter):
    // [n_pad, 384] int8 rows, then [n_pad] fp32 row scales, n_pad = n_local rounded up to 128
    const void* q8 = nullptr;
    double q8_err = 0.0, q8_norm = 0.0;   // max_r |x_r - xhat_r|, max_r |xhat_r| (rounded up)

    // postings (caller-owned)
    const uint64_t* term_ptr = nullptr;
    const void* postings = nullptr;
    const double* idf = nullptr;
    int64_t n_terms = 0, nnz = 0;
    // BM25 constants; bm_lut_ld = longest document + 1 (selects the scan variant whose shared
    // c[len] table needs no fallback)
    int bm_lut_ld = 0;
    int bm_list_k = 0;            // depth of the BM25 top list of the current call (sets the scan's geometry)
    int bm_ctas_per_sm = 0;       // 1: the scan runs beside the dense scan (search chain), one CTA per SM; else 2
    int bm_rows = 0;              // token capacity of a query batch (rows of the bounds table); 0 = B * 64
    double* bm_ctab = nullptr;    // device float64 [2048]: c[len] = k1*(1 - b + b*len/avgdl), built at lrx_set_postings
    double bm_avgdl = 0.0, bm_k1 = 1.5, bm_b = 0.75;

    // workspaces (handle-owned, grown on demand)
    void* ws_dense_part = nullptr;   size_t ws_dense_part_bytes = 0;    // per-CTA key lists
    void* ws_bm_part = nullptr;      size_t ws_bm_part_bytes = 0;       // per-chunk key lists
    void* ws_bm_max = nullptr;       size_t ws_bm_max_bytes = 0;        // per-CTA max
    void* ws_misc = nullptr;         size_t ws_misc_bytes = 0;          // search chain scratch
    void* ws_host = nullptr;         size_t ws_host_bytes = 0;          // pinned staging
    void* ws_io = nullptr;           size_t ws_io_bytes = 0;            // device staging
    void* ws_rm = nullptr;           size_t ws_rm_bytes = 0;            // index removal / replacement: doc map or bits, tile table

    // peer exchange (lrx_exchange_*): this rank's region, the peers' (IPC-mapped), a device copy of
    // the pointer table, the per-call sequence number
    void* xchg = nullptr;            size_t xchg_slot = 0, xchg_bytes = 0;
    void* xchg_peer[LRX_MAX_WORLD] = {nullptr};
    void** xchg_peer_dev = nullptr;
    bool xchg_ready = false;
    int xchg_timeout_ms = 2000;          // bounded spin of the fusion kernel on a peer's flag
    unsigned int* pack_done = nullptr;   // device counter of pack_exchange_kernel (last CTA done)

    // captured launch chains (api.cu: run_planned)
    bool capturing = false;
    lrx_plan* cap_plan = nullptr;
    cudaStream_t cap = nullptr;          // capture origin (the user's stream may be the legacy default one)
    uint64_t ws_epoch = 1, plan_clock = 0;
    std::vector<lrx_plan*> plans;
    std::vector<std::vector<uint64_t>> seen_keys, eager_keys;
    int bm_rows_cfg = 0;                 // lrx_set_query_capacity (device-pointer entry points)
    lrx_pending pend;

    // K1 encoder state (packed weights, activation workspaces, tensor maps): encoder.cu
    void* encoder = nullptr;
};

namespace lrx {

// Fast-pass score error bound used by the exactness guard (DESIGN.md): the scan scores with
// fp16 x fp16 products (exact) accumulated in fp32 by the tensor cores -- 24 accumulation steps
// per quarter row plus 4 fp32 adds, each off by at most one unit in the last place of a partial
// sum <= 1 for L2-normalised rows: <= 28 * 2^-23 = 3.4e-6; tripled for margin.
constexpr double kDenseEps = 1.0e-5;

constexpr int kDim = LRX_DIM;
constexpr int kRowBytes = LRX_DIM * 2;

// dense.cu
int dense_scan_grid(const lrx_handle* h);
int dense_default_width(int K);
cudaError_t launch_dense_topk(lrx_handle* h, const void* q, int B, int K, int width,
                              double* exact, float* D, int64_t* I, int32_t* flags);
bool dense_q8_applies(const lrx_handle* h, int B, int K, int width);
int64_t dense_q8_bytes(int64_t n_local);
cudaError_t launch_dense_q8_build(lrx_handle* h, void* buf, double* bounds_out);
cudaError_t launch_dense_at(lrx_handle* h, const void* q, int B, const int64_t* ids, int n,
                            double* out);

// dense_batched.cu
cudaError_t launch_dense_topk_batched(lrx_handle* h, const void* q, int B, int K, int stride,
                                      double* exact, float* D, int64_t* I, int32_t* flags);

// bm25.cu
cudaError_t launch_bm25(lrx_handle* h, const int32_t* q_terms, const int32_t* q_ptr, int B,
                        const int64_t* cand_ids, int n_cand, double* cand_scores, double* out_max,
                        int K, double* top_scores, int64_t* top_ids);

cudaError_t launch_bm25_bounds(lrx_handle* h, const int32_t* q_terms, const int32_t* q_ptr, int B,
                               cudaStream_t st);
cudaError_t launch_bm25_scan(lrx_handle* h, const int32_t* q_terms, const int32_t* q_ptr, int B,
                             double* out_max, int K, double* top_scores, int64_t* top_ids,
                             cudaStream_t st);
struct BmAtParams;
cudaError_t bm25_at_params(lrx_handle* h, const int32_t* q_terms, const int32_t* q_ptr, int B,
                           BmAtParams* P);
cudaError_t launch_bm25_at(lrx_handle* h, const int32_t* q_terms, const int32_t* q_ptr, int B,
                           const int64_t* ids, int n, double* out, cudaStream_t st);
cudaError_t launch_bm25_pack(lrx_handle* h, const uint32_t* doc_tf, int64_t nnz, const uint32_t* doc_len,
                             void* out, int* host_overflow);
// host_bad: 1 = a tf / length over 16 bits or an appended doc id out of range, 2 = a CSR end does
// not match nnz / nnz_add (nothing launched)
cudaError_t launch_bm25_append(lrx_handle* h, const uint64_t* old_ptr, const void* old_post, int64_t n_terms,
                               int64_t nnz, int64_t n_docs_old, const uint64_t* add_ptr, const uint32_t* add,
                               int64_t n_terms_out, int64_t nnz_add, const uint32_t* doc_len,
                               int64_t n_docs_out, uint64_t* ptr_out, void* post_out, int* host_bad);
// host_bad: 1 = the removal plan does not describe the postings (see lrx_bm25_remove_postings),
// 2 = a CSR end does not match the counts (nothing launched)
cudaError_t launch_bm25_remove(lrx_handle* h, const uint64_t* term_ptr, const void* post, int64_t n_terms,
                               int64_t nnz, int64_t n_docs_old, const uint32_t* removed, int64_t n_removed,
                               const uint64_t* rem_ptr, const uint32_t* rem_doc, const int32_t* term_map,
                               const uint64_t* ptr_out, int64_t n_terms_out, void* post_out, int* host_bad);
// host_bad: 1 = the replacement plan does not describe the postings (see lrx_bm25_replace_postings),
// 2 = a CSR end does not match the counts (nothing launched)
cudaError_t launch_bm25_replace(lrx_handle* h, const uint64_t* term_ptr, const void* post, int64_t n_terms,
                                int64_t nnz, int64_t n_docs, const uint32_t* replaced, int64_t n_rep,
                                const uint64_t* rem_ptr, const uint32_t* rem_doc, const int32_t* term_map,
                                const uint64_t* ins_ptr, const uint32_t* ins_doc_tf, int64_t nnz_ins,
                                const uint32_t* doc_len, const uint64_t* ptr_out, int64_t n_terms_out,
                                void* post_out, int* host_bad);
cudaError_t launch_bm25_lut(lrx_handle* h, double avgdl, double k1, double b, int max_len);
cudaError_t launch_bm25_divcheck(lrx_handle* h, double avgdl, double k1, double b, int n_tf, int n_len,
                                 unsigned long long* host_mismatches);

// fuse.cu
cudaError_t launch_pack_exchange(lrx_handle* h, const int32_t* q_terms, const int32_t* q_ptr, int B, int K,
                                 int mode, const double* dense_exact, const int64_t* dense_ids,
                                 const double* bm_scores, const int64_t* bm_ids, const double* maxbm,
                                 const int32_t* flags, const void* q, void* local_block, bool to_peers,
                                 size_t o_max, size_t o_flags);
// blocks: `world` packed blocks `stride` bytes apart -- this rank's exchange region (exchange) or the
// local block (world == 1)
cudaError_t launch_fuse(lrx_handle* h, const void* blocks, size_t stride, size_t o_max, size_t o_flags,
                        bool exchange, int world, int B, int K, int k, int mode, const double* weights,
                        int64_t* ids, double* score, double* sem, double* kw, int32_t* status);

// encoder.cu
cudaError_t encoder_set_weights(lrx_handle* h, const lrx_bert_weights* w);
cudaError_t encoder_forward(lrx_handle* h, const int32_t* ids, const int32_t* lens, int B, int S,
                            float* out_f32, void* out_f16);
cudaError_t encoder_forward_host(lrx_handle* h, const int32_t* host_ids, const int32_t* host_lens,
                                 int B, int S, float* host_out);
void encoder_free(lrx_handle* h);
// attention_kernel alone on qkv [B*S, 1152] -> ctx [B*S, 384], launched per chunk as encoder_forward
// launches it (lrx_debug_attention); synchronises the handle's stream
cudaError_t encoder_debug_attention(lrx_handle* h, const void* qkv, const int32_t* lens, int B, int S, void* ctx);
// tc_gemm.cu
cudaError_t gemm_f16_adhoc(lrx_handle* h, const void* a, const void* w, int M, int N, int K, int epi,
                           const float* bias, const void* residual, const float* gamma,
                           const float* beta, float eps, void* out);

// Launch with the programmatic-stream-serialization attribute: the kernel's CTAs may be scheduled
// while the previous kernel of the stream still runs; it must call pdl_wait() before it reads
// anything that kernel wrote (common.cuh).
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl_if(bool pdl, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem,
                                 cudaStream_t st, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem,
                              cudaStream_t st, Args... args) {
    return launch_pdl_if(true, kernel, grid, block, smem, st, args...);
}

// One process-wide lock for the per-device "function attribute already set" tables of the
// launchers: handles are locked one by one, but two handles on one device (clone_view) share them.
std::recursive_mutex& attr_mutex();

// profiling hooks (no-ops unless lrx_profile_enable(h, 1))
void prof_begin(lrx_handle* h, int which, cudaStream_t st = nullptr);   // nullptr: h->stream
void prof_end(lrx_handle* h, int which, cudaStream_t st = nullptr);

// shared helper: grow a device workspace
cudaError_t ensure_ws(lrx_handle* h, void** p, size_t* have, size_t need);

}  // namespace lrx
