/*
 * lrx.h -- C ABI of the B200-native hybrid-retrieval hot path.
 *
 * Drop-in boundary for MET4L-DS/Legal-RAG-engine's `RetrievalEngine`
 * (reference: src/retrieval/retrieval_engine.py:23-96, create_vector_store.py:14-83,
 * src/retrieval/orchestrator.py:38-62).  The reference has no FFI of its own: every
 * FLOP of this path runs inside three PyPI wheels.  Each entry point below names the
 * reference call site it replaces; INTEGRATION.md shows the ctypes stub a maintainer
 * would add to the reference.
 *
 * Conventions
 *  - plain C types only; every function returns 0 on success or a negative LRX_E* code;
 *    lrx_last_error() returns the message of the last failure (handle-owned storage,
 *    or a process-wide slot when the handle is NULL).
 *  - one handle per GPU rank.  The handle owns its workspaces and the CUDA stream
 *    binding; it never frees caller memory.  Every entry point calls cudaSetDevice,
 *    so a handle may be created on one host thread and used (sequentially) from
 *    another (reference: src/server/app.py:65-70 vs :110-120).
 *  - pointers named dev_* are device pointers on the handle's GPU; host_* are host
 *    pointers (pinned or pageable).  Nothing here falls back to the CPU: a missing
 *    GPU or a non-sm_100 device is LRX_E_DEVICE at lrx_open.
 *  - ids are GLOBAL chunk ids (int64) = id_base + local row; -1 pads short lists.
 *  - all kernels run on the stream set with lrx_set_stream (default: the legacy
 *    default stream), so PyTorch code can order them with its own work.
 */
#ifndef LRX_H
#define LRX_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LRX_DIM 384                 /* all-MiniLM-L6-v2 embedding width */
#define LRX_MAX_BATCH 64            /* sub-queries per lrx_search_* call */
#define LRX_MAX_DEPTH 256           /* max candidate depth K (= 2k) per list */
#define LRX_MAX_QUERY_TERMS 64      /* default token capacity per sub-query of the device-pointer entry
                                     * points (raise it with lrx_set_query_capacity); the host-buffer
                                     * entry points size the capacity from the batch: no limit */
#define LRX_MAX_WORLD 16            /* shards (GPUs of one box) in a peer exchange */
#define LRX_IPC_HANDLE_BYTES 64     /* sizeof(cudaIpcMemHandle_t) */

enum {
    LRX_OK = 0,
    LRX_E_ARG = -1,        /* bad argument */
    LRX_E_DEVICE = -2,     /* no CUDA device / not sm_100 */
    LRX_E_CUDA = -3,       /* CUDA runtime error (message has the detail) */
    LRX_E_STATE = -4,      /* corpus / postings / weights not set */
    LRX_E_AMBIGUOUS = -5,  /* exactness guard could not be met (see DESIGN.md) */
    LRX_E_NOMEM = -6,
    LRX_E_PEER = -7        /* a peer shard did not publish its block in time */
};

enum { LRX_FUSE_LINEAR = 0, LRX_FUSE_RRF = 1 };

typedef struct lrx_handle lrx_handle;

typedef struct lrx_config {
    int32_t device;        /* CUDA ordinal */
    int32_t dim;           /* must be LRX_DIM */
    int32_t rank;          /* shard index of this handle (0 when unsharded) */
    int32_t world;         /* number of shards (1 when unsharded) */
} lrx_config;

/* ---- lifetime ---------------------------------------------------------- */
int lrx_open(const lrx_config* cfg, lrx_handle** out);
int lrx_close(lrx_handle* h);
const char* lrx_last_error(const lrx_handle* h);
int lrx_set_stream(lrx_handle* h, void* cuda_stream);
/* ABI / build identification: "lrx <version> sm_100a". */
const char* lrx_version(void);

/* ---- index residency (replaces faiss.read_index + pickle.load(bm25.pkl),
 *      retrieval_engine.py:36-47; the data stay owned by the caller) ------- */
/* Row-major fp16 [n_local, 384] chunk matrix (768 B/row, 16-byte aligned). */
int lrx_set_corpus(lrx_handle* h, const void* dev_x_fp16, int64_t n_local, int64_t id_base,
                   int32_t dim);
/* Optional int8 pre-filter of K2 (up to 4 queries, K <= 64): the scan streams an int8 SHADOW of
 * the matrix -- per-row scaled int8 rows, 388 B/row instead of 768 -- and the exact float64
 * re-score of the merged candidate list reads the fp16 rows; the exactness guard uses the
 * rigorous error bound of the shadow, so results stay bit-identical to the plain scan (a query
 * whose candidates the bound cannot separate falls back to the fp16 scan through the widening
 * retry).  The shadow lives in caller-owned device memory of lrx_dense_prefilter_bytes(n_local)
 * bytes, 16-byte aligned.  lrx_build_dense_prefilter quantises the matrix set by lrx_set_corpus
 * into it (synchronous), returns host_bounds_out[2] = {max row error norm, max row norm} and
 * enables the pre-filter; lrx_set_dense_prefilter attaches a shadow built through another handle
 * over the same matrix (dev_buf NULL: back to the plain fp16 scan).  lrx_set_corpus detaches it.
 * (No counterpart in the reference: faiss.IndexFlatIP scans fp32 rows, retrieval_engine.py:64.) */
int64_t lrx_dense_prefilter_bytes(int64_t n_local);
int lrx_build_dense_prefilter(lrx_handle* h, void* dev_buf, int64_t bytes, double* host_bounds_out);
int lrx_set_dense_prefilter(lrx_handle* h, const void* dev_buf, int64_t bytes,
                            const double* host_bounds);
/* Term-major CSR postings restricted to this shard's documents, doc ids LOCAL and
 * ascending within a term.  dev_postings: nnz 8-byte entries {u32 doc_local, u16 tf,
 * u16 doc_len} (lrx_bm25_build_postings fills them from (doc, tf) pairs and the document
 * lengths), 16-byte aligned and readable up to nnz rounded up to an even count (the scan
 * moves 16-byte units).  The query-independent BM25Okapi factor
 *   impact(tf, len) = tf*(k1+1) / (tf + k1*(1 - b + b*len/avgdl))          (float64)
 * is recomputed by the scan from (tf, len) and the GLOBAL avgdl given here, with rank_bm25's
 * float64 operation order.  dev_idf: GLOBAL idf per term (rank_bm25 semantics: epsilon
 * floor applied).  max_doc_len <= 65535.  Replaces pickle.load(bm25.pkl). */
int lrx_set_postings(lrx_handle* h, const uint64_t* dev_term_ptr, const void* dev_postings,
                     const double* dev_idf, int64_t n_terms, int64_t nnz, double avgdl, double k1,
                     double b, int32_t max_doc_len);
/* Index build (create_vector_store.py:60-61, the BM25Okapi constructor's per-document
 * frequency tables): dev_doc_tf = nnz pairs {u32 doc_local, u32 tf} in CSR order ->
 * dev_postings_out (nnz x 8 bytes).  LRX_E_ARG if a tf or a length exceeds 65535. */
int lrx_bm25_build_postings(lrx_handle* h, const uint32_t* dev_doc_tf, int64_t nnz,
                            const uint32_t* dev_doc_len, void* dev_postings_out);
/* Index append (the reference has none: it rebuilds, create_vector_store.py:14-83).  Current index:
 * dev_term_ptr [n_terms+1] + dev_postings (nnz 8-byte entries, as lrx_set_postings takes them) over
 * local documents [0, n_docs_old).  Appended documents: dev_add_ptr [n_terms_out+1] +
 * dev_add_doc_tf {u32 doc_local, u32 tf}[nnz_add], their own term-major CSR (n_terms_out >= n_terms,
 * ids >= n_terms are new terms), doc_local in [n_docs_old, n_docs_out).  dev_doc_len [n_docs_out].
 * Writes dev_term_ptr_out [n_terms_out+1] and dev_postings_out (nnz + nnz_add entries, rounded up to
 * an even count, 16-byte aligned, pad zeroed): term t's current postings, then its appended ones --
 * byte for byte what lrx_bm25_build_postings makes of the whole corpus's CSR.  The outputs must not
 * overlap the inputs.  The handle's index is not touched: pass the outputs to lrx_set_postings with
 * the new idf / avgdl.  Synchronous.  LRX_E_ARG when a tf or a document length exceeds 65535, an
 * appended doc id is out of range, or term_ptr[n_terms] != nnz / add_ptr[n_terms_out] != nnz_add. */
int lrx_bm25_append_postings(lrx_handle* h, const uint64_t* dev_term_ptr, const void* dev_postings,
                             int64_t n_terms, int64_t nnz, int64_t n_docs_old,
                             const uint64_t* dev_add_ptr, const uint32_t* dev_add_doc_tf,
                             int64_t n_terms_out, int64_t nnz_add, const uint32_t* dev_doc_len,
                             int64_t n_docs_out, uint64_t* dev_term_ptr_out, void* dev_postings_out);
/* Index removal (the reference has none: it rebuilds the store).  Current index: dev_term_ptr
 * [n_terms+1] + dev_postings (nnz 8-byte entries) over local documents [0, n_docs_old).  Removed:
 * dev_removed_docs [n_removed], strictly ascending; per old term t its removed documents
 * dev_rem_doc[dev_rem_ptr[t] .. dev_rem_ptr[t+1]), ascending (nnz_rem = rem_ptr[n_terms]);
 * dev_term_map [n_terms]: t's new id, -1 for a term left without postings; dev_term_ptr_out
 * [n_terms_out+1]: the new CSR's pointers (from the surviving document frequencies).  Writes
 * dev_postings_out (nnz - nnz_rem entries, rounded up to an even count, 16-byte aligned, pad
 * zeroed): every surviving posting under its term's new id, its document renumbered to
 * d - |{r in removed : r < d}|, tf and length copied -- byte for byte what lrx_bm25_build_postings
 * makes of the rebuilt CSR.  The outputs must not overlap the inputs.  The handle's index is not
 * touched: pass the outputs to lrx_set_postings with the new idf / avgdl.  Synchronous.  LRX_E_ARG,
 * with nothing else changed, when the CSR ends do not match the counts, a removed list is not
 * strictly ascending or holds a document that is not a removed posting of its term, a posting of a
 * removed document is missing from its term's list, term_map is not a bijection from the terms
 * with survivors onto [0, n_terms_out), or a term's survivors do not fill its output range. */
int lrx_bm25_remove_postings(lrx_handle* h, const uint64_t* dev_term_ptr, const void* dev_postings,
                             int64_t n_terms, int64_t nnz, int64_t n_docs_old,
                             const uint32_t* dev_removed_docs, int64_t n_removed,
                             const uint64_t* dev_rem_ptr, const uint32_t* dev_rem_doc,
                             const int32_t* dev_term_map, const uint64_t* dev_term_ptr_out,
                             int64_t n_terms_out, void* dev_postings_out);
/* Index replacement (the reference has none: it rebuilds the store).  The text of some documents
 * changes; document ids do not.  Current index: dev_term_ptr [n_terms+1] + dev_postings (nnz 8-byte
 * entries) over local documents [0, n_docs).  Replaced: dev_replaced_docs [n_replaced], strictly
 * ascending; per old term t its postings of replaced documents dev_rem_doc[dev_rem_ptr[t] ..
 * dev_rem_ptr[t+1]), ascending (dropped; nnz_rem = rem_ptr[n_terms]); dev_term_map [n_terms]: t's new
 * id, -1 for a word left without postings; per new term u its inserted entries dev_ins_doc_tf
 * {u32 doc, u32 tf}[dev_ins_ptr[u] .. dev_ins_ptr[u+1]), doc ascending, every doc a replaced one
 * (nnz_ins = ins_ptr[n_terms_out]); dev_doc_len [n_docs]: the lengths after the edit;
 * dev_term_ptr_out [n_terms_out+1]: the new CSR's pointers.  Writes dev_postings_out (nnz - nnz_rem +
 * nnz_ins entries, rounded up to an even count, 16-byte aligned, pad zeroed): under each new id, the
 * kept postings of its old term (copied verbatim) merged by document with its inserted entries --
 * byte for byte what lrx_bm25_build_postings makes of the rebuilt CSR.  The outputs must not overlap
 * the inputs.  The handle's index is not touched: pass the outputs to lrx_set_postings with the new
 * idf / avgdl.  Synchronous.  LRX_E_ARG, with nothing else changed, when the CSR ends do not match the
 * counts, a dropped list is not strictly ascending or holds a document that is not a replaced posting
 * of its term, a posting of a replaced document is missing from its term's list, an inserted list is
 * not strictly ascending or holds a document that is not replaced, a tf is outside [1, 65535] or a
 * length over 65535, term_map is not injective into [0, n_terms_out), or a new id's range is not its
 * kept plus inserted count (or is empty). */
int lrx_bm25_replace_postings(lrx_handle* h, const uint64_t* dev_term_ptr, const void* dev_postings,
                              int64_t n_terms, int64_t nnz, int64_t n_docs,
                              const uint32_t* dev_replaced_docs, int64_t n_replaced,
                              const uint64_t* dev_rem_ptr, const uint32_t* dev_rem_doc,
                              const int32_t* dev_term_map, const uint64_t* dev_ins_ptr,
                              const uint32_t* dev_ins_doc_tf, int64_t nnz_ins, const uint32_t* dev_doc_len,
                              const uint64_t* dev_term_ptr_out, int64_t n_terms_out, void* dev_postings_out);

/* ---- K1: encoder (replaces SentenceTransformer("all-MiniLM-L6-v2").encode followed by
 *      faiss.normalize_L2; retrieval_engine.py:28,61-62, create_vector_store.py:33-34,45,51) --
 * Weights: DEVICE pointers to float32 tensors in the HuggingFace BertModel state_dict layout
 * (nn.Linear weight = [out, in]); the library packs its own fp16 copies, so the caller may
 * free them when lrx_set_encoder_weights returns.  Fixed architecture: hidden 384, 12 heads,
 * FFN 1536, 6 layers, LayerNorm eps 1e-12, exact-erf GELU, token type 0. */
#define LRX_BERT_LAYERS 6
typedef struct lrx_bert_layer {
    const float *wq, *bq, *wk, *bk, *wv, *bv;   /* attention.self.{query,key,value}  [384,384],[384] */
    const float *wo, *bo;                       /* attention.output.dense           [384,384],[384] */
    const float *ln1_g, *ln1_b;                 /* attention.output.LayerNorm       [384]           */
    const float *w1, *b1;                       /* intermediate.dense               [1536,384],[1536] */
    const float *w2, *b2;                       /* output.dense                     [384,1536],[384] */
    const float *ln2_g, *ln2_b;                 /* output.LayerNorm                 [384]           */
} lrx_bert_layer;
typedef struct lrx_bert_weights {
    int32_t vocab_size;        /* 30522 for all-MiniLM-L6-v2 */
    int32_t max_positions;     /* 512 */
    const float* word_emb;     /* embeddings.word_embeddings        [vocab, 384] */
    const float* pos_emb;      /* embeddings.position_embeddings    [max_positions, 384] */
    const float* type_emb;     /* embeddings.token_type_embeddings  [2, 384] (row 0 used) */
    const float *emb_ln_g, *emb_ln_b;
    lrx_bert_layer layers[LRX_BERT_LAYERS];
} lrx_bert_weights;
int lrx_set_encoder_weights(lrx_handle* h, const lrx_bert_weights* w);
/* dev_ids int32 [B,S] WordPiece ids ([CLS] ... [SEP], 0-padded), dev_lens int32 [B] = number of
 * attended tokens per sequence (the attention mask is a prefix mask, as the tokenizer emits).
 * Outputs (either may be NULL): float32 [B,384] and fp16 [B,384] unit vectors (the fp16 copy is
 * the query operand of lrx_dense_topk / lrx_search_*). */
int lrx_encode(lrx_handle* h, const int32_t* dev_ids, const int32_t* dev_lens, int32_t B, int32_t S,
               float* dev_out_f32, void* dev_out_f16);
/* Host-buffer form: H2D of ids/lens, the forward pass, D2H of the embeddings, synchronised. */
int lrx_encode_host(lrx_handle* h, const int32_t* host_ids, const int32_t* host_lens, int32_t B,
                    int32_t S, float* host_out_f32);
/* The tensor-core GEMM stage on its own: out[M,N] = epi(A[M,K] * W[N,K]^T), fp16 row-major
 * operands, fp32 accumulation.  epi: 0 +bias -> fp16, 1 +bias, GELU(erf) -> fp16,
 * 2 +bias +residual, LayerNorm (N == 384) -> fp16, 3 raw accumulators -> float32.
 * K % 64 == 0, N % 128 == 0. */
int lrx_gemm_f16(lrx_handle* h, const void* dev_a, const void* dev_w, int32_t M, int32_t N, int32_t K,
                 int32_t epi, const float* dev_bias, const void* dev_residual,
                 const float* dev_gamma, const float* dev_beta, float eps, void* dev_out);

/* ---- stage kernels (device pointers) ----------------------------------- */
/* K2: replaces IndexFlatIP.search(x, K)  (retrieval_engine.py:64).
 * dev_q_fp16 [B,384]; outputs [B,K]: exact float64 score, float32 D, int64 I,
 * best first, (score desc, id asc); pads (-inf, -FLT_MAX, -1).
 * dev_flags [B]: 0 = exact, 1 = exactness guard failed (caller should retry with
 * lrx_dense_topk_ex and a larger width). */
int lrx_dense_topk(lrx_handle* h, const void* dev_q_fp16, int32_t B, int32_t K,
                   double* dev_exact, float* dev_D, int64_t* dev_I, int32_t* dev_flags);
int lrx_dense_topk_ex(lrx_handle* h, const void* dev_q_fp16, int32_t B, int32_t K,
                      int32_t width, double* dev_exact, float* dev_D, int64_t* dev_I,
                      int32_t* dev_flags);
/* K2b: the same search for LARGE batches (B up to 4096; FAISS's BLAS regime, nq >= 20) on the
 * tensor cores: two tcgen05 GEMM passes (tile maxima -> per-query threshold; candidates above
 * it) + exact float64 re-score.  Same outputs and ordering as lrx_dense_topk.  stride: pass 1
 * samples every stride-th 256-row tile (0 = automatic; above 524 288 rows the stride is raised so
 * that at most 16 384 chunks are sampled).  When fewer than 2K sampled 32-row chunks hold rows the
 * batch runs the lrx_dense_topk scan instead.  dev_flags[b] = 1: more than 1024 rows scored within
 * the band of query b's K-th score (many near-identical rows: a stride-1 rerun is flagged too) --
 * answer query b with lrx_dense_topk_ex and a larger width. */
int lrx_dense_topk_batched(lrx_handle* h, const void* dev_q_fp16, int32_t B, int32_t K, int32_t stride,
                           double* dev_exact, float* dev_D, int64_t* dev_I, int32_t* dev_flags);
/* Exact inner products at given global ids (ids outside the shard or -1 -> -inf). */
int lrx_dense_at(lrx_handle* h, const void* dev_q_fp16, int32_t B, const int64_t* dev_ids,
                 int32_t n, double* dev_out);

/* Token capacity of a query batch for the DEVICE-pointer entry points (lrx_bm25, lrx_search_sharded):
 * the library cannot see dev_q_ptr[B] from the host, so the rows of its per-token tables are sized
 * from this figure; 0 (default) = B * LRX_MAX_QUERY_TERMS.  Every token
 * is scored, in order, as the reference does (retrieval_engine.py:67-68 has no limit).  A batch with
 * MORE tokens than the capacity is never scored short silently: lrx_bm25 returns NaN maxima and the
 * search entry points set bit 2 of the status words.  The host-buffer entry points size the
 * capacity from host_q_ptr themselves. */
int lrx_set_query_capacity(lrx_handle* h, int32_t max_total_terms);

/* K3: replaces BM25Okapi.get_scores + max()  (retrieval_engine.py:68,74).
 * dev_q_terms: concatenated term ids (-1 = out of vocabulary), dev_q_ptr [B+1].
 * Emits (i) exact scores at dev_cand_ids [B,n_cand] (may be NULL / n_cand 0; ids outside
 * the shard or -1 give 0), (ii) dev_max [B]: max over the shard's POSITIVE scores, 0 when
 * none, (iii) the shard's top-K positive-score list [B,K] (score desc, id asc; pads
 * (0,-1)); K may be 0. */
int lrx_bm25(lrx_handle* h, const int32_t* dev_q_terms, const int32_t* dev_q_ptr, int32_t B,
             const int64_t* dev_cand_ids, int32_t n_cand, double* dev_cand_scores,
             double* dev_max, int32_t K, double* dev_top_scores, int64_t* dev_top_ids);

/* ---- K5: the whole of RetrievalEngine.search for a batch of sub-queries, on one GPU or on the
 * row shards of one box (world > 1) with the candidate exchange fused into the kernels.
 * Each shard runs K2 + K3 and packs, per sub-query, its candidate records (the dense list and, in
 * rrf mode, the BM25 list), its BM25 maximum and its exactness flag into one block.  At world > 1
 * every rank owns an exchange region (two parities x world slots of one packed block, sequence
 * flags and the call counter); the packing kernel stores the rank's block straight into the slot
 * `rank` of EVERY peer's region over NVLink (peer memory opened through CUDA IPC), its last CTA
 * publishes the call's sequence number with a release store, and the fusion kernel (K4) acquires
 * the world flags before it merges.  The sequence number lives on the device, so the whole chain
 * is one captured CUDA graph replayed per batch: no collective library call, no host
 * synchronisation, one launch.  Calls must be made in the same order by all ranks (SPMD), each on
 * its own stream.  world == 1 needs no exchange: the same call then serves every shard count.
 * Outputs [B,k]: ids (-1 pad), fused score, semantic, keyword (replicated on every rank);
 * dev_status[b]: 0 ok, bit 0 = exactness guard (rerun with a larger width), bit 1 = token capacity
 * exceeded, -1 = a peer's block did not arrive within the exchange timeout.
 *   lrx_exchange_export  allocates this rank's region for batches up to (B_max, k_max) and
 *                        returns its IPC handle (LRX_IPC_HANDLE_BYTES bytes);
 *   lrx_exchange_import  takes all ranks' handles in rank order (exchanged by the host, e.g. one
 *                        torch.distributed all-gather at start-up) and opens the peers' regions;
 *   lrx_search_sharded   K2 + K3 on this shard, exchange, K4: the replicated fused result. */
int lrx_exchange_export(lrx_handle* h, int32_t B_max, int32_t k_max, void* host_handle_out);
int lrx_exchange_import(lrx_handle* h, const void* host_handles_all);
int lrx_search_sharded(lrx_handle* h, const void* dev_q_fp16, const int32_t* dev_q_terms,
                       const int32_t* dev_q_ptr, const double* dev_weights, int32_t B, int32_t k,
                       int32_t mode, int32_t width, int64_t* dev_ids, double* dev_score,
                       double* dev_sem, double* dev_kw, int32_t* dev_status);

/* Bounded spin of the fusion kernel on a peer's sequence flag (default 2000 ms); expiry is reported
 * as status -1 / LRX_E_PEER, never as a hung GPU. */
int lrx_set_exchange_timeout(lrx_handle* h, int32_t milliseconds);

/* Host-buffer form of the whole search: copies the inputs in, runs K2..K4 (exchange included when
 * the handle is a shard, world > 1: every rank makes the same call), copies the results out and
 * synchronises; widens the dense candidate lists and reruns when the exactness guard trips (the
 * status is replicated, so all ranks rerun together).  This is the call `RetrievalEngine.search` /
 * `search_batch` makes (retrieval_engine.py:59).  Any number of tokens per query. */
int lrx_search_batch_host(lrx_handle* h, const void* host_q_fp16, const int32_t* host_q_terms,
                          const int32_t* host_q_ptr, const double* host_weights, int32_t B,
                          int32_t k, int32_t mode, int64_t* host_ids, double* host_score,
                          double* host_sem, double* host_kw);

/* Split form for pipelining: _begin stages the inputs in pinned memory and enqueues H2D + the chain
 * + D2H on the handle's stream and returns at once; _end synchronises, checks the status words
 * (rerunning wider if needed) and copies the results out.  One search in flight per handle; several
 * handles over the same index (same corpus / postings pointers, each with its own stream and
 * exchange region) keep several batches in flight on one GPU. */
int lrx_search_host_begin(lrx_handle* h, const void* host_q_fp16, const int32_t* host_q_terms,
                          const int32_t* host_q_ptr, const double* host_weights, int32_t B, int32_t k,
                          int32_t mode);
int lrx_search_text_host_begin(lrx_handle* h, const int32_t* host_tok_ids, const int32_t* host_tok_lens,
                               int32_t S, const int32_t* host_q_terms, const int32_t* host_q_ptr,
                               const double* host_weights, int32_t B, int32_t k, int32_t mode);
int lrx_search_host_end(lrx_handle* h, int64_t* host_ids, double* host_score, double* host_sem,
                        double* host_kw);

/* The whole of RetrievalEngine.search for a batch of query STRINGS already tokenised on the host
 * (world >= 1; a shard encodes the strings redundantly): H2D of WordPiece ids [B,S] + lens [B] and of the BM25 term ids, K1 (encoder) ->
 * K2 -> K3 -> K4, D2H of the fused results, synchronised.  Replaces retrieval_engine.py:59-96
 * end to end; `search_batch` with B = 4 is the orchestrator fan-out (orchestrator.py:38-62). */
int lrx_search_text_host(lrx_handle* h, const int32_t* host_tok_ids, const int32_t* host_tok_lens,
                         int32_t S, const int32_t* host_q_terms, const int32_t* host_q_ptr,
                         const double* host_weights, int32_t B, int32_t k, int32_t mode,
                         int64_t* host_ids, double* host_score, double* host_sem, double* host_kw);

/* Test hook for K3: the scan divides with the branch-free fast path of the float64 division
 * (same FMA sequence as the compiler's, without the exponent-range test); this counts the
 * (tf, len) pairs in [0,n_tf) x [0,n_len) whose BM25 factor differs from the IEEE division. */
int lrx_debug_bm25_divcheck(lrx_handle* h, double avgdl, double k1, double b, int32_t n_tf,
                            int32_t n_len, uint64_t* host_mismatches);

/* Test hook for K1: the encoder's attention kernel alone, launched as the GEMM chain launches it
 * (per activation chunk, same grid, block and shared memory).  dev_qkv_fp16 [B*S, 1152] = Q | K | V
 * per token, head h at columns 32h .. 32h + 31 of each 384-wide block; dev_lens [B] (clamped to
 * [0, S]); dev_ctx_fp16 [B*S, 384] = softmax(Q K^T / sqrt(32), keys < len) V per head, rows >= len
 * zero.  1 <= B <= 2^20, 1 <= S <= 512.  Synchronises the handle's stream. */
int lrx_debug_attention(lrx_handle* h, const void* dev_qkv_fp16, const int32_t* dev_lens, int32_t B,
                        int32_t S, void* dev_ctx_fp16);

/* Number of kernels launched by this handle since lrx_open (bench.py's gpu_launches). */
int64_t lrx_launch_count(const lrx_handle* h);


/* Per-kernel timing for bench.py's roofline line: when enabled, CUDA events are recorded
 * on the launch stream around every launch of the two streaming kernels
 * (which = 0: dense_scan_kernel, 1: bm25_scan_kernel).  lrx_profile_read synchronises,
 * returns the summed device time and launch count since the last read, and resets. */
int lrx_profile_enable(lrx_handle* h, int32_t on);
int lrx_profile_read(lrx_handle* h, int32_t which, double* total_ms, int64_t* n_launches);

#ifdef __cplusplus
}
#endif
#endif /* LRX_H */
