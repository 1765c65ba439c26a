// K4: cross-shard merge of candidate records + score fusion.
//
// linear : reference src/retrieval/retrieval_engine.py:71-96, operation for
//          operation in float64 (no FMA contraction) -- candidates are the dense
//          top-2k only, semantic = float32-rounded inner product, keyword =
//          bm25/max_bm25, stable descending sort (ties keep flat-IP order).
// rrf    : README.md:39,82-83 (no upstream code): sum of 1/(60+rank) over the dense
//          and BM25 lists, order (rrf desc, id asc).  See oracle/fusion.py.
//
// One CTA per sub-query; every shard runs the same deterministic merge on the
// exchanged records, so the result is replicated bit for bit.  The shards' lists arrive
// sorted, so merging is rank arithmetic (binary searches), not sorting.
#include "common.cuh"
#include "handle.h"
#include "bm25_at.cuh"

namespace lrx {

constexpr int kFuseThreads = 128;
constexpr int kFuseMaxIn = 2048;   // world * K records per list
constexpr int kFuseMaxK = LRX_MAX_DEPTH;

// Where a shard's packed block `[B][2][K] records | [B] max | [B] flags` goes.
//   world == 1    : `local` (handle workspace).
//   peer exchange : slot `rank` of parity `seq & 1` in EVERY shard's exchange region
//     (region = data [2][world][slot] | flags u64 [2][world] | ctr u64 | done u32), stored over
//     NVLink, then a release store of the call's sequence number into the flag word.  The
//     sequence number lives ON THE DEVICE (`ctr` in this rank's own region, advanced by the last
//     CTA of this kernel), so the launch is the same for every call: a CUDA graph can replay it.
struct PackDst {
    unsigned char* local;          // non-peer destination (or NULL)
    void* const* peers;            // [world] exchange regions (device table), NULL = no peer exchange
    int rank, world;
    size_t slot;                   // bytes per slot
    size_t o_max, o_flags;         // byte offsets of [B] max / [B] flags inside a block
};

__device__ __forceinline__ void st_rec(lrx_record* p, const lrx_record& r) {
    p->id = r.id; p->dense = r.dense; p->bm25 = r.bm25;
}

// One WARP per (query, list position) i = (b, j): record 0 = dense candidate j of query b with its
// BM25 score (`kw = bm25[idx] / max_bm25`, retrieval_engine.py:82: looked up here by
// bm25_score_at, the scan's float64 operations in token order); record 1 (rrf) = BM25 hit j with
// its exact dense score (shown as "semantic": one float64 dot product by the warp).  The records go
// straight to their destination(s); the last CTA to finish appends the shard's [B] maxima and
// exactness flags and -- peer exchange -- publishes the sequence number to every shard.
__global__ void pack_exchange_kernel(int B, int K, int mode, const double* __restrict__ dense_exact,
                                     const int64_t* __restrict__ dense_ids,
                                     const double* __restrict__ bm_scores,
                                     const int64_t* __restrict__ bm_ids,
                                     const double* __restrict__ maxbm, const int32_t* __restrict__ flags,
                                     const unsigned char* __restrict__ x, int64_t n_rows,
                                     const __half* __restrict__ q, const BmAtParams A, const PackDst D,
                                     unsigned int* __restrict__ done /* zero between launches */) {
    pdl_trigger();                       // the fusion kernel may be scheduled (it waits for us)
    pdl_wait();                          // the dense merge's candidates are visible
    const int i = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    // this call's sequence number and parity (peer exchange): ctr is advanced by the LAST CTA only
    // after every CTA has read it (its atomicAdd on `done` comes after the read)
    unsigned long long seq = 0;
    unsigned long long* ctr = nullptr;
    if (D.peers != nullptr) {
        unsigned char* own = reinterpret_cast<unsigned char*>(D.peers[D.rank]);
        ctr = reinterpret_cast<unsigned long long*>(own + 2 * (size_t)D.world * D.slot +
                                                    2 * (size_t)D.world * sizeof(unsigned long long));
        seq = *reinterpret_cast<volatile unsigned long long*>(ctr) + 1ull;
    }
    const size_t slot_off = ((size_t)(seq & 1ull) * D.world + D.rank) * D.slot;
    if (i < B * K) {
        const int b = i / K, j = i - b * K;
        lrx_record r0, r1;
        r0.id = dense_ids[i];
        r0.dense = dense_exact[i];
        r0.bm25 = bm25_score_at(A, b, r0.id, lane);          // 0 for -1 pads
        r1.id = -1;
        r1.dense = -INFINITY;
        r1.bm25 = 0.0;
        if (mode == LRX_FUSE_RRF && bm_ids[i] >= 0) {
            r1.id = bm_ids[i];
            r1.bm25 = bm_scores[i];
            const int64_t row = r1.id - A.id_base;
            if (row >= 0 && row < n_rows) {
                const uint2* rowp = reinterpret_cast<const uint2*>(x + row * (int64_t)(LRX_DIM * 2));
                const uint2* qp = reinterpret_cast<const uint2*>(q + (size_t)b * LRX_DIM);
                double acc = 0.0;
#pragma unroll
                for (int s = 0; s < 3; ++s) {
                    const uint2 v = rowp[s * 32 + lane], w = qp[s * 32 + lane];
                    const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&v.x));
                    const float2 c = __half22float2(*reinterpret_cast<const __half2*>(&v.y));
                    const float2 e = __half22float2(*reinterpret_cast<const __half2*>(&w.x));
                    const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w.y));
                    acc = fma((double)a.x, (double)e.x, acc);
                    acc = fma((double)a.y, (double)e.y, acc);
                    acc = fma((double)c.x, (double)f.x, acc);
                    acc = fma((double)c.y, (double)f.y, acc);
                }
#pragma unroll
                for (int lb = 16; lb > 0; lb >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, lb);
                r1.dense = acc;
            }
        }
        const size_t o0 = (((size_t)b * 2 + 0) * K + j) * sizeof(lrx_record);
        const size_t o1 = (((size_t)b * 2 + 1) * K + j) * sizeof(lrx_record);
        if (D.peers == nullptr) {
            if (lane == 0) {
                st_rec(reinterpret_cast<lrx_record*>(D.local + o0), r0);
                st_rec(reinterpret_cast<lrx_record*>(D.local + o1), r1);
            }
        } else {
            for (int w = lane; w < D.world; w += 32) {        // lane w stores to shard w
                unsigned char* dst = reinterpret_cast<unsigned char*>(D.peers[w]) + slot_off;
                st_rec(reinterpret_cast<lrx_record*>(dst + o0), r0);
                st_rec(reinterpret_cast<lrx_record*>(dst + o1), r1);
            }
        }
    }
    // ---- last CTA done: maxima + flags, then (peer exchange) the sequence flags
    __threadfence_system();              // this thread's record stores before the counter
    __syncthreads();
    __shared__ int s_last;
    if (threadIdx.x == 0) s_last = (atomicAdd(done, 1u) == gridDim.x - 1) ? 1 : 0;
    __syncthreads();
    if (!s_last) return;
    __threadfence();                     // the other CTAs' stores (their fences precede their atomics)
    const int n_dst = (D.peers == nullptr) ? 1 : D.world;
    for (int t = threadIdx.x; t < n_dst * B; t += blockDim.x) {
        const int w = t / B, b = t - w * B;
        unsigned char* dst = (D.peers == nullptr)
            ? D.local : reinterpret_cast<unsigned char*>(D.peers[w]) + slot_off;
        reinterpret_cast<double*>(dst + D.o_max)[b] = maxbm[b];
        reinterpret_cast<int32_t*>(dst + D.o_flags)[b] = flags[b];
    }
    __threadfence_system();
    __syncthreads();
    if (D.peers != nullptr && threadIdx.x < D.world) {
        unsigned char* base = reinterpret_cast<unsigned char*>(D.peers[threadIdx.x]);
        unsigned long long* flag = reinterpret_cast<unsigned long long*>(base + 2 * (size_t)D.world * D.slot) +
                                   (size_t)(seq & 1ull) * D.world + D.rank;
        asm volatile("st.release.sys.global.u64 [%0], %1;" :: "l"(flag), "l"(seq) : "memory");
    }
    if (threadIdx.x == 0) {
        if (ctr != nullptr) *ctr = seq;
        *done = 0u;                      // ready for the next launch (stream order)
    }
}

// key = order image (64) | ~id (32) | source slot (32): sorts by (value desc, id asc)
__device__ __forceinline__ u128 rec_key(double v, int64_t id, uint32_t src) {
    return ((u128)f64_ord(v) << 64) | ((u128)(uint32_t)(~(uint32_t)id) << 32) | (u128)src;
}

// Number of keys greater than `key` in a DESCENDING run of n keys (empty keys = 0 at its end).
__device__ __forceinline__ int count_greater_sorted(const u128* run, int n, u128 key) {
    int lo = 0, hi = n;                  // first position whose key is <= `key`
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (run[mid] > key) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// No sorting networks here: every list that arrives is already sorted per shard (K2's re-score and
// K3's merge emit (score desc, id asc)), so the rank of a record in the merged order is a sum of
// binary searches, and the final order of the <= 2K fused scores is a rank by counting.  Keys are
// unique (they end in the source slot), so ranks are a permutation.
//
// Input: `world` packed blocks `stride` bytes apart -- with `exchange`, one parity of this rank's
// exchange region (data [2][world][stride] | flags u64 [2][world] | ctr u64), else the local block.
__global__ void __launch_bounds__(kFuseThreads)
fuse_kernel(const unsigned char* __restrict__ blocks, size_t stride, size_t o_max, size_t o_flags,
            bool exchange, int world, int B, int K, int k, int mode,
            const double* __restrict__ weights, int64_t* __restrict__ out_ids,
            double* __restrict__ out_score, double* __restrict__ out_sem,
            double* __restrict__ out_kw, int32_t* __restrict__ out_status,
            long long timeout_ns, int self) {
    pdl_wait();                                  // the packing / exchange kernel has finished
    extern __shared__ __align__(16) unsigned char fuse_dyn[];
    u128* keys = reinterpret_cast<u128*>(fuse_dyn);   // [kFuseMaxIn]
    __shared__ lrx_record dsel[kFuseMaxK];      // global dense top-K
    __shared__ lrx_record ssel[kFuseMaxK];      // global BM25 top-K (rrf)
    __shared__ double fscore[2 * kFuseMaxK];
    __shared__ int out_slot[2 * kFuseMaxK];     // fused rank -> union slot
    __shared__ int n_dense, n_sparse, n_fused;
    const int b = blockIdx.x;
    const int tid = threadIdx.x;
    const int n_in = world * K;
    if (tid == 0) { n_dense = 0; n_sparse = 0; n_fused = 0; }
    // peer exchange: the blocks of the other shards were stored into this GPU's memory by THEIR
    // kernels.  The call's sequence number is the counter this rank's packing kernel has just
    // advanced; its parity selects the half of the region.  Acquire every shard's sequence flag
    // before touching its block (bounded spin: a lost peer surfaces as status -1, not as a hung GPU).
    __shared__ int wait_failed;
    if (tid == 0) wait_failed = 0;
    __syncthreads();
    if (exchange) {
        const size_t data_bytes = 2 * (size_t)world * stride;
        const unsigned long long* fl = reinterpret_cast<const unsigned long long*>(blocks + data_bytes);
        const unsigned long long seq = __ldcg(fl + 2 * world);           // ctr
        blocks += (size_t)(seq & 1ull) * world * stride;
        if (tid < world && tid != self) {
            const unsigned long long* wf = fl + (size_t)(seq & 1ull) * world + tid;
            long long t0;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
            unsigned long long v;
            for (;;) {
                asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(wf) : "memory");
                if (v >= seq) break;
                long long t1;
                asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
                if (t1 - t0 > timeout_ns) { wait_failed = 1; break; }
                __nanosleep(100);
            }
        }
    }
    __syncthreads();

    // max_bm25 = max(scores) if max(scores) > 0 else 1.0   (retrieval_engine.py:74)
    double maxbm = 0.0;
    int status = 0;
#pragma unroll 1                                 // unrolled, its loads in flight set the kernel's register count
    for (int w = 0; w < world; ++w) {
        const unsigned char* bw = blocks + w * stride;
        const double mv = __ldcg(reinterpret_cast<const double*>(bw + o_max) + b);
        if (mv != mv) status |= 2;               // NaN: a shard saw more query tokens than its capacity
        maxbm = fmax(maxbm, mv);
        status |= __ldcg(reinterpret_cast<const int32_t*>(bw + o_flags) + b);
    }
    if (!(maxbm > 0.0)) maxbm = 1.0;

    // by value, through L2 (ld.cg): the records may have been written by another GPU
    auto rec_at = [&](int list, int src) -> lrx_record {
        const int w = src / K, j = src - w * K;
        const lrx_record* r =
            reinterpret_cast<const lrx_record*>(blocks + w * stride) + ((size_t)b * 2 + list) * K + j;
        lrx_record out;
        out.id = __ldcg(&r->id);
        out.dense = __ldcg(&r->dense);
        out.bm25 = __ldcg(&r->bm25);
        return out;
    };
    // merged top-K of the shards' sorted lists `list` (0 dense, 1 BM25) into sel[]; count in *n_sel
    auto merge_lists = [&](int list, lrx_record* sel, int* n_sel) {
        __syncthreads();                                      // keys[] free
        for (int i = tid; i < n_in; i += kFuseThreads) {
            const lrx_record r = rec_at(list, i);
            keys[i] = (r.id >= 0) ? rec_key(list ? r.bm25 : r.dense, r.id, (uint32_t)i) : (u128)0;
        }
        __syncthreads();
        for (int i = tid; i < n_in; i += kFuseThreads) {
            const u128 key = keys[i];
            if (key == 0) continue;
            const int w_own = i / K;
            int rank = i - w_own * K;                         // position in its own sorted run
            for (int w = 0; w < world && rank < K; ++w)
                if (w != w_own) rank += count_greater_sorted(keys + w * K, K, key);
            if (rank < K) {
                sel[rank] = rec_at(list, i);
                atomicAdd(n_sel, 1);
            }
        }
        __syncthreads();
    };
    // rank by counting of the n keys in keys[]: out_slot[rank] = low 32 bits of the key
    auto order_keys = [&](int n) {
        __syncthreads();
        for (int i = tid; i < n; i += kFuseThreads) {
            const u128 key = keys[i];
            if (key == 0) continue;
            int rank = 0;
            for (int j = 0; j < n; ++j) rank += (keys[j] > key) ? 1 : 0;
            out_slot[rank] = (int)(uint32_t)key;
            atomicAdd(&n_fused, 1);
        }
        __syncthreads();
    };

    merge_lists(0, dsel, &n_dense);
    const int nd = n_dense;

    if (mode == LRX_FUSE_LINEAR) {
        const double w = weights[b];
        const double one_m_w = __dsub_rn(1.0, w);
        for (int j = tid; j < nd; j += kFuseThreads) {
            const double sem = (double)__double2float_rn(dsel[j].dense);   // float(dist)
            const double kw = __ddiv_rn(dsel[j].bm25, maxbm);
            const double s = __dadd_rn(__dmul_rn(sem, one_m_w), __dmul_rn(kw, w));
            fscore[j] = s;
            // stable descending sort: ties keep flat-IP order j
            keys[j] = ((u128)f64_ord(s) << 64) | ((u128)(uint32_t)(~(uint32_t)j) << 32) | (u128)(uint32_t)j;
        }
        order_keys(nd);
        const int n_out = min(k, n_fused);
        for (int i = tid; i < k; i += kFuseThreads) {
            const size_t o = (size_t)b * k + i;
            if (i < n_out) {
                const int j = out_slot[i];
                out_ids[o] = dsel[j].id;
                out_score[o] = fscore[j];
                out_sem[o] = (double)__double2float_rn(dsel[j].dense);
                out_kw[o] = __ddiv_rn(dsel[j].bm25, maxbm);
            } else {
                out_ids[o] = -1;
                out_score[o] = 0.0;
                out_sem[o] = 0.0;
                out_kw[o] = 0.0;
            }
        }
    } else {
        merge_lists(1, ssel, &n_sparse);
        const int ns = n_sparse;
        // union slots: [0, nd) dense entries, [nd, nd + ns) BM25 entries (unused when the
        // document is already in the dense list).  Dense term first: 0.0 + 1/(60 + rank).
        for (int j = tid; j < nd + ns; j += kFuseThreads)
            fscore[j] = (j < nd) ? __dadd_rn(0.0, __ddiv_rn(1.0, 60.0 + (double)(j + 1))) : -1.0;
        __syncthreads();
        for (int r = tid; r < ns; r += kFuseThreads) {
            const double term = __ddiv_rn(1.0, 60.0 + (double)(r + 1));
            int hit = -1;
            for (int j = 0; j < nd; ++j)
                if (dsel[j].id == ssel[r].id) hit = j;
            if (hit >= 0) fscore[hit] = __dadd_rn(fscore[hit], term);      // unique hit per r
            else fscore[nd + r] = __dadd_rn(0.0, term);
        }
        __syncthreads();
        for (int i = tid; i < nd + ns; i += kFuseThreads) {
            u128 key = 0;
            if (fscore[i] > 0.0) {
                const int64_t id = (i < nd) ? dsel[i].id : ssel[i - nd].id;
                key = rec_key(fscore[i], id, (uint32_t)i);
            }
            keys[i] = key;
        }
        order_keys(nd + ns);
        const int n_out = min(k, n_fused);
        for (int i = tid; i < k; i += kFuseThreads) {
            const size_t o = (size_t)b * k + i;
            if (i < n_out) {
                const int src = out_slot[i];
                const lrx_record& r = (src < nd) ? dsel[src] : ssel[src - nd];
                out_ids[o] = r.id;
                out_score[o] = fscore[src];
                out_sem[o] = (double)__double2float_rn(r.dense);
                out_kw[o] = __ddiv_rn(r.bm25, maxbm);
            } else {
                out_ids[o] = -1;
                out_score[o] = 0.0;
                out_sem[o] = 0.0;
                out_kw[o] = 0.0;
            }
        }
    }
    if (tid == 0) out_status[b] = wait_failed ? -1 : status;
}

cudaError_t launch_pack_exchange(lrx_handle* h, const int32_t* q_terms, const int32_t* q_ptr, int B, int K,
                                 int mode, const double* dense_exact, const int64_t* dense_ids,
                                 const double* bm_scores, const int64_t* bm_ids, const double* maxbm,
                                 const int32_t* flags, const void* q, void* local_block, bool to_peers,
                                 size_t o_max, size_t o_flags) {
    BmAtParams A;
    cudaError_t e = bm25_at_params(h, q_terms, q_ptr, B, &A);
    if (e != cudaSuccess) return e;
    PackDst D;
    D.local = (unsigned char*)local_block;
    D.peers = to_peers ? (void* const*)h->xchg_peer_dev : nullptr;
    D.rank = h->rank; D.world = h->world; D.slot = h->xchg_slot;
    D.o_max = o_max; D.o_flags = o_flags;
    const int n = B * K;
    // a plain launch: the kernel follows the join of the two chains (its griddepcontrol.wait is a
    // no-op); the fusion kernel behind it is the programmatic dependent
    pack_exchange_kernel<<<(n + 7) / 8, 256, 0, h->stream>>>(
        B, K, mode, dense_exact, dense_ids, bm_scores, bm_ids, maxbm, flags, (const unsigned char*)h->x,
        h->n_local, (const __half*)q, A, D, h->pack_done);
    h->launches++;
    return cudaGetLastError();
}

cudaError_t launch_fuse(lrx_handle* h, const void* blocks, size_t stride, size_t o_max, size_t o_flags,
                        bool exchange, int world, int B, int K, int k, int mode, const double* weights,
                        int64_t* ids, double* score, double* sem, double* kw, int32_t* status) {
    {
        std::lock_guard<std::recursive_mutex> attr_guard(attr_mutex());   // the flags below are process-wide
        static bool attr_dev[64] = {false};   // function attributes are per device
        bool& attr = attr_dev[h->device & 63];
        if (!attr) {
            cudaError_t e = cudaFuncSetAttribute(fuse_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                 (int)(kFuseMaxIn * sizeof(u128)));
            if (e != cudaSuccess) return e;
            attr = true;
        }
    }
    if (world * K > kFuseMaxIn || K > kFuseMaxK) return cudaErrorInvalidValue;
    cudaError_t e = launch_pdl(fuse_kernel, dim3(B), dim3(kFuseThreads), kFuseMaxIn * sizeof(u128), h->stream,
                               (const unsigned char*)blocks, stride, o_max, o_flags, exchange, world, B, K, k,
                               mode, weights, ids, score, sem, kw, status,
                               (long long)h->xchg_timeout_ms * 1000000ll, h->rank);
    h->launches++;
    return e;
}

}  // namespace lrx
