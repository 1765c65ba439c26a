// K2b: flat inner-product top-K for LARGE query batches (B = 64 ... 4096) on the tensor cores.
//
// Replaces faiss IndexFlatIP.search(x, K) for nq >= 20, where FAISS switches from its
// per-query scan to BLAS sgemm blocks (reference call site: src/retrieval/retrieval_engine.py:64;
// config C3, B = 1024).  scores[B, N] = Q[B,384] * X[N,384]^T never exists in HBM: the GEMM
// tiles live in TMEM and are reduced on the way out.
//
// Two tensor-core passes with the same persistent kernel (dense_tc_kernel<PASS>):
//   pass 1  over every `stride`-th 256-row tile: per (query, 32-row chunk) the MAXIMUM score.
//           The K-th largest chunk maximum T[q] (tilemax_kth_kernel) is a lower bound of the
//           K-th best score: K distinct rows reach it.
//   pass 2  over all tiles: every (query, row) with score >= T[q] - slack is appended to the
//           query's candidate list (a few hundred per query): a private region per (query, CTA,
//           column half), and once that region is full a per-query overflow list of kDbCap slots.
// dense_rescore_list_kernel then re-scores the candidates EXACTLY in float64 (oracle/flat_ip.py),
// orders them by (score desc, id asc) and emits the best K.  With slack = 2 * kTcEps a row that
// was not appended is strictly below the K-th best exact score, so the result is bit-exact; the
// only failure mode is more than kDbCap candidates for a query (flag).  Where fewer than 2K
// sampled chunks hold rows, T would be loose (or -FLT_MAX: chunks past the corpus end rank too),
// so such a batch goes to the streaming scan (K2a) instead.  Chunk stores keep similar chunks next
// to one another, so a query's candidates can crowd into a few regions: the overflow list keeps
// that from flagging it.
//
// Kernel shape (one CTA per SM, 320 threads, warp-specialised like tc_gemm.cu):
//   A operand = 128 queries x 384, loaded once by TMA and RESIDENT in shared memory (96 KB);
//   B operand = 256 chunk rows x 64 per stage, 3-stage TMA ring (SWIZZLE_128B);
//   tcgen05.mma cta_group::1 kind::f16, UMMA 128 x 256 x 16, fp32 accumulators in TMEM,
//   DOUBLE-BUFFERED (2 x 256 columns) so the epilogue of tile i overlaps the MMAs of tile i+1;
//   8 epilogue warps, thread = (query, column half): pipelined tcgen05.ld of 32 columns, running
//   max / compare.  CTA pairs (cluster of 2) multicast the chunk tiles to each other.
// CTA c serves query tile (c % n_mt) and walks chunk tiles (c / n_mt), (c / n_mt) + G, ... so the
// n_mt CTAs that need the same chunk tile touch it at about the same time (one HBM read, L2 hits).
//
// Roofline: tensor pipe.  flops per launch = 2 * B_padded * 384 * rows scanned.
#include <cfloat>

#include "handle.h"
#include "tc.cuh"

namespace lrx {

cudaError_t make_tmap_f16(CUtensorMap* out, const void* ptr, int64_t rows, int64_t cols, int64_t ld,
                          int box_rows);

constexpr int kDbQ = 128;             // queries per CTA (UMMA M)
constexpr int kDbN = 256;             // chunk rows per tile (UMMA N)
constexpr int kDbK = 64;              // halves per k-block (128 B, one swizzle row)
constexpr int kDbKB = kDim / kDbK;    // 6 k-blocks
constexpr int kDbStages = 3;
constexpr int kDbABytes = kDbQ * kDbK * 2;    // 16 KB per k-block of the query tile
constexpr int kDbBBytes = kDbN * kDbK * 2;    // 32 KB per stage
constexpr int kDbEpiWarps = 8;          // two per TMEM lane quarter: column halves of a tile
constexpr int kDbThreads = (kDbEpiWarps + 2) * 32;
constexpr size_t kDbSmem = (size_t)kDbKB * kDbABytes + (size_t)kDbStages * kDbBBytes + 1024 + 256;
constexpr int kDbCap = 1024;          // candidates re-scored per query, at most
constexpr int kDbMaxRegions = 2 * 160; // candidate regions per query (2 per CTA of its query tile)
// |tensor-core fp32 score - exact| for unit fp16 vectors: 384 exact products accumulated in
// fp32 (possibly truncating) in 24 instructions -> well below 1e-5
constexpr float kTcEps = 1e-5f;

struct DbParams {
    int B;                 // valid queries
    int64_t n_rows;
    int n_tiles;           // ceil(n_rows / 256)
    int n_mt;              // query tiles
    int stride;            // pass 1: every stride-th tile
    float* tilemax;        // [n_mt*128][n_samp]       (pass 1 out)
    int n_samp;
    const float* thr;      // [n_mt*128]               (pass 2 in)
    // candidate lists of pass 2: one private region per (query, CTA of the query tile, column half),
    // filled by the ONE thread that owns it with a counter it keeps in a register -- no atomics.  (A
    // list per query behind one atomicAdd put a dependent L2 round trip, taken inside a divergent
    // branch, on every candidate: at 1 M rows 15 % of the (warp, chunk) pairs hit it and the pass ran
    // at 35 % tensor-pipe activity, 1.20 ms for 0.71 ms of MMAs.)
    int n_regions;         // 2 * CTAs per query tile
    int region_cap;        // slots per region
    int* cnt;              // [n_mt*128][n_regions] candidates found (may exceed region_cap: overflow)
    // [n_mt*128][n_regions * region_cap + kDbCap] local row ids: the query's regions, then its
    // overflow list, where a full region's further candidates go behind one atomicAdd (rare: a
    // region fills only where similar rows cluster)
    uint32_t* cand;
    int* ov_cnt;           // [n_mt*128] candidates spilled (may exceed kDbCap); tilemax_kth_kernel zeroes it
};

__host__ __device__ inline size_t db_cand_per_query(int n_regions, int region_cap) {
    return (size_t)n_regions * region_cap + kDbCap;
}

// CS: cluster size.  The CS CTAs of a cluster serve CS different query tiles and walk the SAME chunk
// tiles: each loads 1/CS of a tile's rows and multicasts them to all (one L2 read per cluster).
template <int PASS, int CS>
__global__ void __launch_bounds__(kDbThreads, 1)
dense_tc_kernel(const __grid_constant__ CUtensorMap tma_q, const __grid_constant__ CUtensorMap tma_x,
                const DbParams P) {
    constexpr uint16_t kMask = (uint16_t)((1u << CS) - 1u);
    const uint32_t crank = (CS > 1) ? cluster_ctarank() : 0u;
    extern __shared__ unsigned char db_raw[];
    unsigned char* base = reinterpret_cast<unsigned char*>(
        (reinterpret_cast<uintptr_t>(db_raw) + 1023) & ~(uintptr_t)1023);
    unsigned char* sA = base;
    unsigned char* sB = base + kDbKB * kDbABytes;
    uint64_t* full = reinterpret_cast<uint64_t*>(sB + kDbStages * kDbBBytes);
    uint64_t* empty = full + kDbStages;
    uint64_t* a_full = empty + kDbStages;
    uint64_t* t_full = a_full + 1;       // [2] accumulator ready
    uint64_t* t_empty = t_full + 2;      // [2] accumulator drained
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(t_empty + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int m_tile = blockIdx.x % P.n_mt;
    const int group = blockIdx.x / P.n_mt;
    const int n_groups = gridDim.x / P.n_mt;
    const int step = (PASS == 1) ? P.stride : 1;
    // this CTA's tiles: t = (group + i * n_groups) * step
    const int n_units = (P.n_tiles + step - 1) / step;
    const int my_units = (n_units > group) ? (n_units - group + n_groups - 1) / n_groups : 0;

    constexpr int kProducerWarp = kDbEpiWarps, kMmaWarp = kDbEpiWarps + 1;
    if (warp == kProducerWarp && lane == 0) {
        tma_prefetch_desc(&tma_q);
        tma_prefetch_desc(&tma_x);
        for (int s = 0; s < kDbStages; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], CS);
        }
        mbar_init(a_full, 1);
        for (int b = 0; b < 2; ++b) {
            mbar_init(&t_full[b], 1);
            mbar_init(&t_empty[b], kDbEpiWarps);
        }
        fence_barrier_init();
    }
    if (warp == kMmaWarp) {
        tmem_alloc(tmem_slot, 512);
        tmem_relinquish();
    }
    tc_fence_before();
    __syncthreads();
    if (CS > 1) cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == kProducerWarp) {
        if (lane == 0) {
            // the query tile, once
            mbar_arrive_expect_tx(a_full, (uint32_t)(kDbKB * kDbABytes));
            for (int kb = 0; kb < kDbKB; ++kb)
                tma_load_2d(sA + kb * kDbABytes, &tma_q, kb * kDbK, m_tile * kDbQ, a_full);
            uint32_t it = 0;
            for (int u = 0; u < my_units; ++u) {
                const int tile = (group + u * n_groups) * step;
                for (int kb = 0; kb < kDbKB; ++kb, ++it) {
                    const int s = (int)(it % kDbStages);
                    const uint32_t ph = (it / kDbStages) & 1u;
                    mbar_wait(&empty[s], ph ^ 1u);
                    mbar_arrive_expect_tx(&full[s], (uint32_t)kDbBBytes);
                    if (CS > 1)
                        tma_load_2d_mc(sB + s * kDbBBytes + crank * (kDbBBytes / CS), &tma_x, kb * kDbK,
                                       tile * kDbN + (int)crank * (kDbN / CS), &full[s], kMask);
                    else
                        tma_load_2d(sB + s * kDbBBytes, &tma_x, kb * kDbK, tile * kDbN, &full[s]);
                }
            }
        }
    } else if (warp == kMmaWarp) {
        if (lane == 0) {
            constexpr uint32_t idesc = umma_idesc_f16(kDbQ, kDbN);
            mbar_wait(a_full, 0);
            uint32_t it = 0;
            for (int u = 0; u < my_units; ++u) {
                const int buf = u & 1;
                const uint32_t use = (uint32_t)(u >> 1);
                mbar_wait(&t_empty[buf], (use & 1u) ^ 1u);     // epilogue drained this buffer
                tc_fence_after();
                for (int kb = 0; kb < kDbKB; ++kb, ++it) {
                    const int s = (int)(it % kDbStages);
                    const uint32_t ph = (it / kDbStages) & 1u;
                    mbar_wait(&full[s], ph);
                    tc_fence_after();
                    const uint32_t a_addr = smem_u32(sA + kb * kDbABytes);
                    const uint32_t b_addr = smem_u32(sB + s * kDbBBytes);
#pragma unroll
                    for (int k = 0; k < kDbK / 16; ++k)
                        umma_f16(tmem_base + buf * kDbN, umma_desc_sw128(a_addr + k * 32),
                                 umma_desc_sw128(b_addr + k * 32), idesc, (kb > 0 || k > 0) ? 1u : 0u);
                    if (CS > 1) umma_commit_mc(&empty[s], kMask);
                    else umma_commit(&empty[s]);
                }
                umma_commit(&t_full[buf]);
            }
        }
    } else {
        // ===== epilogue: 8 warps; thread = query (TMEM lane 32*(warp&3)+lane), column half (warp>>2)
        const int quarter = warp & 3, half = warp >> 2;
        constexpr int HB = kDbN / 2, NCH = HB / 32;
        const int ql = quarter * 32 + lane;
        const int q = m_tile * kDbQ + ql;
        const bool q_ok = q < P.B;
        const uint32_t trow = tmem_base + ((uint32_t)(quarter * 32) << 16) + half * HB;
        float thr = 0.f;
        if (PASS == 2) thr = q_ok ? P.thr[q] : FLT_MAX;
        uint32_t rb[2][32];
        const int region = group * 2 + half;
        int my_cnt = 0;                                      // candidates of (q, region) so far
        uint32_t* q_cand = P.cand + (size_t)q * db_cand_per_query(P.n_regions, P.region_cap);
        uint32_t* my_cand = q_cand + (size_t)region * P.region_cap;
        for (int u = 0; u < my_units; ++u) {
            const int buf = u & 1;
            const uint32_t use = (uint32_t)(u >> 1);
            const int tile = (group + u * n_groups) * step;
            const int64_t row0 = (int64_t)tile * kDbN + half * HB;
            const int valid = (int)max((int64_t)0, min((int64_t)HB, P.n_rows - row0));
            mbar_wait(&t_full[buf], use & 1u);
            tc_fence_after();
            tmem_ld32(trow + buf * kDbN, rb[0]);
            tmem_wait_ld();
#pragma unroll
            for (int ch = 0; ch < NCH; ++ch) {
                if (ch + 1 < NCH) tmem_ld32(trow + buf * kDbN + (ch + 1) * 32, rb[(ch + 1) & 1]);
                const uint32_t(&r)[32] = rb[ch & 1];
                const int c = ch * 32;
                if (PASS == 1) {
                    // maximum of every 32-row chunk: 8 samples per tile for the threshold
                    float mx = -FLT_MAX;
#pragma unroll
                    for (int j = 0; j < 32; ++j)
                        if (c + j < valid) mx = fmaxf(mx, __uint_as_float(r[j]));
                    P.tilemax[(size_t)q * P.n_samp + (size_t)(tile / step) * (kDbN / 32) + half * NCH + ch] = mx;
                } else {
                    // fast path: the chunk's maximum by 3-input max (16 instructions for 32 scores); rows
                    // past the end of the corpus (last tile only) are masked out in the rare path
                    float best = __uint_as_float(r[0]);
#pragma unroll
                    for (int j = 1; j + 1 < 32; j += 2)
                        asm("max.f32 %0, %0, %1, %2;" : "+f"(best) : "f"(__uint_as_float(r[j])), "f"(__uint_as_float(r[j + 1])));
                    best = fmaxf(best, __uint_as_float(r[31]));
                    if (best >= thr) {
                        // rare (a few candidates per tile and warp) and therefore SMALL: a hit mask,
                        // then one 4-byte row id per set bit.  (The first form, 32 unrolled
                        // compare-and-store bodies per chunk, was 3 000 instructions of cold code:
                        // every hit streamed them through the instruction cache, ~1 500 cycles on the
                        // critical path of an epilogue-bound pipeline -- 1 M rows: 35 % tensor-pipe
                        // activity with the hits, 77 % of peak without.)
                        uint32_t mask = 0u;
#pragma unroll
                        for (int j = 0; j < 32; ++j) mask |= (__uint_as_float(r[j]) >= thr) ? (1u << j) : 0u;
                        const int left = valid - c;
                        mask &= (left >= 32) ? 0xffffffffu : (left > 0 ? ((1u << left) - 1u) : 0u);
#pragma unroll 1
                        while (mask != 0u) {
                            const int j = __ffs((int)mask) - 1;
                            mask &= mask - 1u;
                            const uint32_t row = (uint32_t)(row0 + c + j);
                            if (my_cnt < P.region_cap) {
                                my_cand[my_cnt] = row;
                            } else {
                                const int o = atomicAdd(&P.ov_cnt[q], 1);
                                if (o < kDbCap) q_cand[(size_t)P.n_regions * P.region_cap + o] = row;
                            }
                            ++my_cnt;
                        }
                    }
                }
                tmem_wait_ld();
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&t_empty[buf]);
        }
        if (PASS == 2) P.cnt[(size_t)q * P.n_regions + region] = my_cnt;
    }
    tc_fence_before();
    __syncthreads();
    if (CS > 1) cluster_sync_all();
    if (warp == kMmaWarp) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

// T[q] = (K-th largest tile maximum) - slack; -FLT_MAX when fewer than K tiles were sampled.
// One CTA per query.  Only the K-th largest of up to 16 384 values is needed, so this is a radix
// SELECT over the order images (four 8-bit passes: shared-memory histogram of the keys that match
// the prefix found so far, then warp 0 walks the 256 bins from the top), not a sort.  Also resets
// the query's overflow counter for pass 2.
__global__ void __launch_bounds__(256)
tilemax_kth_kernel(const float* __restrict__ tilemax, int n_samp, int K, float slack,
                   float* __restrict__ thr, int* __restrict__ ov_cnt) {
    extern __shared__ uint32_t tm_keys[];
    __shared__ uint32_t hist[256];
    __shared__ uint32_t s_prefix, s_rank;
    const int q = blockIdx.x, tid = threadIdx.x, lane = tid & 31;
    for (int i = tid; i < n_samp; i += 256) tm_keys[i] = f32_ord(tilemax[(size_t)q * n_samp + i]);
    if (tid == 0) { s_prefix = 0u; s_rank = (uint32_t)K; }   // rank counted from the largest, 1-based
    __syncthreads();
    if (K <= n_samp) {
        for (int pass = 3; pass >= 0; --pass) {
            hist[tid] = 0u;
            __syncthreads();
            const uint32_t prefix = s_prefix;
            const int hs = 8 * (pass + 1);                   // bits above this byte
            for (int i = tid; i < n_samp; i += 256) {
                const uint32_t key = tm_keys[i];
                if (pass == 3 || (key >> hs) == (prefix >> hs)) atomicAdd(&hist[(key >> (8 * pass)) & 255u], 1u);
            }
            __syncthreads();
            if (tid < 32) {
                // lane l owns bins 255 - 8l .. 248 - 8l (descending); exclusive prefix over lanes
                uint32_t local = 0;
#pragma unroll
                for (int j = 0; j < 8; ++j) local += hist[255 - (8 * lane + j)];
                uint32_t incl = local;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const uint32_t v = __shfl_up_sync(0xffffffffu, incl, d);
                    if (lane >= d) incl += v;
                }
                const uint32_t before = incl - local, rank = s_rank;
                if (before < rank && rank <= incl) {         // the K-th key falls into this lane's bins
                    uint32_t cum = before;
                    for (int j = 0; j < 8; ++j) {
                        const uint32_t bin = 255u - (uint32_t)(8 * lane + j);
                        const uint32_t c = hist[bin];
                        if (rank <= cum + c) {
                            s_prefix = prefix | (bin << (8 * pass));
                            s_rank = rank - cum;
                            break;
                        }
                        cum += c;
                    }
                }
            }
            __syncthreads();
        }
    }
    if (tid == 0) {
        thr[q] = (K <= n_samp) ? ord_f32(s_prefix) - slack : -FLT_MAX;
        ov_cnt[q] = 0;
    }
}

// Exact float64 re-score of a query's (unsorted) candidate list, best K out.  Each warp takes four
// candidates per pass, all twelve row loads in flight before the first reduction; the order is a
// rank by counting on the unique (exact score, id) keys -- a few hundred candidates, no sort.
constexpr int kRlThreads = 256;
__global__ void __launch_bounds__(kRlThreads)
dense_rescore_list_kernel(const unsigned char* __restrict__ x, int64_t id_base,
                          const __half* __restrict__ q, const uint32_t* __restrict__ cand,
                          const int* __restrict__ cnt, const int* __restrict__ ov_cnt, int n_regions,
                          int region_cap, int K, double* __restrict__ out_exact,
                          float* __restrict__ out_D, int64_t* __restrict__ out_I,
                          int32_t* __restrict__ out_flag) {
    __shared__ u128 keys[kDbCap];
    __shared__ u128 best[LRX_MAX_DEPTH];
    __shared__ int pre[kDbMaxRegions + 2];                   // candidates before region r
    const int qi = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // the query's regions, concatenated, then its overflow list as region n_regions (it follows the
    // regions in memory): candidate i lives in the region r with pre[r] <= i < pre[r+1]
    if (tid == 0) {
        int acc = 0;
        for (int r = 0; r < n_regions; ++r) {
            pre[r] = acc;
            acc += min(cnt[(size_t)qi * n_regions + r], region_cap);
        }
        pre[n_regions] = acc;
        pre[n_regions + 1] = acc + ov_cnt[qi];
    }
    __syncthreads();
    const int total = pre[n_regions + 1];
    const int n = min(total, kDbCap);
    const uint32_t* qcand = cand + (size_t)qi * db_cand_per_query(n_regions, region_cap);
    auto cand_at = [&](int i) -> uint32_t {
        int lo = 0, hi = n_regions + 1;                      // last r with pre[r] <= i
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if (pre[mid] <= i) lo = mid; else hi = mid;
        }
        return qcand[(size_t)lo * region_cap + (i - pre[lo])];
    };
    const uint2* qp = reinterpret_cast<const uint2*>(q + (size_t)qi * kDim);
    uint2 qv[3];
#pragma unroll
    for (int s = 0; s < 3; ++s) qv[s] = qp[s * 32 + lane];
    for (int j = tid; j < K && j < LRX_MAX_DEPTH; j += kRlThreads) best[j] = 0;
    constexpr int kWarps = kRlThreads / 32;
    for (int j0 = warp * 4; j0 < n; j0 += kWarps * 4) {
        uint32_t row[4];
        uint2 rv[4][3];
#pragma unroll
        for (int c = 0; c < 4; ++c)
            row[c] = (j0 + c < n) ? cand_at(j0 + c) : 0u;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const uint2* rowp = reinterpret_cast<const uint2*>(x + (int64_t)row[c] * kRowBytes);
#pragma unroll
            for (int s = 0; s < 3; ++s)
                rv[c][s] = (j0 + c < n) ? rowp[s * 32 + lane] : make_uint2(0u, 0u);
        }
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            double acc = 0.0;
#pragma unroll
            for (int s = 0; s < 3; ++s) {
                const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&rv[c][s].x));
                const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&rv[c][s].y));
                const float2 e = __half22float2(*reinterpret_cast<const __half2*>(&qv[s].x));
                const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&qv[s].y));
                acc = fma((double)a.x, (double)e.x, acc);
                acc = fma((double)a.y, (double)e.y, acc);
                acc = fma((double)b.x, (double)f.x, acc);
                acc = fma((double)b.y, (double)f.y, acc);
            }
#pragma unroll
            for (int lb = 16; lb > 0; lb >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, lb);
            if (lane == 0 && j0 + c < n) keys[j0 + c] = make_key128(acc, row[c]);
        }
    }
    __syncthreads();
    for (int j = tid; j < n; j += kRlThreads) {
        const u128 key = keys[j];
        int rank = 0;
        for (int i = 0; i < n && rank < K; ++i) rank += (keys[i] > key) ? 1 : 0;
        if (rank < K) best[rank] = key;
    }
    __syncthreads();
    for (int j = tid; j < K; j += kRlThreads) {
        const u128 key = (j < LRX_MAX_DEPTH) ? best[j] : (u128)0;
        const size_t o = (size_t)qi * K + j;
        if (key != 0) {
            const double e = key128_score(key);
            out_exact[o] = e;
            out_D[o] = (float)e;
            out_I[o] = id_base + (int64_t)key128_row(key);
        } else {
            out_exact[o] = -INFINITY;
            out_D[o] = -3.4028234663852886e38f;
            out_I[o] = -1;
        }
    }
    if (tid == 0) out_flag[qi] = (total > kDbCap) ? 1 : 0;
}

int dense_batched_max_stride(int64_t n_rows, int K) {
    // keep at least 16K sampled 32-row chunks so T is a tight bound
    const int64_t n_tiles = (n_rows + kDbN - 1) / kDbN;
    int s = (int)(n_tiles * (kDbN / 32) / (16 * (int64_t)K));
    if (s < 1) s = 1;
    if (s > 8) s = 8;
    return s;
}

cudaError_t launch_dense_topk_batched(lrx_handle* h, const void* q, int B, int K, int stride,
                                      double* exact, float* D, int64_t* I, int32_t* flags) {
    std::lock_guard<std::recursive_mutex> attr_guard(attr_mutex());   // the flags below are process-wide
    static bool attr_dev[64] = {false};   // function attributes are per device
    bool& attr = attr_dev[h->device & 63];
    cudaError_t e;
    if (!attr) {
        const void* ks[] = {(const void*)dense_tc_kernel<1, 1>, (const void*)dense_tc_kernel<2, 1>,
                            (const void*)dense_tc_kernel<1, 2>, (const void*)dense_tc_kernel<2, 2>,
                            (const void*)dense_tc_kernel<1, 4>, (const void*)dense_tc_kernel<2, 4>};
        for (const void* k : ks) {
            e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kDbSmem);
            if (e != cudaSuccess) return e;
        }
        e = cudaFuncSetAttribute(tilemax_kth_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 65536);
        if (e != cudaSuccess) return e;
        attr = true;
    }
    const int64_t n = h->n_local;
    const int n_tiles = (int)((n + kDbN - 1) / kDbN);
    int n_mt = (B + kDbQ - 1) / kDbQ;
    // cluster of query tiles sharing every chunk tile (padded query tiles are zero rows)
    const int cs = (n_mt >= 2) ? 2 : 1;
    n_mt = (n_mt + cs - 1) / cs * cs;
    const int Bp = n_mt * kDbQ;
    if (stride < 1) stride = dense_batched_max_stride(n, K);
    constexpr int kChunks = kDbN / 32;
    int n_samp = (n_tiles + stride - 1) / stride * kChunks;
    if (n_samp > 16384) {                      // shared-memory sort limit of tilemax_kth_kernel
        stride = (n_tiles * kChunks + 16383) / 16384;
        n_samp = (n_tiles + stride - 1) / stride * kChunks;
    }
    // sampled chunks that hold rows: 8 per sampled tile, fewer when the last tile is sampled.  The
    // others have maximum -FLT_MAX; with fewer than 2K valid ones T is loose (the lists overflow) or
    // -FLT_MAX (every row a candidate)
    int64_t valid = (int64_t)((n_tiles + stride - 1) / stride) * kChunks;
    if ((n_tiles - 1) % stride == 0) valid -= kChunks - (n - (int64_t)(n_tiles - 1) * kDbN + 31) / 32;
    if (valid < 2 * (int64_t)K) {
        // small corpus for this K: no useful threshold -- the streaming kernel, 64 queries a time
        for (int b0 = 0; b0 < B; b0 += LRX_MAX_BATCH) {
            const int nb = (B - b0 < LRX_MAX_BATCH) ? (B - b0) : LRX_MAX_BATCH;
            e = launch_dense_topk(h, (const __half*)q + (size_t)b0 * kDim, nb, K, dense_default_width(K),
                                  exact + (size_t)b0 * K, D + (size_t)b0 * K, I + (size_t)b0 * K, flags + b0);
            if (e != cudaSuccess) return e;
        }
        return cudaSuccess;
    }
    int grid = (h->num_sms / n_mt) * n_mt;
    if (grid < n_mt) grid = n_mt;
    // workspace: tilemax | thr | cnt | cand
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off = (off + bytes + 255) / 256 * 256; return o; };
    const size_t o_tm = take((size_t)Bp * n_samp * sizeof(float));
    const size_t o_thr = take((size_t)Bp * sizeof(float));
    const int n_regions = 2 * (grid / n_mt);
    if (n_regions > kDbMaxRegions) return cudaErrorInvalidConfiguration;
    int region_cap = 16;                       // >= 2048 slots per query over its regions: an even
    while (region_cap * n_regions < 2048) region_cap <<= 1;   // spread fills a few percent of a region
    const size_t o_cnt = take((size_t)Bp * n_regions * sizeof(int));
    const size_t o_cand = take((size_t)Bp * db_cand_per_query(n_regions, region_cap) * sizeof(uint32_t));
    const size_t o_ov_cnt = take((size_t)Bp * sizeof(int));
    e = ensure_ws(h, &h->ws_dense_part, &h->ws_dense_part_bytes, off);
    if (e != cudaSuccess) return e;
    char* W = (char*)h->ws_dense_part;
    CUtensorMap tq, tx;
    e = make_tmap_f16(&tq, q, B, kDim, kDim, kDbQ);
    if (e != cudaSuccess) return e;
    e = make_tmap_f16(&tx, h->x, n, kDim, kDim, kDbN / cs);
    if (e != cudaSuccess) return e;
    DbParams P;
    P.B = B; P.n_rows = n; P.n_tiles = n_tiles; P.n_mt = n_mt; P.stride = stride;
    P.tilemax = (float*)(W + o_tm); P.n_samp = n_samp; P.thr = (const float*)(W + o_thr);
    P.cnt = (int*)(W + o_cnt); P.cand = (uint32_t*)(W + o_cand);
    P.n_regions = n_regions; P.region_cap = region_cap;
    P.ov_cnt = (int*)(W + o_ov_cnt);
    auto launch = [&](int pass) -> cudaError_t {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(grid);
        cfg.blockDim = dim3(kDbThreads);
        cfg.dynamicSmemBytes = kDbSmem;
        cfg.stream = h->stream;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = cs;
        at[0].val.clusterDim.y = 1;
        at[0].val.clusterDim.z = 1;
        cfg.attrs = at;
        cfg.numAttrs = 1;
        if (cs == 4) return pass == 1 ? cudaLaunchKernelEx(&cfg, dense_tc_kernel<1, 4>, tq, tx, P)
                                      : cudaLaunchKernelEx(&cfg, dense_tc_kernel<2, 4>, tq, tx, P);
        if (cs == 2) return pass == 1 ? cudaLaunchKernelEx(&cfg, dense_tc_kernel<1, 2>, tq, tx, P)
                                      : cudaLaunchKernelEx(&cfg, dense_tc_kernel<2, 2>, tq, tx, P);
        return pass == 1 ? cudaLaunchKernelEx(&cfg, dense_tc_kernel<1, 1>, tq, tx, P)
                         : cudaLaunchKernelEx(&cfg, dense_tc_kernel<2, 1>, tq, tx, P);
    };
    prof_begin(h, 0);
    e = launch(1);
    prof_end(h, 0);
    h->launches++;
    if (e != cudaSuccess) return e;
    tilemax_kth_kernel<<<Bp, 256, (size_t)next_pow2(n_samp > 2 ? n_samp : 2) * sizeof(uint32_t), h->stream>>>(
        P.tilemax, n_samp, K, 2.0f * kTcEps, (float*)(W + o_thr), P.ov_cnt);
    h->launches++;
    e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    prof_begin(h, 0);
    e = launch(2);
    prof_end(h, 0);
    h->launches++;
    if (e != cudaSuccess) return e;
    dense_rescore_list_kernel<<<B, kRlThreads, 0, h->stream>>>(
        (const unsigned char*)h->x, h->id_base, (const __half*)q, P.cand, P.cnt, P.ov_cnt, n_regions,
        region_cap, K, exact, D, I, flags);
    h->launches++;
    return cudaGetLastError();
}

}  // namespace lrx
