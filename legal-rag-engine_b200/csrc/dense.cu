// K2a: flat inner-product scan of the fp16 chunk matrix fused with top-k select.
//
// Replaces faiss IndexFlatIP.search (reference: src/retrieval/retrieval_engine.py:64)
// for small query batches (the B <= 4 sub-queries of one fan-out).
//
// Kernels:
//   dense_scan_kernel   HBM-bound: streams the [n,384] fp16 matrix once through a 2-stage
//                       shared-memory ring filled by 1-D bulk async copies (TMA engine,
//                       mbarrier byte counting, L2 evict-first), scores up to 4 queries per row
//                       on the tensor cores (mma.sync m16n8k16, fp16 x fp16 -> fp32: products
//                       exact, accumulation within the guard band kDenseEps) and keeps a per-CTA
//                       top-`width` candidate list in shared memory (threshold test per (row,
//                       query), register sorting networks when a buffer fills, thresholds shared
//                       grid-wide).  Scores never touch HBM.  256 threads, 133 KB: one BM25 scan
//                       CTA fits beside it on the SM (api.cu runs the two scans side by side).
//   dense_scan_q8_kernel  the same scan over an int8 SHADOW of the matrix (388 B/row for 768; the
//                       default when lrx_build_dense_prefilter has run): mma.sync m16n8k32 s8 on
//                       two int8 digits per query element, per-row fp32 scales, 128-row tiles, one
//                       barrier per tile; see the block comment in front of it for the guard band
//                       that keeps the results bit-identical.  dense_q8_build_kernel builds the shadow.
//   dense_merge_rescore_kernel  one CTA per query merges the per-CTA lists (merge.cuh) and
//                       re-scores the `width` survivors EXACTLY in float64 (exact
//                       and order independent, see oracle/flat_ip.py), orders them by
//                       (score desc, id asc), emits the best K and the guard flag.
//
// Algorithmic HBM bytes per launch: dense_scan_kernel n_local * 768, dense_scan_q8_kernel n_pad * 388.
#include "common.cuh"
#include "handle.h"
#include "merge.cuh"

#include <cmath>
#include <cstring>

namespace lrx {

constexpr int kScanThreads = 256;                  // 8 warps: the SM is shared with a BM25 scan CTA
constexpr int kTileRows = 64;                      // 4 rows per warp per tile
constexpr int kTileBytes = kTileRows * kRowBytes;  // 49152
constexpr int kStages = 2;                         // 2, 3 and 4 measure the same; 2 leaves shared
                                                   // memory for a co-resident BM25 CTA
constexpr int kCap = 1024;                         // candidate buffer entries per query
constexpr int kSoftCap = 256;                      // prune once a buffer holds more than this minus a
                                                   // tile: sorting 256 keys costs ~3 us, 1024 keys ~40 us,
                                                   // and the threshold tightens 4x per prune either way
constexpr int kMaxWidth = 512;                     // max per-CTA list length
constexpr int kMaxMerged = 2048;                   // max merged list (int8 pre-filter, deep lists)
static size_t merge_smem_bytes(int merged_width) {
    return (size_t)kMergeCap * sizeof(uint64_t) + (size_t)merged_width * (2 * sizeof(u128) + sizeof(uint64_t));
}
// candidate buffer entries per query: up to 4 queries per pass 1024 each, 5..8 queries 512 each (the
// same 32 KB: a CTA of the BM25 scan must keep fitting beside this kernel's CTA; lists up to 256 wide)
__host__ __device__ constexpr int scan_cap(int nq) { return nq > 4 ? 512 : kCap; }

struct ScanSmem {
    // ring first (16-byte aligned bulk-copy destinations)
    unsigned char ring[kStages][kTileBytes];
    float part[2][kTileRows][8];   // [k half][row][query] partial scores of one tile
    uint64_t full[kStages];
    int tile_of[kStages];          // tile held (or being loaded) by every stage
    int count[8];
    uint32_t tau[8];
    uint64_t keys[1];   // [NQ][scan_cap(NQ)], sized at launch
};

// ---- register sorting networks of the fast prune (two keys per lane, 64 keys per warp)
__device__ __forceinline__ uint64_t shfl_xor_u64(uint64_t v, int m) {
    const uint32_t lo = __shfl_xor_sync(0xffffffffu, (uint32_t)v, m);
    const uint32_t hi = __shfl_xor_sync(0xffffffffu, (uint32_t)(v >> 32), m);
    return ((uint64_t)hi << 32) | lo;
}
// one compare-exchange layer over the 64 keys of a warp, element index i = 2 * lane + r,
// partner i ^ j; `desc` = the pair's first element keeps the larger key
template <int J>
__device__ __forceinline__ void warp64_layer(uint64_t& v0, uint64_t& v1, int lane, bool desc0, bool desc1) {
    if (J == 1) {
        const uint64_t hi = max(v0, v1), lo = min(v0, v1);
        v0 = desc0 ? hi : lo;
        v1 = desc0 ? lo : hi;
    } else {
        const int lj = J >> 1;
        const bool first = (lane & lj) == 0;
        const uint64_t o0 = shfl_xor_u64(v0, lj), o1 = shfl_xor_u64(v1, lj);
        v0 = (desc0 == first) ? max(v0, o0) : min(v0, o0);
        v1 = (desc1 == first) ? max(v1, o1) : min(v1, o1);
    }
}
// bitonic merge of a bitonic 64-key sequence into descending order
__device__ __forceinline__ void warp64_merge_desc(uint64_t& v0, uint64_t& v1, int lane) {
    warp64_layer<32>(v0, v1, lane, true, true);
    warp64_layer<16>(v0, v1, lane, true, true);
    warp64_layer<8>(v0, v1, lane, true, true);
    warp64_layer<4>(v0, v1, lane, true, true);
    warp64_layer<2>(v0, v1, lane, true, true);
    warp64_layer<1>(v0, v1, lane, true, true);
}
// full descending sort of 64 keys
__device__ __forceinline__ void warp64_sort_desc(uint64_t& v0, uint64_t& v1, int lane) {
    const int i0 = 2 * lane;
#define LRX_L(K, J) warp64_layer<J>(v0, v1, lane, ((i0 & K) == 0), (((i0 + 1) & K) == 0))
    LRX_L(2, 1);
    LRX_L(4, 2); LRX_L(4, 1);
    LRX_L(8, 4); LRX_L(8, 2); LRX_L(8, 1);
    LRX_L(16, 8); LRX_L(16, 4); LRX_L(16, 2); LRX_L(16, 1);
    LRX_L(32, 16); LRX_L(32, 8); LRX_L(32, 4); LRX_L(32, 2); LRX_L(32, 1);
#undef LRX_L
    warp64_merge_desc(v0, v1, lane);
}

template <int NQ>
__device__ __forceinline__ void scan_prune(uint64_t* keys, int* count, uint32_t* tau, int width,
                                           int tid, unsigned int* tau_g) {
    constexpr int cap = scan_cap(NQ);
    int nmax = width;
#pragma unroll
    for (int q = 0; q < NQ; ++q) nmax = max(nmax, count[q]);
    if (width == 64 && nmax <= 256) {
        // fast path (the default list width, pruned at the soft cap): two warps per query, each
        // sorts two 64-key quarters in registers; the best 64 of two descending runs A, B are the
        // bitonic sequence max(A[i], B[63 - i]), sorted by one bitonic merge -- once inside the
        // warp (B reversed by a shuffle), once across the two warps through shared memory.  Four
        // queries at a time (8 warps): a pass of 5..8 queries takes two rounds.
        const int lane = tid & 31, warp = tid >> 5;
#pragma unroll 1
        for (int qb = 0; qb < NQ; qb += 4) {
        const int q = qb + (warp & 3), half = warp >> 2;     // 8 warps: (query, half)
        uint64_t* kq = keys + q * cap;
        const bool active = q < NQ;
        const int n = active ? count[q] : 0;
        uint64_t v0 = 0ull, v1 = 0ull;
        if (active) {
            const int i0 = half * 128 + 2 * lane;
            v0 = (i0 < n) ? kq[i0] : 0ull;
            v1 = (i0 + 1 < n) ? kq[i0 + 1] : 0ull;
            uint64_t w0 = (i0 + 64 < n) ? kq[i0 + 64] : 0ull;
            uint64_t w1 = (i0 + 65 < n) ? kq[i0 + 65] : 0ull;
            warp64_sort_desc(v0, v1, lane);
            warp64_sort_desc(w0, w1, lane);
            // B[63 - 2l] and B[62 - 2l] live in lane 31 - l as its second and first key
            const uint64_t r0 = __shfl_sync(0xffffffffu, w1, 31 - lane);
            const uint64_t r1 = __shfl_sync(0xffffffffu, w0, 31 - lane);
            v0 = max(v0, r0);
            v1 = max(v1, r1);
            warp64_merge_desc(v0, v1, lane);
        }
        __syncthreads();                                     // all reads of keys done
        if (active && half == 1) {
            kq[64 + 2 * lane] = v0;
            kq[64 + 2 * lane + 1] = v1;
        }
        __syncthreads();
        if (active && half == 0) {
            const uint64_t* other = kq + 64;
            v0 = max(v0, other[63 - 2 * lane]);
            v1 = max(v1, other[62 - 2 * lane]);
            warp64_merge_desc(v0, v1, lane);
            kq[2 * lane] = v0;
            kq[2 * lane + 1] = v1;
        }
        __syncthreads();
        }
    } else {
        // general path (wider lists): sort only as many slots as are in use (power of two >= the
        // fullest buffer, >= width; unused ones padded with the empty key), all NQ buffers at once.
        // Bitonic sort with the 64-key stages in registers: chunks of 64 are sorted by one warp
        // each (alternating direction), and of every later merge only the steps at distance >= 64
        // go through shared memory -- 10 block-wide steps for 1024 keys instead of 55.
        const int n2 = min(cap, next_pow2(nmax));
#pragma unroll
        for (int q = 0; q < NQ; ++q) {
            const int n = count[q];
            for (int i = tid; i < n2; i += kScanThreads)
                if (i >= n) keys[q * cap + i] = 0ull;
        }
        __syncthreads();
        if (n2 < 128) {
            block_bitonic_sort_desc<uint64_t>(keys, n2, NQ, cap, tid, kScanThreads);
        } else {
            const int lane = tid & 31, warp = tid >> 5;
            const int chunks = n2 >> 6, total = chunks * NQ;
            // one pass over the 64-key chunks: sort (first = true) or bitonic-merge them, written
            // back descending when the chunk lies in a descending block of size k, else ascending
            auto chunk_pass = [&](int k, bool first) {
                for (int c = warp; c < total; c += kScanThreads / 32) {
                    const int q = c / chunks, ch = c - q * chunks;
                    uint64_t* kc = keys + q * cap + ch * 64;
                    uint64_t v0 = kc[2 * lane], v1 = kc[2 * lane + 1];
                    if (first) warp64_sort_desc(v0, v1, lane); else warp64_merge_desc(v0, v1, lane);
                    const bool desc = ((ch * 64) & k) == 0;
                    __syncwarp();
                    kc[desc ? 2 * lane : 63 - 2 * lane] = v0;
                    kc[desc ? 2 * lane + 1 : 62 - 2 * lane] = v1;
                }
                __syncthreads();
            };
            chunk_pass(64, true);
            const int half = n2 >> 1, lh = 31 - __clz(half);
            for (int k = 128; k <= n2; k <<= 1) {
                for (int j = k >> 1; j >= 64; j >>= 1) {
                    for (int t = tid; t < half * NQ; t += kScanThreads) {
                        const int q = t >> lh, u = t & (half - 1);
                        const int i = ((u & ~(j - 1)) << 1) | (u & (j - 1));
                        const int p = i | j;
                        uint64_t* kk = keys + q * cap;
                        const uint64_t a = kk[i], b = kk[p];
                        const bool desc = ((i & k) == 0);
                        if (desc ? (a < b) : (a > b)) { kk[i] = b; kk[p] = a; }
                    }
                    __syncthreads();
                }
                chunk_pass(k, false);
            }
        }
    }
    if (tid < NQ) {
        const int c = min(count[tid], width);
        count[tid] = c;
        if (c == width) {
            // `width` rows of this CTA reach this score: no row below it, anywhere, can be among
            // the best `width` -- share it with every CTA of the grid (threshold warm-up once
            // per grid instead of once per CTA)
            const uint32_t t = max(tau[tid], (uint32_t)(keys[tid * cap + width - 1] >> 32));
            tau[tid] = t;
            atomicMax(tau_g + tid, t);
        }
    }
    __syncthreads();
}

template <int NQ>
__global__ void __launch_bounds__(kScanThreads, 2)          // <= 128 registers: see kScanThreads
dense_scan_kernel(const unsigned char* __restrict__ x, int64_t n_rows,
                  const __half* __restrict__ q, int n_q, int width,
                  uint64_t* __restrict__ part /* [grid][NQ][width] */,
                  unsigned int* __restrict__ tau_g /* [4] shared thresholds, zero at launch */) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    ScanSmem& sm = *reinterpret_cast<ScanSmem*>(smem_raw);
    uint64_t* keys = sm.keys;

    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int warp = tid >> 5;

    // width <= 128: prune at 256 entries; wider lists keep the full buffer
    constexpr int cap = scan_cap(NQ);
    const int soft_cap = (2 * width <= kSoftCap) ? kSoftCap : cap;
    // Tiles are static, blockIdx + i * grid: at any moment the grid reads one contiguous ~7 MB
    // window of the matrix.  (Measured: claiming tiles from a grid-wide counter
    // costs 25 % -- one contended atomic per 48 KB -- and re-filling a stage BEFORE the tile's
    // per-row tests instead of after the closing barrier costs 30 %; 32-row tiles cost 50 %; a
    // variant without the k split -- 8 rows per warp over the whole k, half of each MMA redundant,
    // one barrier per tile, no partial sums -- measures the same but needs 122 registers, which
    // leaves no margin for the BM25 CTA on the same SM.)
    const int n_tiles = (int)((n_rows + kTileRows - 1) / kTileRows);

    if (tid == 0) {
        for (int s = 0; s < kStages; ++s) mbar_init(&sm.full[s], 1);
        fence_barrier_init();
    }
    if (tid < 8) {
        sm.count[tid] = 0;
        sm.tau[tid] = 0u;   // ordinal 0: every finite score passes
    }
    __syncthreads();

    auto issue = [&](int tile, int s) {                      // thread 0 only
        sm.tile_of[s] = tile;
        if (tile >= n_tiles) return;
        const int64_t row0 = (int64_t)tile * kTileRows;
        const int rows = (int)min((int64_t)kTileRows, n_rows - row0);
        const uint32_t bytes = (uint32_t)rows * kRowBytes;
        mbar_arrive_expect_tx(&sm.full[s], bytes);
        bulk_g2s_hint(sm.ring[s], x + row0 * kRowBytes, bytes, &sm.full[s], l2_policy_evict_first());
    };
    int next_tile = (int)blockIdx.x + kStages * (int)gridDim.x;   // thread 0: the next tile to load
    if (tid == 0) {
        for (int s = 0; s < kStages; ++s) issue((int)blockIdx.x + s * (int)gridDim.x, s);
    }
    __syncthreads();                                         // tile_of[] visible

    // ---- scoring on the tensor cores (mma.sync m16n8k16, fp16 x fp16 -> fp32): a tile is four
    //      16-row blocks x two 192-column halves, one (block, half) per warp.  The 8 "n"
    //      columns are the <= 4 queries plus zero padding.  Lane (g = lane / 4, t = lane % 4) reads
    //      16 contiguous bytes of rows g and g + 8 per 32-column chunk -- two MMAs' worth -- and
    //      holds the query's halves at the SAME columns, so A and B agree on a (permuted) k order.
    const int g = lane >> 2, t = lane & 3;
    const int mblk = warp & 3, kh = (warp >> 2) & 1;
    constexpr bool mma_warp = true;
    uint32_t qb[6][4];                                           // query g, chunks 6*kh .. 6*kh + 5
#pragma unroll
    for (int j = 0; j < 6; ++j) {
        const uint4 v = (g < n_q && mma_warp)
            ? *reinterpret_cast<const uint4*>(q + (size_t)g * kDim + (6 * kh + j) * 32 + 8 * t)
            : make_uint4(0u, 0u, 0u, 0u);
        qb[j][0] = v.x; qb[j][1] = v.y; qb[j][2] = v.z; qb[j][3] = v.w;
    }
    const uint32_t a_off = (uint32_t)((mblk * 16 + g) * kRowBytes + (6 * kh) * 64 + 16 * t);

    for (int it = 0;; ++it) {
        const int s = it % kStages;
        const uint32_t parity = (uint32_t)((it / kStages) & 1);
        const int tile = sm.tile_of[s];
        if (tile >= n_tiles) break;                          // a CTA's tiles come in increasing order
        const int64_t row0 = (int64_t)tile * kTileRows;
        const int rows = (int)min((int64_t)kTileRows, n_rows - row0);

        mbar_wait(&sm.full[s], parity);

        if (mma_warp) {
            float c0[4] = {0.f, 0.f, 0.f, 0.f}, c1[4] = {0.f, 0.f, 0.f, 0.f};   // two accumulation chains
            const unsigned char* base = sm.ring[s] + a_off;
            uint4 xa[6], xb[6];
#pragma unroll
            for (int j = 0; j < 6; ++j) {
                xa[j] = *reinterpret_cast<const uint4*>(base + j * 64);                  // row g
                xb[j] = *reinterpret_cast<const uint4*>(base + 8 * kRowBytes + j * 64);  // row g + 8
            }
#pragma unroll
            for (int j = 0; j < 6; ++j) {
                asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 "
                             "{%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                             : "+f"(c0[0]), "+f"(c0[1]), "+f"(c0[2]), "+f"(c0[3])
                             : "r"(xa[j].x), "r"(xb[j].x), "r"(xa[j].y), "r"(xb[j].y),
                               "r"(qb[j][0]), "r"(qb[j][1]));
                asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 "
                             "{%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                             : "+f"(c1[0]), "+f"(c1[1]), "+f"(c1[2]), "+f"(c1[3])
                             : "r"(xa[j].z), "r"(xb[j].z), "r"(xa[j].w), "r"(xb[j].w),
                               "r"(qb[j][2]), "r"(qb[j][3]));
            }
            // lane t holds queries 2t, 2t + 1 of rows g and g + 8; columns >= NQ are padding
            if (2 * t < NQ) {
                *reinterpret_cast<float2*>(&sm.part[kh][mblk * 16 + g][2 * t]) =
                    make_float2(c0[0] + c1[0], c0[1] + c1[1]);
                *reinterpret_cast<float2*>(&sm.part[kh][mblk * 16 + g + 8][2 * t]) =
                    make_float2(c0[2] + c1[2], c0[3] + c1[3]);
            }
        }
        __syncthreads();                       // partial scores visible

        // ---- one thread per (row, query): sum of the two halves, threshold test, rare append to
        //      the shared buffer
#pragma unroll
        for (int i = tid; i < kTileRows * NQ; i += kScanThreads) {
            const int row_in_tile = i / NQ, qi = i % NQ;
            const float sc = sm.part[0][row_in_tile][qi] + sm.part[1][row_in_tile][qi];
            if (row_in_tile < rows && qi < n_q) {
                const uint32_t o = f32_ord(sc);
                if (o >= sm.tau[qi]) {
                    const int pos = atomicAdd(&sm.count[qi], 1);
                    keys[qi * cap + pos] =
                        ((uint64_t)o << 32) | (uint32_t)(~(uint32_t)(row0 + row_in_tile));
                }
            }
        }
        // ---- block barrier: partial sums consumed, pruning decided uniformly
        bool need = false;
#pragma unroll
        for (int qi = 0; qi < NQ; ++qi) need |= (sm.count[qi] > soft_cap - kTileRows);
        const int any = __syncthreads_or(need ? 1 : 0);
        if (tid == 0) {                        // re-fill the stage with the CTA's next tile
            issue(next_tile, s);
            next_tile += (int)gridDim.x;
        }
        if (any) scan_prune<NQ>(keys, sm.count, sm.tau, width, tid, tau_g);
        else if (tid < NQ) {
            // pick up thresholds published by other CTAs (read by the next tile's tests: the
            // barrier of the next iteration orders it; a stale value is only conservative)
            const uint32_t tg = *(volatile unsigned int*)(tau_g + tid);
            if (tg > sm.tau[tid]) sm.tau[tid] = tg;
        }
    }

    // ---- final: sorted per-CTA lists out
    __syncthreads();
    scan_prune<NQ>(keys, sm.count, sm.tau, width, tid, tau_g);
    for (int i = tid; i < NQ * width; i += kScanThreads) {
        const int qi = i / width;
        const int j = i - qi * width;
        const uint64_t k = (j < sm.count[qi]) ? keys[qi * cap + j] : 0ull;
        part[((size_t)blockIdx.x * NQ + qi) * width + j] = k;
    }
}

// ---------------------------------------------------------------------------
// K2a with an int8 pre-filter (lrx_build_dense_prefilter): the scan streams a SHADOW of the matrix
// -- int8 rows with one fp32 scale per row, 388 bytes per row instead of 768 -- and the exact
// float64 re-score of the merged candidate list reads the fp16 rows as before.  Results stay
// bit-exact: the guard band of the exactness test becomes the rigorous bound
//     |x.q - A(x, q)|  <=  E * |q| + X * |q - qhat| + rounding,
// E = max_r |x_r - xhat_r|, X = max_r |xhat_r| (measured when the shadow is built), qhat the
// two-digit int8 image of the query (q ~= cq * (256 * hi + lo): its error is 1/256 of a row's).
// The band is ~0.0085 for unit vectors instead of 1e-5, so the MERGED list is four times the
// per-CTA list (256 candidates by default; per-CTA lists stay 64 wide and keep the register
// prune), and the bound on every row outside the merged list is the larger of its last key and
// the last key of every per-CTA list that is full (a full list may have dropped rows below it).
//
// dense_scan_q8_kernel: 128-row tiles (48 KB of int8 rows + 512 B of scales per stage, two bulk
// copies on one mbarrier), one 16-row block per warp over the WHOLE k = 384 (no partial sums, one
// block barrier per tile), mma.sync m16n8k32 s8 x s8 -> s32 (exact): the 8 "n" columns are the
// hi and lo digits of the <= 4 queries, so lane (g, t) ends up with both digit sums of query t for
// rows g and g + 8 and tests them against the threshold straight from registers.
// Algorithmic HBM bytes per launch: n_pad * 388.
constexpr int kQ8TileRows = 128;
constexpr int kQ8RowBytes = kDim;                            // 384
constexpr int kQ8TileBytes = kQ8TileRows * kQ8RowBytes;      // 49152

__host__ __device__ inline int64_t q8_pad_rows(int64_t n) {
    return (n + kQ8TileRows - 1) / kQ8TileRows * kQ8TileRows;
}

// The two int8 digits of one query element; `inv` = 127 / max|q| (0 for an all-zero query).  Explicit
// round-to-nearest intrinsics: the scan and the re-score kernel must agree bit for bit on the
// digits (no FMA contraction).
__device__ __forceinline__ void q8_digits(float v, float inv, int& hi, int& lo) {
    const float s = __fmul_rn(v, inv);
    hi = max(-127, min(127, __float2int_rn(s)));
    lo = max(-127, min(127, __float2int_rn(__fmul_rn(__fsub_rn(s, (float)hi), 256.f))));
}
__device__ __forceinline__ float q8_inv(float mx) { return mx > 0.f ? __fdiv_rn(127.f, mx) : 0.f; }
__device__ __forceinline__ float q8_cq(float mx) { return __fmul_rn(mx, 1.0f / 32512.0f); }   // max / (127 * 256)
// the 12 elements lane `lane` holds of a 384-wide fp16 vector: 4 consecutive ones per 128-column third
__device__ __forceinline__ void q8_load12(const __half* __restrict__ v, int lane, float* out) {
    const uint2* p = reinterpret_cast<const uint2*>(v);
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        const uint2 w = p[j * 32 + lane];
        const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&w.x));
        const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&w.y));
        out[4 * j + 0] = a.x; out[4 * j + 1] = a.y; out[4 * j + 2] = b.x; out[4 * j + 3] = b.y;
    }
}
__device__ __forceinline__ float warp_max_abs12(const float* v) {
    float mx = 0.f;
#pragma unroll
    for (int i = 0; i < 12; ++i) mx = fmaxf(mx, fabsf(v[i]));
#pragma unroll
    for (int lb = 16; lb > 0; lb >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, lb));
    return mx;
}
__device__ __forceinline__ double warp_sum_f64(double v) {
#pragma unroll
    for (int lb = 16; lb > 0; lb >>= 1) v += __shfl_xor_sync(0xffffffffu, v, lb);
    return v;
}
__device__ __forceinline__ uint32_t pack_s8x4(int a, int b, int c, int d) {
    return (uint32_t)(a & 0xff) | ((uint32_t)(b & 0xff) << 8) | ((uint32_t)(c & 0xff) << 16) |
           ((uint32_t)(d & 0xff) << 24);
}

// Shadow build: one warp per row.  bounds[0], bounds[1]: ordered images of max_r |x_r - xhat_r|^2 and
// max_r |xhat_r|^2 in float64 (every product below is exact in float64; the sums of 384 squares are
// off by < 1e-13 relative, the host rounds the bounds up).
__global__ void __launch_bounds__(256)
dense_q8_build_kernel(const unsigned char* __restrict__ x, int64_t n_rows, int64_t n_pad,
                      unsigned char* __restrict__ rows8, float* __restrict__ scales,
                      unsigned long long* __restrict__ bounds) {
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (row >= n_pad) return;
    uint32_t* dst = reinterpret_cast<uint32_t*>(rows8 + row * kQ8RowBytes);
    if (row >= n_rows) {                                     // padding of the last tile
#pragma unroll
        for (int j = 0; j < 3; ++j) dst[j * 32 + lane] = 0u;
        if (lane == 0) scales[row] = 0.f;
        return;
    }
    float v[12];
    q8_load12(reinterpret_cast<const __half*>(x + row * kRowBytes), lane, v);
    const float mx = warp_max_abs12(v);
    const float scale = __fdiv_rn(mx, 127.f), inv = q8_inv(mx);
    double err2 = 0.0, n2 = 0.0;
    int xi[12];
#pragma unroll
    for (int i = 0; i < 12; ++i) {
        xi[i] = max(-127, min(127, __float2int_rn(__fmul_rn(v[i], inv))));
        const double xh = (double)scale * (double)xi[i];
        const double e = (double)v[i] - xh;
        err2 = fma(e, e, err2);
        n2 = fma(xh, xh, n2);
    }
    err2 = warp_sum_f64(err2);
    n2 = warp_sum_f64(n2);
    // Odd rows are stored with their 64-byte chunks swapped pairwise (chunk c at 64 * (c ^ 1)): the
    // scan's lanes of rows g and g + 1 then read the two different halves of a 128-byte line for the
    // same logical columns, and a quarter warp's 16-byte loads cover all 32 banks (rows are 384 B =
    // 0 mod 128 apart: unswizzled, every pair of rows collided -- 2 wavefronts per load instead of 1).
    const int sw = (int)(row & 1) << 4;                      // word index ^ 16 = byte offset ^ 64
#pragma unroll
    for (int j = 0; j < 3; ++j)
        dst[(j * 32 + lane) ^ sw] = pack_s8x4(xi[4 * j], xi[4 * j + 1], xi[4 * j + 2], xi[4 * j + 3]);
    if (lane == 0) {
        scales[row] = scale;
        atomicMax(bounds + 0, (unsigned long long)f64_ord(err2));
        atomicMax(bounds + 1, (unsigned long long)f64_ord(n2));
    }
}

template <int NT>
struct ScanQ8Smem {
    unsigned char ring[kStages][kQ8TileBytes];   // 16-byte aligned bulk-copy destinations
    float scale[kStages][kQ8TileRows];
    signed char qd[8 * NT][kDim];                // query digits: row 2 * query (hi), 2 * query + 1 (lo)
    float cq[4 * NT];
    uint64_t full[kStages];
    int tile_of[kStages];
    int count[8];
    uint32_t tau[8];
    uint64_t keys[1];   // [4 * NT][scan_cap(4 * NT)], sized at launch
};

__device__ __forceinline__ void mma_s8(int* c, uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3,
                                       uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k32.row.col.s32.s8.s8.s32 "
                 "{%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+r"(c[0]), "+r"(c[1]), "+r"(c[2]), "+r"(c[3])
                 : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

// NT = 1: up to 4 queries (one 8-column MMA tile of digits, B fragments in registers); NT = 2: 5..8
// queries (two tiles; the second tile's -- and, to stay under 128 registers beside a BM25 CTA, the
// first tile's -- B fragments are re-read from shared memory per chunk), 512 candidate slots each.
template <int NT>
__global__ void __launch_bounds__(kScanThreads, 2)
dense_scan_q8_kernel(const unsigned char* __restrict__ rows8, const float* __restrict__ scales,
                     int64_t n_rows, const __half* __restrict__ q, int n_q, int width,
                     uint64_t* __restrict__ part /* [grid][NQ][width] */,
                     unsigned int* __restrict__ tau_g /* [8] shared thresholds, zero at launch */) {
    constexpr int NQ = 4 * NT;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    ScanQ8Smem<NT>& sm = *reinterpret_cast<ScanQ8Smem<NT>*>(smem_raw);
    uint64_t* keys = sm.keys;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int cap = scan_cap(NQ);
    const int soft_cap = (width <= 64) ? kSoftCap : cap;    // a tile appends up to 128 keys per query
    const int n_tiles = (int)((n_rows + kQ8TileRows - 1) / kQ8TileRows);   // the shadow is padded to whole tiles

    if (tid == 0) {
        for (int s = 0; s < kStages; ++s) mbar_init(&sm.full[s], 1);
        fence_barrier_init();
    }
    if (tid < 8) {
        sm.count[tid] = 0;
        sm.tau[tid] = 0u;
    }
    __syncthreads();
    auto issue = [&](int tile, int s) {                      // thread 0 only
        sm.tile_of[s] = tile;
        if (tile >= n_tiles) return;
        const int64_t row0 = (int64_t)tile * kQ8TileRows;
        mbar_arrive_expect_tx(&sm.full[s], (uint32_t)(kQ8TileBytes + kQ8TileRows * sizeof(float)));
        const uint64_t pol = l2_policy_evict_first();
        bulk_g2s_hint(sm.ring[s], rows8 + row0 * kQ8RowBytes, kQ8TileBytes, &sm.full[s], pol);
        bulk_g2s_hint(sm.scale[s], scales + row0, (uint32_t)(kQ8TileRows * sizeof(float)), &sm.full[s], pol);
    };
    int next_tile = (int)blockIdx.x + kStages * (int)gridDim.x;
    if (tid == 0)
        for (int s = 0; s < kStages; ++s) issue((int)blockIdx.x + s * (int)gridDim.x, s);

    // ---- query digits (every CTA redoes the <= 8 queries: 3 K elements), warp w = query w
    {
        uint32_t* qrow = reinterpret_cast<uint32_t*>(&sm.qd[0][0]);
        if (warp < NQ) {
            uint32_t* hi_row = qrow + (2 * warp) * (kDim / 4);
            uint32_t* lo_row = qrow + (2 * warp + 1) * (kDim / 4);
            if (warp < n_q) {
                float v[12];
                q8_load12(q + (size_t)warp * kDim, lane, v);
                const float mx = warp_max_abs12(v);
                const float inv = q8_inv(mx);
                int hi[12], lo[12];
#pragma unroll
                for (int i = 0; i < 12; ++i) q8_digits(v[i], inv, hi[i], lo[i]);
#pragma unroll
                for (int j = 0; j < 3; ++j) {
                    hi_row[j * 32 + lane] = pack_s8x4(hi[4 * j], hi[4 * j + 1], hi[4 * j + 2], hi[4 * j + 3]);
                    lo_row[j * 32 + lane] = pack_s8x4(lo[4 * j], lo[4 * j + 1], lo[4 * j + 2], lo[4 * j + 3]);
                }
                if (lane == 0) sm.cq[warp] = q8_cq(mx);
            } else {
#pragma unroll
                for (int j = 0; j < 3; ++j) { hi_row[j * 32 + lane] = 0u; lo_row[j * 32 + lane] = 0u; }
                if (lane == 0) sm.cq[warp] = 0.f;
            }
        }
    }
    __syncthreads();                                         // digits, tile_of[] visible

    // B fragments: lane (g, t) holds 16 bytes per 64-column chunk of digit row g at the SAME columns
    // as its A bytes, so A and B agree on a (permuted) k order -- no ldmatrix, no swizzle.
    const int g = lane >> 2, t = lane & 3;
    uint4 qb[NT == 1 ? 6 : 1];
    if (NT == 1) {
#pragma unroll
        for (int j = 0; j < 6; ++j) qb[NT == 1 ? j : 0] = *reinterpret_cast<const uint4*>(&sm.qd[g][j * 64 + 16 * t]);
    }
    float cq[NT];
#pragma unroll
    for (int u = 0; u < NT; ++u) cq[u] = sm.cq[4 * u + t];
    const uint32_t a_off = (uint32_t)((warp * 16 + g) * kQ8RowBytes + 16 * t);

    for (int it = 0;; ++it) {
        const int s = it % kStages;
        const uint32_t parity = (uint32_t)((it / kStages) & 1);
        const int tile = sm.tile_of[s];
        if (tile >= n_tiles) break;
        const int64_t row0 = (int64_t)tile * kQ8TileRows;
        mbar_wait(&sm.full[s], parity);

        int c0[NT][4], c1[NT][4];                            // two accumulation chains per digit tile
#pragma unroll
        for (int u = 0; u < NT; ++u)
#pragma unroll
            for (int i = 0; i < 4; ++i) c0[u][i] = c1[u][i] = 0;
        {
            const unsigned char* base = sm.ring[s] + a_off;
            uint4 xa[6], xb[6];
#pragma unroll
            for (int j = 0; j < 6; ++j) {                    // logical chunk j of an odd row sits at j ^ 1
                xa[j] = *reinterpret_cast<const uint4*>(base + ((j ^ (g & 1)) * 64));                    // row g
                xb[j] = *reinterpret_cast<const uint4*>(base + 8 * kQ8RowBytes + ((j ^ (g & 1)) * 64));  // row g + 8
            }
#pragma unroll
            for (int j = 0; j < 6; ++j) {
#pragma unroll
                for (int u = 0; u < NT; ++u) {
                    const uint4 b = (NT == 1) ? qb[NT == 1 ? j : 0]
                                              : *reinterpret_cast<const uint4*>(&sm.qd[8 * u + g][j * 64 + 16 * t]);
                    mma_s8(c0[u], xa[j].x, xb[j].x, xa[j].y, xb[j].y, b.x, b.y);
                    mma_s8(c1[u], xa[j].z, xb[j].z, xa[j].w, xb[j].w, b.z, b.w);
                }
            }
        }
        // lane (g, t): digit sums (hi, lo) of queries t (and 4 + t) for rows g and g + 8 of the warp's
        // block.  |256 * hi + lo| <= 257 * 384 * 127^2 < 2^31.
#pragma unroll
        for (int u = 0; u < NT; ++u) {
            const int qi = 4 * u + t;
            if (qi < n_q) {
                const int r0 = warp * 16 + g;
                const uint32_t tau = sm.tau[qi];
#pragma unroll
                for (int hrow = 0; hrow < 2; ++hrow) {
                    const int r = r0 + 8 * hrow;
                    const int D = (c0[u][2 * hrow] + c1[u][2 * hrow]) * 256 +
                                  (c0[u][2 * hrow + 1] + c1[u][2 * hrow + 1]);
                    const float sc = __fmul_rn(__fmul_rn(sm.scale[s][r], cq[u]), (float)D);
                    const uint32_t o = f32_ord(sc);
                    if (o >= tau && row0 + r < n_rows) {
                        const int pos = atomicAdd(&sm.count[qi], 1);
                        keys[qi * cap + pos] = ((uint64_t)o << 32) | (uint32_t)(~(uint32_t)(row0 + r));
                    }
                }
            }
        }
        // ---- the one block barrier of a tile: the stage is consumed, the appends are visible, and
        //      pruning is decided uniformly (a thread reads count[] after its own appends, so the
        //      last appender of a query sees its final value; the OR makes every thread agree)
        bool need = false;
#pragma unroll
        for (int qi = 0; qi < NQ; ++qi) need |= (sm.count[qi] > soft_cap - kQ8TileRows);
        const int any = __syncthreads_or(need ? 1 : 0);
        if (tid == 0) {                        // re-fill the stage with the CTA's next tile
            issue(next_tile, s);
            next_tile += (int)gridDim.x;
        }
        if (any) scan_prune<NQ>(keys, sm.count, sm.tau, width, tid, tau_g);
        else if (tid < NQ) {
            // thresholds published by other CTAs; the next tile's tests may still read the old
            // value: a stale threshold is only conservative
            const uint32_t tg = *(volatile unsigned int*)(tau_g + tid);
            if (tg > sm.tau[tid]) sm.tau[tid] = tg;
        }
    }

    __syncthreads();
    scan_prune<NQ>(keys, sm.count, sm.tau, width, tid, tau_g);
    for (int i = tid; i < NQ * width; i += kScanThreads) {
        const int qi = i / width;
        const int j = i - qi * width;
        const uint64_t k = (j < sm.count[qi]) ? keys[qi * cap + j] : 0ull;
        part[((size_t)blockIdx.x * NQ + qi) * width + j] = k;
    }
}

// ---------------------------------------------------------------------------
// Exact float64 inner product of one fp16 row with one fp16 query, by a warp.
__device__ __forceinline__ double warp_exact_dot(const unsigned char* __restrict__ x, int64_t row,
                                                 const __half* __restrict__ qv, int lane) {
    const uint2* rowp = reinterpret_cast<const uint2*>(x + row * kRowBytes);
    const uint2* qp = reinterpret_cast<const uint2*>(qv);
    double acc = 0.0;
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        const uint2 v = rowp[j * 32 + lane];
        const uint2 w = qp[j * 32 + lane];
        const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&v.x));
        const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&v.y));
        const float2 c = __half22float2(*reinterpret_cast<const __half2*>(&w.x));
        const float2 d = __half22float2(*reinterpret_cast<const __half2*>(&w.y));
        acc = fma((double)a.x, (double)c.x, acc);
        acc = fma((double)a.y, (double)c.y, acc);
        acc = fma((double)b.x, (double)d.x, acc);
        acc = fma((double)b.y, (double)d.y, acc);
    }
#pragma unroll
    for (int lb = 16; lb > 0; lb >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, lb);
    return acc;
}

// Merge of the per-CTA lists of one query + exact re-score of the survivors, one CTA per query:
//   merge_lists_block  -> the best `width` fp32-scored keys, in shared memory
//   re-score           each warp takes 4 survivors per pass, all 12 row loads in flight before
//                      the first reduction; exact float64 dot products (order independent)
//   order              rank by counting on (exact score desc, id asc); emit the best K + guard flag
//   lists are `list_width` long, the merged list `width` (>= list_width; longer only behind the int8
//   pre-filter); q8_norm >= 0: the scan scored the int8 shadow, the guard band is computed per query
__global__ void __launch_bounds__(kMergeThreads, 1)
dense_merge_rescore_kernel(const uint64_t* __restrict__ part, int n_lists, int list_stride, int list_width,
                           const unsigned char* __restrict__ x, int64_t n_rows, int64_t id_base,
                           const __half* __restrict__ q, int width, int K, double eps,
                           double q8_err, double q8_norm,
                           double* __restrict__ out_exact, float* __restrict__ out_D,
                           int64_t* __restrict__ out_I, int32_t* __restrict__ out_flag) {
    // dynamic shared memory (merge_smem_bytes): buf [kMergeCap] u64 | keys [width] u128 |
    // sorted [width] u128 | merged [width] u64
    extern __shared__ __align__(128) unsigned char merge_raw[];
    uint64_t* buf = reinterpret_cast<uint64_t*>(merge_raw);
    u128* keys = reinterpret_cast<u128*>(merge_raw + kMergeCap * sizeof(uint64_t));
    u128* sorted = keys + width;
    uint64_t* merged = reinterpret_cast<uint64_t*>(sorted + width);
    __shared__ int s_count, s_overflow;
    __shared__ uint64_t s_bound;
    __shared__ unsigned long long s_full;       // largest last key of a per-CTA list that is full
    __shared__ double s_eps;
    const int qi = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) s_full = 0ull;
    if (warp == 1) {
        // guard band of this query (see dense_scan_q8_kernel): the digits are recomputed with the
        // scan's own operations, the norms in float64
        double e = eps;
        if (q8_norm >= 0.0) {
            float v[12];
            q8_load12(q + (size_t)qi * kDim, lane, v);
            const float mx = warp_max_abs12(v);
            const float inv = q8_inv(mx);
            const double cq = (double)q8_cq(mx);
            double nq = 0.0, ne = 0.0;
#pragma unroll
            for (int i = 0; i < 12; ++i) {
                int hi, lo;
                q8_digits(v[i], inv, hi, lo);
                const double d = (double)v[i] - cq * (double)(256 * hi + lo);
                nq = fma((double)v[i], (double)v[i], nq);
                ne = fma(d, d, ne);
            }
            nq = sqrt(warp_sum_f64(nq));
            ne = sqrt(warp_sum_f64(ne));
            e = (q8_err * nq + q8_norm * ne + 2.0e-7 * q8_norm * (nq + ne)) * (1.0 + 1.0e-6) + 1.0e-12;
        }
        if (lane == 0) s_eps = e;
    }
    merge_lists_block<uint64_t>(part, n_lists, list_stride, qi, list_width, width, buf, merged, &s_count,
                                &s_overflow, &s_bound);
    for (int l = tid; l < n_lists; l += kMergeThreads) {
        const uint64_t last = part[((size_t)qi + (size_t)l * list_stride) * list_width + list_width - 1];
        if (last != 0ull) atomicMax(&s_full, (unsigned long long)last);
    }

    constexpr int kWarps = kMergeThreads / 32;
    for (int j0 = warp * 4; j0 < width; j0 += kWarps * 4) {
        uint64_t kk[4];
        uint2 rv[4][3];
#pragma unroll
        for (int c = 0; c < 4; ++c) kk[c] = (j0 + c < width) ? merged[j0 + c] : 0ull;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const uint2* rowp = reinterpret_cast<const uint2*>(
                x + (int64_t)(kk[c] ? key64_row(kk[c]) : 0u) * kRowBytes);
#pragma unroll
            for (int s = 0; s < 3; ++s)
                rv[c][s] = (kk[c] && n_rows > 0) ? rowp[s * 32 + lane] : make_uint2(0u, 0u);
        }
        const uint2* qp = reinterpret_cast<const uint2*>(q + (size_t)qi * kDim);
        uint2 qv[3];
#pragma unroll
        for (int s = 0; s < 3; ++s) qv[s] = qp[s * 32 + lane];
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
            if (lane == 0 && j0 + c < width)
                keys[j0 + c] = kk[c] ? make_key128(acc, key64_row(kk[c])) : (u128)0;
        }
    }
    for (int j = tid; j < width; j += kMergeThreads) sorted[j] = 0;
    __syncthreads();
    for (int j = tid; j < width; j += kMergeThreads) {
        const u128 key = keys[j];
        if (key != 0) sorted[merge_rank_of<u128>(keys, width, key)] = key;
    }
    __syncthreads();
    for (int j = tid; j < K; j += kMergeThreads) {
        const u128 key = (j < width) ? sorted[j] : (u128)0;
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
    if (tid == 0) {
        int flag = 0;
        // Rows outside the merged list: keys of the per-CTA lists that did not make it (below the
        // merged list's last key, which is non-empty then) and rows a CTA dropped -- by its
        // threshold or by a prune, both only once its list was full, and all below that list's
        // final last key.  Their fast score is <= s_out, hence their exact score <= s_out + eps;
        // they must lose strictly to the K-th exact score.  Neither bound present: every row is
        // in the merged list and the result is exact as it stands.
        const uint64_t last = merged[width - 1];
        const uint64_t out_key = (last > (uint64_t)s_full) ? last : (uint64_t)s_full;
        if (out_key != 0ull) {
            const int kk = (K < width) ? K : width;
            const u128 kth = sorted[kk - 1];
            if (kth == 0 || K > width) {
                flag = 1;
            } else {
                const double s_out = (double)key64_score(out_key);
                flag = (s_out + s_eps < key128_score(kth)) ? 0 : 1;
            }
        }
        out_flag[qi] = flag;
    }
}

// exact scores at given global ids; one warp per (query, id)
__global__ void dense_at_kernel(const unsigned char* __restrict__ x, int64_t n_rows,
                                int64_t id_base, const __half* __restrict__ q,
                                const int64_t* __restrict__ ids, int n, double* __restrict__ out) {
    const int qi = blockIdx.y;
    const int lane = threadIdx.x & 31;
    const int j = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (j >= n) return;
    const int64_t id = ids[(size_t)qi * n + j];
    const int64_t row = id - id_base;
    double e = -INFINITY;
    if (id >= 0 && row >= 0 && row < n_rows) e = warp_exact_dot(x, row, q + (size_t)qi * kDim, lane);
    if (lane == 0) out[(size_t)qi * n + j] = e;
}

// ---------------------------------------------------------------------------
static size_t scan_smem_bytes(int nq) {
    return offsetof(ScanSmem, keys) + (size_t)nq * kCap * sizeof(uint64_t);
}

int dense_scan_grid(const lrx_handle* h) {
    // (tiles of the fp16 scan; the int8 scan's 128-row tiles run on the same grid -- a CTA without a
    // tile of its own emits empty lists)
    const int64_t n_tiles = (h->n_local + kTileRows - 1) / kTileRows;
    return (int)((n_tiles < h->num_sms) ? (n_tiles > 0 ? n_tiles : 1) : h->num_sms);
}

template <int NQ>
static cudaError_t launch_scan(lrx_handle* h, const __half* q, int n_q, int width, uint64_t* part,
                               int grid) {
    std::lock_guard<std::recursive_mutex> attr_guard(attr_mutex());   // the flags below are process-wide
    static bool attr_dev[64] = {false};   // function attributes are per device
    bool& attr = attr_dev[h->device & 63];
    // always the 4-query footprint (133 KB): it is what keeps the grid at ONE CTA per SM.  With the
    // smaller buffers of NQ = 1 / 2 two CTAs fit an SM and the block scheduler pairs them up, leaving
    // half of the SMs -- and of the HBM request streams -- idle (measured: batch 1 over 1 M rows
    // 0.181 ms against 0.124 ms for batch 4).
    const size_t smem = scan_smem_bytes(4);
    if (!attr) {
        cudaError_t e = cudaFuncSetAttribute(dense_scan_kernel<NQ>,
                                             cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        // the SM's L1 / shared-memory split is fixed while a CTA is resident: ask for all of it as
        // shared memory so that a BM25 scan CTA (90 KB) can join this kernel's CTA (133 KB)
        e = cudaFuncSetAttribute(dense_scan_kernel<NQ>, cudaFuncAttributePreferredSharedMemoryCarveout,
                                 cudaSharedmemCarveoutMaxShared);
        if (e != cudaSuccess) return e;
        attr = true;
    }
    // shared thresholds live behind the per-CTA lists in the same workspace
    unsigned int* tau_g = reinterpret_cast<unsigned int*>(part + (size_t)grid * 8 * width);
    cudaError_t e0 = cudaMemsetAsync(tau_g, 0, 8 * sizeof(unsigned int), h->stream);
    if (e0 != cudaSuccess) return e0;
    prof_begin(h, 0);
    dense_scan_kernel<NQ><<<grid, kScanThreads, smem, h->stream>>>(
        (const unsigned char*)h->x, h->n_local, q, n_q, width, part, tau_g);
    prof_end(h, 0);
    h->launches++;
    return cudaGetLastError();
}

// ---- int8 pre-filter
bool dense_q8_applies(const lrx_handle* h, int B, int K, int width) {
    // up to 8 queries per pass (the hi / lo digits of 4 queries fill the 8 columns of one MMA tile;
    // 5..8 queries take two tiles), lists up to 128 wide per CTA -- a widened retry beyond that goes
    // back to the fp16 scan and its 1e-5 band
    if (h->q8 == nullptr || h->n_local <= 0 || B > 8) return false;
    if (K <= 64) return width <= 128;
    // deep lists: only at the default width (a retry goes to the fp16 scan) and on shards large
    // enough that every CTA's share of the best K is far below its 64-entry list
    return width == dense_default_width(K) && width <= 256 && h->n_local >= 32768;
}

int64_t dense_q8_bytes(int64_t n_local) {
    const int64_t n_pad = q8_pad_rows(n_local);
    return n_pad * (kQ8RowBytes + (int64_t)sizeof(float));
}

// quantise h->x into buf (rows, then scales), bounds_out = {E, X} rounded up
cudaError_t launch_dense_q8_build(lrx_handle* h, void* buf, double* bounds_out) {
    const int64_t n_pad = q8_pad_rows(h->n_local);
    bounds_out[0] = bounds_out[1] = 0.0;
    if (n_pad == 0) return cudaSuccess;
    unsigned long long* dev_bounds = nullptr;
    cudaError_t e = cudaMalloc((void**)&dev_bounds, 2 * sizeof(unsigned long long));
    if (e != cudaSuccess) return e;
    e = cudaMemsetAsync(dev_bounds, 0, 2 * sizeof(unsigned long long), h->stream);
    unsigned char* rows8 = (unsigned char*)buf;
    float* scales = (float*)(rows8 + n_pad * kQ8RowBytes);
    if (e == cudaSuccess) {
        dense_q8_build_kernel<<<(unsigned)((n_pad + 7) / 8), 256, 0, h->stream>>>(
            (const unsigned char*)h->x, h->n_local, n_pad, rows8, scales, dev_bounds);
        h->launches++;
        e = cudaGetLastError();
    }
    unsigned long long hb[2] = {0ull, 0ull};
    if (e == cudaSuccess)
        e = cudaMemcpyAsync(hb, dev_bounds, sizeof(hb), cudaMemcpyDeviceToHost, h->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    cudaFree(dev_bounds);
    if (e != cudaSuccess) return e;
    for (int i = 0; i < 2; ++i) {
        double sq = 0.0;
        if (hb[i] != 0ull) {                                 // inverse of f64_ord for a non-negative value
            const unsigned long long u = hb[i] & 0x7fffffffffffffffull;
            memcpy(&sq, &u, sizeof(sq));
        }
        bounds_out[i] = sqrt(sq) * (1.0 + 1.0e-9);
    }
    return cudaSuccess;
}

template <int NT>
static cudaError_t launch_scan_q8(lrx_handle* h, const __half* q, int n_q, int width, uint64_t* part,
                                  int grid) {
    std::lock_guard<std::recursive_mutex> attr_guard(attr_mutex());
    static bool attr_dev[64] = {false};
    bool& attr = attr_dev[h->device & 63];
    // about the footprint of the fp16 scan (135 / 138 KB): one CTA per SM, a BM25 scan CTA fits beside it
    const size_t smem = offsetof(ScanQ8Smem<NT>, keys) + (size_t)4 * kCap * sizeof(uint64_t);
    if (!attr) {
        cudaError_t e = cudaFuncSetAttribute(dense_scan_q8_kernel<NT>,
                                             cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        e = cudaFuncSetAttribute(dense_scan_q8_kernel<NT>, cudaFuncAttributePreferredSharedMemoryCarveout,
                                 cudaSharedmemCarveoutMaxShared);
        if (e != cudaSuccess) return e;
        attr = true;
    }
    unsigned int* tau_g = reinterpret_cast<unsigned int*>(part + (size_t)grid * 8 * width);
    cudaError_t e0 = cudaMemsetAsync(tau_g, 0, 8 * sizeof(unsigned int), h->stream);
    if (e0 != cudaSuccess) return e0;
    const int64_t n_pad = q8_pad_rows(h->n_local);
    const unsigned char* rows8 = (const unsigned char*)h->q8;
    const float* scales = (const float*)(rows8 + n_pad * kQ8RowBytes);
    prof_begin(h, 0);
    dense_scan_q8_kernel<NT><<<grid, kScanThreads, smem, h->stream>>>(rows8, scales, h->n_local, q, n_q, width,
                                                                       part, tau_g);
    prof_end(h, 0);
    h->launches++;
    return cudaGetLastError();
}

int dense_default_width(int K) {
    int w = next_pow2(K + 32);
    if (w < 64) w = 64;
    return w;
}

cudaError_t launch_dense_topk(lrx_handle* h, const void* qv, int B, int K, int width,
                              double* exact, float* D, int64_t* I, int32_t* flags) {
    const int grid = dense_scan_grid(h);
    cudaError_t e;
    // per-CTA lists for up to 8 queries per pass
    e = ensure_ws(h, &h->ws_dense_part, &h->ws_dense_part_bytes,
                  (size_t)grid * 8 * width * sizeof(uint64_t) + 64);
    if (e != cudaSuccess) return e;
    std::lock_guard<std::recursive_mutex> attr_guard(attr_mutex());   // the flags below are process-wide
    static bool attr_dev[64] = {false};   // function attributes are per device
    bool& attr = attr_dev[h->device & 63];
    if (!attr) {
        e = cudaFuncSetAttribute(dense_merge_rescore_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)merge_smem_bytes(kMaxMerged));
        if (e != cudaSuccess) return e;
        attr = true;
    }
    uint64_t* part = (uint64_t*)h->ws_dense_part;
    const __half* q = (const __half*)qv;
    if (dense_q8_applies(h, B, K, width)) {
        // int8 pre-filter: short per-CTA lists, a long merged list.  K <= 64: lists `width` long (64,
        // 128 on a retry), merged list four times that.  Deeper (config C5, K = 200): lists of 64 --
        // a CTA holds 1 / 148 of the rows and ~K / 148 of the best K; a CTA that holds more fills its
        // list, which the guard sees -- and a merged list of 2048 (the band needs ~10 K candidates).
        const int list_width = (K <= 64) ? width : 64;
        const int merged_width = (K <= 64) ? ((4 * width < kMaxWidth) ? 4 * width : kMaxWidth) : kMaxMerged;
        e = (B > 4) ? launch_scan_q8<2>(h, q, B, list_width, part, grid)
                    : launch_scan_q8<1>(h, q, B, list_width, part, grid);
        if (e != cudaSuccess) return e;
        dense_merge_rescore_kernel<<<B, kMergeThreads, merge_smem_bytes(merged_width), h->stream>>>(
            part, grid, (B > 4) ? 8 : 4, list_width, (const unsigned char*)h->x, h->n_local, h->id_base, q, merged_width, K,
            kDenseEps, h->q8_err, h->q8_norm, exact, D, I, flags);
        h->launches++;
        return cudaGetLastError();
    }
    // One matrix pass serves up to 8 queries: the MMA tile has 8 columns either way (SURVEY 8(d)
    // budgets ONE read of the matrix per batch).  5..8 queries take the 8-query instantiation (512
    // candidate slots per query, lists up to 256 wide); up to 4 the 4-query one -- the 1- and 2-query
    // instantiations measured SLOWER (batch 1 over 1 M rows: 0.179 ms against 0.124 ms for batch 4).
    const int per_pass = (B > 4 && width <= 256) ? 8 : 4;
    for (int b0 = 0; b0 < B; b0 += per_pass) {
        const int nq = (B - b0 < per_pass) ? (B - b0) : per_pass;
        const int NQ = nq > 4 ? 8 : 4;
        e = (NQ == 8) ? launch_scan<8>(h, q + (size_t)b0 * kDim, nq, width, part, grid)
                      : launch_scan<4>(h, q + (size_t)b0 * kDim, nq, width, part, grid);
        if (e != cudaSuccess) return e;
        // list l of query qi of this pass: part[(l * NQ + qi) * width]
        dense_merge_rescore_kernel<<<nq, kMergeThreads, merge_smem_bytes(width), h->stream>>>(
            part, grid, NQ, width, (const unsigned char*)h->x, h->n_local, h->id_base,
            q + (size_t)b0 * kDim, width, K, kDenseEps, 0.0, -1.0, exact + (size_t)b0 * K, D + (size_t)b0 * K,
            I + (size_t)b0 * K, flags + b0);
        h->launches++;
        e = cudaGetLastError();
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

cudaError_t launch_dense_at(lrx_handle* h, const void* q, int B, const int64_t* ids, int n,
                            double* out) {
    if (n <= 0 || B <= 0) return cudaSuccess;
    dim3 grid((n + 3) / 4, B);
    dense_at_kernel<<<grid, 128, 0, h->stream>>>((const unsigned char*)h->x, h->n_local,
                                                 h->id_base, (const __half*)q, ids, n, out);
    h->launches++;
    return cudaGetLastError();
}

}  // namespace lrx
