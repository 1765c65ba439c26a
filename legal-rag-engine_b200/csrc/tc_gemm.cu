// K1 GEMMs: out[M,N] = epilogue(A[M,K] * W[N,K]^T) on the 5th-gen tensor cores.
//
// Replaces the torch-CPU sgemm calls inside SentenceTransformer.encode
// (reference: src/retrieval/retrieval_engine.py:61, create_vector_store.py:45): the six
// BertLayer projections of all-MiniLM-L6-v2.  fp16 operands, fp32 accumulation in TMEM.
//
// Persistent CTAs, each walking 128 x BN output tiles, 320 threads (kGemmThreads), warp-specialised:
//   warp 8   TMA producer: 2-D tiled loads (SWIZZLE_128B) of the A tile (128 x 64 halves)
//            and the W tile (BN x 64 halves) into a shared-memory ring (GemmCfg::kStages deep),
//            completion counted on full[] mbarriers, slots recycled through empty[] mbarriers;
//            for K = 384 on the big plans the CTA's A tile stays resident (ARES) and clusters
//            of 2 multicast W (CS).
//   warp 9   allocates TMEM and issues tcgen05.mma (UMMA 128 x N x 16, cta_group::1) from ONE
//            lane: 4 k-steps per stage; tcgen05.commit releases the stage / publishes the
//            accumulator.
//   warps 0-7 epilogue (kEpiWarps): thread = output row (TMEM lane 32 (warp & 3) + lane) x column
//            half (warp >> 2): tcgen05.ld 32 columns at a time, then
//              EPI_BIAS        + bias                              -> fp16   (QKV projection)
//              EPI_BIAS_GELU   + bias, GELU (fitted tanh form)     -> fp16   (FFN up)
//              EPI_BIAS_RES_LN + bias + residual, LayerNorm(384)   -> fp16   (attention output /
//                              FFN down; BN = 384 = the whole row, each half's sums meet in
//                              shared memory; the pre-norm row is parked in TMEM between
//                              the three passes with tcgen05.st)
//              EPI_F32         raw fp32 accumulators                         (tests / K2b)
//
// Roofline: tensor pipe.  flops per launch = 2*M*N*K.
#include <cstdio>

#include "handle.h"
#include "tc.cuh"

namespace lrx {

constexpr int kBM = 128;
constexpr int kGemmCluster = 2;                   // cluster size along M when clusters apply (gemm_plan)
constexpr int kBK = 64;
constexpr int kEpiWarps = 8;                      // two per TMEM lane quarter: column halves
constexpr int kGemmThreads = (kEpiWarps + 2) * 32;   // + TMA producer warp + MMA warp
constexpr int kABytes = kBM * kBK * 2;   // 16 KB

struct GemmEpi {
    const float* bias;        // [N]
    const __half* residual;   // [M, ld_res]      (LN epilogue)
    const float* gamma;       // [N]
    const float* beta;        // [N]
    void* out;                // fp16 [M, ld_out] (fp32 for EPI_F32)
    int ld_out, ld_res;
    int M;                    // valid rows
    float eps;
    int pdl_early;            // let the next kernel be scheduled at this kernel's start (else at its end)
};

constexpr int kAResKB = 6;                        // k-blocks of a RESIDENT A tile (K = 384)

// ARES: the 128 x 384 A tile of the CTA's row block stays in shared memory (96 KB) while the CTA
// walks the n-blocks, so only W streams through the ring (K == 384 GEMMs); otherwise A and W
// both stream (K = 1536).
// CS: cluster size along M.  The CS CTAs of a cluster need the same W tile at the same time: each
// loads 1/CS of it and MULTICASTS it to all, so L2 sees one request per cluster instead of one per
// CTA (the W tiles are the hot spot: every CTA of the grid reads the same few hundred lines).
template <int BN, bool ARES, int CS>
struct GemmCfg {
    static constexpr int kBoxB = (CS > 1) ? BN / CS : ((BN > 256) ? 128 : BN);   // rows per TMA box of W
    static constexpr int kBBytes = BN * kBK * 2;
    static constexpr int kStageBytes = (ARES ? 0 : kABytes) + kBBytes;
    static constexpr int kResBytes = ARES ? kAResKB * kABytes : 0;
    // epilogue side: bias (whole vector, N <= 1536) / gamma / beta / LayerNorm partial sums, and one 2 KB staging
    // tile (32 rows x 32 halves, SWIZZLE_64B) per epilogue warp for the TMA stores / residual loads
    static constexpr int kParamBytes = 1536 * 4 + 2 * 384 * 4 + 2 * 2 * 128 * 4;
    // one staging tile per epilogue warp, two for the bias / GELU epilogues (BN <= 256); the
    // LayerNorm GEMMs (BN = 384) need the space for a third ring stage
    static constexpr int kIoTile = (BN <= 256) ? 4096 : 2048;
    static constexpr int kIoBytes = kEpiWarps * kIoTile + 2048 /*align*/;
    static constexpr int kBarBytes = 512;
    static constexpr int kBudget = 224 * 1024 - 1024 - kBarBytes - kParamBytes - kIoBytes;
    static constexpr int kStagesRaw = (kBudget - kResBytes) / kStageBytes;
    static constexpr int kStages = kStagesRaw > 8 ? 8 : kStagesRaw;
    static constexpr int kAcc = (2 * BN <= 512) ? 2 : 1;              // TMEM accumulator buffers
    static constexpr int kTmemCols = (kAcc * BN <= 128) ? 128 : (kAcc * BN <= 256 ? 256 : 512);
    static constexpr size_t kSmem = (size_t)kResBytes + (size_t)kStages * kStageBytes + 1024 /*align*/ +
                                    kBarBytes + kParamBytes + kIoBytes;
};

// GELU(x) = x * Phi(x) (exact-erf form), evaluated as 0.5 x (1 + tanh(u(x))) with
//   u(x) = x (c1 + c3 x^2 + c5 x^4),  x^2 clamped to 64,
// the coefficients fitted (minimax over |x| <= 8, tools/gelu_fit.py) to the ERF form, not the usual
// "tanh approximation" constants: |0.5 x (1 + tanh u) - x Phi(x)| <= 2.6e-5 with an exact tanh (the
// textbook constants: 4.7e-4).  Past |x| = 8 tanh(u) is +-1 in any precision and the result is x or
// 0.  Two elements at a time so that the hyperbolic tangent is ONE packed tanh.approx.f16x2 (absolute
// error 2^-11: 2.4e-4 |x| on the result, the size of the fp16 rounding of the output): 9 FP32
// instructions + half a MUFU per element.  The first form (Abramowitz-Stegun 7.1.26: a reciprocal, a
// packed exponential and a degree-5 polynomial, 16 FP32 + 1.25 MUFU per element) made the FFN-up
// epilogue 1.9x as long as the MMAs of its tile -- the kernel ran at 29 % tensor-pipe activity.
__device__ __forceinline__ float2 gelu2(float x0, float x1) {
    constexpr float c1 = 7.97507884e-01f, c3 = 3.70056460e-02f, c5 = -3.51516789e-04f;
    const float s0 = fminf(x0 * x0, 64.0f), s1 = fminf(x1 * x1, 64.0f);
    const float u0 = x0 * fmaf(s0, fmaf(s0, c5, c3), c1);
    const float u1 = x1 * fmaf(s1, fmaf(s1, c5, c3), c1);
    const __half2 arg = __floats2half2_rn(u0, u1);
    uint32_t th;
    asm("tanh.approx.f16x2 %0, %1;" : "=r"(th) : "r"(*reinterpret_cast<const uint32_t*>(&arg)));
    const float2 t = __half22float2(*reinterpret_cast<const __half2*>(&th));
    const float h0 = 0.5f * x0, h1 = 0.5f * x1;
    return make_float2(fmaf(h0, t.x, h0), fmaf(h1, t.y, h1));
}
__device__ __forceinline__ void epi_bar() { asm volatile("bar.sync 1, 256;" ::: "memory"); }

// Staging tile of one epilogue warp: 32 rows x 32 halves (64 B per row) in the SWIZZLE_64B layout
// of the TMA tensor maps: 16-byte chunk j of row r sits at chunk (j ^ ((r >> 1) & 3)).  Lane r
// owns row r, so every quarter-warp touches 8 distinct bank groups (conflict-free).
__device__ __forceinline__ void stage_put_row(unsigned char* tile, int r, const float (&v)[32]) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const __half2 h0 = __floats2half2_rn(v[8 * j + 0], v[8 * j + 1]);
        const __half2 h1 = __floats2half2_rn(v[8 * j + 2], v[8 * j + 3]);
        const __half2 h2 = __floats2half2_rn(v[8 * j + 4], v[8 * j + 5]);
        const __half2 h3 = __floats2half2_rn(v[8 * j + 6], v[8 * j + 7]);
        uint4 u;
        u.x = *reinterpret_cast<const uint32_t*>(&h0);
        u.y = *reinterpret_cast<const uint32_t*>(&h1);
        u.z = *reinterpret_cast<const uint32_t*>(&h2);
        u.w = *reinterpret_cast<const uint32_t*>(&h3);
        *reinterpret_cast<uint4*>(tile + r * 64 + ((j ^ ((r >> 1) & 3)) << 4)) = u;
    }
}
__device__ __forceinline__ void stage_get_row(const unsigned char* tile, int r, uint4 (&dst)[4]) {
#pragma unroll
    for (int j = 0; j < 4; ++j)
        dst[j] = *reinterpret_cast<const uint4*>(tile + r * 64 + ((j ^ ((r >> 1) & 3)) << 4));
}
// whole warp: publish the staged tile with one TMA store (rows beyond the tensor are clipped)
__device__ __forceinline__ void stage_store(const CUtensorMap* m, int col, int row, const unsigned char* tile,
                                            int lane) {
    fence_proxy_async();            // generic-proxy writes -> visible to the async proxy
    __syncwarp();
    if (lane == 0) {
        tma_store_2d(m, col, row, tile);
        bulk_commit();
    }
}
// whole warp: every store has read its tile / every store but the latest has
__device__ __forceinline__ void stage_acquire(int lane) {
    if (lane == 0) bulk_wait_read();
    __syncwarp();
}
__device__ __forceinline__ void stage_acquire1(int lane) {
    if (lane == 0) bulk_wait_read1();
    __syncwarp();
}

// Persistent: CTA c owns output tiles c, c + grid, ... (n-block fastest, so CTAs running side by
// side share the A rows in L2).  The shared-memory ring flows across tiles; with two TMEM
// accumulators (BN <= 256) the epilogue of tile i overlaps the MMAs of tile i + 1.
template <int BN, int EPI, bool ARES, int CS>
__global__ void __launch_bounds__(kGemmThreads, 1)
tc_gemm_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_b,
               const __grid_constant__ CUtensorMap tma_out, const __grid_constant__ CUtensorMap tma_res,
               int num_k_blocks, int m_tiles, int n_tiles, GemmEpi ep) {
    using Cfg = GemmCfg<BN, ARES, CS>;
    constexpr uint16_t kMask = (uint16_t)((1u << CS) - 1u);
    const uint32_t crank = (CS > 1) ? cluster_ctarank() : 0u;
    constexpr int kStages = Cfg::kStages;
    constexpr int kAcc = Cfg::kAcc;
    extern __shared__ unsigned char gemm_smem_raw[];
    unsigned char* base = reinterpret_cast<unsigned char*>(
        (reinterpret_cast<uintptr_t>(gemm_smem_raw) + 1023) & ~(uintptr_t)1023);
    unsigned char* sA = base;                                        // ARES: [6][16 KB]; else [stages][16 KB]
    unsigned char* sB = base + (ARES ? Cfg::kResBytes : kStages * kABytes);
    unsigned char* sEnd = base + Cfg::kResBytes + kStages * Cfg::kStageBytes;
    uint64_t* full = reinterpret_cast<uint64_t*>(sEnd);
    uint64_t* empty = full + kStages;
    uint64_t* t_full = empty + kStages;      // [kAcc] accumulator complete
    uint64_t* t_empty = t_full + 2;          // [kAcc] accumulator drained by the epilogue
    uint64_t* a_full = t_empty + 2;          // ARES: resident A tile landed
    uint64_t* a_empty = a_full + 1;          // ARES: every MMA of the row block has read it
    uint64_t* r_full = a_empty + 1;          // [kEpiWarps][2] residual chunk landed (LayerNorm epilogue)
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(r_full + 2 * kEpiWarps);
    float* s_bias = reinterpret_cast<float*>(sEnd + Cfg::kBarBytes);                      // [N <= 1536]
    float* s_gamma = s_bias + 1536;                                                     // [384]
    float* s_beta = s_gamma + 384;                                                        // [384]
    float* s_part = s_beta + 384;                                                         // [2][2][128]
    unsigned char* s_io = reinterpret_cast<unsigned char*>(
        (reinterpret_cast<uintptr_t>(s_part + 2 * 2 * 128) + 2047) & ~(uintptr_t)2047);   // [kEpiWarps][2][2 KB]

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int total_tiles = m_tiles * n_tiles;
    constexpr int kProducerWarp = kEpiWarps, kMmaWarp = kEpiWarps + 1;

    // Programmatic dependent launch: from the trigger on, CTAs of the next kernel of the stream may
    // take an SM as soon as one is free, run their prologue and wait.  A grid that leaves SMs idle
    // (fewer row blocks than SMs) triggers at once -- 0.566 -> 0.521 ms for 64 sequences of 128
    // tokens; a full grid triggers when its CTA is done, so that the successor's CTAs do not sit on
    // the SMs it is still using -- 6.01 -> 5.73 ms for 1024 sequences (at once: 6.15).
    if (ep.pdl_early) pdl_trigger();
    if (warp == kProducerWarp && lane == 0) {
        tma_prefetch_desc(&tma_a);
        tma_prefetch_desc(&tma_b);
        for (int s = 0; s < kStages; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], CS);          // released by the MMA warp of every CTA of the cluster
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(&t_full[b], 1);
            mbar_init(&t_empty[b], kEpiWarps);
        }
        mbar_init(a_full, 1);
        mbar_init(a_empty, 1);
        for (int w = 0; w < 2 * kEpiWarps; ++w) mbar_init(&r_full[w], 1);
        tma_prefetch_desc(&tma_out);
        fence_barrier_init();
    }
    if (warp == kMmaWarp) {
        tmem_alloc(tmem_slot, Cfg::kTmemCols);
        tmem_relinquish();
    }
    tc_fence_before();
    __syncthreads();
    if (CS > 1) cluster_sync_all();            // peers' barriers are initialised before any multicast
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    pdl_wait();                                // the previous kernel's outputs are complete and visible

    if (warp == kProducerWarp) {
        // ===== TMA producer
        if (lane == 0) {
            uint32_t it = 0;
            if (ARES) {
                int mi = 0;
                for (int m_blk = blockIdx.x; m_blk < m_tiles; m_blk += gridDim.x, ++mi) {
                    mbar_wait(a_empty, ((uint32_t)mi & 1u) ^ 1u);     // previous row block retired
                    mbar_arrive_expect_tx(a_full, (uint32_t)Cfg::kResBytes);
                    for (int kb = 0; kb < kAResKB; ++kb)
                        tma_load_2d(sA + kb * kABytes, &tma_a, kb * kBK, m_blk * kBM, a_full);
                    for (int n_blk = 0; n_blk < n_tiles; ++n_blk) {
                        for (int kb = 0; kb < kAResKB; ++kb, ++it) {
                            const int s = (int)(it % kStages);
                            const uint32_t ph = (it / kStages) & 1u;
                            mbar_wait(&empty[s], ph ^ 1u);
                            mbar_arrive_expect_tx(&full[s], (uint32_t)Cfg::kStageBytes);
                            if (CS > 1) {
                                tma_load_2d_mc(sB + s * Cfg::kBBytes + crank * (Cfg::kBoxB * kBK * 2), &tma_b,
                                               kb * kBK, n_blk * BN + (int)crank * Cfg::kBoxB, &full[s], kMask);
                            } else {
#pragma unroll
                                for (int nb = 0; nb < BN / Cfg::kBoxB; ++nb)
                                    tma_load_2d(sB + s * Cfg::kBBytes + nb * (Cfg::kBoxB * kBK * 2), &tma_b,
                                                kb * kBK, n_blk * BN + nb * Cfg::kBoxB, &full[s]);
                            }
                        }
                    }
                }
            } else {
                for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
                    const int m_blk = tile / n_tiles, n_blk = tile - m_blk * n_tiles;
                    for (int kb = 0; kb < num_k_blocks; ++kb, ++it) {
                        const int s = (int)(it % kStages);
                        const uint32_t ph = (it / kStages) & 1u;
                        mbar_wait(&empty[s], ph ^ 1u);
                        mbar_arrive_expect_tx(&full[s], (uint32_t)Cfg::kStageBytes);
                        tma_load_2d(sA + s * kABytes, &tma_a, kb * kBK, m_blk * kBM, &full[s]);
                        if (CS > 1) {
                            tma_load_2d_mc(sB + s * Cfg::kBBytes + crank * (Cfg::kBoxB * kBK * 2), &tma_b,
                                           kb * kBK, n_blk * BN + (int)crank * Cfg::kBoxB, &full[s], kMask);
                        } else {
#pragma unroll
                            for (int nb = 0; nb < BN / Cfg::kBoxB; ++nb)
                                tma_load_2d(sB + s * Cfg::kBBytes + nb * (Cfg::kBoxB * kBK * 2), &tma_b, kb * kBK,
                                            n_blk * BN + nb * Cfg::kBoxB, &full[s]);
                        }
                    }
                }
            }
        }
    } else if (warp == kMmaWarp) {
        // ===== MMA issuer (one lane)
        if (lane == 0) {
            constexpr int N0 = (BN > 256) ? 256 : BN;
            constexpr int N1 = BN - N0;
            constexpr uint32_t idesc0 = umma_idesc_f16(kBM, N0);
            constexpr uint32_t idesc1 = umma_idesc_f16(kBM, N1 > 0 ? N1 : 16);
            uint32_t it = 0;
            int u = 0;
            // tiles in the order the producer feeds them: ARES -> row block by row block
            const int n_mine = ARES ? ((m_tiles > (int)blockIdx.x) ? (m_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0) * n_tiles
                                    : ((total_tiles > (int)blockIdx.x) ? (total_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0);
            for (; u < n_mine; ++u) {
                const int buf = u % kAcc;
                const uint32_t use = (uint32_t)(u / kAcc);
                if (ARES && (u % n_tiles) == 0) {
                    mbar_wait(a_full, (uint32_t)(u / n_tiles) & 1u);
                    tc_fence_after();
                }
                mbar_wait(&t_empty[buf], (use & 1u) ^ 1u);    // epilogue has drained this accumulator
                tc_fence_after();
                const uint32_t tacc = tmem_base + buf * BN;
                for (int kb = 0; kb < num_k_blocks; ++kb, ++it) {
                    const int s = (int)(it % kStages);
                    const uint32_t ph = (it / kStages) & 1u;
                    mbar_wait(&full[s], ph);
                    tc_fence_after();
                    const uint32_t a_addr = smem_u32(sA + (ARES ? kb : s) * kABytes);
                    const uint32_t b_addr = smem_u32(sB + s * Cfg::kBBytes);
#pragma unroll
                    for (int k = 0; k < kBK / 16; ++k) {
                        const uint64_t ad = umma_desc_sw128(a_addr + k * 32);
                        const uint64_t bd = umma_desc_sw128(b_addr + k * 32);
                        const uint32_t acc = (kb > 0 || k > 0) ? 1u : 0u;
                        umma_f16(tacc, ad, bd, idesc0, acc);
                        if (N1 > 0) {
                            const uint64_t bd1 = umma_desc_sw128(b_addr + N0 * 128 + k * 32);
                            umma_f16(tacc + N0, ad, bd1, idesc1, acc);
                        }
                    }
                    if (CS > 1) umma_commit_mc(&empty[s], kMask);   // slot free in every CTA of the cluster
                    else umma_commit(&empty[s]);              // smem slot free when the MMAs retire
                }
                umma_commit(&t_full[buf]);                    // accumulator complete
                if (ARES && (u % n_tiles) == n_tiles - 1) umma_commit(a_empty);   // A tile may be replaced
            }
        }
    } else {
        // ===== epilogue: 8 warps; thread = output row (TMEM lane 32*(warp&3)+lane), column half
        //       (warp >> 2).  Per-column parameters are staged in shared memory (float4 broadcast
        //       loads instead of one global load per element).
        const int quarter = warp & 3, half = warp >> 2;
        const int et = threadIdx.x;                      // 0..255
        constexpr int HB = BN / 2;                       // columns per half
        if (EPI != 3) {
            for (int i = et; i < n_tiles * BN; i += 256) s_bias[i] = ep.bias[i];
            if (EPI == 2) {
                for (int i = et; i < 384; i += 256) {
                    s_gamma[i] = ep.gamma[i];
                    s_beta[i] = ep.beta[i];
                }
            }
            epi_bar();
        }
        const int n_mine = ARES ? ((m_tiles > (int)blockIdx.x) ? (m_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0) * n_tiles
                                : ((total_tiles > (int)blockIdx.x) ? (total_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0);
        // this warp's staging tiles: two, used in turn by the bias / GELU epilogues, so that a chunk is
        // written while the TMA store of the chunk before still reads its tile (with one tile every
        // 32-column chunk waited for the previous store's read: ~1 000 cycles each, serial -- the FFN-up
        // kernel spent 36 us on 10 us of MMAs)
        unsigned char* tile_io = s_io + warp * Cfg::kIoTile;
        uint32_t st_n = 0;
        uint32_t res_n = 0;                               // residual chunks requested so far (phase)
        for (int u = 0; u < n_mine; ++u) {
            int m_blk, n_blk;
            if (ARES) {
                m_blk = blockIdx.x + (u / n_tiles) * gridDim.x;
                n_blk = u % n_tiles;
            } else {
                const int tile = blockIdx.x + u * gridDim.x;
                m_blk = tile / n_tiles;
                n_blk = tile - m_blk * n_tiles;
            }
            const int buf = u % kAcc;
            const uint32_t use = (uint32_t)(u / kAcc);
            const int n0 = n_blk * BN;
            const float* bias = s_bias + n0;
            mbar_wait(&t_full[buf], use & 1u);
            tc_fence_after();
            const int row = quarter * 32 + lane;
            const int64_t grow = (int64_t)m_blk * kBM + row;
            const bool ok = grow < ep.M;
            const uint32_t trow = tmem_base + ((uint32_t)(quarter * 32) << 16) + buf * BN + half * HB;
            const int cb = half * HB;                    // first column of this thread's half
            float v[32];
            // TMEM loads are software-pipelined: the load of chunk c + 1 is in flight while
            // chunk c is processed (tcgen05.wait::ld comes after the math).
            constexpr int NCH = HB / 32;
            uint32_t rb[2][32];
            if (EPI == 3) {
                float* out = reinterpret_cast<float*>(ep.out) + grow * ep.ld_out + n0 + cb;
                tmem_ld32(trow, rb[0]);
                tmem_wait_ld();
#pragma unroll
                for (int ch = 0; ch < NCH; ++ch) {
                    if (ch + 1 < NCH) tmem_ld32(trow + (ch + 1) * 32, rb[(ch + 1) & 1]);
                    const uint32_t(&r)[32] = rb[ch & 1];
                    if (ok) {
                        float4* o4 = reinterpret_cast<float4*>(out + ch * 32);
#pragma unroll
                        for (int j = 0; j < 8; ++j)
                            o4[j] = make_float4(__uint_as_float(r[4 * j]), __uint_as_float(r[4 * j + 1]),
                                                __uint_as_float(r[4 * j + 2]), __uint_as_float(r[4 * j + 3]));
                    }
                    tmem_wait_ld();
                }
            } else if (EPI == 0 || EPI == 1) {
                const int row_w = m_blk * kBM + quarter * 32;         // first output row of this warp
                tmem_ld32(trow, rb[0]);
                tmem_wait_ld();
#pragma unroll
                for (int ch = 0; ch < NCH; ++ch) {
                    if (ch + 1 < NCH) tmem_ld32(trow + (ch + 1) * 32, rb[(ch + 1) & 1]);
                    const uint32_t(&r)[32] = rb[ch & 1];
                    const int c = ch * 32;
#pragma unroll
                    for (int j4 = 0; j4 < 8; ++j4) {
                        const float4 bb = *reinterpret_cast<const float4*>(bias + cb + c + 4 * j4);
                        const float x0 = __uint_as_float(r[4 * j4 + 0]) + bb.x;
                        const float x1 = __uint_as_float(r[4 * j4 + 1]) + bb.y;
                        const float x2 = __uint_as_float(r[4 * j4 + 2]) + bb.z;
                        const float x3 = __uint_as_float(r[4 * j4 + 3]) + bb.w;
                        if (EPI == 1) {
                            const float2 ga = gelu2(x0, x1), gb = gelu2(x2, x3);
                            v[4 * j4 + 0] = ga.x; v[4 * j4 + 1] = ga.y;
                            v[4 * j4 + 2] = gb.x; v[4 * j4 + 3] = gb.y;
                        } else {
                            v[4 * j4 + 0] = x0; v[4 * j4 + 1] = x1;
                            v[4 * j4 + 2] = x2; v[4 * j4 + 3] = x3;
                        }
                    }
                    stage_acquire1(lane);                             // the store before the previous one has read its tile
                    unsigned char* tile_w = tile_io + (st_n & 1u) * 2048;
                    ++st_n;
                    stage_put_row(tile_w, lane, v);
                    stage_store(&tma_out, n0 + cb + c, row_w, tile_w, lane);
                    tmem_wait_ld();
                }
            } else {
                // bias + residual, LayerNorm over the whole row (BN == N == 384): each thread owns
                // half a row, the two halves exchange their partial sums through shared memory
                const int row_w = m_blk * kBM + quarter * 32;
                float* part = s_part + (u & 1) * 2 * 2 * 128;       // [stat][half][row]
                float sum = 0.f;
                // residual chunks come in through the warp's staging tile (TMA, coalesced): chunk
                // ch + 1 is requested as soon as every lane holds chunk ch in registers
                // (chunk ch + 1 is requested as soon as every lane holds chunk ch in registers)
                auto res_request = [&](int ch) {
                    if (lane == 0) {
                        mbar_arrive_expect_tx(&r_full[warp], 2048u);
                        tma_load_2d(tile_io, &tma_res, cb + ch * 32, row_w, &r_full[warp]);
                    }
                };
                stage_acquire(lane);                                 // last tile's output store has read it
                res_request(0);
                tmem_ld32(trow, rb[0]);
                tmem_wait_ld();
#pragma unroll
                for (int ch = 0; ch < NCH; ++ch) {
                    uint4 rr[4];
                    mbar_wait(&r_full[warp], res_n & 1u);
                    ++res_n;
                    stage_get_row(tile_io, lane, rr);
                    __syncwarp();
                    if (ch + 1 < NCH) {
                        res_request(ch + 1);
                        tmem_ld32(trow + (ch + 1) * 32, rb[(ch + 1) & 1]);
                    }
                    uint32_t(&r)[32] = rb[ch & 1];
                    const int c = ch * 32;
                    const __half2* rh = reinterpret_cast<const __half2*>(rr);
#pragma unroll
                    for (int j4 = 0; j4 < 8; ++j4) {
                        const float4 bb = *reinterpret_cast<const float4*>(bias + cb + c + 4 * j4);
                        const float2 f0 = __half22float2(rh[2 * j4]), f1 = __half22float2(rh[2 * j4 + 1]);
                        const float x0 = __uint_as_float(r[4 * j4 + 0]) + bb.x + f0.x;
                        const float x1 = __uint_as_float(r[4 * j4 + 1]) + bb.y + f0.y;
                        const float x2 = __uint_as_float(r[4 * j4 + 2]) + bb.z + f1.x;
                        const float x3 = __uint_as_float(r[4 * j4 + 3]) + bb.w + f1.y;
                        sum += (x0 + x1) + (x2 + x3);
                        r[4 * j4 + 0] = __float_as_uint(x0);
                        r[4 * j4 + 1] = __float_as_uint(x1);
                        r[4 * j4 + 2] = __float_as_uint(x2);
                        r[4 * j4 + 3] = __float_as_uint(x3);
                    }
                    tmem_wait_ld();                       // chunk ch + 1 has landed ...
                    tmem_st32(trow + c, r);               // ... before this buffer's registers are reused
                }
                part[half * 128 + row] = sum;
                tmem_wait_st();
                epi_bar();
                const float mean = (part[row] + part[128 + row]) * (1.0f / BN);
                float var = 0.f;
                tmem_ld32(trow, rb[0]);
                tmem_wait_ld();
#pragma unroll
                for (int ch = 0; ch < NCH; ++ch) {
                    if (ch + 1 < NCH) tmem_ld32(trow + (ch + 1) * 32, rb[(ch + 1) & 1]);
                    const uint32_t(&r)[32] = rb[ch & 1];
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const float d = __uint_as_float(r[j]) - mean;
                        var = fmaf(d, d, var);
                    }
                    tmem_wait_ld();
                }
                part[256 + half * 128 + row] = var;
                epi_bar();
                const float rstd = 1.0f / sqrtf((part[256 + row] + part[256 + 128 + row]) * (1.0f / BN) + ep.eps);
                tmem_ld32(trow, rb[0]);
                tmem_wait_ld();
#pragma unroll
                for (int ch = 0; ch < NCH; ++ch) {
                    if (ch + 1 < NCH) tmem_ld32(trow + (ch + 1) * 32, rb[(ch + 1) & 1]);
                    const uint32_t(&r)[32] = rb[ch & 1];
                    const int c = ch * 32;
#pragma unroll
                    for (int j4 = 0; j4 < 8; ++j4) {
                        const float4 gg = *reinterpret_cast<const float4*>(s_gamma + cb + c + 4 * j4);
                        const float4 be = *reinterpret_cast<const float4*>(s_beta + cb + c + 4 * j4);
                        v[4 * j4 + 0] = (__uint_as_float(r[4 * j4 + 0]) - mean) * rstd * gg.x + be.x;
                        v[4 * j4 + 1] = (__uint_as_float(r[4 * j4 + 1]) - mean) * rstd * gg.y + be.y;
                        v[4 * j4 + 2] = (__uint_as_float(r[4 * j4 + 2]) - mean) * rstd * gg.z + be.z;
                        v[4 * j4 + 3] = (__uint_as_float(r[4 * j4 + 3]) - mean) * rstd * gg.w + be.w;
                    }
                    stage_acquire(lane);
                    stage_put_row(tile_io, lane, v);
                    stage_store(&tma_out, cb + c, row_w, tile_io, lane);
                    tmem_wait_ld();
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&t_empty[buf]);        // accumulator may be overwritten
        }
        stage_acquire(lane);                                  // shared memory outlives its last store
    }
    tc_fence_before();
    __syncthreads();
    if (!ep.pdl_early) pdl_trigger();          // this CTA's work is done
    if (CS > 1) cluster_sync_all();            // nobody leaves while a peer may still multicast to it
    if (warp == kMmaWarp) {
        tc_fence_after();
        tmem_dealloc(tmem_base, Cfg::kTmemCols);
    }
}

// ---------------------------------------------------------------- host side
typedef CUresult (*PFN_tmapEncodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                        const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                        const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                        CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_tmapEncodeTiled get_encode_fn() {
    static PFN_tmapEncodeTiled fn = nullptr;
    if (fn == nullptr) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = (PFN_tmapEncodeTiled)p;
    }
    return fn;
}

// fp16 row-major [rows, cols] with leading dimension ld (elements); box = 64 cols x box_rows,
// SWIZZLE_128B; out-of-range rows/cols read as zero.
cudaError_t make_tmap_f16(CUtensorMap* out, const void* ptr, int64_t rows, int64_t cols, int64_t ld,
                          int box_rows) {
    PFN_tmapEncodeTiled fn = get_encode_fn();
    if (fn == nullptr) return cudaErrorNotSupported;
    if (rows <= 0) rows = 1;
    cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t gstride[1] = {(cuuint64_t)ld * 2};
    cuuint32_t box[2] = {(cuuint32_t)kBK, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(ptr), gdim, gstride, box,
                    estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                    CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? cudaSuccess : cudaErrorInvalidValue;
}

// fp16 row-major [rows, cols]: the epilogue's staging-tile view, box = 32 cols x 32 rows,
// SWIZZLE_64B (TMA stores of outputs, TMA loads of the LayerNorm residual).
cudaError_t make_tmap_io_f16(CUtensorMap* out, const void* ptr, int64_t rows, int64_t cols, int64_t ld) {
    PFN_tmapEncodeTiled fn = get_encode_fn();
    if (fn == nullptr) return cudaErrorNotSupported;
    if (rows <= 0) rows = 1;
    cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t gstride[1] = {(cuuint64_t)ld * 2};
    cuuint32_t box[2] = {32, 32};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(ptr), gdim, gstride, box,
                    estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B,
                    CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? cudaSuccess : cudaErrorInvalidValue;
}

template <int BN, int EPI, bool ARES, int CS>
static cudaError_t launch_cfg(lrx_handle* h, const CUtensorMap& ta, const CUtensorMap& tb,
                              const CUtensorMap& tout, const CUtensorMap& tres, int M,
                              int N, int K, const GemmEpi& ep) {
    std::lock_guard<std::recursive_mutex> attr_guard(attr_mutex());   // the flags below are process-wide
    static bool attr_dev[64] = {false};   // function attributes are per device
    bool& attr = attr_dev[h->device & 63];
    auto kern = tc_gemm_kernel<BN, EPI, ARES, CS>;
    constexpr size_t smem = GemmCfg<BN, ARES, CS>::kSmem;
    if (!attr) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        attr = true;
    }
    int m_tiles = (M + kBM - 1) / kBM;
    const int n_tiles = N / BN;
    if (CS > 1) m_tiles = (m_tiles + CS - 1) / CS * CS;     // padded row blocks: loads zero-fill, stores are guarded
    const int units = ARES ? m_tiles : m_tiles * n_tiles;
    int grid = units < h->num_sms ? units : h->num_sms;
    if (CS > 1) grid = grid / CS * CS;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(kGemmThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = h->stream;
    // programmatic dependent launch: this kernel's CTAs may take an SM as soon as the previous
    // kernel's CTA leaves it and run their prologue (barriers, TMEM, descriptor prefetch) while the
    // rest of that grid drains; they wait (griddepcontrol.wait) before touching activations
    cudaLaunchAttribute at[2];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = CS;
    at[0].val.clusterDim.y = 1;
    at[0].val.clusterDim.z = 1;
    at[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = 2;
    GemmEpi ep2 = ep;
    ep2.pdl_early = (units < h->num_sms) ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kern, ta, tb, tout, tres, K / kBK, m_tiles, n_tiles, ep2);
}

// Which variant runs (the W tensor map's box must match: gemm_box_rows_w).
struct GemmPlan { int bn; bool ares; int cs; };
GemmPlan gemm_plan(int num_sms, int M, int N, int K, int epi) {
    GemmPlan p;
    p.bn = (epi == 2) ? 384 : (N % 192 == 0 ? 192 : (N % 256 == 0 ? 256 : 128));
    const int m_tiles = (M + kBM - 1) / kBM;
    const bool big = m_tiles >= num_sms / 2;                 // enough row blocks to fill the SMs
    p.ares = (K == kAResKB * kBK) && (big || N / p.bn == 1);
    // clusters need every CTA of a cluster to walk the same n sequence: A-resident (n inner loop),
    // or a single n-block
    p.cs = (big && (p.ares || N / p.bn == 1)) ? kGemmCluster : 1;
    return p;
}

template <int BN, int EPI>
static cudaError_t launch_one(lrx_handle* h, const CUtensorMap& ta, const CUtensorMap& tb,
                              const CUtensorMap& tout, const CUtensorMap& tres, int M,
                              int N, int K, const GemmEpi& ep) {
    const GemmPlan p = gemm_plan(h->num_sms, M, N, K, EPI);
    if (p.cs > 1) {
        if (p.ares) return launch_cfg<BN, EPI, true, kGemmCluster>(h, ta, tb, tout, tres, M, N, K, ep);
        return launch_cfg<BN, EPI, false, kGemmCluster>(h, ta, tb, tout, tres, M, N, K, ep);
    }
    if (p.ares) return launch_cfg<BN, EPI, true, 1>(h, ta, tb, tout, tres, M, N, K, ep);
    return launch_cfg<BN, EPI, false, 1>(h, ta, tb, tout, tres, M, N, K, ep);
}

// W-operand TMA box rows for a GEMM of this shape (the plan the launcher will pick)
int gemm_box_rows_w(int num_sms, int M, int N, int K, int epi) {
    const GemmPlan p = gemm_plan(num_sms, M, N, K, epi);
    if (p.cs > 1) return p.bn / p.cs;
    return p.bn > 256 ? 128 : p.bn;
}

// epi: 0 bias, 1 bias+GELU, 2 bias+residual+LayerNorm (N must be 384), 3 raw fp32.
// `tb` must have been built with gemm_box_rows_w(...) rows per box; `tout` / `tres` are
// make_tmap_io_f16 views of the fp16 output / residual (ignored by epi 3 / epi != 2).
cudaError_t launch_tc_gemm(lrx_handle* h, const CUtensorMap& ta, const CUtensorMap& tb,
                           const CUtensorMap& tout, const CUtensorMap& tres, int M, int N, int K, int epi,
                           const float* bias, const float* gamma, const float* beta, float eps,
                           void* out, int ld_out) {
    if (M <= 0) return cudaSuccess;
    if (K % kBK != 0 || N % 128 != 0 || epi < 0 || epi > 3) return cudaErrorInvalidValue;
    if (epi != 3 && N > 1536) return cudaErrorInvalidValue;      // bias vector staged whole in smem
    GemmEpi ep;
    ep.bias = bias; ep.residual = nullptr; ep.gamma = gamma; ep.beta = beta;
    ep.out = out; ep.ld_out = ld_out; ep.ld_res = 0; ep.M = M; ep.eps = eps;
    const int bn = gemm_plan(h->num_sms, M, N, K, epi).bn;
    cudaError_t e = cudaErrorInvalidValue;
#define LRX_GEMM_CASE(BN_, EPI_) \
    if (bn == BN_ && epi == EPI_) e = launch_one<BN_, EPI_>(h, ta, tb, tout, tres, M, N, K, ep)
    if (epi == 2) {
        if (N != 384) return cudaErrorInvalidValue;
        e = launch_one<384, 2>(h, ta, tb, tout, tres, M, N, K, ep);
    }
    LRX_GEMM_CASE(256, 0); LRX_GEMM_CASE(192, 0); LRX_GEMM_CASE(128, 0);
    LRX_GEMM_CASE(256, 1); LRX_GEMM_CASE(192, 1); LRX_GEMM_CASE(128, 1);
    LRX_GEMM_CASE(256, 3); LRX_GEMM_CASE(192, 3); LRX_GEMM_CASE(128, 3);
#undef LRX_GEMM_CASE
    h->launches++;
    return e;
}

// One-off form (tests, stage benchmarks): builds the two tensor maps per call.
cudaError_t gemm_f16_adhoc(lrx_handle* h, const void* a, const void* w, int M, int N, int K, int epi,
                           const float* bias, const void* residual, const float* gamma,
                           const float* beta, float eps, void* out) {
    CUtensorMap ta, tb, tout, tres;
    cudaError_t e = make_tmap_f16(&ta, a, M, K, K, 128);
    if (e != cudaSuccess) return e;
    e = make_tmap_f16(&tb, w, N, K, K, gemm_box_rows_w(h->num_sms, M, N, K, epi));
    if (e != cudaSuccess) return e;
    tout = ta;
    tres = ta;
    if (epi != 3) {
        e = make_tmap_io_f16(&tout, out, M, N, N);
        if (e != cudaSuccess) return e;
    }
    if (epi == 2) {
        e = make_tmap_io_f16(&tres, residual, M, N, N);
        if (e != cudaSuccess) return e;
    }
    return launch_tc_gemm(h, ta, tb, tout, tres, M, N, K, epi, bias, gamma, beta, eps, out, N);
}

}  // namespace lrx
