// K1: all-MiniLM-L6-v2 forward = SentenceTransformer.encode + faiss.normalize_L2
// (reference: src/retrieval/retrieval_engine.py:61-62, create_vector_store.py:45,51).
//
//   BertEmbeddings   word[id] + position[s] + token_type[0], LayerNorm(eps 1e-12)
//   6 x BertLayer    QKV projection (tc_gemm, +bias) -> 12-head attention (this file)
//                    -> output projection + residual + LayerNorm (tc_gemm, fused epilogue)
//                    -> FFN up + exact-erf GELU (tc_gemm) -> FFN down + residual + LayerNorm
//   Pooling          sum(h * mask) / max(sum(mask), 1e-9)
//   Normalize        x / max(||x||_2, 1e-12)      (sentence-transformers Normalize module)
//   normalize_L2     x * (1 / sqrt(||x||^2))      (faiss, applied again by the reference)
//
// Activations are fp16 [tokens, width] row-major in handle-owned workspaces, processed in
// chunks of whole sequences sized so one chunk's working set stays L2-resident; all
// statistics (LayerNorm, softmax, pooling, norms) are fp32.
#include <cmath>
#include <cstdlib>
#include <cstring>

#include "handle.h"
#include "tc.cuh"

namespace lrx {

constexpr int kHidden = 384;
constexpr int kHeads = 12;
constexpr int kHeadDim = 32;
constexpr int kFfn = 1536;
constexpr int kQkv = 3 * kHidden;
constexpr int kLayers = 6;
constexpr float kLnEps = 1e-12f;
// tokens per chunk: 148 row tiles of 128 = one full wave of the LayerNorm GEMMs (whose tile is
// the whole 384-wide row); ~7.7 KB of activations per token, consecutive kernels hit in L2
constexpr int64_t kChunkTokens = 148 * 128;
// the GEMMs of the chain are launched with programmatic stream serialization (tc_gemm.cu); for the
// small kernels between them it bought nothing (A/B, tools/ab) and they stay plain launches
constexpr bool kEncPdlSmall = false;

// tc_gemm.cu
cudaError_t make_tmap_f16(CUtensorMap* out, const void* ptr, int64_t rows, int64_t cols, int64_t ld,
                          int box_rows);
cudaError_t make_tmap_io_f16(CUtensorMap* out, const void* ptr, int64_t rows, int64_t cols, int64_t ld);
cudaError_t launch_tc_gemm(lrx_handle* h, const CUtensorMap& ta, const CUtensorMap& tb,
                           const CUtensorMap& tout, const CUtensorMap& tres, int M, int N, int K, int epi,
                           const float* bias, const float* gamma, const float* beta, float eps,
                           void* out, int ld_out);
int gemm_box_rows_w(int num_sms, int M, int N, int K, int epi);

struct EncLayer {
    __half* wqkv;   // [1152, 384]
    __half* wo;     // [384, 384]
    __half* w1;     // [1536, 384]
    __half* w2;     // [384, 1536]
    float *bqkv, *bo, *b1, *b2, *ln1_g, *ln1_b, *ln2_g, *ln2_b;
    // W tensor maps for the two launch plans: [0] small batches, [1] full waves (clusters)
    CUtensorMap t_wqkv[2], t_wo[2], t_w1[2], t_w2[2];
};

struct Encoder {
    int vocab = 0, max_pos = 0;
    float *word = nullptr, *pos = nullptr, *type0 = nullptr, *eln_g = nullptr, *eln_b = nullptr;
    EncLayer L[kLayers];
    void* blob = nullptr;      // one allocation holding every packed weight
    // activation workspaces for `cap` tokens
    int64_t cap = 0;
    void* act = nullptr;
    __half *x = nullptr, *x1 = nullptr, *qkv = nullptr, *ctx = nullptr, *ff = nullptr;
    CUtensorMap t_x, t_x1, t_ctx, t_ff;              // A-operand views (128-row boxes, SWIZZLE_128B)
    CUtensorMap io_x, io_x1, io_qkv, io_ff;          // epilogue views (32 x 32 boxes, SWIZZLE_64B)
    void* small_ws = nullptr;  // encoder_small_kernel: per-group scratch (qkv, ctx, ff, pre-LayerNorm sums)
    size_t small_ws_bytes = 0;
    void* io = nullptr;        // host-form staging (ids, lens, out)
    size_t io_bytes = 0;
    void* io_host = nullptr;
    size_t io_host_bytes = 0;
};

// ------------------------------------------------------------ weight packing
__global__ void f32_to_f16_kernel(const float* __restrict__ src, __half* __restrict__ dst, int64_t n) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (int64_t)gridDim.x * blockDim.x)
        dst[i] = __float2half_rn(src[i]);
}

// ---------------------------------------------------------------- embeddings
// one warp per token; lane owns columns j*128 + lane*4 + {0..3}, j = 0..2
__global__ void __launch_bounds__(256)
embed_ln_kernel(const int32_t* __restrict__ ids, int64_t n_tokens, int S, int vocab, int max_pos,
                const float* __restrict__ word, const float* __restrict__ pos,
                const float* __restrict__ type0, const float* __restrict__ g,
                const float* __restrict__ b, __half* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int64_t tok = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    pdl_trigger();
    pdl_wait();                                // the previous chunk's pooling has read x
    if (tok >= n_tokens) return;
    int id = ids[tok];
    id = (id < 0 || id >= vocab) ? 0 : id;
    int s = (int)(tok % S);
    s = (s >= max_pos) ? max_pos - 1 : s;
    float v[12];
    float sum = 0.f;
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        const int c = j * 128 + lane * 4;
        const float4 w = __ldg(reinterpret_cast<const float4*>(word + (size_t)id * kHidden + c));
        const float4 p = __ldg(reinterpret_cast<const float4*>(pos + (size_t)s * kHidden + c));
        const float4 t = __ldg(reinterpret_cast<const float4*>(type0 + c));
        v[4 * j + 0] = w.x + p.x + t.x;
        v[4 * j + 1] = w.y + p.y + t.y;
        v[4 * j + 2] = w.z + p.z + t.z;
        v[4 * j + 3] = w.w + p.w + t.w;
        sum += v[4 * j] + v[4 * j + 1] + v[4 * j + 2] + v[4 * j + 3];
    }
#pragma unroll
    for (int lb = 16; lb > 0; lb >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, lb);
    const float mean = sum * (1.0f / kHidden);
    float var = 0.f;
#pragma unroll
    for (int i = 0; i < 12; ++i) {
        const float d = v[i] - mean;
        var = fmaf(d, d, var);
    }
#pragma unroll
    for (int lb = 16; lb > 0; lb >>= 1) var += __shfl_xor_sync(0xffffffffu, var, lb);
    const float rstd = 1.0f / sqrtf(var * (1.0f / kHidden) + kLnEps);
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        const int c = j * 128 + lane * 4;
        const float4 gg = __ldg(reinterpret_cast<const float4*>(g + c));
        const float4 bb = __ldg(reinterpret_cast<const float4*>(b + c));
        const __half2 h0 = __floats2half2_rn((v[4 * j + 0] - mean) * rstd * gg.x + bb.x,
                                             (v[4 * j + 1] - mean) * rstd * gg.y + bb.y);
        const __half2 h1 = __floats2half2_rn((v[4 * j + 2] - mean) * rstd * gg.z + bb.z,
                                             (v[4 * j + 3] - mean) * rstd * gg.w + bb.w);
        uint2 u;
        u.x = *reinterpret_cast<const uint32_t*>(&h0);
        u.y = *reinterpret_cast<const uint32_t*>(&h1);
        *reinterpret_cast<uint2*>(out + tok * kHidden + c) = u;
    }
}

// ----------------------------------------------------------------- attention
// One CTA per (head, sequence): K and V of the head staged row-major in shared memory (80-byte
// rows: conflict-free ldmatrix), each warp owns 16-query tiles; QK^T and P*V on mma.sync
// m16n8k16 (fp16 in, fp32 accumulate) with the B fragments fetched by ldmatrix.x4 (V through
// .trans, so no transposed copy is ever written); online softmax over 64-key blocks in fp32 in
// the exp2 domain (one MUFU.EX2 per score).  Keys >= len are masked out; query rows >= len
// (padding) produce zeros.
constexpr int kAttnThreads = 256;
constexpr int kKPad = 40;    // halves per K / V row in smem (32 + 8)

__device__ __forceinline__ void mma16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0,
                                         uint32_t b1) {
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, "
        "{%0,%1,%2,%3};"
        : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t pack_h2(float a, float b) {
    const __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<const uint32_t*>(&h);
}
__device__ __forceinline__ void ldsm_x4(uint32_t (&r)[4], const void* p) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(smem_u32(p)));
}
__device__ __forceinline__ void ldsm_x4_t(uint32_t (&r)[4], const void* p) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(smem_u32(p)));
}
__device__ __forceinline__ float ex2(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

__global__ void __launch_bounds__(kAttnThreads)
attention_kernel(const __half* __restrict__ qkv, const int32_t* __restrict__ lens, int S,
                 __half* __restrict__ ctx) {
    extern __shared__ __align__(16) unsigned char attn_raw[];
    // (no early trigger here: the next kernel is a GEMM of one 200 KB CTA per SM, and this grid
    // has several waves of small CTAs still to place)
    pdl_wait();                                // the QKV projection is complete
    const int head = blockIdx.x;
    const int seq = blockIdx.y;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, t = lane & 3;
    int len = lens[seq];
    len = len < 0 ? 0 : (len > S ? S : len);
    const int Sk = (len + 63) & ~63;                 // staged keys (multiple of 64)
    __half* sK = reinterpret_cast<__half*>(attn_raw);            // [Sk][kKPad]
    __half* sV = sK + (size_t)Sk * kKPad;                         // [Sk][kKPad]
    const __half* base = qkv + (size_t)seq * S * kQkv + head * kHeadDim;

    // ---- stage K and V (row-major, padded) with 16-byte async copies; rows >= len are zero-filled
    for (int i = tid; i < Sk * 4; i += kAttnThreads) {
        const int s = i >> 2, part = i & 3;          // 4 x 16-byte parts per 64-byte row
        const int sr = s < len ? s : 0;
        const uint32_t nbytes = s < len ? 16u : 0u;
        const __half* kp = base + (size_t)sr * kQkv + kHidden + part * 8;
        asm volatile("cp.async.ca.shared.global [%0], [%1], 16, %2;"
                     ::"r"(smem_u32(sK + s * kKPad + part * 8)), "l"(kp), "r"(nbytes) : "memory");
        asm volatile("cp.async.ca.shared.global [%0], [%1], 16, %2;"
                     ::"r"(smem_u32(sV + s * kKPad + part * 8)), "l"(kp + kHidden), "r"(nbytes) : "memory");
    }
    asm volatile("cp.async.commit_group;" ::: "memory");

    // softmax in the exp2 domain: p = 2^((s - m) * scale * log2(e)), the scale folded into one FFMA
    const float scale2 = 0.17677669529663687f * 1.4426950408889634f;
    // ldmatrix lane roles: matrix (lane >> 3), row (lane & 7)
    const int lm = lane >> 3, lr = lane & 7;
    const int n_qtiles = (S + 15) >> 4;
    // Q fragments (A operand) of a 16-query tile, two k-steps over d = 0..31
    uint32_t qa[2][4];
    auto load_q = [&](int qt) {
        const int r0 = qt * 16 + g, r1 = r0 + 8;
#pragma unroll
        for (int ks = 0; ks < 2; ++ks) {
            const __half* q0p = base + (size_t)r0 * kQkv + ks * 16 + 2 * t;
            const __half* q1p = base + (size_t)r1 * kQkv + ks * 16 + 2 * t;
            qa[ks][0] = (r0 < len) ? __ldg(reinterpret_cast<const uint32_t*>(q0p)) : 0u;
            qa[ks][1] = (r1 < len) ? __ldg(reinterpret_cast<const uint32_t*>(q1p)) : 0u;
            qa[ks][2] = (r0 < len) ? __ldg(reinterpret_cast<const uint32_t*>(q0p + 8)) : 0u;
            qa[ks][3] = (r1 < len) ? __ldg(reinterpret_cast<const uint32_t*>(q1p + 8)) : 0u;
        }
    };
    if (warp < n_qtiles) load_q(warp);               // in flight together with the K / V copies
    asm volatile("cp.async.wait_all;" ::: "memory");
    __syncthreads();
    for (int qt = warp; qt < n_qtiles; qt += kAttnThreads / 32) {
        const int q0 = qt * 16;
        const int r0 = q0 + g, r1 = q0 + g + 8;
        __half* o0 = ctx + ((size_t)seq * S + r0) * kHidden + head * kHeadDim;
        __half* o1 = ctx + ((size_t)seq * S + r1) * kHidden + head * kHeadDim;
        if (qt != warp) load_q(qt);
        if (q0 >= len) {                              // padding tile: zeros
#pragma unroll
            for (int nd = 0; nd < 4; ++nd) {
                if (r0 < S) *reinterpret_cast<uint32_t*>(o0 + nd * 8 + 2 * t) = 0u;
                if (r1 < S) *reinterpret_cast<uint32_t*>(o1 + nd * 8 + 2 * t) = 0u;
            }
            continue;
        }
        float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f;
        float o[4][4];
#pragma unroll
        for (int nd = 0; nd < 4; ++nd)
#pragma unroll
            for (int i = 0; i < 4; ++i) o[nd][i] = 0.f;

        for (int kb = 0; kb < Sk; kb += 64) {
            float sc[8][4];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
#pragma unroll
                for (int i = 0; i < 4; ++i) sc[j][i] = 0.f;
                // K rows kb + 8j .. +7, the four 8-wide d blocks: {b0,b1} of k-step 0, then of k-step 1
                uint32_t kf[4];
                ldsm_x4(kf, sK + (kb + j * 8 + lr) * kKPad + lm * 8);
                mma16816(sc[j], qa[0], kf[0], kf[1]);
                mma16816(sc[j], qa[1], kf[2], kf[3]);
            }
            // mask (last block only) + block max, on the raw scores
            if (kb + 64 > len) {
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const int key = kb + j * 8 + 2 * t;
                    if (key >= len) { sc[j][0] = -INFINITY; sc[j][2] = -INFINITY; }
                    if (key + 1 >= len) { sc[j][1] = -INFINITY; sc[j][3] = -INFINITY; }
                }
            }
            float bm0 = -INFINITY, bm1 = -INFINITY;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                bm0 = fmaxf(bm0, fmaxf(sc[j][0], sc[j][1]));
                bm1 = fmaxf(bm1, fmaxf(sc[j][2], sc[j][3]));
            }
            bm0 = fmaxf(bm0, __shfl_xor_sync(0xffffffffu, bm0, 1));
            bm0 = fmaxf(bm0, __shfl_xor_sync(0xffffffffu, bm0, 2));
            bm1 = fmaxf(bm1, __shfl_xor_sync(0xffffffffu, bm1, 1));
            bm1 = fmaxf(bm1, __shfl_xor_sync(0xffffffffu, bm1, 2));
            const float mn0 = fmaxf(m0, bm0), mn1 = fmaxf(m1, bm1);   // finite: key kb < len
            const float a0 = ex2((m0 - mn0) * scale2), a1 = ex2((m1 - mn1) * scale2);
            m0 = mn0; m1 = mn1;
            const float nm0 = -mn0 * scale2, nm1 = -mn1 * scale2;
            float ps0 = 0.f, ps1 = 0.f;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                sc[j][0] = ex2(fmaf(sc[j][0], scale2, nm0));
                sc[j][1] = ex2(fmaf(sc[j][1], scale2, nm0));
                sc[j][2] = ex2(fmaf(sc[j][2], scale2, nm1));
                sc[j][3] = ex2(fmaf(sc[j][3], scale2, nm1));
                ps0 += sc[j][0] + sc[j][1];
                ps1 += sc[j][2] + sc[j][3];
            }
            l0 = l0 * a0 + ps0;
            l1 = l1 * a1 + ps1;
#pragma unroll
            for (int nd = 0; nd < 4; ++nd) {
                o[nd][0] *= a0; o[nd][1] *= a0;
                o[nd][2] *= a1; o[nd][3] *= a1;
            }
            // O += P * V   (P from the score fragments; V fragments through ldmatrix.trans)
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
                uint32_t pa[4];
                pa[0] = pack_h2(sc[2 * kk][0], sc[2 * kk][1]);
                pa[1] = pack_h2(sc[2 * kk][2], sc[2 * kk][3]);
                pa[2] = pack_h2(sc[2 * kk + 1][0], sc[2 * kk + 1][1]);
                pa[3] = pack_h2(sc[2 * kk + 1][2], sc[2 * kk + 1][3]);
#pragma unroll
                for (int np = 0; np < 2; ++np) {
                    // matrices: (keys 0-7, d block 2np), (keys 8-15, 2np), (keys 0-7, 2np+1), (keys 8-15, 2np+1)
                    uint32_t vf[4];
                    ldsm_x4_t(vf, sV + (kb + kk * 16 + (lm & 1) * 8 + lr) * kKPad + (2 * np + (lm >> 1)) * 8);
                    mma16816(o[2 * np], pa, vf[0], vf[1]);
                    mma16816(o[2 * np + 1], pa, vf[2], vf[3]);
                }
            }
        }
        // row sums across the quad, normalise, store
        l0 += __shfl_xor_sync(0xffffffffu, l0, 1);
        l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
        l1 += __shfl_xor_sync(0xffffffffu, l1, 1);
        l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
        const float i0 = 1.0f / l0, i1 = 1.0f / l1;
#pragma unroll
        for (int nd = 0; nd < 4; ++nd) {
            if (r0 < S)
                *reinterpret_cast<uint32_t*>(o0 + nd * 8 + 2 * t) =
                    (r0 < len) ? pack_h2(o[nd][0] * i0, o[nd][1] * i0) : 0u;
            if (r1 < S)
                *reinterpret_cast<uint32_t*>(o1 + nd * 8 + 2 * t) =
                    (r1 < len) ? pack_h2(o[nd][2] * i1, o[nd][3] * i1) : 0u;
        }
    }
}

// ------------------------------------------------------------------- pooling
// One CTA (128 threads x 3 columns) per sequence: masked mean, Normalize, normalize_L2.
__device__ __forceinline__ float block_sum_128(float v, float* red) {
#pragma unroll
    for (int lb = 16; lb > 0; lb >>= 1) v += __shfl_xor_sync(0xffffffffu, v, lb);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    return red[0] + red[1] + red[2] + red[3];
}

__global__ void __launch_bounds__(128)
pool_normalize_kernel(const __half* __restrict__ x, const int32_t* __restrict__ lens, int S,
                      float* __restrict__ out_f32, __half* __restrict__ out_f16) {
    __shared__ float red[4];
    pdl_trigger();
    pdl_wait();                                // the last layer's output is complete
    const int seq = blockIdx.x;
    const int tid = threadIdx.x;
    int len = lens[seq];
    len = len < 0 ? 0 : (len > S ? S : len);
    float acc[3] = {0.f, 0.f, 0.f};
    const __half* p = x + (size_t)seq * S * kHidden;
    for (int s = 0; s < len; ++s) {
#pragma unroll
        for (int j = 0; j < 3; ++j) acc[j] += __half2float(p[(size_t)s * kHidden + j * 128 + tid]);
    }
    const float denom = fmaxf((float)len, 1e-9f);          // torch.clamp(sum_mask, min=1e-9)
    float sq = 0.f;
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        acc[j] = acc[j] / denom;
        sq = fmaf(acc[j], acc[j], sq);
    }
    sq = block_sum_128(sq, red);
    const float nrm = fmaxf(sqrtf(sq), 1e-12f);            // F.normalize(p=2, eps=1e-12)
    float sq2 = 0.f;
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        acc[j] = acc[j] / nrm;
        sq2 = fmaf(acc[j], acc[j], sq2);
    }
    sq2 = block_sum_128(sq2, red);
    if (sq2 > 0.f) {                                       // faiss.normalize_L2
        const float inv = 1.0f / sqrtf(sq2);
#pragma unroll
        for (int j = 0; j < 3; ++j) acc[j] *= inv;
    }
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        const size_t o = (size_t)seq * kHidden + j * 128 + tid;
        if (out_f32 != nullptr) out_f32[o] = acc[j];
        if (out_f16 != nullptr) out_f16[o] = __float2half_rn(acc[j]);
    }
}

// ------------------------------------- query-sized sequences: one cluster per group, one launch
// A query batch (the 1-4 strings of a fan-out, a few dozen tokens each) through the 31-launch
// tcgen05 chain above costs 0.37 ms of launch and pipeline start-up latencies for 0.2 GFLOP of work,
// all of it on the one or two SMs that own the batch's single 128-row tile.  encoder_small_kernel
// runs the WHOLE forward pass -- embeddings, 6 layers, pooling, both normalisations -- as one
// launch, and spreads it: sequences are independent, so every GROUP of sequences with at most
// M = 16 MT tokens (MT = 2: S <= 32, MT = 4: S <= 64) gets its own cluster of 8 CTAs, and inside a
// cluster every GEMM is split over the 64 warps by output COLUMNS (sm_tile_mma below):
//   * a warp owns half of the group's rows x up to 6 column tiles of 8; its weights are fetched as
//     16-byte loads per lane straight into mma.sync B fragments (A and B agree on a permuted k
//     order, as in dense.cu: no ldmatrix, no swizzle), four 32-k chunks ahead of the MMAs, the first
//     four chunks of a phase before the cluster barrier in front of it;
//   * the group's activations X [M x 384] live in every CTA's shared memory (replicated); A
//     operands written by other CTAs (attention output, FFN activations) are staged by cp.async;
//   * QKV: 144 column tiles = 16 warp pairs x 5 + 16 x 4, FFN up: 192 = 32 x 6, attention output:
//     48 = 16 x 2 + 16 x 1; FFN down (K = 1536) is 48 column tiles x 4 k quarters whose partial
//     sums meet in the LayerNorm IN A FIXED ORDER, so the result does not depend on timing;
//   * slices meet in an L2-resident scratch, a cluster barrier (release / acquire) separates
//     producer and consumer steps: 5 per layer; LayerNorm runs redundantly in every CTA (fp32);
//   * attention: one (sequence, head) pair per warp, mma.sync QK^T / PV with one-shot softmax.
// Every row's arithmetic is the same whatever the batch, the padded length or the row's place in
// the tile, so a sequence's embedding does not depend on what it was batched with (the serving
// front coalesces requests, tests/test_gpu_engine.py::test_micro_batching_front_...).
constexpr int kSmCtas = 8;
constexpr int kSmThreads = 256;
constexpr int kSmWarps = kSmThreads / 32;
constexpr int kSmLd = 416;              // halves per staged row: 832 B = 64 mod 128, so the 16-byte
                                        // fragment loads of 2 rows x 4 lanes cover all 32 banks
constexpr int kSmAttnWarps = 5;         // warps per CTA that take attention pairs (their K / V staging
                                        // shares the A-staging tile)
constexpr int kSmMaxGroups = 128;       // groups per launch (scratch: 0.45 / 0.9 MB each)

template <int MT>
struct SmGeom {
    static constexpr int M = 16 * MT;
    static constexpr size_t tile_bytes = (size_t)M * kSmLd * 2;
    static constexpr size_t smem = 2 * tile_bytes;
    static constexpr size_t o_qkv = 0;
    static constexpr size_t o_ctx = o_qkv + (size_t)M * kQkv * 2;
    static constexpr size_t o_ff = o_ctx + (size_t)M * kHidden * 2;
    static constexpr size_t o_y = o_ff + (size_t)M * kFfn * 2;
    static constexpr size_t o_ypart = o_y + (size_t)M * kHidden * 4;
    static constexpr size_t scratch = o_ypart + 4 * (size_t)M * kHidden * 4;
};
static_assert(kSmAttnWarps * 2 * 32 * kKPad * 2 <= (int)SmGeom<2>::tile_bytes, "attention staging (MT = 2)");
static_assert(kSmAttnWarps * 2 * 64 * kKPad * 2 <= (int)SmGeom<4>::tile_bytes, "attention staging (MT = 4)");

struct SmallLayer {
    const __half *wqkv, *wo, *w1, *w2;
    const float *bqkv, *bo, *b1, *b2, *ln1_g, *ln1_b, *ln2_g, *ln2_b;
};
struct SmallParams {
    const int32_t* ids;
    const int32_t* lens;
    int B, S, spg, vocab, max_pos;      // spg: sequences per group
    const float *word, *pos, *type0, *eln_g, *eln_b;
    SmallLayer L[kLayers];
    unsigned char* scratch;             // [groups][SmGeom::scratch]
    float* out_f32;
    __half* out_f16;
};

__device__ __forceinline__ float gelu_erf(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752f)); }
__device__ __forceinline__ uint4 ldcg_u4(const void* p) { return __ldcg(reinterpret_cast<const uint4*>(p)); }

// A warp's tile of one GEMM phase: MW row blocks of 16 (rows mrow0 ..) x nu <= 6 column tiles of 8,
// K = 384 in 12 chunks of 32, k-pipelined: the B fragments of chunk ch + kSmPd are fetched straight
// from L2 (one 16-byte load per lane and column tile: W row n0 + g, k = kbase + 32 ch + 8 t .. + 8)
// while chunk ch is multiplied.  A is read from shared memory once per phase and warp (only the
// warp's own rows).  The first version gave every warp ALL rows of 8 columns at a time and re-read
// the whole A tile per 8 columns: 1536 shared-memory wavefront cycles per unit and SM, three times
// the tensor time.
constexpr int kSmPd = 4;                // chunks of B in flight
constexpr int kSmNu = 6;                // column tiles per warp, at most
struct SmB {
    uint4 r[kSmPd][kSmNu];
};
// w0: this lane's pointer into column tile 0 (row n0 + g, k = kbase + 8 t); tiles are 8 rows of W
// (8 * ldw halves) apart
__device__ __forceinline__ void sm_b_fetch(SmB& B, int slot_ch, int ch, const __half* __restrict__ w0,
                                           int ldw, int nu) {
#pragma unroll
    for (int j = 0; j < kSmNu; ++j)
        if (j < nu) B.r[slot_ch][j] = __ldg(reinterpret_cast<const uint4*>(w0 + (size_t)j * 8 * ldw + 32 * ch));
}
__device__ __forceinline__ void sm_b_prefetch(SmB& B, const __half* __restrict__ w0, int ldw, int nu) {
#pragma unroll
    for (int ch = 0; ch < kSmPd; ++ch) sm_b_fetch(B, ch, ch, w0, ldw, nu);
}
// acc[mw][j] = A[mrow0 + 16 mw .. + 16, 0:384] * W[tile j]^T; B holds chunks 0 .. kSmPd - 1 on entry
template <int MW>
__device__ __forceinline__ void sm_tile_mma(const __half* a_tile, int mrow0, SmB& B, const __half* __restrict__ w0,
                                            int ldw, int nu, int g, int t, float (&acc)[MW][kSmNu][4]) {
#pragma unroll
    for (int mw = 0; mw < MW; ++mw)
#pragma unroll
        for (int j = 0; j < kSmNu; ++j)
#pragma unroll
            for (int i = 0; i < 4; ++i) acc[mw][j][i] = 0.f;
    const __half* a_lane = a_tile + (size_t)(mrow0 + g) * kSmLd + 8 * t;
#pragma unroll
    for (int ch = 0; ch < 12; ++ch) {
        uint32_t lo[MW][4], hi[MW][4];
#pragma unroll
        for (int mw = 0; mw < MW; ++mw) {
            const uint4 a0 = *reinterpret_cast<const uint4*>(a_lane + (size_t)(16 * mw) * kSmLd + 32 * ch);
            const uint4 a1 = *reinterpret_cast<const uint4*>(a_lane + (size_t)(16 * mw + 8) * kSmLd + 32 * ch);
            lo[mw][0] = a0.x; lo[mw][1] = a1.x; lo[mw][2] = a0.y; lo[mw][3] = a1.y;
            hi[mw][0] = a0.z; hi[mw][1] = a1.z; hi[mw][2] = a0.w; hi[mw][3] = a1.w;
        }
#pragma unroll
        for (int j = 0; j < kSmNu; ++j) {
            if (j < nu) {
                const uint4 bb = B.r[ch % kSmPd][j];
#pragma unroll
                for (int mw = 0; mw < MW; ++mw) {
                    mma16816(acc[mw][j], lo[mw], bb.x, bb.y);
                    mma16816(acc[mw][j], hi[mw], bb.z, bb.w);
                }
            }
        }
        if (ch + kSmPd < 12) sm_b_fetch(B, ch % kSmPd, ch + kSmPd, w0, ldw, nu);
    }
}

// LayerNorm of row `r`: v[12] = the lane's 12 values (columns j*128 + lane*4 ..), result -> xs row
__device__ __forceinline__ void sm_ln_row(float (&v)[12], const float* __restrict__ gam,
                                          const float* __restrict__ bet, __half* xrow, int lane) {
    float sum = 0.f;
#pragma unroll
    for (int i = 0; i < 12; ++i) sum += v[i];
#pragma unroll
    for (int lb = 16; lb > 0; lb >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, lb);
    const float mean = sum * (1.0f / kHidden);
    float var = 0.f;
#pragma unroll
    for (int i = 0; i < 12; ++i) { const float d = v[i] - mean; var = fmaf(d, d, var); }
#pragma unroll
    for (int lb = 16; lb > 0; lb >>= 1) var += __shfl_xor_sync(0xffffffffu, var, lb);
    const float rstd = 1.0f / sqrtf(var * (1.0f / kHidden) + kLnEps);
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        const int c = j * 128 + lane * 4;
        const float4 gg = __ldg(reinterpret_cast<const float4*>(gam + c));
        const float4 bb = __ldg(reinterpret_cast<const float4*>(bet + c));
        uint2 u;
        u.x = pack_h2((v[4 * j] - mean) * rstd * gg.x + bb.x, (v[4 * j + 1] - mean) * rstd * gg.y + bb.y);
        u.y = pack_h2((v[4 * j + 2] - mean) * rstd * gg.z + bb.z, (v[4 * j + 3] - mean) * rstd * gg.w + bb.w);
        *reinterpret_cast<uint2*>(xrow + c) = u;
    }
}

// attention of ONE (sequence, head) pair by one warp, S <= 16 MT keys: attention_kernel's arithmetic
// (one softmax block) on warp-private staging.  qkv / ctx: the group's scratch, row0 = the
// sequence's first row in it.
template <int MT>
__device__ __forceinline__ void sm_attention_pair(const __half* qkv, int row0, int head, int S, int len,
                                                  __half* sK, __half* sV, __half* ctx, int lane) {
    constexpr int NKB = 2 * MT;                              // 8-key blocks
    const int g = lane >> 2, t = lane & 3;
    const __half* base = qkv + (size_t)row0 * kQkv + head * kHeadDim;
    __syncwarp();                                            // the previous pair's reads are done
    for (int i = lane; i < 16 * MT * 4; i += 32) {
        const int s = i >> 2, part = i & 3;
        const int sr = s < len ? s : 0;
        const uint32_t nbytes = s < len ? 16u : 0u;
        const __half* kp = base + (size_t)sr * kQkv + kHidden + part * 8;
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;"
                     ::"r"(smem_u32(sK + s * kKPad + part * 8)), "l"(kp), "r"(nbytes) : "memory");
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;"
                     ::"r"(smem_u32(sV + s * kKPad + part * 8)), "l"(kp + kHidden), "r"(nbytes) : "memory");
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
    const float scale2 = 0.17677669529663687f * 1.4426950408889634f;
    const int lm = lane >> 3, lr = lane & 7;
    const int n_qtiles = (S + 15) >> 4;
    bool staged = false;
    for (int qt = 0; qt < n_qtiles; ++qt) {
        const int q0 = qt * 16;
        const int r0 = q0 + g, r1 = q0 + g + 8;
        __half* o0 = ctx + (size_t)(row0 + r0) * kHidden + head * kHeadDim;
        __half* o1 = ctx + (size_t)(row0 + r1) * kHidden + head * kHeadDim;
        if (q0 >= len) {                                      // padding tile: zeros
#pragma unroll
            for (int nd = 0; nd < 4; ++nd) {
                if (r0 < S) *reinterpret_cast<uint32_t*>(o0 + nd * 8 + 2 * t) = 0u;
                if (r1 < S) *reinterpret_cast<uint32_t*>(o1 + nd * 8 + 2 * t) = 0u;
            }
            continue;
        }
        uint32_t qa[2][4];
#pragma unroll
        for (int ks = 0; ks < 2; ++ks) {
            const __half* q0p = base + (size_t)r0 * kQkv + ks * 16 + 2 * t;
            const __half* q1p = base + (size_t)r1 * kQkv + ks * 16 + 2 * t;
            qa[ks][0] = (r0 < len) ? __ldcg(reinterpret_cast<const uint32_t*>(q0p)) : 0u;
            qa[ks][1] = (r1 < len) ? __ldcg(reinterpret_cast<const uint32_t*>(q1p)) : 0u;
            qa[ks][2] = (r0 < len) ? __ldcg(reinterpret_cast<const uint32_t*>(q0p + 8)) : 0u;
            qa[ks][3] = (r1 < len) ? __ldcg(reinterpret_cast<const uint32_t*>(q1p + 8)) : 0u;
        }
        if (!staged) {
            asm volatile("cp.async.wait_all;" ::: "memory");
            __syncwarp();
            staged = true;
        }
        float sc[NKB][4];
#pragma unroll
        for (int j = 0; j < NKB; ++j) {
#pragma unroll
            for (int i = 0; i < 4; ++i) sc[j][i] = 0.f;
            uint32_t kf[4];
            ldsm_x4(kf, sK + (j * 8 + lr) * kKPad + lm * 8);
            mma16816(sc[j], qa[0], kf[0], kf[1]);
            mma16816(sc[j], qa[1], kf[2], kf[3]);
        }
#pragma unroll
        for (int j = 0; j < NKB; ++j) {                      // mask keys >= len
            const int key = j * 8 + 2 * t;
            if (key >= len) { sc[j][0] = -INFINITY; sc[j][2] = -INFINITY; }
            if (key + 1 >= len) { sc[j][1] = -INFINITY; sc[j][3] = -INFINITY; }
        }
        float m0 = -INFINITY, m1 = -INFINITY;
#pragma unroll
        for (int j = 0; j < NKB; ++j) {
            m0 = fmaxf(m0, fmaxf(sc[j][0], sc[j][1]));
            m1 = fmaxf(m1, fmaxf(sc[j][2], sc[j][3]));
        }
        m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 1));
        m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 2));
        m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 1));
        m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 2));
        const float nm0 = -m0 * scale2, nm1 = -m1 * scale2;   // finite: key 0 < len
        float l0 = 0.f, l1 = 0.f;
#pragma unroll
        for (int j = 0; j < NKB; ++j) {
            sc[j][0] = ex2(fmaf(sc[j][0], scale2, nm0));
            sc[j][1] = ex2(fmaf(sc[j][1], scale2, nm0));
            sc[j][2] = ex2(fmaf(sc[j][2], scale2, nm1));
            sc[j][3] = ex2(fmaf(sc[j][3], scale2, nm1));
            l0 += sc[j][0] + sc[j][1];
            l1 += sc[j][2] + sc[j][3];
        }
        float o[4][4];
#pragma unroll
        for (int nd = 0; nd < 4; ++nd)
#pragma unroll
            for (int i = 0; i < 4; ++i) o[nd][i] = 0.f;
#pragma unroll
        for (int kk = 0; kk < MT; ++kk) {
            uint32_t pa[4];
            pa[0] = pack_h2(sc[2 * kk][0], sc[2 * kk][1]);
            pa[1] = pack_h2(sc[2 * kk][2], sc[2 * kk][3]);
            pa[2] = pack_h2(sc[2 * kk + 1][0], sc[2 * kk + 1][1]);
            pa[3] = pack_h2(sc[2 * kk + 1][2], sc[2 * kk + 1][3]);
#pragma unroll
            for (int np = 0; np < 2; ++np) {
                uint32_t vf[4];
                ldsm_x4_t(vf, sV + (kk * 16 + (lm & 1) * 8 + lr) * kKPad + (2 * np + (lm >> 1)) * 8);
                mma16816(o[2 * np], pa, vf[0], vf[1]);
                mma16816(o[2 * np + 1], pa, vf[2], vf[3]);
            }
        }
        l0 += __shfl_xor_sync(0xffffffffu, l0, 1);
        l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
        l1 += __shfl_xor_sync(0xffffffffu, l1, 1);
        l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
        const float i0 = 1.0f / l0, i1 = 1.0f / l1;
#pragma unroll
        for (int nd = 0; nd < 4; ++nd) {
            if (r0 < S)
                *reinterpret_cast<uint32_t*>(o0 + nd * 8 + 2 * t) =
                    (r0 < len) ? pack_h2(o[nd][0] * i0, o[nd][1] * i0) : 0u;
            if (r1 < S)
                *reinterpret_cast<uint32_t*>(o1 + nd * 8 + 2 * t) =
                    (r1 < len) ? pack_h2(o[nd][2] * i1, o[nd][3] * i1) : 0u;
        }
    }
    if (!staged) asm volatile("cp.async.wait_all;" ::: "memory");   // len == 0: nothing was consumed
}

template <int MT>
__global__ void __launch_bounds__(kSmThreads, 1)
encoder_small_kernel(const SmallParams P) {
    using G = SmGeom<MT>;
    constexpr int M = G::M;
    extern __shared__ __align__(16) unsigned char sm_raw[];
    __half* xs = reinterpret_cast<__half*>(sm_raw);                       // [M][kSmLd] activations X
    __half* as = reinterpret_cast<__half*>(sm_raw + G::tile_bytes);       // [M][kSmLd] staged A operand
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, t = lane & 3;
    const int c = (int)cluster_ctarank();
    const int grp = blockIdx.x / kSmCtas;
    const int seq0 = grp * P.spg;
    const int nseq = min(P.spg, P.B - seq0);
    const int T = nseq * P.S;                                // rows in use
    unsigned char* sc_base = P.scratch + (size_t)grp * G::scratch;
    __half* s_qkv = reinterpret_cast<__half*>(sc_base + G::o_qkv);
    __half* s_ctx = reinterpret_cast<__half*>(sc_base + G::o_ctx);
    __half* s_ff = reinterpret_cast<__half*>(sc_base + G::o_ff);
    float* s_y = reinterpret_cast<float*>(sc_base + G::o_y);
    float* s_yp = reinterpret_cast<float*>(sc_base + G::o_ypart);
    constexpr int MW = MT / 2;                               // 16-row blocks per warp
    const int mrow0 = (warp & 1) * 16 * MW;                  // the warp's rows
    const int ng = c * 4 + (warp >> 1);                      // its column group in the cluster, 0..31
    SmB Bf;                                                  // B fragments in flight
    float acc[MW][kSmNu][4];
    // column tiles (of 8) per phase: QKV 144 = 16 groups x 5 + 16 x 4; output projection 48 = 16 x 2 +
    // 16 x 1; FFN up 192 = 32 x 6; FFN down: CTA c owns k quarter c & 3 of tiles (c >> 2) * 24 .. + 24
    const int qkv_t0 = ng < 16 ? 5 * ng : 80 + 4 * (ng - 16), qkv_nu = ng < 16 ? 5 : 4;
    const int out_t0 = ng < 16 ? 2 * ng : 32 + (ng - 16), out_nu = ng < 16 ? 2 : 1;
    const int up_t0 = 6 * ng;
    const int kq = c & 3;
    const int dn_t0 = (c >> 2) * 24 + 6 * (warp >> 1);
    auto w_lane = [&](const __half* w, int tile0, int ldw, int kbase) {
        return w + (size_t)(8 * tile0 + g) * ldw + kbase + 8 * t;
    };
    // the first GEMM's first weights go out before anything else
    sm_b_prefetch(Bf, w_lane(P.L[0].wqkv, qkv_t0, kHidden, 0), kHidden, qkv_nu);

    // ---- embeddings + LayerNorm, every row of X in every CTA (rows >= T: zeros)
    for (int r = warp; r < M; r += kSmWarps) {
        __half* xrow = xs + (size_t)r * kSmLd;
        if (r >= T) {
            for (int cc = lane * 4; cc < kHidden; cc += 128) *reinterpret_cast<uint2*>(xrow + cc) = make_uint2(0u, 0u);
            continue;
        }
        int id = P.ids[(size_t)seq0 * P.S + r];
        id = (id < 0 || id >= P.vocab) ? 0 : id;
        int sp = r % P.S;
        sp = (sp >= P.max_pos) ? P.max_pos - 1 : sp;
        float v[12];
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            const int cc = j * 128 + lane * 4;
            const float4 w = __ldg(reinterpret_cast<const float4*>(P.word + (size_t)id * kHidden + cc));
            const float4 p = __ldg(reinterpret_cast<const float4*>(P.pos + (size_t)sp * kHidden + cc));
            const float4 ty = __ldg(reinterpret_cast<const float4*>(P.type0 + cc));
            v[4 * j + 0] = w.x + p.x + ty.x;
            v[4 * j + 1] = w.y + p.y + ty.y;
            v[4 * j + 2] = w.z + p.z + ty.z;
            v[4 * j + 3] = w.w + p.w + ty.w;
        }
        sm_ln_row(v, P.eln_g, P.eln_b, xrow, lane);
    }
    __syncthreads();

    for (int l = 0; l < kLayers; ++l) {
        const SmallLayer& L = P.L[l];
        // ---- (1) QKV projection -> scratch qkv (fp16)
        sm_tile_mma<MW>(xs, mrow0, Bf, w_lane(L.wqkv, qkv_t0, kHidden, 0), kHidden, qkv_nu, g, t, acc);
#pragma unroll
        for (int j = 0; j < kSmNu; ++j) {
            if (j < qkv_nu) {
                const int col = 8 * (qkv_t0 + j) + 2 * t;
                const float2 bb = __ldg(reinterpret_cast<const float2*>(L.bqkv + col));
#pragma unroll
                for (int mw = 0; mw < MW; ++mw) {
                    const int r0 = mrow0 + 16 * mw + g;
                    *reinterpret_cast<uint32_t*>(s_qkv + (size_t)r0 * kQkv + col) =
                        pack_h2(acc[mw][j][0] + bb.x, acc[mw][j][1] + bb.y);
                    *reinterpret_cast<uint32_t*>(s_qkv + (size_t)(r0 + 8) * kQkv + col) =
                        pack_h2(acc[mw][j][2] + bb.x, acc[mw][j][3] + bb.y);
                }
            }
        }
        // the output projection's first weights travel under the attention (32-row groups; with 64
        // rows the attention needs the registers)
        if (MT == 2) sm_b_prefetch(Bf, w_lane(L.wo, out_t0, kHidden, 0), kHidden, out_nu);
        cluster_sync_all();
        // ---- (2) attention: (sequence, head) pairs over kSmAttnWarps warps per CTA
        if (warp < kSmAttnWarps) {
            __half* sK = as + (size_t)warp * (2 * 16 * MT * kKPad);
            __half* sV = sK + 16 * MT * kKPad;
            for (int p = c * kSmAttnWarps + warp; p < nseq * kHeads; p += kSmCtas * kSmAttnWarps) {
                const int sq = p / kHeads, head = p - sq * kHeads;
                int len = P.lens[seq0 + sq];
                len = len < 0 ? 0 : (len > P.S ? P.S : len);
                sm_attention_pair<MT>(s_qkv, sq * P.S, head, P.S, len, sK, sV, s_ctx, lane);
            }
        }
        cluster_sync_all();
        // ---- (3) output projection + residual -> scratch y (fp32); A = ctx staged from the scratch
        for (int i = tid; i < M * 48; i += kSmThreads) {
            const int r = i / 48, part = i - r * 48;
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;"
                         ::"r"(smem_u32(as + (size_t)r * kSmLd + part * 8)), "l"(s_ctx + (size_t)r * kHidden + part * 8)
                         : "memory");
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
        if (MT != 2) sm_b_prefetch(Bf, w_lane(L.wo, out_t0, kHidden, 0), kHidden, out_nu);
        asm volatile("cp.async.wait_all;" ::: "memory");
        __syncthreads();
        sm_tile_mma<MW>(as, mrow0, Bf, w_lane(L.wo, out_t0, kHidden, 0), kHidden, out_nu, g, t, acc);
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            if (j < out_nu) {
                const int col = 8 * (out_t0 + j) + 2 * t;
                const float2 bb = __ldg(reinterpret_cast<const float2*>(L.bo + col));
#pragma unroll
                for (int mw = 0; mw < MW; ++mw) {
                    const int r0 = mrow0 + 16 * mw + g;
                    const float2 x0 = __half22float2(*reinterpret_cast<const __half2*>(xs + (size_t)r0 * kSmLd + col));
                    const float2 x1 = __half22float2(*reinterpret_cast<const __half2*>(xs + (size_t)(r0 + 8) * kSmLd + col));
                    *reinterpret_cast<float2*>(s_y + (size_t)r0 * kHidden + col) =
                        make_float2(acc[mw][j][0] + bb.x + x0.x, acc[mw][j][1] + bb.y + x0.y);
                    *reinterpret_cast<float2*>(s_y + (size_t)(r0 + 8) * kHidden + col) =
                        make_float2(acc[mw][j][2] + bb.x + x1.x, acc[mw][j][3] + bb.y + x1.y);
                }
            }
        }
        // FFN up's first weights travel under the barrier + LayerNorm
        sm_b_prefetch(Bf, w_lane(L.w1, up_t0, kHidden, 0), kHidden, 6);
        cluster_sync_all();
        // ---- (4) LayerNorm 1 (every CTA, all rows; the loads of four rows in flight together) -> X;
        //          FFN up + GELU -> scratch ff (fp16)
#pragma unroll 1
        for (int rb = 0; rb < M / kSmWarps; rb += 4) {
            float v[4][12];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int r = warp + kSmWarps * (rb + i);
#pragma unroll
                for (int j = 0; j < 3; ++j) {
                    const float4 q = __ldcg(reinterpret_cast<const float4*>(s_y + (size_t)r * kHidden + j * 128 + lane * 4));
                    v[i][4 * j] = q.x; v[i][4 * j + 1] = q.y; v[i][4 * j + 2] = q.z; v[i][4 * j + 3] = q.w;
                }
            }
#pragma unroll
            for (int i = 0; i < 4; ++i)
                sm_ln_row(v[i], L.ln1_g, L.ln1_b, xs + (size_t)(warp + kSmWarps * (rb + i)) * kSmLd, lane);
        }
        __syncthreads();
        sm_tile_mma<MW>(xs, mrow0, Bf, w_lane(L.w1, up_t0, kHidden, 0), kHidden, 6, g, t, acc);
#pragma unroll
        for (int j = 0; j < kSmNu; ++j) {
            const int col = 8 * (up_t0 + j) + 2 * t;
            const float2 bb = __ldg(reinterpret_cast<const float2*>(L.b1 + col));
#pragma unroll
            for (int mw = 0; mw < MW; ++mw) {
                const int r0 = mrow0 + 16 * mw + g;
                *reinterpret_cast<uint32_t*>(s_ff + (size_t)r0 * kFfn + col) =
                    pack_h2(gelu_erf(acc[mw][j][0] + bb.x), gelu_erf(acc[mw][j][1] + bb.y));
                *reinterpret_cast<uint32_t*>(s_ff + (size_t)(r0 + 8) * kFfn + col) =
                    pack_h2(gelu_erf(acc[mw][j][2] + bb.x), gelu_erf(acc[mw][j][3] + bb.y));
            }
        }
        sm_b_prefetch(Bf, w_lane(L.w2, dn_t0, kFfn, kq * kHidden), kFfn, 6);
        cluster_sync_all();
        // ---- (5) FFN down: partial sums over this CTA's k quarter -> scratch ypart[kq] (fp32)
        for (int i = tid; i < M * 48; i += kSmThreads) {
            const int r = i / 48, part = i - r * 48;
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;"
                         ::"r"(smem_u32(as + (size_t)r * kSmLd + part * 8)),
                           "l"(s_ff + (size_t)r * kFfn + kq * kHidden + part * 8)
                         : "memory");
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
        asm volatile("cp.async.wait_all;" ::: "memory");
        __syncthreads();
        sm_tile_mma<MW>(as, mrow0, Bf, w_lane(L.w2, dn_t0, kFfn, kq * kHidden), kFfn, 6, g, t, acc);
        {
            float* yp = s_yp + (size_t)kq * M * kHidden;
#pragma unroll
            for (int j = 0; j < kSmNu; ++j) {
                const int col = 8 * (dn_t0 + j) + 2 * t;
#pragma unroll
                for (int mw = 0; mw < MW; ++mw) {
                    const int r0 = mrow0 + 16 * mw + g;
                    *reinterpret_cast<float2*>(yp + (size_t)r0 * kHidden + col) = make_float2(acc[mw][j][0], acc[mw][j][1]);
                    *reinterpret_cast<float2*>(yp + (size_t)(r0 + 8) * kHidden + col) = make_float2(acc[mw][j][2], acc[mw][j][3]);
                }
            }
        }
        cluster_sync_all();
        // ---- (6) the four k quarters in order + bias + residual, LayerNorm 2 -> X (two rows' loads
        //          in flight together)
#pragma unroll 1
        for (int rb = 0; rb < M / kSmWarps; rb += 2) {
            float v[2][12];
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const int r = warp + kSmWarps * (rb + i);
                const __half* xrow = xs + (size_t)r * kSmLd;
#pragma unroll
                for (int j = 0; j < 3; ++j) {
                    const int cc = j * 128 + lane * 4;
                    const size_t o = (size_t)r * kHidden + cc;
                    const float4 p0 = __ldcg(reinterpret_cast<const float4*>(s_yp + o));
                    const float4 p1 = __ldcg(reinterpret_cast<const float4*>(s_yp + (size_t)M * kHidden + o));
                    const float4 p2 = __ldcg(reinterpret_cast<const float4*>(s_yp + 2 * (size_t)M * kHidden + o));
                    const float4 p3 = __ldcg(reinterpret_cast<const float4*>(s_yp + 3 * (size_t)M * kHidden + o));
                    const float4 bb = __ldg(reinterpret_cast<const float4*>(L.b2 + cc));
                    const float2 xa = __half22float2(*reinterpret_cast<const __half2*>(xrow + cc));
                    const float2 xb = __half22float2(*reinterpret_cast<const __half2*>(xrow + cc + 2));
                    v[i][4 * j + 0] = (((p0.x + p1.x) + p2.x) + p3.x) + bb.x + xa.x;
                    v[i][4 * j + 1] = (((p0.y + p1.y) + p2.y) + p3.y) + bb.y + xa.y;
                    v[i][4 * j + 2] = (((p0.z + p1.z) + p2.z) + p3.z) + bb.z + xb.x;
                    v[i][4 * j + 3] = (((p0.w + p1.w) + p2.w) + p3.w) + bb.w + xb.y;
                }
            }
#pragma unroll
            for (int i = 0; i < 2; ++i)
                sm_ln_row(v[i], L.ln2_g, L.ln2_b, xs + (size_t)(warp + kSmWarps * (rb + i)) * kSmLd, lane);
        }
        if (l + 1 < kLayers) sm_b_prefetch(Bf, w_lane(P.L[l + 1].wqkv, qkv_t0, kHidden, 0), kHidden, qkv_nu);
        __syncthreads();
    }

    // ---- pooling + Normalize + normalize_L2: sequence i of the group on CTA i % 8
    __shared__ float red[kSmWarps];
    auto block_sum = [&](float v) -> float {
#pragma unroll
        for (int lb = 16; lb > 0; lb >>= 1) v += __shfl_xor_sync(0xffffffffu, v, lb);
        __syncthreads();
        if (lane == 0) red[warp] = v;
        __syncthreads();
        float s = 0.f;
#pragma unroll
        for (int i = 0; i < kSmWarps; ++i) s += red[i];
        return s;
    };
    for (int sq = c; sq < nseq; sq += kSmCtas) {
        int len = P.lens[seq0 + sq];
        len = len < 0 ? 0 : (len > P.S ? P.S : len);
        const bool two = tid + 256 < kHidden;
        float a0 = 0.f, a1 = 0.f;
        for (int sidx = 0; sidx < len; ++sidx) {
            const __half* row = xs + (size_t)(sq * P.S + sidx) * kSmLd;
            a0 += __half2float(row[tid]);
            if (two) a1 += __half2float(row[tid + 256]);
        }
        const float denom = fmaxf((float)len, 1e-9f);          // torch.clamp(sum_mask, min=1e-9)
        a0 = a0 / denom; a1 = a1 / denom;
        const float nrm = fmaxf(sqrtf(block_sum(a0 * a0 + (two ? a1 * a1 : 0.f))), 1e-12f);   // F.normalize
        a0 = a0 / nrm; a1 = a1 / nrm;
        const float sq2 = block_sum(a0 * a0 + (two ? a1 * a1 : 0.f));
        if (sq2 > 0.f) {                                       // faiss.normalize_L2
            const float inv = 1.0f / sqrtf(sq2);
            a0 *= inv; a1 *= inv;
        }
        const size_t o = (size_t)(seq0 + sq) * kHidden;
        if (P.out_f32 != nullptr) { P.out_f32[o + tid] = a0; if (two) P.out_f32[o + tid + 256] = a1; }
        if (P.out_f16 != nullptr) {
            P.out_f16[o + tid] = __float2half_rn(a0);
            if (two) P.out_f16[o + tid + 256] = __float2half_rn(a1);
        }
    }
}

// ------------------------------------------------------------------ host side
static size_t rup(size_t v, size_t a) { return (v + a - 1) / a * a; }

void encoder_free(lrx_handle* h) {
    Encoder* e = (Encoder*)h->encoder;
    if (e == nullptr) return;
    if (e->blob) cudaFree(e->blob);
    if (e->act) cudaFree(e->act);
    if (e->small_ws) cudaFree(e->small_ws);
    if (e->io) cudaFree(e->io);
    if (e->io_host) cudaFreeHost(e->io_host);
    delete e;
    h->encoder = nullptr;
}

static cudaError_t conv(cudaStream_t st, const float* src, __half* dst, int64_t n) {
    f32_to_f16_kernel<<<256, 256, 0, st>>>(src, dst, n);
    return cudaGetLastError();
}

#define ENC_CK(expr)                          \
    do {                                      \
        cudaError_t _e = (expr);              \
        if (_e != cudaSuccess) return _e;     \
    } while (0)

cudaError_t encoder_set_weights(lrx_handle* h, const lrx_bert_weights* w) {
    encoder_free(h);
    Encoder* e = new Encoder();
    h->encoder = e;
    e->vocab = w->vocab_size;
    e->max_pos = w->max_positions;
    // ---- one blob: fp32 tables + per-layer fp16 matrices + fp32 vectors
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off = rup(off + bytes, 256); return o; };
    const size_t o_word = take((size_t)e->vocab * kHidden * 4);
    const size_t o_pos = take((size_t)e->max_pos * kHidden * 4);
    const size_t o_type = take(kHidden * 4);
    const size_t o_eg = take(kHidden * 4), o_eb = take(kHidden * 4);
    size_t o_l[kLayers][12];
    for (int l = 0; l < kLayers; ++l) {
        o_l[l][0] = take((size_t)kQkv * kHidden * 2);
        o_l[l][1] = take((size_t)kHidden * kHidden * 2);
        o_l[l][2] = take((size_t)kFfn * kHidden * 2);
        o_l[l][3] = take((size_t)kHidden * kFfn * 2);
        o_l[l][4] = take(kQkv * 4);
        o_l[l][5] = take(kHidden * 4);
        o_l[l][6] = take(kFfn * 4);
        o_l[l][7] = take(kHidden * 4);
        for (int i = 8; i < 12; ++i) o_l[l][i] = take(kHidden * 4);
    }
    ENC_CK(cudaMalloc(&e->blob, off));
    char* B = (char*)e->blob;
    cudaStream_t st = h->stream;
    auto cpy = [&](size_t o, const float* src, size_t n) {
        return cudaMemcpyAsync(B + o, src, n * 4, cudaMemcpyDeviceToDevice, st);
    };
    e->word = (float*)(B + o_word); ENC_CK(cpy(o_word, w->word_emb, (size_t)e->vocab * kHidden));
    e->pos = (float*)(B + o_pos);   ENC_CK(cpy(o_pos, w->pos_emb, (size_t)e->max_pos * kHidden));
    e->type0 = (float*)(B + o_type); ENC_CK(cpy(o_type, w->type_emb, kHidden));
    e->eln_g = (float*)(B + o_eg);  ENC_CK(cpy(o_eg, w->emb_ln_g, kHidden));
    e->eln_b = (float*)(B + o_eb);  ENC_CK(cpy(o_eb, w->emb_ln_b, kHidden));
    for (int l = 0; l < kLayers; ++l) {
        const lrx_bert_layer& s = w->layers[l];
        EncLayer& d = e->L[l];
        d.wqkv = (__half*)(B + o_l[l][0]);
        d.wo = (__half*)(B + o_l[l][1]);
        d.w1 = (__half*)(B + o_l[l][2]);
        d.w2 = (__half*)(B + o_l[l][3]);
        d.bqkv = (float*)(B + o_l[l][4]);
        d.bo = (float*)(B + o_l[l][5]);
        d.b1 = (float*)(B + o_l[l][6]);
        d.b2 = (float*)(B + o_l[l][7]);
        d.ln1_g = (float*)(B + o_l[l][8]);
        d.ln1_b = (float*)(B + o_l[l][9]);
        d.ln2_g = (float*)(B + o_l[l][10]);
        d.ln2_b = (float*)(B + o_l[l][11]);
        const int64_t hh = (int64_t)kHidden * kHidden;
        ENC_CK(conv(st, s.wq, d.wqkv, hh));
        ENC_CK(conv(st, s.wk, d.wqkv + hh, hh));
        ENC_CK(conv(st, s.wv, d.wqkv + 2 * hh, hh));
        ENC_CK(conv(st, s.wo, d.wo, hh));
        ENC_CK(conv(st, s.w1, d.w1, (int64_t)kFfn * kHidden));
        ENC_CK(conv(st, s.w2, d.w2, (int64_t)kHidden * kFfn));
        ENC_CK(cpy(o_l[l][4], s.bq, kHidden));
        ENC_CK(cpy(o_l[l][4] + kHidden * 4, s.bk, kHidden));
        ENC_CK(cpy(o_l[l][4] + 2 * kHidden * 4, s.bv, kHidden));
        ENC_CK(cpy(o_l[l][5], s.bo, kHidden));
        ENC_CK(cpy(o_l[l][6], s.b1, kFfn));
        ENC_CK(cpy(o_l[l][7], s.b2, kHidden));
        ENC_CK(cpy(o_l[l][8], s.ln1_g, kHidden));
        ENC_CK(cpy(o_l[l][9], s.ln1_b, kHidden));
        ENC_CK(cpy(o_l[l][10], s.ln2_g, kHidden));
        ENC_CK(cpy(o_l[l][11], s.ln2_b, kHidden));
        for (int pl = 0; pl < 2; ++pl) {
            const int Mp = pl ? (int)kChunkTokens : 128;
            ENC_CK(make_tmap_f16(&d.t_wqkv[pl], d.wqkv, kQkv, kHidden, kHidden,
                                 gemm_box_rows_w(h->num_sms, Mp, kQkv, kHidden, 0)));
            ENC_CK(make_tmap_f16(&d.t_wo[pl], d.wo, kHidden, kHidden, kHidden,
                                 gemm_box_rows_w(h->num_sms, Mp, kHidden, kHidden, 2)));
            ENC_CK(make_tmap_f16(&d.t_w1[pl], d.w1, kFfn, kHidden, kHidden,
                                 gemm_box_rows_w(h->num_sms, Mp, kFfn, kHidden, 1)));
            ENC_CK(make_tmap_f16(&d.t_w2[pl], d.w2, kHidden, kFfn, kFfn,
                                 gemm_box_rows_w(h->num_sms, Mp, kHidden, kFfn, 2)));
        }
    }
    h->launches += 6 * kLayers;
    return cudaStreamSynchronize(st);   // the caller may free its fp32 copies on return
}

static cudaError_t encoder_reserve(Encoder* e, int64_t tokens) {
    if (tokens <= e->cap) return cudaSuccess;
    if (e->act) { ENC_CK(cudaFree(e->act)); e->act = nullptr; e->cap = 0; }
    const int64_t cap = (int64_t)rup((size_t)tokens, 128);
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off = rup(off + bytes, 1024); return o; };
    const size_t o_x = take((size_t)cap * kHidden * 2), o_x1 = take((size_t)cap * kHidden * 2);
    const size_t o_qkv = take((size_t)cap * kQkv * 2), o_ctx = take((size_t)cap * kHidden * 2);
    const size_t o_ff = take((size_t)cap * kFfn * 2);
    ENC_CK(cudaMalloc(&e->act, off));
    ENC_CK(cudaMemset(e->act, 0, off));
    char* A = (char*)e->act;
    e->x = (__half*)(A + o_x); e->x1 = (__half*)(A + o_x1); e->qkv = (__half*)(A + o_qkv);
    e->ctx = (__half*)(A + o_ctx); e->ff = (__half*)(A + o_ff);
    ENC_CK(make_tmap_f16(&e->t_x, e->x, cap, kHidden, kHidden, 128));
    ENC_CK(make_tmap_f16(&e->t_x1, e->x1, cap, kHidden, kHidden, 128));
    ENC_CK(make_tmap_f16(&e->t_ctx, e->ctx, cap, kHidden, kHidden, 128));
    ENC_CK(make_tmap_f16(&e->t_ff, e->ff, cap, kFfn, kFfn, 128));
    ENC_CK(make_tmap_io_f16(&e->io_x, e->x, cap, kHidden, kHidden));
    ENC_CK(make_tmap_io_f16(&e->io_x1, e->x1, cap, kHidden, kHidden));
    ENC_CK(make_tmap_io_f16(&e->io_qkv, e->qkv, cap, kQkv, kQkv));
    ENC_CK(make_tmap_io_f16(&e->io_ff, e->ff, cap, kFfn, kFfn));
    e->cap = cap;
    return cudaSuccess;
}


// Query-sized sequences (S <= 64): the whole forward pass as ONE launch, a cluster of 8 CTAs per
// group of sequences (at most 32 / 64 tokens); kSmMaxGroups groups per launch.
template <int MT>
static cudaError_t encoder_forward_small(lrx_handle* h, Encoder* e, const int32_t* ids, const int32_t* lens,
                                         int B, int S, float* out_f32, void* out_f16) {
    using G = SmGeom<MT>;
    const int spg = G::M / S;                                  // sequences per group, >= 1
    const int groups_all = (B + spg - 1) / spg;
    const int groups_max = groups_all < kSmMaxGroups ? groups_all : kSmMaxGroups;
    const size_t need = (size_t)groups_max * G::scratch;
    if (e->small_ws_bytes < need) {
        if (h->capturing) return cudaErrorStreamCaptureUnsupported;
        ENC_CK(cudaStreamSynchronize(h->stream));
        if (e->small_ws) cudaFree(e->small_ws);
        e->small_ws = nullptr; e->small_ws_bytes = 0;
        h->ws_epoch++;
        ENC_CK(cudaMalloc(&e->small_ws, need));
        // rows of the scratch that no sequence owns are read (row-wise, never mixed with real rows)
        // but never written: keep them finite
        ENC_CK(cudaMemsetAsync(e->small_ws, 0, need, h->stream));
        e->small_ws_bytes = need;
    }
    {
        std::lock_guard<std::recursive_mutex> attr_guard(attr_mutex());   // the flags below are process-wide
        static bool attr_dev[64] = {false};   // function attributes are per device
        bool& attr = attr_dev[h->device & 63];
        if (!attr) {
            ENC_CK(cudaFuncSetAttribute(encoder_small_kernel<MT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (int)G::smem));
            attr = true;
        }
    }
    SmallParams P;
    P.S = S; P.spg = spg; P.vocab = e->vocab; P.max_pos = e->max_pos;
    P.word = e->word; P.pos = e->pos; P.type0 = e->type0; P.eln_g = e->eln_g; P.eln_b = e->eln_b;
    for (int l = 0; l < kLayers; ++l) {
        const EncLayer& s = e->L[l];
        SmallLayer& d = P.L[l];
        d.wqkv = s.wqkv; d.wo = s.wo; d.w1 = s.w1; d.w2 = s.w2;
        d.bqkv = s.bqkv; d.bo = s.bo; d.b1 = s.b1; d.b2 = s.b2;
        d.ln1_g = s.ln1_g; d.ln1_b = s.ln1_b; d.ln2_g = s.ln2_g; d.ln2_b = s.ln2_b;
    }
    P.scratch = (unsigned char*)e->small_ws;
    for (int g0 = 0; g0 < groups_all; g0 += groups_max) {
        const int ng = (groups_all - g0) < groups_max ? (groups_all - g0) : groups_max;
        const int b0 = g0 * spg;
        P.ids = ids + (size_t)b0 * S; P.lens = lens + b0;
        P.B = (B - b0) < ng * spg ? (B - b0) : ng * spg;
        P.out_f32 = out_f32 ? out_f32 + (size_t)b0 * kHidden : nullptr;
        P.out_f16 = out_f16 ? (__half*)out_f16 + (size_t)b0 * kHidden : nullptr;
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(kSmCtas * ng);
        cfg.blockDim = dim3(kSmThreads);
        cfg.dynamicSmemBytes = G::smem;
        cfg.stream = h->stream;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = kSmCtas;
        at[0].val.clusterDim.y = 1;
        at[0].val.clusterDim.z = 1;
        cfg.attrs = at;
        cfg.numAttrs = 1;
        ENC_CK(cudaLaunchKernelEx(&cfg, encoder_small_kernel<MT>, P));
        h->launches++;
    }
    return cudaSuccess;
}

// attention_kernel over nb sequences of S tokens, as the GEMM chain runs it (encoder_forward) and as
// lrx_debug_attention tests it: one CTA per (head, sequence), K / V of all S padded keys reserved in
// dynamic shared memory -- 80 KB at S = 512, past the 48 KB default, hence the one-time opt-in.
static int chunk_sequences(int B, int S) {
    int n = (int)(kChunkTokens / S);
    if (n < 1) n = 1;
    return n > B ? B : n;
}

static cudaError_t launch_attention(lrx_handle* h, const __half* qkv, const int32_t* lens, int nb, int S,
                                    __half* ctx) {
    {
        std::lock_guard<std::recursive_mutex> attr_guard(attr_mutex());   // the flags below are process-wide
        static bool attr_dev[64] = {false};   // function attributes are per device
        bool& attr = attr_dev[h->device & 63];
        if (!attr) {
            ENC_CK(cudaFuncSetAttribute(attention_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        96 * 1024));
            attr = true;
        }
    }
    const int Sk = (S + 63) & ~63;
    const size_t smem = (size_t)Sk * kKPad * 2 * 2;
    ENC_CK(launch_pdl_if(kEncPdlSmall, attention_kernel, dim3(kHeads, nb), dim3(kAttnThreads), smem, h->stream,
                         qkv, lens, S, ctx));
    h->launches++;
    return cudaSuccess;
}

cudaError_t encoder_debug_attention(lrx_handle* h, const void* qkv, const int32_t* lens, int B, int S, void* ctx) {
    const int spc = chunk_sequences(B, S);
    for (int b0 = 0; b0 < B; b0 += spc) {
        const int nb = (B - b0 < spc) ? (B - b0) : spc;
        const size_t row0 = (size_t)b0 * S;
        ENC_CK(launch_attention(h, (const __half*)qkv + row0 * kQkv, lens + b0, nb, S,
                                (__half*)ctx + row0 * kHidden));
    }
    return cudaStreamSynchronize(h->stream);
}

// Which path.  Sequences of at most 64 tokens in batches of at most 64 groups take the cluster
// kernel -- its result for a sequence does not depend on the batch, the padded length or the tile
// variant, so everything a serving front coalesces (serving.py: at most 64 queries per batch)
// embeds exactly as it would alone; bulk work (index build) takes the tcgen05 GEMM chain.  A B200
// holds 14 clusters of 8 at a time: up to 14 groups of 32 rows run as one wave (0.16 ms), more
// sequences are packed into 64-row groups (0.26 ms per wave; from about 30 groups on the chain
// would be faster -- 0.4 ms for 64 x 32 tokens against 0.74 -- which is the price of the invariance).
// 0: chain, 2 / 4: cluster kernel with 32- / 64-row groups.
static int small_path(int B, int S) {
    if (S > 64) return 0;
    if (S <= 32) {
        const int spg = 32 / S;
        if ((B + spg - 1) / spg <= 14) return 2;
    }
    const int spg4 = 64 / S;
    return ((B + spg4 - 1) / spg4 <= 64) ? 4 : 0;
}

cudaError_t encoder_forward(lrx_handle* h, const int32_t* ids, const int32_t* lens, int B, int S,
                            float* out_f32, void* out_f16) {
    Encoder* e = (Encoder*)h->encoder;
    const int sp = small_path(B, S);
    if (sp == 2) return encoder_forward_small<2>(h, e, ids, lens, B, S, out_f32, out_f16);
    if (sp == 4) return encoder_forward_small<4>(h, e, ids, lens, B, S, out_f32, out_f16);
    const int seq_per_chunk = chunk_sequences(B, S);
    if ((int64_t)seq_per_chunk * S > e->cap) {
        // the activation workspace moves: not inside a capture, and captured chains are retired
        if (h->capturing) return cudaErrorStreamCaptureUnsupported;
        h->ws_epoch++;
    }
    ENC_CK(encoder_reserve(e, (int64_t)seq_per_chunk * S));
    cudaStream_t st = h->stream;
    for (int b0 = 0; b0 < B; b0 += seq_per_chunk) {
        const int nb = (B - b0 < seq_per_chunk) ? (B - b0) : seq_per_chunk;
        const int64_t T = (int64_t)nb * S;
        const int32_t* cid = ids + (size_t)b0 * S;
        const int32_t* clen = lens + b0;
        ENC_CK(launch_pdl_if(kEncPdlSmall, embed_ln_kernel, dim3((unsigned)((T + 7) / 8)), dim3(256), 0, st, cid, T, S, e->vocab,
                          e->max_pos, (const float*)e->word, (const float*)e->pos, (const float*)e->type0,
                          (const float*)e->eln_g, (const float*)e->eln_b, e->x));
        h->launches++;
        // which W tensor-map set matches the plan the GEMM launcher picks for this many rows
        const int pl = ((int)((T + 127) / 128) >= h->num_sms / 2) ? 1 : 0;
        for (int l = 0; l < kLayers; ++l) {
            EncLayer& L = e->L[l];
            ENC_CK(launch_tc_gemm(h, e->t_x, L.t_wqkv[pl], e->io_qkv, e->io_qkv, (int)T, kQkv, kHidden, 0,
                                  L.bqkv, nullptr, nullptr, 0.f, e->qkv, kQkv));
            ENC_CK(launch_attention(h, e->qkv, clen, nb, S, e->ctx));
            ENC_CK(launch_tc_gemm(h, e->t_ctx, L.t_wo[pl], e->io_x1, e->io_x, (int)T, kHidden, kHidden, 2,
                                  L.bo, L.ln1_g, L.ln1_b, kLnEps, e->x1, kHidden));
            ENC_CK(launch_tc_gemm(h, e->t_x1, L.t_w1[pl], e->io_ff, e->io_ff, (int)T, kFfn, kHidden, 1,
                                  L.b1, nullptr, nullptr, 0.f, e->ff, kFfn));
            ENC_CK(launch_tc_gemm(h, e->t_ff, L.t_w2[pl], e->io_x, e->io_x1, (int)T, kHidden, kFfn, 2,
                                  L.b2, L.ln2_g, L.ln2_b, kLnEps, e->x, kHidden));
        }
        ENC_CK(launch_pdl_if(kEncPdlSmall, pool_normalize_kernel, dim3(nb), dim3(128), 0, st, (const __half*)e->x, clen, S,
                          out_f32 ? out_f32 + (size_t)b0 * kHidden : (float*)nullptr,
                          out_f16 ? (__half*)out_f16 + (size_t)b0 * kHidden : (__half*)nullptr));
        h->launches++;
    }
    return cudaSuccess;
}

cudaError_t encoder_forward_host(lrx_handle* h, const int32_t* host_ids, const int32_t* host_lens,
                                 int B, int S, float* host_out) {
    Encoder* e = (Encoder*)h->encoder;
    const size_t b_ids = rup((size_t)B * S * 4, 256), b_len = rup((size_t)B * 4, 256);
    const size_t b_out = rup((size_t)B * kHidden * 4, 256);
    const size_t total = b_ids + b_len + b_out;
    if (e->io_bytes < total) {
        if (e->io) cudaFree(e->io);
        if (e->io_host) cudaFreeHost(e->io_host);
        e->io = nullptr; e->io_host = nullptr; e->io_bytes = 0;
        ENC_CK(cudaMalloc(&e->io, total * 2));
        ENC_CK(cudaMallocHost(&e->io_host, total * 2));
        e->io_bytes = total * 2;
    }
    char* hp = (char*)e->io_host;
    char* dp = (char*)e->io;
    memcpy(hp, host_ids, (size_t)B * S * 4);
    memcpy(hp + b_ids, host_lens, (size_t)B * 4);
    ENC_CK(cudaMemcpyAsync(dp, hp, b_ids + b_len, cudaMemcpyHostToDevice, h->stream));
    ENC_CK(encoder_forward(h, (const int32_t*)dp, (const int32_t*)(dp + b_ids), B, S,
                           (float*)(dp + b_ids + b_len), nullptr));
    ENC_CK(cudaMemcpyAsync(hp + b_ids + b_len, dp + b_ids + b_len, (size_t)B * kHidden * 4,
                           cudaMemcpyDeviceToHost, h->stream));
    ENC_CK(cudaStreamSynchronize(h->stream));
    memcpy(host_out, hp + b_ids + b_len, (size_t)B * kHidden * 4);
    return cudaSuccess;
}

}  // namespace lrx
