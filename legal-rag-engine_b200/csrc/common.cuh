// Shared device helpers: mbarrier / bulk-copy PTX, order-preserving keys,
// block-wide bitonic sort, threshold-buffer top-k.  sm_100a only.
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace lrx {

typedef unsigned __int128 u128;

// ---------------------------------------------------------------- PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// Bounded wait: a pipeline bug traps (surfaces as a CUDA error) instead of
// hanging the GPU box.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t spins = 0;
    while (!mbar_try_wait(bar, parity)) {
        if (++spins > (1u << 24)) __trap();   // each failed try_wait already sleeps in HW
    }
}
// Programmatic dependent launch: a kernel launched with launch_pdl() (handle.h) may start while
// its predecessor in the stream still runs; pdl_wait() blocks until the predecessor grid has
// completed and its memory is visible (a no-op under a normal launch), pdl_trigger() lets the
// successor's CTAs be scheduled from now on (a no-op without such a successor).
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// 1-D bulk async copy global -> shared (TMA engine, no tensor map), completion counted in bytes on
// an mbarrier, dst/src 16-byte aligned, bytes % 16 == 0; with an L2 eviction-priority hint: a stream
// that is read once should not push the small structures other kernels keep re-reading (tables,
// bounds, thresholds) out of L2.
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ void bulk_g2s_hint(void* dst, const void* src, uint32_t bytes, uint64_t* bar,
                                              uint64_t policy) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
        ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
        : "memory");
}

// ------------------------------------------------------- order-preserving keys
// Unsigned images of IEEE values whose integer order equals the float order.
__device__ __forceinline__ uint32_t f32_ord(float f) {
    const uint32_t u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float ord_f32(uint32_t o) {
    return __uint_as_float((o & 0x80000000u) ? (o & 0x7fffffffu) : ~o);
}
__device__ __forceinline__ uint64_t f64_ord(double d) {
    const uint64_t u = (uint64_t)__double_as_longlong(d);
    return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}
__device__ __forceinline__ double ord_f64(uint64_t o) {
    return __longlong_as_double((long long)((o >> 63) ? (o & 0x7fffffffffffffffull) : ~o));
}
// (score desc, row asc)  <=>  key desc.  Key 0 is "empty".
__device__ __forceinline__ uint64_t make_key64(float s, uint32_t row) {
    return ((uint64_t)f32_ord(s) << 32) | (uint32_t)(~row);
}
__device__ __forceinline__ uint32_t key64_row(uint64_t k) { return ~(uint32_t)k; }
__device__ __forceinline__ float key64_score(uint64_t k) { return ord_f32((uint32_t)(k >> 32)); }
__device__ __forceinline__ u128 make_key128(double s, uint32_t row) {
    return ((u128)f64_ord(s) << 32) | (u128)(uint32_t)(~row);
}
__device__ __forceinline__ uint32_t key128_row(u128 k) { return ~(uint32_t)k; }
__device__ __forceinline__ double key128_score(u128 k) { return ord_f64((uint64_t)(k >> 32)); }

// --------------------------------------------------------------- bitonic sort
// Sorts `nbuf` independent arrays of `n` keys (n a power of two, arrays `stride`
// apart in shared memory) in DESCENDING order with all threads of the block.
// Caller must __syncthreads() after the last write to keys; returns synced.
template <typename KeyT>
__device__ __forceinline__ void block_bitonic_sort_desc(KeyT* keys, int n, int nbuf, int stride,
                                                        int tid, int nthreads) {
    const int half = n >> 1;
    const int total = half * nbuf;
    const int lh = 31 - __clz(half);                  // half is a power of two
    for (int k = 2; k <= n; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int t = tid; t < total; t += nthreads) {
                const int buf = t >> lh;
                const int u = t & (half - 1);
                const int i = ((u & ~(j - 1)) << 1) | (u & (j - 1));
                const int p = i | j;
                KeyT* kk = keys + (size_t)buf * stride;
                const KeyT a = kk[i], b = kk[p];
                const bool desc = ((i & k) == 0);
                if (desc ? (a < b) : (a > b)) {
                    kk[i] = b;
                    kk[p] = a;
                }
            }
            __syncthreads();
        }
    }
}

// Descending bitonic sort of n (power of two) keys in shared memory by ONE warp:
// ordering between stages is a __syncwarp, no block barrier.
template <typename KeyT>
__device__ __forceinline__ void warp_bitonic_sort_desc(KeyT* keys, int n, int lane) {
    const int half = n >> 1;
    for (int k = 2; k <= n; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int u = lane; u < half; u += 32) {
                const int i = ((u & ~(j - 1)) << 1) | (u & (j - 1));
                const int p = i | j;
                const KeyT a = keys[i], b = keys[p];
                const bool desc = ((i & k) == 0);
                if (desc ? (a < b) : (a > b)) {
                    keys[i] = b;
                    keys[p] = a;
                }
            }
            __syncwarp();
        }
    }
}

__host__ __device__ __forceinline__ int next_pow2(int v) {
    int p = 1;
    while (p < v) p <<= 1;
    return p;
}

}  // namespace lrx
