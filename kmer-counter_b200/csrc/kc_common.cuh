// kc_common.cuh -- shared device/host helpers for libkc_b200 (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#ifndef __CUDA_ARCH__
#define KC_HOST_ONLY 1
#endif

namespace kc {

constexpr int kMaxWords = 4;        // KMer128: 4 x uint64 (KMerSizes.h:25-28)
constexpr int kRadixBits = 8;
constexpr int kRadixBins = 1 << kRadixBits;

// ---------------------------------------------------------------- key type
// A key is W 64-bit words, word 0 most significant (GPUHandler.cu:247-298 order).
template <int W>
struct alignas(W == 2 || W == 4 ? 16 : 8) Key {
    uint64_t w[W];
};

template <int W>
__host__ __device__ __forceinline__ bool key_eq(const Key<W> &a, const Key<W> &b) {
    bool e = true;
#pragma unroll
    for (int i = 0; i < W; i++) e = e && (a.w[i] == b.w[i]);
    return e;
}

template <int W>
__host__ __device__ __forceinline__ bool key_lt(const Key<W> &a, const Key<W> &b) {
#pragma unroll
    for (int i = 0; i < W; i++) {
        if (a.w[i] < b.w[i]) return true;
        if (a.w[i] > b.w[i]) return false;
    }
    return false;
}

template <int W>
__host__ __device__ __forceinline__ bool key_is_zero(const Key<W> &a) {
    uint64_t o = 0;
#pragma unroll
    for (int i = 0; i < W; i++) o |= a.w[i];
    return o == 0;
}

// ------------------------------------------------------------- small utils
// SMs of the current device (grids of grid-stride kernels are a multiple of it)
inline int sm_count() {
    static int cached[64] = {0};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
    if (cached[dev] == 0) {
        int n = 0;
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        cached[dev] = n > 0 ? n : 148;
    }
    return cached[dev];
}

__host__ __device__ __forceinline__ uint64_t div_up(uint64_t a, uint64_t b) { return (a + b - 1) / b; }

__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31; }
__device__ __forceinline__ uint32_t lanemask_lt() {
    uint32_t m;
    asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
    return m;
}

// streaming (read-once / write-once) global accesses: keep them out of L1
__device__ __forceinline__ uint64_t ld_stream_u64(const uint64_t *p) {
    uint64_t v;
    asm volatile("ld.global.nc.L1::no_allocate.u64 %0, [%1];" : "=l"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ void st_stream_u64(uint64_t *p, uint64_t v) {
    asm volatile("st.global.L1::no_allocate.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

template <int W>
__device__ __forceinline__ Key<W> ld_key(const uint64_t *base, uint64_t idx) {
    Key<W> k;
    if constexpr (W == 2) {
        ulonglong2 v = *reinterpret_cast<const ulonglong2 *>(base + idx * 2);
        k.w[0] = v.x; k.w[1] = v.y;
    } else if constexpr (W == 4) {
        ulonglong2 v0 = *reinterpret_cast<const ulonglong2 *>(base + idx * 4);
        ulonglong2 v1 = *reinterpret_cast<const ulonglong2 *>(base + idx * 4 + 2);
        k.w[0] = v0.x; k.w[1] = v0.y; k.w[2] = v1.x; k.w[3] = v1.y;
    } else {
#pragma unroll
        for (int i = 0; i < W; i++) k.w[i] = base[idx * W + i];
    }
    return k;
}

template <int W>
__device__ __forceinline__ void st_key(uint64_t *base, uint64_t idx, const Key<W> &k) {
    if constexpr (W == 2) {
        *reinterpret_cast<ulonglong2 *>(base + idx * 2) = make_ulonglong2(k.w[0], k.w[1]);
    } else if constexpr (W == 4) {
        *reinterpret_cast<ulonglong2 *>(base + idx * 4) = make_ulonglong2(k.w[0], k.w[1]);
        *reinterpret_cast<ulonglong2 *>(base + idx * 4 + 2) = make_ulonglong2(k.w[2], k.w[3]);
    } else {
#pragma unroll
        for (int i = 0; i < W; i++) base[idx * W + i] = k.w[i];
    }
}

// --------------------------------------------- decoupled look-back (chained scan)
// One 64-bit status word per tile: top 2 bits = state, low 62 bits = value.
// Tiles take their index from an atomic ticket, so every predecessor of a
// waiting tile is already running: the spin below always makes progress.
constexpr uint64_t kLbEmpty = 0, kLbAggregate = 1ull << 62, kLbInclusive = 2ull << 62;
constexpr uint64_t kLbValueMask = (1ull << 62) - 1;

__device__ __forceinline__ uint64_t ld_acquire_u64(const uint64_t *p) {
    uint64_t v;
    asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_u64(uint64_t *p, uint64_t v) {
    asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_u32(const uint32_t *p) {
    uint32_t v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_u32(uint32_t *p, uint32_t v) {
    asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// Decoupled look-back, called by ALL 32 lanes of one warp of the tile. Publishes `aggregate`,
// returns the exclusive prefix over all earlier tiles to every lane, then publishes the inclusive
// value. A window of 32 predecessors is read per round instead of one status word (a tile whose
// predecessors have only published their aggregates walks back 32 at a time, not one L2 round
// trip each).
__device__ __forceinline__ uint64_t lookback_exclusive_warp(uint64_t *status, uint32_t tile, uint64_t aggregate) {
    const uint32_t lane = threadIdx.x & 31;
    if (tile == 0) {
        if (lane == 0) st_release_u64(&status[0], kLbInclusive | aggregate);
        return 0;
    }
    if (lane == 0) st_release_u64(&status[tile], kLbAggregate | aggregate);
    uint64_t excl = 0;
    int64_t base = (int64_t)tile - 1;
    while (true) {
        const int64_t t = base - (int64_t)lane;
        const uint64_t s = t >= 0 ? ld_acquire_u64(&status[t]) : kLbInclusive;      // before tile 0: inclusive, 0
        const uint64_t st = s & ~kLbValueMask;
        const uint32_t inc = __ballot_sync(0xffffffffu, st == kLbInclusive);
        const uint32_t emp = __ballot_sync(0xffffffffu, st == kLbEmpty);
        const uint32_t fi = inc ? (uint32_t)__ffs(inc) - 1 : 32u;                    // nearest predecessor with an inclusive value
        const uint32_t need = fi < 31 ? (2u << fi) - 1u : 0xffffffffu;               // lanes 0 .. fi
        if (emp & need) { __nanosleep(20); continue; }
        uint64_t v = lane <= fi ? (s & kLbValueMask) : 0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        excl += v;
        if (fi < 32) break;
        base -= 32;
    }
    if (lane == 0) st_release_u64(&status[tile], kLbInclusive | (excl + aggregate));
    return excl;
}

// ------------------------------------------------------- TMA bulk copy + mbarrier
__device__ __forceinline__ uint32_t smem_u32(const void *p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t phase) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(phase)
        : "memory");
}
// 1-D bulk copy global -> shared through the TMA unit; bytes % 16 == 0, both 16-B aligned
__device__ __forceinline__ void tma_load_1d(void *smem_dst, const void *gmem_src, uint32_t bytes, uint64_t *bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
            smem_u32(smem_dst)),
        "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}

}  // namespace kc

// ------------------------------------------------------------ host error macros
#define KC_CUDA_TRY(ctx, expr)                                                               \
    do {                                                                                     \
        cudaError_t _e = (expr);                                                             \
        if (_e != cudaSuccess) {                                                             \
            (ctx)->set_error(KC_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, \
                             __LINE__);                                                      \
            cudaGetLastError();  /* a refused call's error must not surface at the next launch check */ \
            return KC_ERR_CUDA;                                                              \
        }                                                                                    \
    } while (0)
