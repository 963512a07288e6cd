// kc_extract.cu -- extraction into the fixed slot array (sort path).
#include "kc_internal.h"

namespace kc {

template <int W>
struct StoreSink : SinkBase {
    uint64_t *keys;
    __device__ __forceinline__ void operator()(int, uint64_t slot, Key<W> key, bool valid) const {
        if (!valid) {
#pragma unroll
            for (int i = 0; i < W; i++) key.w[i] = 0;
        }
        st_key<W>(keys, slot, key);
    }
};

bool extract_plan(const void *d_reads, uint64_t n_reads, uint32_t L, uint32_t k, uint32_t flags,
                  unsigned long long *d_n_invalid, ExtractParams *out, uint32_t stage_bytes_target) {
    if (k == 0 || k > 128 || L < k || L > 4096) return false;
    if (flags & kPlanCanonical) flags |= kPlanStrict;      // a canonical key is exactly k bases
    const bool strict = (flags & kPlanStrict) != 0;
    ExtractParams p{};
    p.reads = static_cast<const uint8_t *>(d_reads);
    p.n_reads = n_reads;
    p.L = L;
    p.k = k;
    p.nk = L - k + 1;
    p.nw = (L + 31) / 32;
    p.nb4 = (L + 3) / 4;
    uint32_t groups = stage_bytes_target / (16u * L);   // default ~12.5 KB of reads per stage
    p.tile_reads = 16u * (groups ? groups : 1u);
    p.n_tiles = (uint32_t)((n_reads + p.tile_reads - 1) / p.tile_reads);
    p.nk_magic = (uint32_t)((1ull << 32) / p.nk + 1);
    p.nb4_magic = p.nb4 == 1 ? 0xffffffffu : (uint32_t)((1ull << 32) / p.nb4 + 1);
    p.segs_per_read = (p.nk + 17) / 18;                    // ~18 positions per thread-segment (<= 32: one 64-bit lookahead word)
    p.seg_len = (p.nk + p.segs_per_read - 1) / p.segs_per_read;
    uint32_t m = k % 32;
    bool masked = strict ? (m != 0) : (m >= 1 && m <= 28);   // SURVEY F4
    p.last_mask = masked ? (~0ull << (64 - 2 * m)) : ~0ull;
    p.plan_flags = flags & (kPlanStrict | kPlanCanonical);
    p.n_invalid = d_n_invalid;
    extract_smem_layout(p);
    if (p.smem_total > 200 * 1024) return false;
    *out = p;
    return true;
}

template <int W, class Sink>
static cudaError_t launch_extract(const ExtractParams &p, Sink sink, int n_sms, cudaStream_t s) {
    if (p.n_tiles == 0) return cudaSuccess;
    auto kern = extract_kernel_for<W, Sink>(p);
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem_total);
    if (e != cudaSuccess) return e;
    int per_sm = 1;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kExtractThreads, p.smem_total);
    if (e != cudaSuccess) return e;
    if (per_sm < 1) per_sm = 1;
    if (per_sm > 4) per_sm = 4;
    uint32_t grid = (uint32_t)n_sms * per_sm;      // persistent: a whole number of CTAs per SM
    if (grid > p.n_tiles) grid = p.n_tiles;
    kern<<<grid, kExtractThreads, p.smem_total, s>>>(p, sink);
    return cudaGetLastError();
}

cudaError_t launch_extract_store(const ExtractParams &p, int W, uint64_t *d_keys, int n_sms, cudaStream_t s) {
    switch (W) {
        case 1: return launch_extract<1>(p, StoreSink<1>{{}, d_keys}, n_sms, s);
        case 2: return launch_extract<2>(p, StoreSink<2>{{}, d_keys}, n_sms, s);
        case 3: return launch_extract<3>(p, StoreSink<3>{{}, d_keys}, n_sms, s);
        case 4: return launch_extract<4>(p, StoreSink<4>{{}, d_keys}, n_sms, s);
    }
    return cudaErrorInvalidValue;
}

}  // namespace kc
