// kc_spectrum.cu -- count spectrum (histogram of record counts) and count-range filtering of runs.
//
// Both read a finished run (keys, counts) and never touch the counting kernels.
//   histogram: one pass over the counts. Counts of real data pile up in a few low bins, so a warp
//              first merges its lanes' equal bins (__match_any_sync, one atomic per distinct bin),
//              then adds into a per-block shared-memory histogram of the low bins or, above them,
//              straight into the uint64 device histogram. Only non-zero shared bins are flushed.
//   filter:    stable compaction in two passes, so the output is sized exactly and no tile waits on
//              another: survivors per tile, an exclusive scan of the tile totals (one block), then
//              every tile ranks its survivors with a block scan and writes them at its offset.
#include "kc_internal.h"

namespace kc {

namespace {

constexpr int kHistThreads = 256;
constexpr int kHistItems = 4;                       // counts per thread per grid-stride step
constexpr uint32_t kHistSmemBins = 4096;            // 16 KB of shared bins per block (counts 0..4095): 8 blocks fit an SM

constexpr int kFiltThreads = 256;
constexpr int kFiltItems = 8;
constexpr int kFiltTile = kFiltThreads * kFiltItems;
constexpr int kScanThreads = 1024;

__device__ __forceinline__ void hist_add(uint32_t bin, uint32_t *s_hist, uint32_t smem_bins,
                                         unsigned long long *g_hist) {
    const uint32_t peers = __match_any_sync(__activemask(), bin);
    if ((peers & lanemask_lt()) == 0) {             // the lowest lane of each group of equal bins
        const uint32_t v = __popc(peers);
        if (bin < smem_bins) atomicAdd(&s_hist[bin], v);
        else atomicAdd(&g_hist[bin], (unsigned long long)v);
    }
}

__global__ void __launch_bounds__(kHistThreads) histogram_kernel(const uint32_t *__restrict__ counts, uint64_t n,
                                                                 uint32_t n_bins, uint32_t smem_bins,
                                                                 unsigned long long *__restrict__ g_hist) {
    extern __shared__ uint32_t s_hist[];
    for (uint32_t b = threadIdx.x; b < smem_bins; b += kHistThreads) s_hist[b] = 0;
    __syncthreads();
    const uint32_t top = n_bins - 1;
    const uint64_t step = (uint64_t)gridDim.x * kHistThreads * kHistItems;
    for (uint64_t base = (uint64_t)blockIdx.x * kHistThreads * kHistItems; base < n; base += step) {
        uint32_t c[kHistItems];
#pragma unroll
        for (int j = 0; j < kHistItems; j++) {      // all loads first, coalesced: consecutive threads, consecutive counts
            const uint64_t i = base + (uint64_t)j * kHistThreads + threadIdx.x;
            c[j] = i < n ? __ldcs(counts + i) : 0xffffffffu;
        }
#pragma unroll
        for (int j = 0; j < kHistItems; j++) {
            const uint64_t i = base + (uint64_t)j * kHistThreads + threadIdx.x;
            if (i < n) hist_add(c[j] < top ? c[j] : top, s_hist, smem_bins, g_hist);
        }
    }
    __syncthreads();
    for (uint32_t b = threadIdx.x; b < smem_bins; b += kHistThreads) {
        const uint32_t v = s_hist[b];
        if (v) atomicAdd(&g_hist[b], (unsigned long long)v);
    }
}

__device__ __forceinline__ bool in_range(uint32_t c, uint32_t lo, uint32_t hi) { return c >= lo && c <= hi; }

// survivors of every tile
__global__ void __launch_bounds__(kFiltThreads) filter_count_kernel(const uint32_t *__restrict__ counts, uint64_t n,
                                                                    uint32_t lo, uint32_t hi,
                                                                    uint32_t *__restrict__ tile_n) {
    constexpr int WARPS = kFiltThreads / 32;
    __shared__ uint32_t s_warp[WARPS];
    const uint64_t base = (uint64_t)blockIdx.x * kFiltTile;
    uint32_t mine = 0;
#pragma unroll
    for (int j = 0; j < kFiltItems; j++) {
        const uint64_t i = base + (uint64_t)j * kFiltThreads + threadIdx.x;
        mine += (i < n && in_range(counts[i], lo, hi)) ? 1u : 0u;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, o);
    if ((threadIdx.x & 31) == 0) s_warp[threadIdx.x >> 5] = mine;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t t = 0;
#pragma unroll
        for (int w = 0; w < WARPS; w++) t += s_warp[w];
        tile_n[blockIdx.x] = t;
    }
}

// exclusive scan of the tile totals in place (one block; thread t owns a contiguous segment);
// *d_total = survivors in all
__global__ void __launch_bounds__(kScanThreads) filter_scan_kernel(uint64_t *__restrict__ tile_off,
                                                                   const uint32_t *__restrict__ tile_n, uint64_t tiles,
                                                                   unsigned long long *__restrict__ d_total) {
    constexpr int WARPS = kScanThreads / 32;
    __shared__ uint64_t s_warp[WARPS];
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint64_t per = div_up(tiles, (uint64_t)kScanThreads);
    const uint64_t b = (uint64_t)tid * per, e = b + per < tiles ? b + per : tiles;
    uint64_t sum = 0;
    for (uint64_t t = b; t < e; t++) sum += tile_n[t];
    uint64_t incl = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint64_t v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= (uint32_t)o) incl += v;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    uint64_t woff = 0, total = 0;
#pragma unroll
    for (int w = 0; w < WARPS; w++) {
        if (w < (int)warp) woff += s_warp[w];
        total += s_warp[w];
    }
    uint64_t run = woff + incl - sum;
    for (uint64_t t = b; t < e; t++) {
        const uint32_t v = tile_n[t];
        tile_off[t] = run;
        run += v;
    }
    if (tid == 0) *d_total = total;
}

// survivors of every tile, in order, at the tile's offset: keys only loaded for survivors
template <int W>
__global__ void __launch_bounds__(kFiltThreads) filter_write_kernel(const uint64_t *__restrict__ keys,
                                                                    const uint32_t *__restrict__ counts, uint64_t n,
                                                                    uint32_t lo, uint32_t hi,
                                                                    const uint64_t *__restrict__ tile_off,
                                                                    uint64_t *__restrict__ out_keys,
                                                                    uint32_t *__restrict__ out_counts) {
    constexpr int WARPS = kFiltThreads / 32;
    __shared__ uint32_t s_cnt[kFiltItems * WARPS];
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint64_t base = (uint64_t)blockIdx.x * kFiltTile;
    uint32_t c[kFiltItems], ballots[kFiltItems];
#pragma unroll
    for (int j = 0; j < kFiltItems; j++) {
        const uint64_t i = base + (uint64_t)j * kFiltThreads + tid;
        c[j] = i < n ? counts[i] : 0;
        ballots[j] = __ballot_sync(0xffffffffu, i < n && in_range(c[j], lo, hi));
        if (lane == 0) s_cnt[j * WARPS + warp] = __popc(ballots[j]);
    }
    __syncthreads();
    // exclusive scan of the ITEMS x WARPS survivor counts (index order = j-major = record order), one warp
    if (warp == 0) {
        uint32_t total = 0;
        for (int c0 = 0; c0 < kFiltItems * WARPS; c0 += 32) {
            const uint32_t v = (c0 + lane < kFiltItems * WARPS) ? s_cnt[c0 + lane] : 0;
            uint32_t incl = v;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= (uint32_t)o) incl += t;
            }
            if (c0 + lane < kFiltItems * WARPS) s_cnt[c0 + lane] = total + incl - v;
            total += __shfl_sync(0xffffffffu, incl, 31);
        }
    }
    __syncthreads();
    const uint64_t obase = tile_off[blockIdx.x];
    const uint32_t lt = lanemask_lt();
#pragma unroll
    for (int j = 0; j < kFiltItems; j++) {
        if (ballots[j] & (1u << lane)) {
            const uint64_t i = base + (uint64_t)j * kFiltThreads + tid;
            const uint64_t o = obase + s_cnt[j * WARPS + warp] + __popc(ballots[j] & lt);
            st_key<W>(out_keys, o, ld_key<W>(keys, i));
            out_counts[o] = c[j];
        }
    }
}

}  // namespace

cudaError_t run_histogram(const uint32_t *counts, uint64_t n, uint32_t n_bins, unsigned long long *d_hist, int n_sms,
                          cudaStream_t s, int *n_launches) {
    cudaError_t e = cudaMemsetAsync(d_hist, 0, (uint64_t)n_bins * 8, s);
    if (e != cudaSuccess || n == 0) return e;
    const uint32_t smem_bins = n_bins < kHistSmemBins ? n_bins : kHistSmemBins;
    const uint64_t per_block = (uint64_t)kHistThreads * kHistItems;
    const uint64_t want = div_up(n, per_block), cap = (uint64_t)n_sms * 8;
    const uint32_t grid = (uint32_t)(want < cap ? want : cap);
    histogram_kernel<<<grid, kHistThreads, smem_bins * 4, s>>>(counts, n, n_bins, smem_bins, d_hist);
    if (n_launches) *n_launches += 1;
    return cudaGetLastError();
}

uint64_t filter_workspace_bytes(uint64_t n) {
    const uint64_t tiles = div_up(n ? n : 1, (uint64_t)kFiltTile);
    return 256 + tiles * 8 + tiles * 4;
}

cudaError_t filter_count(const uint32_t *counts, uint64_t n, uint32_t lo, uint32_t hi, void *ws,
                         unsigned long long *d_total, cudaStream_t s, int *n_launches) {
    if (n == 0) return cudaMemsetAsync(d_total, 0, 8, s);
    const uint64_t tiles = div_up(n, (uint64_t)kFiltTile);
    if (tiles >= (1ull << 31)) return cudaErrorInvalidValue;
    uint64_t *tile_off = reinterpret_cast<uint64_t *>(static_cast<uint8_t *>(ws) + 256);
    uint32_t *tile_n = reinterpret_cast<uint32_t *>(tile_off + tiles);
    filter_count_kernel<<<(uint32_t)tiles, kFiltThreads, 0, s>>>(counts, n, lo, hi, tile_n);
    filter_scan_kernel<<<1, kScanThreads, 0, s>>>(tile_off, tile_n, tiles, d_total);
    if (n_launches) *n_launches += 2;
    return cudaGetLastError();
}

cudaError_t filter_write(const uint64_t *keys, const uint32_t *counts, uint64_t n, int W, uint32_t lo, uint32_t hi,
                         const void *ws, uint64_t *out_keys, uint32_t *out_counts, cudaStream_t s, int *n_launches) {
    if (n == 0) return cudaSuccess;
    const uint64_t tiles = div_up(n, (uint64_t)kFiltTile);
    const uint64_t *tile_off = reinterpret_cast<const uint64_t *>(static_cast<const uint8_t *>(ws) + 256);
    switch (W) {
        case 1: filter_write_kernel<1><<<(uint32_t)tiles, kFiltThreads, 0, s>>>(keys, counts, n, lo, hi, tile_off, out_keys, out_counts); break;
        case 2: filter_write_kernel<2><<<(uint32_t)tiles, kFiltThreads, 0, s>>>(keys, counts, n, lo, hi, tile_off, out_keys, out_counts); break;
        case 3: filter_write_kernel<3><<<(uint32_t)tiles, kFiltThreads, 0, s>>>(keys, counts, n, lo, hi, tile_off, out_keys, out_counts); break;
        case 4: filter_write_kernel<4><<<(uint32_t)tiles, kFiltThreads, 0, s>>>(keys, counts, n, lo, hi, tile_off, out_keys, out_counts); break;
        default: return cudaErrorInvalidValue;
    }
    if (n_launches) *n_launches += 1;
    return cudaGetLastError();
}

}  // namespace kc
