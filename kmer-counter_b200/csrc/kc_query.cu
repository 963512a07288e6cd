// kc_query.cu -- look keys up in a run: the run's bucket index, the per-slot keys of reads, the lookup.
//
// A run is sorted by key, word 0 first. The index cuts it on the top b bits of word 0: offsets[j] is the
// first record whose top b bits are >= j (j = 0 .. 2^b), so the records of bucket j are
// [offsets[j], offsets[j + 1]). b is picked so that a bucket holds 2 to 4 records of uniform keys; a key
// then costs two offset loads, a binary search of one or two probes and a count load, all random.
#include "kc_internal.h"

namespace kc {

// ---------------------------------------------------------------------------- index
// The bits of word 0 a bucket is selected by: about 2 to 4 records per bucket, no more buckets than the
// key has significant bits for, and an index of at most 2^25 + 1 offsets (256 MiB).
int query_index_bits(uint64_t n, int sig_bits) {
    int lg = 0;
    while (lg < 63 && (2ull << lg) <= n) lg++;          // floor(log2 n), 0 for n <= 1
    int b = lg - 1 < 1 ? 1 : lg - 1;
    if (b > 25) b = 25;
    if (b > sig_bits) b = sig_bits;
    return b;
}

// Two passes over a cleared index, each thread's work bounded. Pass 1, over the records: record i (0 .. n,
// record n standing for the bucket past the last) writes the offsets of the buckets in (bucket(i - 1),
// bucket(i)], at most kIndexGap of them. Pass 2, over the buckets: a bucket pass 1 left clear (it lies in a
// longer empty stretch, where keys crowd into few buckets) gets its lower bound by binary search. On
// uniform keys every stretch is short and pass 2 only reads the index; O(n + 2^b) work, no atomics.
constexpr uint64_t kIndexGap = 64;
constexpr uint64_t kIndexClear = ~0ull;

__global__ void __launch_bounds__(256) query_index_records(const uint64_t *__restrict__ keys, int W, uint64_t n,
                                                           uint32_t shift, uint64_t n_buckets, uint64_t *__restrict__ offsets) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i <= n; i += stride) {
        const uint64_t first = i == 0 ? 0 : (keys[(i - 1) * W] >> shift) + 1;
        const uint64_t last = i == n ? n_buckets : keys[i * W] >> shift;
        if (last + 1 - first <= kIndexGap)
            for (uint64_t j = first; j <= last; j++) offsets[j] = i;
    }
}

__global__ void __launch_bounds__(256) query_index_fill(const uint64_t *__restrict__ keys, int W, uint64_t n,
                                                        uint32_t shift, uint64_t n_buckets, uint64_t *__restrict__ offsets) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; j <= n_buckets; j += stride) {
        if (offsets[j] != kIndexClear) continue;
        uint64_t lo = 0, hi = n;                        // first record whose bucket is >= j
        while (lo < hi) {
            const uint64_t mid = (lo + hi) >> 1;
            if ((keys[mid * W] >> shift) < j) lo = mid + 1;
            else hi = mid;
        }
        offsets[j] = lo;
    }
}

cudaError_t query_index(const uint64_t *keys, int W, uint64_t n, int bits, uint64_t *offsets, int n_sms, cudaStream_t s,
                        int *n_launches) {
    const uint64_t n_buckets = 1ull << bits, cap = (uint64_t)n_sms * 16;
    cudaError_t e = cudaMemsetAsync(offsets, 0xff, (n_buckets + 1) * 8, s);
    if (e != cudaSuccess) return e;
    const uint64_t b1 = div_up(n + 1, 256), b2 = div_up(n_buckets + 1, 256);
    query_index_records<<<(uint32_t)(b1 < cap ? b1 : cap), 256, 0, s>>>(keys, W, n, 64u - bits, n_buckets, offsets);
    query_index_fill<<<(uint32_t)(b2 < cap ? b2 : cap), 256, 0, s>>>(keys, W, n, 64u - bits, n_buckets, offsets);
    *n_launches += 2;
    return cudaGetLastError();
}

// ---------------------------------------------------------------------- keys of reads
// Every slot's key and whether its window holds a k-mer. StoreSink cannot tell the two apart: it stores
// key 0 for a window without a k-mer, and key 0 is also the all-A k-mer.
template <int W>
struct KeyValidSink : SinkBase {
    uint64_t *keys;
    uint8_t *valid;
    __device__ __forceinline__ void operator()(int, uint64_t slot, const Key<W> &key, bool v) const {
        st_key<W>(keys, slot, key);
        valid[slot] = v ? 1 : 0;
    }
};

cudaError_t query_extract(const ExtractParams &p, int W, uint64_t *d_keys, uint8_t *d_valid, int n_sms, cudaStream_t s) {
    switch (W) {
        case 1: return launch_extract<1>(p, KeyValidSink<1>{{}, d_keys, d_valid}, n_sms, s);
        case 2: return launch_extract<2>(p, KeyValidSink<2>{{}, d_keys, d_valid}, n_sms, s);
        case 3: return launch_extract<3>(p, KeyValidSink<3>{{}, d_keys, d_valid}, n_sms, s);
        case 4: return launch_extract<4>(p, KeyValidSink<4>{{}, d_keys, d_valid}, n_sms, s);
    }
    return cudaErrorInvalidValue;
}

// ----------------------------------------------------------------------------- lookup
constexpr int kLookupThreads = 256;
// keys per thread, searched in lockstep so that their loads are in flight together. As many as fit in 32
// registers without spills (full occupancy: 8 CTAs of 256 threads per SM); 256-bit keys take 40 (6 CTAs).
template <int W> __host__ __device__ constexpr int lookup_keys_per_thread() { return W == 1 ? 3 : (W == 2 ? 2 : 1); }

// Thread t of block B takes keys B*256*Q + q*256 + t (q < Q): the loads of the query keys, the counts and
// the validity marks are coalesced, and the slots a warp holds for one q are consecutive.
template <int W>
__global__ void __launch_bounds__(kLookupThreads, W == 4 ? 6 : 8) query_lookup_kernel(QueryLookup p) {
    constexpr int Q = lookup_keys_per_thread<W>();
    const uint64_t base = (uint64_t)blockIdx.x * kLookupThreads * Q + threadIdx.x;
    const uint64_t *__restrict__ rk = p.run_keys;
    Key<W> key[Q];
    uint64_t lo[Q], hi[Q];            // a hit leaves lo = hi = its record
    bool ok[Q], found[Q];
#pragma unroll
    for (int q = 0; q < Q; q++) {
        const uint64_t i = base + (uint64_t)q * kLookupThreads;
        ok[q] = i < p.n && (!p.valid || p.valid[i]);
        bool live = ok[q];
        if (i < p.n) key[q] = ld_key<W>(p.keys, i);
        else
#pragma unroll
            for (int w = 0; w < W; w++) key[q].w[w] = 0;
        if (p.tail_bits && (key[q].w[W - 1] & p.tail_bits)) live = false;     // not a k-mer: bits past its k bases
        if (p.fold) key[q] = key_canonical<W>(key[q], p.rc_sh);
        const uint64_t b = key[q].w[0] >> p.shift;
        lo[q] = live ? p.offsets[b] : 0;
        hi[q] = live ? p.offsets[b + 1] : 0;
        found[q] = false;
    }
    // binary search of [lo, hi) with full-key compares, one probe of every key per round
    bool more = true;
    while (more) {
        more = false;
#pragma unroll
        for (int q = 0; q < Q; q++) {
            if (lo[q] < hi[q]) {
                const uint64_t mid = (lo[q] + hi[q]) >> 1;
                const Key<W> m = ld_key<W>(rk, mid);
                if (key_eq<W>(m, key[q])) { found[q] = true; lo[q] = hi[q] = mid; }
                else if (key_lt<W>(m, key[q])) lo[q] = mid + 1;
                else hi[q] = mid;
                more |= lo[q] < hi[q];
            }
        }
    }
    uint32_t cnt[Q];
#pragma unroll
    for (int q = 0; q < Q; q++) cnt[q] = found[q] ? p.run_counts[lo[q]] : 0u;
#pragma unroll
    for (int q = 0; q < Q; q++) {
        const uint64_t i = base + (uint64_t)q * kLookupThreads;
        if (p.counts && i < p.n) p.counts[i] = cnt[q];
        if (p.hits) {
            // the warp's slots are consecutive, so its lanes' reads are runs of lanes: one atomic per run
            const bool hit = ok[q] && cnt[q] >= p.lo && cnt[q] <= p.hi;
            const uint32_t r = i < p.n ? (uint32_t)i / p.nk : 0xffffffffu;
            const uint32_t lane = threadIdx.x & 31;
            const uint32_t prev = __shfl_up_sync(0xffffffffu, r, 1);
            const uint32_t heads = __ballot_sync(0xffffffffu, lane == 0 || prev != r);
            const uint32_t hits = __ballot_sync(0xffffffffu, hit);
            if ((heads >> lane) & 1u) {
                const uint32_t later = lane == 31 ? 0u : heads & (0xffffffffu << (lane + 1));
                const uint32_t end = later ? (uint32_t)__ffs(later) - 1 : 32u;
                const uint32_t seg = (end == 32 ? 0xffffffffu : (1u << end) - 1u) & (0xffffffffu << lane);
                const uint32_t c = __popc(hits & seg);
                if (c) atomicAdd(&p.hits[r], c);
            }
        }
    }
}

template <int W>
static cudaError_t launch_lookup(const QueryLookup &p, cudaStream_t s) {
    const uint64_t per_block = (uint64_t)kLookupThreads * lookup_keys_per_thread<W>();
    query_lookup_kernel<W><<<(uint32_t)div_up(p.n, per_block), kLookupThreads, 0, s>>>(p);
    return cudaGetLastError();
}

cudaError_t query_lookup(const QueryLookup &p, int W, cudaStream_t s) {
    if (p.n == 0) return cudaSuccess;
    switch (W) {
        case 1: return launch_lookup<1>(p, s);
        case 2: return launch_lookup<2>(p, s);
        case 3: return launch_lookup<3>(p, s);
        case 4: return launch_lookup<4>(p, s);
    }
    return cudaErrorInvalidValue;
}

}  // namespace kc
