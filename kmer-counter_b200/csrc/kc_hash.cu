// kc_hash.cu -- open-addressing hash-table counting for 64-bit keys (k <= 32).
//
// Replaces the reference's actual counting step at HEAD: one
// tbb::concurrent_hash_map insert per k-mer occurrence on <= 8 host threads
// (KMerCounter.cpp:61-82, hasher KMerCounter.h:42-52) after a D2H of every raw
// record.  Here the extraction kernel inserts straight into a device table, so
// occurrences never exist in memory at all: per occurrence one 16-byte slot is
// claimed (64-bit CAS on the key) and its count bumped (32-bit RED).
//
// Every 64-bit pattern is a legal key (SURVEY H2), so one pattern -- all ones, the
// poly-T window -- is reserved as the empty marker and counted in a side counter.
#include "kc_internal.h"

namespace kc {

namespace {

constexpr uint64_t kEmptyKey = ~0ull;
constexpr uint32_t kMaxProbe = 1u << 16;

__device__ __forceinline__ uint64_t mix64(uint64_t x) {
    x ^= x >> 33; x *= 0xff51afd7ed558ccdull;
    x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ull;
    x ^= x >> 33;
    return x;
}

// returns 1 when this call claimed a fresh slot
__device__ __forceinline__ uint32_t table_add(const HashTable &t, uint64_t k, uint32_t add) {
    if (k == kEmptyKey) { atomicAdd(&t.side[0], (unsigned long long)add); return 0; }
    const uint64_t mask = t.capacity - 1;
    uint64_t h = mix64(k) & mask;
    for (uint32_t probe = 0; probe < kMaxProbe; probe++) {
        unsigned long long *kp = reinterpret_cast<unsigned long long *>(t.slots + 2 * h);
        uint64_t cur = *reinterpret_cast<volatile unsigned long long *>(kp);
        if (cur == kEmptyKey) cur = atomicCAS(kp, kEmptyKey, k);
        if (cur == kEmptyKey || cur == k) {
            if (add) atomicAdd(reinterpret_cast<uint32_t *>(kp + 1), add);
            return cur == kEmptyKey ? 1u : 0u;
        }
        h = (h + 1) & mask;
    }
    t.side[1] = 1;   // table full: the caller falls back to the sort path
    return 0;
}

struct HashSink : SinkBase {
    HashTable t;
    uint32_t claimed;   // slots this thread claimed (= new distinct keys)
    __device__ __forceinline__ void operator()(int, uint64_t, const Key<1> &key, bool valid) {
        if (valid) claimed += table_add(t, key.w[0], 1u);
    }
    // one atomic per warp: side[3] accumulates the number of distinct keys in the table
    __device__ __forceinline__ void finish() {
        uint32_t c = claimed;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
        if ((threadIdx.x & 31) == 0 && c) atomicAdd(&t.side[3], (unsigned long long)c);
    }
};

__global__ void hash_fill_kernel(ulonglong2 *slots, uint64_t capacity) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < capacity; i += stride)
        slots[i] = make_ulonglong2(kEmptyKey, 0ull);
}

// the reference's zero-count key-0 record (SURVEY F7): present whenever any slot was empty
__global__ void hash_touch_zero_kernel(HashTable t, const unsigned long long *d_n_invalid) {
    if (*d_n_invalid) {
        if (table_add(t, 0ull, 0u)) atomicAdd(&t.side[3], 1ull);
    }
}

__global__ void hash_compact_kernel(HashTable t, uint64_t *__restrict__ out_keys, uint32_t *__restrict__ out_counts,
                                    unsigned long long *__restrict__ d_num) {
    const ulonglong2 *slots = reinterpret_cast<const ulonglong2 *>(t.slots);
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    const uint32_t lane = threadIdx.x & 31;
    const uint64_t start = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t rounds = (t.capacity + stride - 1) / stride;
    for (uint64_t r = 0; r < rounds; r++) {
        const uint64_t i = start + r * stride;
        ulonglong2 s = make_ulonglong2(kEmptyKey, 0ull);
        if (i < t.capacity) s = slots[i];
        const bool live = s.x != kEmptyKey;
        const uint32_t bal = __ballot_sync(0xffffffffu, live);
        if (bal) {
            unsigned long long base = 0;
            if (lane == (uint32_t)(__ffs(bal) - 1)) base = atomicAdd(d_num, (unsigned long long)__popc(bal));
            base = __shfl_sync(0xffffffffu, base, __ffs(bal) - 1);
            if (live) {
                const uint64_t o = base + __popc(bal & lanemask_lt());
                out_keys[o] = s.x;
                out_counts[o] = (uint32_t)s.y;
            }
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0 && t.side[0]) {   // the reserved pattern, counted aside
        const unsigned long long o = atomicAdd(d_num, 1ull);
        out_keys[o] = kEmptyKey;
        out_counts[o] = (uint32_t)t.side[0];
    }
}

}  // namespace

uint64_t hash_table_bytes(uint64_t capacity) { return capacity * 16 + 64; }

cudaError_t hash_clear(HashTable t, cudaStream_t s) {
    cudaError_t e = cudaMemsetAsync(t.side, 0, 32, s);
    if (e != cudaSuccess) return e;
    hash_fill_kernel<<<(uint32_t)sm_count() * 8, 256, 0, s>>>(reinterpret_cast<ulonglong2 *>(t.slots), t.capacity);
    return cudaGetLastError();
}

cudaError_t launch_extract_hash(const ExtractParams &p, HashTable t, int n_sms, cudaStream_t s) {
    if (p.n_tiles == 0) return cudaSuccess;
    auto kern = extract_kernel_for<1, HashSink>(p);
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem_total);
    if (e != cudaSuccess) return e;
    int per_sm = 1;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kExtractThreads, p.smem_total);
    if (e != cudaSuccess) return e;
    if (per_sm < 1) per_sm = 1;
    if (per_sm > 6) per_sm = 6;            // random-access bound: more resident warps hide more latency
    uint32_t grid = (uint32_t)n_sms * per_sm;
    if (grid > p.n_tiles) grid = p.n_tiles;
    kern<<<grid, kExtractThreads, p.smem_total, s>>>(p, HashSink{{}, t, 0u});
    return cudaGetLastError();
}

cudaError_t hash_touch_zero(HashTable t, const unsigned long long *d_n_invalid, cudaStream_t s) {
    hash_touch_zero_kernel<<<1, 1, 0, s>>>(t, d_n_invalid);
    return cudaGetLastError();
}

cudaError_t hash_compact(HashTable t, uint64_t *out_keys, uint32_t *out_counts, unsigned long long *d_num,
                         cudaStream_t s, int *n_launches) {
    cudaError_t e = cudaMemsetAsync(d_num, 0, 8, s);
    if (e != cudaSuccess) return e;
    hash_compact_kernel<<<(uint32_t)sm_count() * 8, 256, 0, s>>>(t, out_keys, out_counts, d_num);
    if (n_launches) *n_launches += 1;
    return cudaGetLastError();
}

}  // namespace kc
