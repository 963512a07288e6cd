// kc_partition.cu -- partitioned hash counting for 64- and 128-bit keys (k <= 64), sm_100a.
//
// This is the B200 replacement for the reference's counting step (one TBB hash
// insert per k-mer occurrence on the host, KMerCounter.cpp:61-82) AND for its
// sort + reduce (GPUHandler.cu:300-360) in one design: keys are partitioned by
// their leading bits (= leading bases, so partitions are key ranges and their
// concatenation is already sorted), then every partition is counted in an
// open-addressing hash table that lives in SHARED MEMORY, its distinct keys are
// sorted there, and the records are written once, in final order.
//
// Why: measured on B200 (tools/ubench), shared-memory atomics run at ~2.8 T ops/s
// and 64-bit shared CAS at ~0.75 T ops/s chip-wide, against ~15 G inserts/s for a
// table in HBM and ~380 G keys/s for ballot-based stable ranking.  A most-
// significant-digit partition needs no stable ranking -- a key's position inside
// its bucket is irrelevant -- so ranking is one shared atomicAdd per key.
//
//   P0  hist1     extract (fused encode) -> level-1 digit histogram      reads R*L
//   PA  scatter1  extract -> keys grouped by level-1 digit (2^b1 buckets) writes 8N
//   H2  hist2     level-2 digit histogram inside each bucket             reads 8N
//   PB  scatter2  keys grouped by the b1+b2 leading bits                 reads 8N, writes 8N
//   PC  finish    per sub-bucket: shared-memory hash count, sort of the distinct keys,
//                 ordered write via decoupled look-back                  reads 8N, writes 12U
#include "kc_internal.h"

namespace kc {

namespace {

constexpr int kMaxBins = 1024;          // bins per level
constexpr int kPbThreads = 256;
constexpr int kPbItems = 16;            // 64-bit keys a PB thread moves per tile (128-bit keys: half as many)
template <int W> struct PbCfg { static constexpr int ITEMS = kPbItems / W, TILE = kPbThreads * ITEMS; };
constexpr int kDefaultTarget = 3072;    // keys per sub-bucket the plan aims for

// exclusive scan of nb (<= 1024) shared counters by THREADS threads; every thread returns the total
template <int THREADS, int MAXBINS = kMaxBins>
__device__ __forceinline__ uint32_t block_scan_bins(const uint32_t *cnt, uint32_t *start, int nb, uint32_t *s_warp) {
    constexpr int PER = MAXBINS / THREADS > 0 ? MAXBINS / THREADS : 1;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    uint32_t v[PER];
    uint32_t sum = 0;
#pragma unroll
    for (int i = 0; i < PER; i++) {
        const int b = tid * PER + i;
        v[i] = b < nb ? cnt[b] : 0;
        sum += v[i];
    }
    uint32_t incl = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    uint32_t off = 0, total = 0;
#pragma unroll
    for (int w = 0; w < THREADS / 32; w++) {
        const uint32_t t = s_warp[w];
        if (w < warp) off += t;
        total += t;
    }
    uint32_t run = off + incl - sum;
#pragma unroll
    for (int i = 0; i < PER; i++) {
        const int b = tid * PER + i;
        if (b < nb) start[b] = run;
        run += v[i];
    }
    __syncthreads();
    return total;
}

// ------------------------------------------------------------------- P0: hist1
template <int W>
struct Hist1Sink : SinkBase {
    static constexpr bool kRolling = true;
    static constexpr bool kTopOnlySweep0 = true;
    __device__ __forceinline__ void top(uint32_t top32, bool valid) {
        if (valid) atomicAdd(&sh[top32 >> (shift1 - 32)], 1u);
    }
    uint32_t *g_hist1;
    int shift1, nb1;
    uint32_t *sh;
    __device__ __forceinline__ void begin(uint8_t *extra) {
        sh = reinterpret_cast<uint32_t *>(extra);
        for (int i = threadIdx.x; i < nb1; i += kExtractThreads) sh[i] = 0;
    }
    __device__ __forceinline__ void operator()(int, uint64_t, const Key<W> &key, bool valid) {
        if (valid) atomicAdd(&sh[key.w[0] >> shift1], 1u);
    }
    __device__ __forceinline__ void finish() {
        __syncthreads();
        for (int i = threadIdx.x; i < nb1; i += kExtractThreads) {
            const uint32_t c = sh[i];
            if (c) atomicAdd(&g_hist1[i], c);
        }
    }
};

// one block: bucket bases, the mutable cursors, and the tile map for H2 / PB
__global__ void __launch_bounds__(1024) scan1_kernel(const uint32_t *__restrict__ hist1, int nb1, uint32_t tile_keys,
                                                     uint32_t *__restrict__ base1, uint32_t *__restrict__ cursor1,
                                                     uint32_t *__restrict__ tile_prefix) {
    __shared__ uint32_t s_a[32], s_b[32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t c = tid < nb1 ? hist1[tid] : 0;
    const uint32_t t = (c + tile_keys - 1) / tile_keys;
    uint32_t ia = c, ib = t;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t xa = __shfl_up_sync(0xffffffffu, ia, o), xb = __shfl_up_sync(0xffffffffu, ib, o);
        if (lane >= o) { ia += xa; ib += xb; }
    }
    if (lane == 31) { s_a[warp] = ia; s_b[warp] = ib; }
    __syncthreads();
    uint32_t oa = 0, ob = 0;
    for (int w = 0; w < warp; w++) { oa += s_a[w]; ob += s_b[w]; }
    if (tid < nb1) {
        base1[tid] = oa + ia - c;
        cursor1[tid] = oa + ia - c;
        tile_prefix[tid] = ob + ib - t;
        if (tid == nb1 - 1) { base1[nb1] = oa + ia; tile_prefix[nb1] = ob + ib; }
    }
}

// ---------------------------------------------------------------- PA: scatter1
template <int W>
struct Scatter1Sink : SinkBase {
    static constexpr int kSweeps = 2;
    static constexpr bool kRolling = true;
    static constexpr bool kTopOnlySweep0 = true;
    __device__ __forceinline__ void top(uint32_t top32, bool valid) {      // sweep 0: count the level-1 digit
        if (valid) atomicAdd(&cnt[top32 >> (shift1 - 32)], 1u);
    }
    uint32_t *g_cursor1;
    uint64_t *out;
    int shift1, nb1;
    // shared
    uint32_t *cnt, *start, *gbase, *s_warp;
    Key<W> *staging;
    uint32_t total;
    uint32_t reserved[kMaxBins / kExtractThreads];     // answers of this thread's reservations (registers)

    static __host__ __device__ uint32_t smem_bytes(uint32_t max_tile_keys) {
        return 3 * kMaxBins * 4 + 64 + max_tile_keys * 8 * W;
    }
    __device__ __forceinline__ void begin(uint8_t *extra) {
        cnt = reinterpret_cast<uint32_t *>(extra);
        start = cnt + kMaxBins;
        gbase = start + kMaxBins;
        s_warp = gbase + kMaxBins;
        staging = reinterpret_cast<Key<W> *>(s_warp + 16);
        for (int i = threadIdx.x; i < nb1; i += kExtractThreads) cnt[i] = 0;
        total = 0;
    }
    __device__ __forceinline__ void operator()(int sw, uint64_t, const Key<W> &key, bool valid) {
        if (!valid) return;
        const uint32_t d = (uint32_t)(key.w[0] >> shift1);
        if (sw == 0) {
            atomicAdd(&cnt[d], 1u);
        } else {
            const uint32_t pos = start[d] + atomicAdd(&cnt[d], 1u);
            staging[pos] = key;
        }
    }
    __device__ __forceinline__ void sweep_end(int sw) {
        if (sw == 0) {
            total = block_scan_bins<kExtractThreads>(cnt, start, nb1, s_warp);
            // reserve the bins' ranges now, look at the answers after the placing sweep: the
            // round trips of the global atomics are hidden behind it
#pragma unroll
            for (int u = 0; u < kMaxBins / kExtractThreads; u++) {
                const int b = u * kExtractThreads + threadIdx.x;
                if (b < nb1) {
                    const uint32_t c = cnt[b];
                    if (c) reserved[u] = atomicAdd(&g_cursor1[b], c);
                    cnt[b] = 0;
                }
            }
            __syncthreads();
        } else {
#pragma unroll
            for (int u = 0; u < kMaxBins / kExtractThreads; u++) {
                const int b = u * kExtractThreads + threadIdx.x;
                if (b < nb1) gbase[b] = reserved[u] - start[b];            // dst = gbase[d] + staging index
            }
            __syncthreads();
            // (not unrolled: unrolled by 4, this loop made PA 5 % slower on a B200, 3.18 -> 3.33 ms at C2)
#pragma unroll 1
            for (uint32_t i = threadIdx.x; i < total; i += kExtractThreads) {
                const Key<W> k = staging[i];
                st_key<W>(out, gbase[k.w[0] >> shift1] + i, k);
            }
            for (int b = threadIdx.x; b < nb1; b += kExtractThreads) cnt[b] = 0;
            __syncthreads();
        }
    }
};

// ------------------------------------------------------------------- H2: hist2
// Level-2 histogram of the grouped keys. The grouped array is dense and a key's own leading
// bits name its sub-bucket, so no tile map is needed: a CTA takes a flat chunk of kH2Chunk keys,
// counts those of the chunk's first bucket (all of them, except where the chunk straddles a
// bucket boundary) in shared memory and flushes nb2 counters once per chunk; stragglers add to
// the global counter directly.
constexpr uint32_t kH2Chunk = 32768;
template <int W>
__global__ void __launch_bounds__(kPbThreads) hist2_kernel(const uint64_t *__restrict__ keys,
                                                           const uint32_t *__restrict__ n_keys_ptr, int b2, int shift2,
                                                           uint32_t *__restrict__ g_hist2) {
    __shared__ uint32_t sh[kMaxBins];
    const uint32_t n = *n_keys_ptr;
    const uint32_t begin = blockIdx.x * kH2Chunk;
    if (begin >= n) return;
    const uint32_t end = begin + kH2Chunk < n ? begin + kH2Chunk : n;
    const uint32_t nb2 = 1u << b2, m2 = nb2 - 1;
    for (uint32_t i = threadIdx.x; i < nb2; i += kPbThreads) sh[i] = 0;
    const uint32_t b0 = (uint32_t)(keys[(size_t)begin * W] >> shift2) >> b2;      // word 0 holds the prefix
    __syncthreads();
    auto add = [&](uint64_t w0) {
        const uint32_t pfx = (uint32_t)(w0 >> shift2);
        if ((pfx >> b2) == b0) atomicAdd(&sh[pfx & m2], 1u);
        else atomicAdd(&g_hist2[pfx], 1u);
    };
    if constexpr (W == 1) {
        // begin is a multiple of the chunk: 16-byte loads of two keys
        const ulonglong2 *k2 = reinterpret_cast<const ulonglong2 *>(keys + begin);
        const uint32_t pairs = (end - begin) >> 1;
#pragma unroll 4
        for (uint32_t i = threadIdx.x; i < pairs; i += kPbThreads) {
            const ulonglong2 v = k2[i];
            add(v.x);
            add(v.y);
        }
        if (((end - begin) & 1u) && threadIdx.x == 0) add(keys[end - 1]);
    } else {
#pragma unroll 4
        for (uint32_t i = begin + threadIdx.x; i < end; i += kPbThreads) add(keys[(size_t)i * W]);
    }
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < nb2; i += kPbThreads) {
        const uint32_t c = sh[i];
        if (c) atomicAdd(&g_hist2[(size_t)b0 * nb2 + i], c);
    }
}

// Exclusive scan over all sub-buckets -> base2 (n+1) and the mutable cursors. One CTA per tile of
// 4096 entries; a CTA gets its offset by summing the entries before its tile itself (at most
// 2 MB out of L2), so there is neither a carried dependency between tiles nor scratch memory.
// The input must not alias the outputs.
constexpr uint32_t kScan2Tile = 4096;
__global__ void __launch_bounds__(1024) scan2_kernel(const uint32_t *__restrict__ hist2, uint32_t n,
                                                     uint32_t *__restrict__ base2, uint32_t *__restrict__ cursor2) {
    __shared__ uint32_t s_w[32];
    __shared__ uint32_t s_carry;
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t t0 = blockIdx.x * kScan2Tile;
    uint32_t acc = 0;
#pragma unroll 8
    for (uint32_t i = tid; i < t0; i += 1024) acc += hist2[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) s_w[warp] = acc;
    __syncthreads();
    if (tid == 0) {
        uint32_t c = 0;
        for (int w = 0; w < 32; w++) c += s_w[w];
        s_carry = c;
    }
    __syncthreads();
    const uint32_t i0 = t0 + tid * 4;
    uint32_t v[4];
#pragma unroll
    for (int u = 0; u < 4; u++) v[u] = i0 + u < n ? hist2[i0 + u] : 0;
    const uint32_t sum = v[0] + v[1] + v[2] + v[3];
    uint32_t incl = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= (uint32_t)o) incl += t;
    }
    __syncthreads();                        // s_w is reused
    if (lane == 31) s_w[warp] = incl;
    __syncthreads();
    uint32_t off = s_carry, tot = 0;
#pragma unroll
    for (uint32_t w = 0; w < 32; w++) {
        const uint32_t x = s_w[w];
        if (w < warp) off += x;
        tot += x;
    }
    uint32_t run = off + incl - sum;
#pragma unroll
    for (int u = 0; u < 4; u++) {
        if (i0 + u < n) { base2[i0 + u] = run; cursor2[i0 + u] = run; }
        run += v[u];
    }
    if (tid == 0 && t0 + kScan2Tile >= n) base2[n] = s_carry + tot;    // the last tile closes the scan
}

// ---------------------------------------------------------------- PB: scatter2
// Level-2 scatter over flat tiles of the grouped array (dense, bucket after bucket): the keys'
// own leading bits name bucket and sub-bucket, so a CTA needs no tile map and its loads are in
// flight from the first instruction. Bins are relative to the bucket of the tile's first key
// and span two buckets when the tile straddles a boundary; a key even further away (tiles
// crossing a bucket of fewer than TILE keys) is placed on its own.
template <int W>
__global__ void __launch_bounds__(kPbThreads) scatter2_kernel(const uint64_t *__restrict__ keys,
                                                              uint64_t *__restrict__ out,
                                                              const uint32_t *__restrict__ n_keys_ptr, int b2, int shift2,
                                                              uint32_t *__restrict__ g_cursor2) {
    constexpr int ITEMS = PbCfg<W>::ITEMS, TILE = PbCfg<W>::TILE;
    __shared__ uint32_t cnt[kMaxBins], start[kMaxBins], gbase[kMaxBins];
    __shared__ uint32_t s_warp[kPbThreads / 32];
    __shared__ Key<W> staging[TILE];
    const uint32_t n = *n_keys_ptr;
    const uint32_t begin = blockIdx.x * (uint32_t)TILE;
    if (begin >= n) return;
    const uint32_t end = begin + TILE < n ? begin + TILE : n;
    Key<W> key[ITEMS];
    uint16_t rank[ITEMS];
#pragma unroll
    for (int i = 0; i < ITEMS; i++) {
        const uint32_t idx = begin + i * kPbThreads + threadIdx.x;
        if (idx < end) key[i] = ld_key<W>(keys, idx);
        else key[i].w[0] = 0;
    }
    const uint32_t nb2 = 1u << b2;
    const uint32_t p0 = ((uint32_t)(keys[(size_t)begin * W] >> shift2) >> b2) << b2;     // first sub-bucket of the first key's bucket
    const uint32_t pl = (uint32_t)(keys[(size_t)(end - 1) * W] >> shift2);
    const uint32_t nb = (pl >> b2) == (p0 >> b2) ? nb2 : 2 * nb2;                         // 2 * nb2 <= kMaxBins
    for (uint32_t i = threadIdx.x; i < nb; i += kPbThreads) cnt[i] = 0;
    __syncthreads();
#pragma unroll
    for (int i = 0; i < ITEMS; i++) {
        const uint32_t idx = begin + i * kPbThreads + threadIdx.x;
        rank[i] = 0xffffu;
        if (idx < end) {
            const uint32_t pfx = (uint32_t)(key[i].w[0] >> shift2);
            const uint32_t rel = pfx - p0;
            if (rel < nb) rank[i] = (uint16_t)atomicAdd(&cnt[rel], 1u);
            else st_key<W>(out, atomicAdd(&g_cursor2[pfx], 1u), key[i]);
        }
    }
    __syncthreads();
    const uint32_t total = block_scan_bins<kPbThreads>(cnt, start, (int)nb, s_warp);
    // reserve the bins' ranges, stage the keys while the atomics are in flight, then look at the answers
    uint32_t reserved[kMaxBins / kPbThreads];
#pragma unroll
    for (int u = 0; u < kMaxBins / kPbThreads; u++) {
        const uint32_t b = u * kPbThreads + threadIdx.x;
        reserved[u] = 0;
        if (b < nb) {
            const uint32_t c = cnt[b];
            if (c) reserved[u] = atomicAdd(&g_cursor2[p0 + b], c);
        }
    }
#pragma unroll
    for (int i = 0; i < ITEMS; i++)
        if (rank[i] != 0xffffu) staging[start[(uint32_t)(key[i].w[0] >> shift2) - p0] + rank[i]] = key[i];
#pragma unroll
    for (int u = 0; u < kMaxBins / kPbThreads; u++) {
        const uint32_t b = u * kPbThreads + threadIdx.x;
        if (b < nb) gbase[b] = reserved[u] - start[b];
    }
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < total; i += kPbThreads) {
        const Key<W> k = staging[i];
        st_key<W>(out, gbase[(uint32_t)(k.w[0] >> shift2) - p0] + i, k);
    }
}

// ------------------------------------------------------------------ PC: finish

struct FinishParams {
    const uint64_t *keys;          // grouped by sub-bucket
    const uint32_t *base2;         // [n_sub + 1]
    uint32_t n_sub;
    int prefix_bits;               // b1 + b2
    uint64_t *tmp_keys;            // distinct keys of sub-bucket j land at tmp[base2[j] ...), sorted
    uint32_t *tmp_counts;
    uint32_t *m_out;               // [n_sub] distinct records of each sub-bucket
    unsigned long long *d_overflow;
    const unsigned long long *d_n_invalid;
    int add_phantom;               // KC_COMPAT_REF: key 0 exists whenever a slot was empty (SURVEY F7)
    const uint32_t *list;          // optional: only these sub-buckets (NULL = all)
    const uint32_t *list_count;
    uint32_t *tmp_start;           // [n_sub] where sub-bucket j's records start in tmp (written here, read by the gather)
    // MULTI mode (merging pre-counted parts from several ranks): source s holds sorted unique
    // (key, count) records, src_off[s][j] .. src_off[s][j+1] are those of sub-bucket j
    uint32_t n_src;
    const uint64_t *src_keys[8];
    const uint32_t *src_counts[8];
    const uint32_t *src_off[8];
};

// keys a thread loads before it starts inserting them (64-bit keys, sweep: 16 -> 7.35 ms, 8 -> 6.41, 4 -> 6.03,
// 2 -> 6.04; 128-bit keys: 4 measured better than 2)
constexpr int kPcBatch = 4;
constexpr float kPcLoad = 2.0f;    // table slots per expected distinct key (first guess)
constexpr int kSortBins = 1024;    // most bins the in-table counting sort uses

__device__ __forceinline__ uint32_t pow2_ceil_u32(uint32_t x) { return x <= 1 ? 1u : 1u << (32 - __clz(x - 1)); }

// ---- table slot primitives: 64-bit keys use a 64-bit shared CAS, 128-bit keys ATOMS.CAS.128
template <int W> __device__ __forceinline__ bool key_all_ones(const Key<W> &k) {
    uint64_t a = ~0ull;
#pragma unroll
    for (int i = 0; i < W; i++) a &= k.w[i];
    return a == ~0ull;
}
template <int W> __device__ __forceinline__ bool key_any_word_ones(const Key<W> &k) {
    bool r = false;
#pragma unroll
    for (int i = 0; i < W; i++) r = r || (k.w[i] == ~0ull);
    return r;
}
template <int W> __device__ __forceinline__ void key_set_ones(Key<W> &k) {
#pragma unroll
    for (int i = 0; i < W; i++) k.w[i] = ~0ull;
}
__device__ __forceinline__ Key<1> slot_claim(Key<1> *slot, const Key<1> &k) {      // returns the previous content
    Key<1> o;
    o.w[0] = atomicCAS(reinterpret_cast<unsigned long long *>(slot), ~0ull, (unsigned long long)k.w[0]);
    return o;
}
__device__ __forceinline__ Key<2> slot_claim(Key<2> *slot, const Key<2> &k) {
    Key<2> o;
    const uint32_t a = smem_u32(slot);
    asm volatile(
        "{\n"
        ".reg .b128 c, n, o;\n"
        "mov.b128 c, {%3, %3};\n"
        "mov.b128 n, {%4, %5};\n"
        "atom.shared.cas.b128 o, [%2], c, n;\n"
        "mov.b128 {%0, %1}, o;\n"
        "}\n"
        : "=l"(o.w[0]), "=l"(o.w[1])
        : "r"(a), "l"(~0ull), "l"(k.w[0]), "l"(k.w[1])
        : "memory");
    return o;
}
template <int W> __device__ __forceinline__ uint32_t key_hash(const Key<W> &k) {
    uint32_t x = (uint32_t)k.w[0] ^ (uint32_t)(k.w[0] >> 29);
    if constexpr (W > 1) x ^= ((uint32_t)k.w[W - 1] ^ (uint32_t)(k.w[W - 1] >> 31)) * 0x85EBCA6Bu;
    return x * 0x9E3779B1u;
}

// One CTA per sub-bucket (round-robin over a persistent grid). Nothing here depends on
// another CTA: a sub-bucket with n keys has at most n distinct keys, so its records are
// written to a private range of a temporary array (position 0 is the phantom's) and a later
// gather closes the gaps.
template <int kPcThreads, int kHcap, bool MULTI, int W>
__global__ void __launch_bounds__(kPcThreads) finish_kernel(FinishParams p) {
    static_assert(!MULTI || W == 1, "merging pre-counted parts is implemented for 64-bit keys");
    constexpr int kLcap = kHcap / 2;
    extern __shared__ __align__(16) uint8_t pc_smem[];
    Key<W> *tk = reinterpret_cast<Key<W> *>(pc_smem);               // table keys   [kHcap]
    Key<W> *lk = tk + kHcap;                                        // list keys    [kLcap]
    uint32_t *tc = reinterpret_cast<uint32_t *>(lk + kLcap);        // table counts [kHcap]
    uint32_t *lc = tc + kHcap;                                      // list counts  [kLcap]
    // once the table has been compacted into the list its arrays are reused by the sort:
    Key<W> *sk = tk;                                                // sorted keys   [kLcap]
    uint32_t *sc = reinterpret_cast<uint32_t *>(tk + kLcap);        // sorted counts [kLcap]
    constexpr int kBins = kHcap / 2 < kSortBins ? kHcap / 2 : kSortBins;
    uint32_t *c3 = tc;                                              // counting-sort bins [kBins]
    uint32_t *s3 = tc + kBins;                                      // their starts
    __shared__ uint32_t s_m, s_ones, s_over, s_maxbin;
    __shared__ uint32_t s_warp[kPcThreads / 32];
    const uint32_t tid = threadIdx.x, lane = tid & 31;

    const uint32_t n_work = p.list ? *p.list_count : p.n_sub;
    float ratio = 0.5f;            // distinct / total of the sub-buckets finished so far (uniform across the CTA)
    for (uint32_t jj = blockIdx.x; jj < n_work; jj += gridDim.x) {
        const uint32_t j = p.list ? p.list[jj] : jj;
        uint32_t begin = 0, end = 0, n_in = 0, start_out = 0, floor_m = 0;
        if constexpr (MULTI) {
            for (uint32_t sidx = 0; sidx < p.n_src; sidx++) {
                const uint32_t ns = p.src_off[sidx][j + 1] - p.src_off[sidx][j];
                n_in += ns;
                floor_m = ns > floor_m ? ns : floor_m;        // every part is key-unique already
                start_out += p.src_off[sidx][j] - p.src_off[sidx][0];   // offsets may be absolute (peer arrays) or slice-relative
            }
        } else {
            begin = p.base2[j];
            end = p.base2[j + 1];
            n_in = end - begin;
            start_out = j == 0 ? 0 : begin + 1;       // position 0 of the temporary array is the phantom's
        }
        const bool phantom = !MULTI && (j == 0) && p.add_phantom && (*p.d_n_invalid != 0);
        if (tid == 0) p.tmp_start[j] = start_out;
        if (n_in == 0 && !phantom) {
            if (tid == 0) p.m_out[j] = 0;
            continue;
        }

        // Hash-count the keys of round r (of 2^round_bits) in a table of `cap` slots and compact
        // the distinct ones into lk/lc. Returns false if more than cap/2 are distinct.
        auto build = [&](uint32_t r, uint32_t round_bits, uint32_t cap, uint32_t &m, uint32_t &ones) -> bool {
            Key<W> empty;
            key_set_ones<W>(empty);
            for (uint32_t i = tid; i < cap; i += kPcThreads) { tk[i] = empty; tc[i] = 0; }
            if (tid == 0) { s_m = 0; s_ones = 0; s_over = 0; }
            __syncthreads();
            const int rshift = 64 - p.prefix_bits - (int)round_bits;
            const uint32_t rmask = (1u << round_bits) - 1;
            const uint32_t hshift = __clz(cap) + 1;                  // 32 - log2(cap)
            uint32_t claims = 0;                                     // slots this thread claimed = new distinct keys
            // a probe sequence longer than this means the table is far beyond half full: abandon the attempt
            const uint32_t max_probes = cap < 64 ? cap : 64;
            auto insert = [&](const Key<W> &k, uint32_t add) {
                uint32_t h = key_hash<W>(k) >> hshift;
                for (uint32_t probes = 0; probes < max_probes; probes++) {
                    Key<W> cur = tk[h];
                    // a slot that looks (even partly: a 128-bit read may tear) empty is settled by the CAS
                    if (key_any_word_ones<W>(cur)) {
                        cur = slot_claim(&tk[h], k);
                        if (key_all_ones<W>(cur)) { claims++; if (add) atomicAdd(&tc[h], add); return; }
                    }
                    if (key_eq<W>(cur, k)) { if (add) atomicAdd(&tc[h], add); return; }
                    h = (h + 1) & (cap - 1);
                }
                s_over = 1;
            };
            if constexpr (MULTI) {
                for (uint32_t sidx = 0; sidx < p.n_src; sidx++) {
                    const uint32_t b = p.src_off[sidx][j], e = p.src_off[sidx][j + 1];
                    for (uint32_t i = b + tid; i < e; i += kPcThreads) {
                        if (*reinterpret_cast<volatile uint32_t *>(&s_over)) break;
                        Key<W> k;
                        k.w[0] = p.src_keys[sidx][i];
                        const uint32_t w = p.src_counts[sidx][i];
                        if (round_bits && ((uint32_t)(k.w[0] >> rshift) & rmask) != r) continue;
                        if (key_all_ones<W>(k)) { atomicAdd(&s_ones, w); continue; }
                        insert(k, w);
                    }
                }
            } else {
                // A sub-bucket far larger than the plan's target holds heavy hitters (skewed input):
                // there the lanes of a warp that carry the same key are combined first (MATCH.ANY) and
                // one of them adds their number, instead of 32 atomics serialising on one counter.
                const bool hot = (end - begin) > 16384u;
                if (!hot) {
                    for (uint32_t i0 = begin; i0 < end; i0 += kPcThreads * kPcBatch) {
                        if (*reinterpret_cast<volatile uint32_t *>(&s_over)) break;
                        Key<W> kk[kPcBatch];
#pragma unroll
                        for (int u = 0; u < kPcBatch; u++) {
                            const uint32_t i = i0 + u * kPcThreads + tid;
                            if (i < end) kk[u] = ld_key<W>(p.keys, i);
                            else kk[u].w[0] = 0;
                        }
#pragma unroll
                        for (int u = 0; u < kPcBatch; u++) {
                            const uint32_t i = i0 + u * kPcThreads + tid;
                            if (i >= end) continue;
                            const Key<W> k = kk[u];
                            if (round_bits && ((uint32_t)(k.w[0] >> rshift) & rmask) != r) continue;
                            if (key_all_ones<W>(k)) { atomicAdd(&s_ones, 1u); continue; }
                            insert(k, 1u);
                        }
                    }
                } else {
                    for (uint32_t i0 = begin; i0 < end; i0 += kPcThreads) {
                        uint32_t ov = *reinterpret_cast<volatile uint32_t *>(&s_over);
                        ov = __shfl_sync(0xffffffffu, ov, 0);           // the whole warp leaves together
                        if (ov) break;
                        const uint32_t i = i0 + tid;
                        Key<W> k;
                        k.w[0] = 0;
                        bool act = i < end;
                        if (act) k = ld_key<W>(p.keys, i);
                        if (act && round_bits && ((uint32_t)(k.w[0] >> rshift) & rmask) != r) act = false;
                        if (act && key_all_ones<W>(k)) { atomicAdd(&s_ones, 1u); act = false; }
                        const uint32_t am = __ballot_sync(0xffffffffu, act);
                        if (act) {
                            uint32_t peers = __match_any_sync(am, (unsigned long long)k.w[0]);
                            if constexpr (W > 1) peers &= __match_any_sync(am, (unsigned long long)k.w[W - 1]);
                            if ((int)lane == __ffs(peers) - 1) insert(k, (uint32_t)__popc(peers));
                        }
                    }
                }
            }
            if (phantom && r == 0 && tid == 0) {                      // key 0 joins with count += 0 (SURVEY F7)
                Key<W> zero;
#pragma unroll
                for (int i = 0; i < W; i++) zero.w[i] = 0;
                insert(zero, 0u);
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) claims += __shfl_xor_sync(0xffffffffu, claims, o);
            if (lane == 0 && claims) atomicAdd(&s_m, claims);
            __syncthreads();
            m = s_m;
            ones = s_ones;
            const bool ok = !s_over && 2 * m <= cap;
            __syncthreads();
            if (!ok) return false;
            if (tid == 0) s_m = 0;
            __syncthreads();
            for (uint32_t i0 = 0; i0 < cap; i0 += kPcThreads) {
                const uint32_t i = i0 + tid;
                const Key<W> k = tk[i];
                const bool live = !key_all_ones<W>(k);
                const uint32_t bal = __ballot_sync(0xffffffffu, live);
                if (bal) {
                    uint32_t b = 0;
                    const int leader = __ffs(bal) - 1;
                    if ((int)lane == leader) b = atomicAdd(&s_m, (uint32_t)__popc(bal));
                    b = __shfl_sync(0xffffffffu, b, leader);
                    if (live) {
                        const uint32_t o = b + __popc(bal & lanemask_lt());
                        lk[o] = k;
                        lc[o] = tc[i];
                    }
                }
            }
            __syncthreads();
            return true;
        };

        // Sort the m (key, count) pairs of lk/lc and write them at ob: counting sort on the
        // next key bits into the (now free) table arrays, then a tiny insertion sort inside each
        // bin; a bitonic network takes over when some bin is crowded.
        auto sort_and_write = [&](uint32_t m, uint32_t ones, uint32_t round_bits, uint64_t ob) {
            uint32_t nb3 = pow2_ceil_u32(m);
            nb3 = nb3 < 64 ? 64 : (nb3 > (uint32_t)kBins ? (uint32_t)kBins : nb3);
            int shift3 = 64 - p.prefix_bits - (int)round_bits - (31 - __clz(nb3));
            if (shift3 < 0) shift3 = 0;
            for (uint32_t i = tid; i < nb3; i += kPcThreads) c3[i] = 0;
            if (tid == 0) s_maxbin = 0;
            __syncthreads();
            constexpr int kPer = (kLcap + kPcThreads - 1) / kPcThreads;
            uint32_t rk[kPer];
#pragma unroll
            for (int u = 0; u < kPer; u++) {
                const uint32_t i = u * kPcThreads + tid;
                if (i < m) rk[u] = atomicAdd(&c3[(uint32_t)(lk[i].w[0] >> shift3) & (nb3 - 1)], 1u);
            }
            __syncthreads();
            uint32_t mx = 0;
            for (uint32_t i = tid; i < nb3; i += kPcThreads) mx = max(mx, c3[i]);
            if (mx > 1) atomicMax(&s_maxbin, mx);
            block_scan_bins<kPcThreads>(c3, s3, (int)nb3, s_warp);
            const uint32_t maxbin = s_maxbin;
            const Key<W> *rk_keys = sk;
            const uint32_t *rk_cnts = sc;
            if (maxbin <= 24) {
#pragma unroll
                for (int u = 0; u < kPer; u++) {
                    const uint32_t i = u * kPcThreads + tid;
                    if (i < m) {
                        const Key<W> k = lk[i];
                        const uint32_t o = s3[(uint32_t)(k.w[0] >> shift3) & (nb3 - 1)] + rk[u];
                        sk[o] = k;
                        sc[o] = lc[i];
                    }
                }
                __syncthreads();
                if (maxbin > 1) {
                    for (uint32_t b = tid; b < nb3; b += kPcThreads) {
                        const uint32_t n = c3[b];
                        if (n < 2) continue;
                        const uint32_t s0 = s3[b];
                        for (uint32_t a = 1; a < n; a++) {        // insertion sort of a handful of keys
                            const Key<W> k = sk[s0 + a];
                            const uint32_t c = sc[s0 + a];
                            uint32_t q = a;
                            while (q > 0 && key_lt<W>(k, sk[s0 + q - 1])) { sk[s0 + q] = sk[s0 + q - 1]; sc[s0 + q] = sc[s0 + q - 1]; q--; }
                            sk[s0 + q] = k;
                            sc[s0 + q] = c;
                        }
                    }
                    __syncthreads();
                }
            } else {
                // crowded bins (keys sharing their next bits): bitonic network over lk/lc
                rk_keys = lk;
                rk_cnts = lc;
                const uint32_t p2 = pow2_ceil_u32(m);
                Key<W> pad;
                key_set_ones<W>(pad);
                for (uint32_t i = m + tid; i < p2; i += kPcThreads) { lk[i] = pad; lc[i] = 0; }
                __syncthreads();
                for (uint32_t size = 2; size <= p2; size <<= 1) {
                    for (uint32_t stride = size >> 1; stride > 0; stride >>= 1) {
                        for (uint32_t t = tid; t < (p2 >> 1); t += kPcThreads) {
                            const uint32_t lo = 2 * t - (t & (stride - 1));
                            const uint32_t hi = lo + stride;
                            const bool up = (lo & size) == 0;
                            const Key<W> a = lk[lo], b = lk[hi];
                            if (key_lt<W>(b, a) == up) {
                                lk[lo] = b; lk[hi] = a;
                                const uint32_t ca = lc[lo]; lc[lo] = lc[hi]; lc[hi] = ca;
                            }
                        }
                        __syncthreads();
                    }
                }
            }
            for (uint32_t i = tid; i < m; i += kPcThreads) {
                st_key<W>(p.tmp_keys, ob + i, rk_keys[i]);
                p.tmp_counts[ob + i] = rk_cnts[i];
            }
            if (ones && tid == 0) {                        // the all-ones key is the largest key there is
                Key<W> top;
                key_set_ones<W>(top);
                st_key<W>(p.tmp_keys, ob + m, top);
                p.tmp_counts[ob + m] = ones;
            }
            __syncthreads();
        };

        const uint64_t ob0 = start_out;
        const uint32_t n = n_in + (phantom ? 1u : 0u);
        // First guess from the distinct/total ratio of the sub-buckets this CTA has finished so
        // far (starts at 1/2): table = twice the expected distinct keys; if that exceeds the
        // largest table the keys are taken in 2^round_bits passes (pass r = keys whose next bits
        // are r). A failed attempt is abandoned early, quadruples the table, then halves the pass.
        uint32_t expect = (uint32_t)((float)n * ratio * 1.25f) + 16;
        if (expect < floor_m) expect = floor_m;
        if (expect > n) expect = n;
        // (at most 4 passes to begin with: an oversized sub-bucket is usually a few heavy hitters, not
        // many distinct keys, and a wrong optimistic guess is abandoned after a couple of thousand keys)
        uint32_t round_bits = 0;
        while ((expect >> round_bits) > (uint32_t)kLcap && round_bits < 2) round_bits++;
        uint32_t cap = pow2_ceil_u32((uint32_t)(kPcLoad * (float)(expect >> round_bits)));
        cap = cap < 256 ? 256 : (cap > (uint32_t)kHcap ? (uint32_t)kHcap : cap);
        while (true) {
            const uint32_t n_rounds = 1u << round_bits;
            uint32_t running = 0;
            bool ok = true;
            for (uint32_t r = 0; r < n_rounds && ok; r++) {
                uint32_t m = 0, ones = 0;
                ok = build(r, round_bits, cap, m, ones);
                if (ok) {
                    sort_and_write(m, ones, round_bits, ob0 + running);
                    running += m + (ones ? 1 : 0);
                }
            }
            if (ok) {
                if (tid == 0) p.m_out[j] = running;
                ratio = 0.5f * ratio + 0.5f * __fdividef((float)running, (float)n);      // steers a guess only
                break;
            }
            if (cap < (uint32_t)kHcap) {
                cap = cap * 4 > (uint32_t)kHcap ? (uint32_t)kHcap : cap * 4;
            } else {
                round_bits += 1;
                if (p.prefix_bits + (int)round_bits > 54 || round_bits > 20) {   // give up: caller re-counts by sorting
                    if (tid == 0) { atomicExch(p.d_overflow, 1ull); p.m_out[j] = 0; }
                    break;
                }
            }
        }
        __syncthreads();
    }
}

// PC's CTA and table shape: 256 threads and 2048 slots, the best of the sweep over CTA and table
// sizes in profiles/r1/finish_variant_sweep.txt
template <bool MULTI, int W>
cudaError_t launch_finish(const FinishParams &fp, int n_sms, uint32_t n_sub, cudaStream_t s) {
    constexpr int THREADS = 256, HCAP = 2048;
    constexpr uint32_t smem = HCAP * (8 * W + 4) + (HCAP / 2) * (8 * W + 4);
    auto kern = finish_kernel<THREADS, HCAP, MULTI, W>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    int per_sm = 1;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, THREADS, smem);
    if (per_sm < 1) per_sm = 1;
    uint32_t grid = (uint32_t)n_sms * per_sm;
    if (grid > n_sub) grid = n_sub;
    kern<<<grid, THREADS, smem, s>>>(fp);
    return cudaGetLastError();
}

// records of sub-bucket j: tmp[src(j) .. src(j) + m_j) -> out[off[j] ...); one warp per sub-bucket
template <int W>
__global__ void __launch_bounds__(256) gather_kernel(const uint64_t *__restrict__ tmp_keys,
                                                     const uint32_t *__restrict__ tmp_counts,
                                                     const uint32_t *__restrict__ tmp_start,
                                                     const uint32_t *__restrict__ off, uint32_t n_sub,
                                                     uint64_t *__restrict__ out_keys,
                                                     uint32_t *__restrict__ out_counts) {
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t warps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t j = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; j < n_sub; j += warps) {
        const uint32_t o0 = off[j], m = off[j + 1] - o0;
        const uint64_t s0 = tmp_start[j];
        for (uint32_t i = lane; i < m; i += 32) {
            st_key<W>(out_keys, o0 + i, ld_key<W>(tmp_keys, s0 + i));
            out_counts[o0 + i] = tmp_counts[s0 + i];
        }
    }
}

}  // namespace

// ------------------------------------------------------------------------ host
struct PartitionPlan {
    int b1, b2;
    uint32_t nb1, nb2, n_sub;
};

static PartitionPlan make_plan(uint64_t n_slots, int sig_bits, int target) {
    int B = 2;
    while (B < 20 && (n_slots >> B) > (uint64_t)target) B++;
    if (B > sig_bits) B = sig_bits;        // never partition on bits that are always zero (masked tail)
    if (B < 2) B = 2;
    PartitionPlan pl;
    pl.b1 = (B + 1) / 2;
    pl.b2 = B - pl.b1;
    pl.nb1 = 1u << pl.b1;
    pl.nb2 = 1u << pl.b2;
    pl.n_sub = pl.nb1 * pl.nb2;
    return pl;
}

// Second half of the partitioned count, run once the number of records is known on the
// host: closes the gaps between the sub-buckets' record ranges.
cudaError_t partition_gather(int W, uint64_t n_slots, int sig_bits, int target_sub, const uint64_t *tmp_keys,
                             const uint32_t *tmp_counts, void *ws, uint64_t *out_keys, uint32_t *out_counts,
                             cudaStream_t s) {
    const PartitionPlan pl = make_plan(n_slots, sig_bits, target_sub > 0 ? target_sub : kDefaultTarget);
    uint32_t *hist1 = reinterpret_cast<uint32_t *>(ws);
    uint32_t *hist2 = hist1 + 4 * (kMaxBins + 8);
    uint32_t *base2 = hist2 + pl.n_sub + 8;
    uint32_t *off = base2 + pl.n_sub + 8;
    uint32_t *tmp_start = off + pl.n_sub + 8 + pl.n_sub + 8;
    if (W == 1) gather_kernel<1><<<(uint32_t)sm_count() * 8, 256, 0, s>>>(tmp_keys, tmp_counts, tmp_start, off, pl.n_sub, out_keys, out_counts);
    else gather_kernel<2><<<(uint32_t)sm_count() * 8, 256, 0, s>>>(tmp_keys, tmp_counts, tmp_start, off, pl.n_sub, out_keys, out_counts);
    return cudaGetLastError();
}

// The plan a chunk of n_slots k-mer slots is counted with, and where the per-sub-bucket
// record offsets (n_sub + 1 entries, valid after partition_count) live inside ws.
void partition_plan_info(uint64_t n_slots, int sig_bits, int target_sub, void *ws, uint32_t *n_sub,
                         uint32_t *prefix_bits, const uint32_t **d_offsets) {
    const PartitionPlan pl = make_plan(n_slots, sig_bits, target_sub > 0 ? target_sub : kDefaultTarget);
    *n_sub = pl.n_sub;
    *prefix_bits = (uint32_t)(pl.b1 + pl.b2);
    if (d_offsets) {
        const uint32_t *hist1 = reinterpret_cast<const uint32_t *>(ws);
        *d_offsets = hist1 + 4 * (kMaxBins + 8) + 2 * (pl.n_sub + 8);
    }
}

uint64_t merge_parts_workspace_bytes(uint32_t n_sub) { return (uint64_t)(4 * (n_sub + 8)) * 4 + 256; }

// Merge pre-counted parts: n_src sources of sorted unique (key, count) records covering the
// same n_sub consecutive sub-buckets (src_off[s] = n_sub + 1 offsets into source s). Equal keys
// are summed in shared-memory tables, sub-bucket by sub-bucket; records land in tmp arrays
// (capacity = total input records + 1), *d_num_out = records. Finish with merge_parts_gather.
cudaError_t merge_parts_count(uint32_t n_src, const uint64_t *const *src_keys, const uint32_t *const *src_counts,
                              const uint32_t *const *src_off, uint32_t n_sub, int prefix_bits, uint64_t *tmp_keys,
                              uint32_t *tmp_counts, unsigned long long *d_num_out, unsigned long long *d_overflow,
                              void *ws, int n_sms, cudaStream_t s, int *n_launches) {
    if (n_src == 0 || n_src > 8) return cudaErrorInvalidValue;
    uint32_t *m_out = reinterpret_cast<uint32_t *>(ws);
    uint32_t *off = m_out + n_sub + 8;
    uint32_t *tmp_start = off + n_sub + 8;
    uint32_t *scratch = tmp_start + n_sub + 8;
    cudaError_t e;
    if ((e = cudaMemsetAsync(d_num_out, 0, 8, s)) != cudaSuccess) return e;
    if ((e = cudaMemsetAsync(d_overflow, 0, 8, s)) != cudaSuccess) return e;
    FinishParams fp{};
    fp.n_sub = n_sub;
    fp.prefix_bits = prefix_bits;
    fp.tmp_keys = tmp_keys;
    fp.tmp_counts = tmp_counts;
    fp.m_out = m_out;
    fp.d_overflow = d_overflow;
    fp.tmp_start = tmp_start;
    fp.n_src = n_src;
    for (uint32_t i = 0; i < n_src; i++) { fp.src_keys[i] = src_keys[i]; fp.src_counts[i] = src_counts[i]; fp.src_off[i] = src_off[i]; }
    if ((e = launch_finish<true, 1>(fp, n_sms, n_sub, s)) != cudaSuccess) return e;
    scan2_kernel<<<(n_sub + kScan2Tile - 1) / kScan2Tile, 1024, 0, s>>>(m_out, n_sub, off, scratch);
    if ((e = cudaMemcpyAsync(d_num_out, off + n_sub, 4, cudaMemcpyDeviceToDevice, s)) != cudaSuccess) return e;
    if (n_launches) *n_launches += 2;
    return cudaGetLastError();
}

cudaError_t merge_parts_gather(uint32_t n_sub, const uint64_t *tmp_keys, const uint32_t *tmp_counts, void *ws,
                               uint64_t *out_keys, uint32_t *out_counts, uint32_t *out_offsets, cudaStream_t s) {
    uint32_t *m_out = reinterpret_cast<uint32_t *>(ws);
    uint32_t *off = m_out + n_sub + 8;
    uint32_t *tmp_start = off + n_sub + 8;
    gather_kernel<1><<<(uint32_t)sm_count() * 8, 256, 0, s>>>(tmp_keys, tmp_counts, tmp_start, off, n_sub, out_keys, out_counts);
    if (out_offsets) {
        cudaError_t e = cudaMemcpyAsync(out_offsets, off, (size_t)(n_sub + 1) * 4, cudaMemcpyDeviceToDevice, s);
        if (e != cudaSuccess) return e;
    }
    return cudaGetLastError();
}

bool partition_two_levels(uint64_t n_slots, int sig_bits, int target_sub) {
    return make_plan(n_slots, sig_bits, target_sub > 0 ? target_sub : kDefaultTarget).b2 > 0;
}

uint64_t partition_workspace_bytes(uint64_t n_slots) {
    (void)n_slots;
    const uint64_t nsub = 1u << 20;
    // hist1, base1, cursor1, tile_prefix | hist2, base2, cursor2 | status | flags
    return 4 * (kMaxBins + 8) * 4 + 3 * (nsub + 8) * 4 + nsub * 8 + 256;
}

// Counts the k-mers of `ep` (W = 1 or 2 words per key) into sorted unique (out_keys, out_counts).
// keys_a / keys_b: scratch of n_slots keys each. *d_num_out = records; *d_overflow != 0
// means a sub-bucket could not be counted (caller falls back to sort + run-length).
template <int W>
static cudaError_t partition_count_w(const ExtractParams &ep_in, uint64_t n_slots, int sig_bits, bool add_phantom,
                                     uint64_t *keys_a, uint64_t *keys_b, uint64_t *out_keys, uint32_t *out_counts,
                                     unsigned long long *d_num_out, unsigned long long *d_overflow,
                                     unsigned long long *d_scratch_invalid, void *ws, int n_sms, int target_sub,
                                     cudaStream_t s, int *n_launches, cudaEvent_t *evs) {
    const PartitionPlan pl = make_plan(n_slots, sig_bits, target_sub > 0 ? target_sub : kDefaultTarget);
    uint8_t *w = static_cast<uint8_t *>(ws);
    uint32_t *hist1 = reinterpret_cast<uint32_t *>(w);
    uint32_t *base1 = hist1 + kMaxBins + 8;
    uint32_t *cursor1 = base1 + kMaxBins + 8;
    uint32_t *tile_prefix = cursor1 + kMaxBins + 8;
    uint32_t *hist2 = tile_prefix + kMaxBins + 8;
    uint32_t *base2 = hist2 + pl.n_sub + 8;
    uint32_t *cursor2 = base2 + pl.n_sub + 8;
    uint32_t *status_scratch = cursor2 + pl.n_sub + 8;       // n_sub + 8 entries, scratch for the second scan
    cudaError_t e;
    const size_t zero_bytes = reinterpret_cast<uint8_t *>(status_scratch) - w;
    if ((e = cudaMemsetAsync(ws, 0, zero_bytes, s)) != cudaSuccess) return e;
    if ((e = cudaMemsetAsync(d_num_out, 0, 8, s)) != cudaSuccess) return e;
    if ((e = cudaMemsetAsync(d_overflow, 0, 8, s)) != cudaSuccess) return e;

    const int shift1 = 64 - pl.b1, shift2 = 64 - pl.b1 - pl.b2;
    // P0: level-1 histogram (invalid-slot count goes to a scratch counter: PA counts it for real)
    {
        // the histogram pass keeps nothing per tile, so it takes larger tiles than PA (fewer barriers
        // per read): 12800 bytes of reads
        ExtractParams ep = ep_in;
        if (!extract_plan(ep_in.reads, ep_in.n_reads, ep_in.L, ep_in.k, ep_in.plan_flags, d_scratch_invalid, &ep, 12800))
            ep = ep_in;
        ep.n_invalid = d_scratch_invalid;
        auto kern = extract_kernel_for<W, Hist1Sink<W>>(ep_in);
        const uint32_t smem = ep.smem_total + kMaxBins * 4;
        if ((e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess) return e;
        int per_sm = 1;
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kExtractThreads, smem);
        per_sm = per_sm < 1 ? 1 : (per_sm > 6 ? 6 : per_sm);
        uint32_t grid = (uint32_t)n_sms * per_sm;
        if (grid > ep.n_tiles) grid = ep.n_tiles;
        Hist1Sink<W> sink{};
        sink.g_hist1 = hist1; sink.shift1 = shift1; sink.nb1 = (int)pl.nb1;
        kern<<<grid, kExtractThreads, smem, s>>>(ep, sink);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
    }
    scan1_kernel<<<1, 1024, 0, s>>>(hist1, (int)pl.nb1, (uint32_t)PbCfg<W>::TILE, base1, cursor1, tile_prefix);
    if (evs) cudaEventRecord(evs[0], s);
    // PA: keys grouped by level-1 digit
    {
        auto kern = extract_kernel_for<W, Scatter1Sink<W>>(ep_in);
        const uint32_t max_tile_keys = ep_in.tile_reads * ep_in.nk;
        const uint32_t smem = ep_in.smem_total + Scatter1Sink<W>::smem_bytes(max_tile_keys);
        if ((e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess) return e;
        int per_sm = 1;
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kExtractThreads, smem);
        per_sm = per_sm < 1 ? 1 : (per_sm > 6 ? 6 : per_sm);
        uint32_t grid = (uint32_t)n_sms * per_sm;
        if (grid > ep_in.n_tiles) grid = ep_in.n_tiles;
        Scatter1Sink<W> sink{};
        sink.g_cursor1 = cursor1; sink.out = keys_a; sink.shift1 = shift1; sink.nb1 = (int)pl.nb1;
        kern<<<grid, kExtractThreads, smem, s>>>(ep_in, sink);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
    }
    if (evs) cudaEventRecord(evs[1], s);
    // H2 + PB over the level-1 buckets
    if (pl.b2 > 0) {
        hist2_kernel<W><<<(uint32_t)div_up(n_slots, (uint64_t)kH2Chunk), kPbThreads, 0, s>>>(keys_a, base1 + pl.nb1, pl.b2, shift2, hist2);
        scan2_kernel<<<(pl.n_sub + kScan2Tile - 1) / kScan2Tile, 1024, 0, s>>>(hist2, pl.n_sub, base2, cursor2);
        if (evs) cudaEventRecord(evs[2], s);
        scatter2_kernel<W><<<(uint32_t)div_up(n_slots, (uint64_t)PbCfg<W>::TILE), kPbThreads, 0, s>>>(
            keys_a, keys_b, base1 + pl.nb1, pl.b2, shift2, cursor2);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
    } else {
        if ((e = cudaMemcpyAsync(base2, base1, (pl.nb1 + 1) * 4, cudaMemcpyDeviceToDevice, s)) != cudaSuccess) return e;
        if (evs) cudaEventRecord(evs[2], s);
    }
    const uint64_t *grouped = pl.b2 > 0 ? keys_b : keys_a;
    if (evs) cudaEventRecord(evs[3], s);
    // PC: count + sort per sub-bucket into the temporary arrays, then offsets of the survivors
    {
        if (out_keys == grouped) return cudaErrorInvalidValue;
        uint32_t *m_out = hist2;                               // the level-2 histogram is dead by now
        FinishParams fp{};
        fp.keys = grouped; fp.base2 = base2; fp.n_sub = pl.n_sub; fp.prefix_bits = pl.b1 + pl.b2;
        fp.tmp_keys = out_keys; fp.tmp_counts = out_counts; fp.m_out = m_out; fp.d_overflow = d_overflow;
        fp.d_n_invalid = ep_in.n_invalid; fp.add_phantom = add_phantom ? 1 : 0;
        fp.tmp_start = status_scratch + pl.n_sub + 8;
        if ((e = launch_finish<false, W>(fp, n_sms, pl.n_sub, s)) != cudaSuccess) return e;
        // off[] (n_sub + 1) overwrites cursor2; its last entry is the number of records
        scan2_kernel<<<(pl.n_sub + kScan2Tile - 1) / kScan2Tile, 1024, 0, s>>>(m_out, pl.n_sub, cursor2, status_scratch);
        if ((e = cudaMemcpyAsync(d_num_out, cursor2 + pl.n_sub, 4, cudaMemcpyDeviceToDevice, s)) != cudaSuccess) return e;
    }
    if (evs) cudaEventRecord(evs[4], s);
    if (n_launches) *n_launches += pl.b2 > 0 ? 8 : 5;
    return cudaSuccess;
}

bool partition_fits(const ExtractParams &ep, int W) {
    constexpr uint64_t kMaxSmemOptin = 227 * 1024;          // a CTA's dynamic shared memory on sm_100
    const uint32_t keys = ep.tile_reads * ep.nk;
    const uint64_t extra = W == 1 ? Scatter1Sink<1>::smem_bytes(keys) : Scatter1Sink<2>::smem_bytes(keys);
    return (W == 1 || W == 2) && ep.smem_total + extra <= kMaxSmemOptin;
}

cudaError_t partition_count(int W, const ExtractParams &ep, uint64_t n_slots, int sig_bits, bool add_phantom,
                            uint64_t *keys_a, uint64_t *keys_b, uint64_t *out_keys, uint32_t *out_counts,
                            unsigned long long *d_num_out, unsigned long long *d_overflow,
                            unsigned long long *d_scratch_invalid, void *ws, int n_sms, int target_sub,
                            cudaStream_t s, int *n_launches, cudaEvent_t *evs /* 5: after P0, PA, H2, PB, PC */) {
    if (W == 1)
        return partition_count_w<1>(ep, n_slots, sig_bits, add_phantom, keys_a, keys_b, out_keys, out_counts, d_num_out,
                                    d_overflow, d_scratch_invalid, ws, n_sms, target_sub, s, n_launches, evs);
    if (W == 2)
        return partition_count_w<2>(ep, n_slots, sig_bits, add_phantom, keys_a, keys_b, out_keys, out_counts, d_num_out,
                                    d_overflow, d_scratch_invalid, ws, n_sms, target_sub, s, n_launches, evs);
    return cudaErrorInvalidValue;
}

}  // namespace kc
