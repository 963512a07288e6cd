// kc_merge.cu -- GPU merge-path merge of two sorted key-unique runs, summing the
// counts of equal keys; and the set operations of two runs (union, intersect,
// subtract) on the same kernels.
//
// Replaces KMerFileMerger::Merge (KMerFileMerger.cpp:49-96: a serial O(M) min-scan
// per output record over file cursors) and the cursor class under it
// (SortedKMerFile.cpp).  M runs are merged as a pairwise tree by the caller.
//
// Kernel 1 cuts the merged sequence into equal diagonals (merge path, ties go
// to run A) and nudges a cut that would separate an equal (A,B) pair.  Kernel 2
// loads one tile of A and B into shared memory; every thread searches its own
// diagonal once and merges its positions serially in registers, folding the B
// half of an equal pair into its A partner; the surviving records are written
// in order at the offset a decoupled look-back over the tiles gives.  Which
// records survive, and with what count, is the tile kernel's OP.
#include "kc_internal.h"

namespace kc {

namespace {

// OP of the tile kernel: kTileMerge is the merge (union, counts summed); the set operations
// kSetUnion .. kSetSubtractCounts take the count mode of keys in both runs as a kernel argument
constexpr int kTileMerge = -1;

// the count of a key present in both runs (kCounts*; the sum wraps at 2^32)
__device__ __forceinline__ uint32_t both_count(uint32_t a, uint32_t b, uint32_t mode) {
    switch (mode) {
        case kCountsMin: return min(a, b);
        case kCountsMax: return max(a, b);
        case kCountsA: return a;
        case kCountsB: return b;
        default: return a + b;
    }
}

constexpr int kMergeThreads = 512;

// items per thread of the tile kernel; a tile is kMergeThreads * IPT positions of the merged sequence.
// Sweep on two runs of 129 M records (tools/merge_test/merge_perf.cu, profiles/r2/merge_sweep_s19.txt):
// 256 x 8 with a one-thread look-back 3.69 ms, with the warp look-back 2.62, 512 x 12: 2.06 (W = 2: 256 x 6
// 4.23 -> 512 x 8 3.77); 512 x 16 and 1024 x 8 are slower again (3.2 / 3.0 ms).
template <int W> struct MergeCfg {
    static constexpr int IPT = W == 1 ? 12 : (W == 2 ? 8 : 4);
    static constexpr int TILE = kMergeThreads * IPT;
};

template <int W>
__global__ void merge_partition_kernel(const uint64_t *__restrict__ ka, uint64_t na, const uint64_t *__restrict__ kb,
                                       uint64_t nb, uint32_t n_tiles, uint64_t *__restrict__ cut_a,
                                       uint64_t *__restrict__ cut_b) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t > n_tiles) return;
    uint64_t diag = (uint64_t)t * MergeCfg<W>::TILE;
    if (diag > na + nb) diag = na + nb;
    uint64_t lo = diag > nb ? diag - nb : 0, hi = diag < na ? diag : na;
    while (lo < hi) {
        const uint64_t mid = (lo + hi) >> 1;
        const Key<W> a = ld_key<W>(ka, mid), b = ld_key<W>(kb, diag - 1 - mid);
        if (!key_lt<W>(b, a)) lo = mid + 1;   // a <= b: a goes first
        else hi = mid;
    }
    uint64_t a = lo, b = diag - lo;
    if (a > 0 && b < nb && key_eq<W>(ld_key<W>(ka, a - 1), ld_key<W>(kb, b))) b++;   // keep equal pairs together
    cut_a[t] = a;
    cut_b[t] = b;
}

// One tile: the A and B pieces between two cuts go to shared memory (coalesced), every thread finds
// where its IPT positions of the merged sequence start (one merge-path search per thread, in shared
// memory) and merges them serially in registers: one key comparison per record. An A record whose
// key is also at the head of B takes B's count; that B record -- always the next position, ties go
// to A -- is dropped. The survivors are compacted through shared memory and written as one
// contiguous piece at the offset a decoupled look-back over the tiles gives.
// (A tile can hold TILE + 1 records: the cut after it was moved to keep an equal pair together;
// the extra record is that pair's B half, the last position, and needs no thread.)
// A set operation (OP != kTileMerge) decides instead whether an A record with a B partner survives
// and with which count, whether an A record without one survives, and whether a B record without
// one does. The B half of a pair never survives, so the extra record and the cuts stay as they are.
template <int W, int OP>
__global__ void __launch_bounds__(kMergeThreads) merge_tile_kernel(
    const uint64_t *__restrict__ ka, const uint32_t *__restrict__ ca, const uint64_t *__restrict__ kb,
    const uint32_t *__restrict__ cb, const uint64_t *__restrict__ cut_a, const uint64_t *__restrict__ cut_b,
    uint32_t n_tiles, uint64_t *__restrict__ out_keys, uint32_t *__restrict__ out_counts,
    unsigned long long *__restrict__ d_num_out, unsigned long long *ticket, uint64_t *status, uint32_t counts) {
    constexpr int IPT = MergeCfg<W>::IPT, TILE = MergeCfg<W>::TILE;
    constexpr int CAP = TILE + 2;
    constexpr int WARPS = kMergeThreads / 32;
    extern __shared__ __align__(16) uint8_t smem_raw[];
    Key<W> *s_in = reinterpret_cast<Key<W> *>(smem_raw);                       // A then B; later the survivors
    uint32_t *s_inc = reinterpret_cast<uint32_t *>(s_in + CAP);                // their counts
    __shared__ uint32_t s_tile, s_warp[WARPS];
    __shared__ uint64_t s_base;

    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) s_tile = (uint32_t)atomicAdd(ticket, 1ull);
    __syncthreads();
    const uint32_t tile = s_tile;
    const uint64_t a0 = cut_a[tile], a1 = cut_a[tile + 1], b0 = cut_b[tile], b1 = cut_b[tile + 1];
    const uint32_t na = (uint32_t)(a1 - a0), nb = (uint32_t)(b1 - b0);

    const uint32_t m = min(na + nb, (uint32_t)TILE);
    const Key<W> *sA = s_in, *sB = s_in + na;
    const uint32_t *cA = s_inc, *cB = s_inc + na;
    for (uint32_t i = tid; i < na + nb; i += kMergeThreads) {
        if (i < na) { s_in[i] = ld_key<W>(ka, a0 + i); s_inc[i] = ca[a0 + i]; }
        else { s_in[i] = ld_key<W>(kb, b0 + (i - na)); s_inc[i] = cb[b0 + (i - na)]; }
    }
    __syncthreads();
    // this thread's positions [d, d + IPT) of the merged sequence start at A[ai], B[bi]
    const uint32_t d = min(tid * IPT, m);
    uint32_t ai, bi;
    {
        uint32_t lo = d > nb ? d - nb : 0, hi = d < na ? d : na;
        while (lo < hi) {
            const uint32_t mid = (lo + hi) >> 1;
            if (!key_lt<W>(sB[d - 1 - mid], sA[mid])) lo = mid + 1;
            else hi = mid;
        }
        ai = lo;
        bi = d - lo;
    }
    Key<W> rk[IPT];
    uint32_t rc[IPT];
    uint32_t keep = 0;                      // bit j: position d + j survives
    Key<W> a_head, b_head, a_prev;
    if (ai < na) a_head = sA[ai];
    if (bi < nb) b_head = sB[bi];
    bool have_prev = ai > 0;
    if (have_prev) a_prev = sA[ai - 1];
#pragma unroll
    for (int j = 0; j < IPT; j++) {
        if (d + j < m) {
            const bool take_a = bi >= nb || (ai < na && !key_lt<W>(b_head, a_head));
            if (take_a) {
                rk[j] = a_head;
                if constexpr (OP == kTileMerge) {
                    uint32_t c = cA[ai];
                    if (bi < nb && key_eq<W>(b_head, a_head)) c += cB[bi];
                    rc[j] = c;
                    keep |= 1u << j;
                } else {
                    const uint32_t c = cA[ai];
                    if (bi < nb && key_eq<W>(b_head, a_head)) {                  // the key is in both runs
                        const uint32_t cb_ = cB[bi];
                        if constexpr (OP == kSetUnion || OP == kSetIntersect) {
                            rc[j] = both_count(c, cb_, counts);
                            keep |= 1u << j;
                        } else if constexpr (OP == kSetSubtractCounts) {
                            rc[j] = c - cb_;
                            if (c > cb_) keep |= 1u << j;
                        }
                    } else if constexpr (OP != kSetIntersect) {                   // only in A
                        rc[j] = c;
                        keep |= 1u << j;
                    }
                }
                a_prev = a_head;
                have_prev = true;
                ai++;
                if (ai < na) a_head = sA[ai];
            } else {
                rk[j] = b_head;
                rc[j] = cB[bi];
                if constexpr (OP == kTileMerge || OP == kSetUnion)       // (only in B, or a pair's B half)
                    if (!(have_prev && key_eq<W>(a_prev, b_head))) keep |= 1u << j;
                bi++;
                if (bi < nb) b_head = sB[bi];
            }
        }
    }
    const uint32_t mine = __popc(keep);
    uint32_t incl = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= (uint32_t)o) incl += t;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();                        // (also: every thread is done reading the inputs)
    uint32_t woff = 0, total = 0;
#pragma unroll
    for (int w = 0; w < WARPS; w++) {
        if (w < (int)warp) woff += s_warp[w];
        total += s_warp[w];
    }
    uint32_t o = woff + incl - mine;
#pragma unroll
    for (int j = 0; j < IPT; j++) {
        if (keep & (1u << j)) {
            s_in[o] = rk[j];
            s_inc[o] = rc[j];
            o++;
        }
    }
    if (warp == 0) {                        // the first warp looks back 32 tiles at a time
        const uint64_t excl = lookback_exclusive_warp(status, tile, total);
        if (lane == 0) {
            s_base = excl;
            if (tile + 1 == n_tiles) *d_num_out = excl + total;
        }
    }
    __syncthreads();
    const uint64_t base = s_base;
    for (uint32_t i = tid; i < total; i += kMergeThreads) {
        st_key<W>(out_keys, base + i, s_in[i]);
        out_counts[base + i] = s_inc[i];
    }
}

template <int W, int OP>
cudaError_t merge_pair_w(const uint64_t *ka, const uint32_t *ca, uint64_t na, const uint64_t *kb, const uint32_t *cb,
                         uint64_t nb, uint32_t counts, uint64_t *out_keys, uint32_t *out_counts,
                         unsigned long long *d_num_out, void *ws, cudaStream_t s, int *n_launches) {
    constexpr int TILE = MergeCfg<W>::TILE;
    constexpr int CAP = TILE + 2;
    const uint64_t total = na + nb;
    const uint32_t n_tiles = (uint32_t)div_up(total, (uint64_t)TILE);
    uint8_t *wsb = static_cast<uint8_t *>(ws);
    unsigned long long *ticket = reinterpret_cast<unsigned long long *>(wsb);
    uint64_t *status = reinterpret_cast<uint64_t *>(wsb + 256);
    uint64_t *cut_a = status + n_tiles;
    uint64_t *cut_b = cut_a + n_tiles + 1;
    cudaError_t e;
    if ((e = cudaMemsetAsync(ws, 0, 256 + (size_t)n_tiles * 8, s)) != cudaSuccess) return e;
    merge_partition_kernel<W><<<(n_tiles + 1 + 127) / 128, 128, 0, s>>>(ka, na, kb, nb, n_tiles, cut_a, cut_b);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    const size_t smem = (size_t)CAP * (sizeof(Key<W>) + 4) + 16;
    auto kern = merge_tile_kernel<W, OP>;
    if ((e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess)
        return e;
    kern<<<n_tiles, kMergeThreads, smem, s>>>(ka, ca, kb, cb, cut_a, cut_b, n_tiles, out_keys, out_counts, d_num_out,
                                              ticket, status, counts);
    if (n_launches) *n_launches += 2;
    return cudaGetLastError();
}

template <int OP>
cudaError_t tile_pass(const uint64_t *ka, const uint32_t *ca, uint64_t na, const uint64_t *kb, const uint32_t *cb,
                      uint64_t nb, int W, uint32_t counts, uint64_t *out_keys, uint32_t *out_counts,
                      unsigned long long *d_num_out, void *ws, cudaStream_t s, int *n_launches) {
    switch (W) {
        case 1: return merge_pair_w<1, OP>(ka, ca, na, kb, cb, nb, counts, out_keys, out_counts, d_num_out, ws, s, n_launches);
        case 2: return merge_pair_w<2, OP>(ka, ca, na, kb, cb, nb, counts, out_keys, out_counts, d_num_out, ws, s, n_launches);
        case 3: return merge_pair_w<3, OP>(ka, ca, na, kb, cb, nb, counts, out_keys, out_counts, d_num_out, ws, s, n_launches);
        case 4: return merge_pair_w<4, OP>(ka, ca, na, kb, cb, nb, counts, out_keys, out_counts, d_num_out, ws, s, n_launches);
    }
    return cudaErrorInvalidValue;
}

}  // namespace

uint64_t merge_workspace_bytes(uint64_t na, uint64_t nb) {
    const uint64_t tiles = div_up(na + nb + 1, (uint64_t)MergeCfg<4>::TILE) + 2;      // (the smallest tile of any width)
    return 256 + tiles * 8 * 3 + 256;
}

cudaError_t merge_pair(const uint64_t *ka, const uint32_t *ca, uint64_t na, const uint64_t *kb, const uint32_t *cb,
                       uint64_t nb, int W, uint64_t *out_keys, uint32_t *out_counts, unsigned long long *d_num_out,
                       void *ws, cudaStream_t s, int *n_launches) {
    if (na + nb == 0) return cudaMemsetAsync(d_num_out, 0, 8, s);
    return tile_pass<kTileMerge>(ka, ca, na, kb, cb, nb, W, 0, out_keys, out_counts, d_num_out, ws, s, n_launches);
}

cudaError_t combine_pair(const uint64_t *ka, const uint32_t *ca, uint64_t na, const uint64_t *kb, const uint32_t *cb,
                         uint64_t nb, int W, uint32_t op, uint32_t counts, uint64_t *out_keys, uint32_t *out_counts,
                         unsigned long long *d_num_out, void *ws, cudaStream_t s, int *n_launches) {
    if (counts > kCountsB || (counts != kCountsSum && (op == kSetSubtract || op == kSetSubtractCounts)))
        return cudaErrorInvalidValue;
    if (op == kSetUnion && counts == kCountsSum)
        return merge_pair(ka, ca, na, kb, cb, nb, W, out_keys, out_counts, d_num_out, ws, s, n_launches);
    if (na + nb == 0) return cudaMemsetAsync(d_num_out, 0, 8, s);
    switch (op) {
        case kSetUnion:
            return tile_pass<kSetUnion>(ka, ca, na, kb, cb, nb, W, counts, out_keys, out_counts, d_num_out, ws, s, n_launches);
        case kSetIntersect:
            return tile_pass<kSetIntersect>(ka, ca, na, kb, cb, nb, W, counts, out_keys, out_counts, d_num_out, ws, s, n_launches);
        case kSetSubtract:
            return tile_pass<kSetSubtract>(ka, ca, na, kb, cb, nb, W, counts, out_keys, out_counts, d_num_out, ws, s, n_launches);
        case kSetSubtractCounts:
            return tile_pass<kSetSubtractCounts>(ka, ca, na, kb, cb, nb, W, counts, out_keys, out_counts, d_num_out, ws, s,
                                                 n_launches);
    }
    return cudaErrorInvalidValue;
}

}  // namespace kc
