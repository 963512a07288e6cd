// kc_super.cu -- super-window counting path (sm_100a). See kc_super.cuh for the design.
//
// What it replaces in the reference: extractKMers' one-record-per-occurrence output
// (GPUHandler.cu:129-233, 8.4x the input), the host hash accumulate (KMerCounter.cpp:61-82)
// and sortKmers + reduceKMers (GPUHandler.cu:300-360). Key semantics are those of
// kc_extract.cuh (SURVEY.md A.2): the key of window p is the 2-bit codes of s[p .. p+span).
#include <math.h>
#include <stdlib.h>

#include "kc_internal.h"
#include "kc_super.cuh"

namespace kc {

namespace {

constexpr uint32_t kNoBin = 0xffffffffu;
constexpr int kSwThreads = 256;
constexpr int kSwMaxSeg = 18;           // windows one thread derives minimizers for
constexpr int kNb1Max = 1024;           // level-1 bins / histogram bins S2 keeps
constexpr int kRsBins = 2048;           // bins a record-scatter tile handles (level 2: two buckets x 1024)

// ---------------------------------------------------------------- minimizer -> bin
// Order of m-mers = order of a 32-bit bijective hash of their 2-bit codes (no ties between
// different m-mers); the bin of a window is a second hash of its smallest m-mer hash. Both are
// functions of the key's bases only, so equal keys always meet in the same bin.
template <uint32_t X> struct ILog2 { static constexpr uint32_t v = 1 + ILog2<(X >> 1)>::v; };
template <> struct ILog2<1> { static constexpr uint32_t v = 0; };

__host__ __device__ __forceinline__ uint32_t mmer_hash(uint32_t mm) {
    uint32_t h = mm * 0x9E3779B1u;
    h ^= h >> 15;
    h *= 0x85EBCA6Bu;
    return h;
}
__device__ __forceinline__ uint32_t bin_of_min(uint32_t mn, uint32_t n_bins) {
    return __umulhi(mn * 0xC2B2AE35u, n_bins);
}

// ===================================================================== S1: scatter
struct SwScatterParams {
    ExtractParams ep;
    uint32_t m, w, nh, nh_stride, seg_len, segs_per_read, cmax, span;
    uint32_t h_off, bin_off, bits_off;  // shared-memory offsets: m-mer hashes, window bins, boundary bitmask
    uint32_t n_bins, bin_cap;
    uint64_t ovf_cap;
    uint32_t *cursor;                   // [n_bins] records appended to each bin so far
    uint8_t *bins;                      // n_bins x bin_cap records of 16W bytes
    uint8_t *ovf;                       // ovf_cap records
    unsigned long long *sc;
};

template <int W, bool CANON>
__global__ void __launch_bounds__(kSwThreads) sw_scatter_kernel(SwScatterParams q) {
    const ExtractParams &p = q.ep;
    extern __shared__ __align__(128) uint8_t smem[];
    const uint32_t stage_bytes = p.stage_bytes;
    uint8_t *stage0 = smem;
    uint64_t *enc = reinterpret_cast<uint64_t *>(smem + p.enc_off);
    uint8_t *enc_b = reinterpret_cast<uint8_t *>(enc);
    const uint32_t enc_row = p.nw + 1;
    uint8_t *bad4 = smem + p.bad_off;
    uint8_t *flag = smem + p.flag_off;
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem + p.bar_off);
    uint32_t *hh = reinterpret_cast<uint32_t *>(smem + q.h_off);
    uint32_t *bid = reinterpret_cast<uint32_t *>(smem + q.bin_off);
    uint32_t *seg_st = reinterpret_cast<uint32_t *>(smem + q.bits_off);       // [tile_reads * segs_per_read]
    uint32_t *seg_bd = seg_st + p.tile_reads * q.segs_per_read;
    __shared__ uint32_t s_nstart;
    const uint32_t tid = threadIdx.x, lane = tid & 31;

    if (tid == 0) {
        s_nstart = 0;
        mbar_init(&bars[0], 1);
        mbar_init(&bars[1], 1);
        mbar_fence_init();
    }
    for (uint32_t i = tid; i < p.tile_reads * enc_row; i += kSwThreads) enc[i] = 0;
    for (uint32_t i = tid; i < p.tile_reads; i += kSwThreads) flag[i] = 0;
    __syncthreads();

    auto tile_reads_of = [&](uint32_t t) -> uint32_t {
        uint64_t first = (uint64_t)t * p.tile_reads;
        uint64_t left = p.n_reads - first;
        return left < p.tile_reads ? (uint32_t)left : p.tile_reads;
    };
    auto issue_load = [&](uint32_t t, uint32_t s) {
        uint32_t bytes = tile_reads_of(t) * p.L;
        const uint8_t *src = p.reads + (uint64_t)t * p.tile_reads * p.L;
        uint8_t *dst = stage0 + s * stage_bytes;
        if ((bytes & 15u) == 0) {
            if (tid == 0) {
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                mbar_expect_tx(&bars[s], bytes);
                tma_load_1d(dst, src, bytes, &bars[s]);
            }
        } else {
            for (uint32_t i = tid; i < bytes; i += kSwThreads) dst[i] = src[i];
        }
    };

    uint32_t phase_bits = 0, stage = 0;
    unsigned long long invalid_local = 0, windows_local = 0, records_local = 0;
    const uint32_t mmask = q.m >= 16 ? 0xffffffffu : ((1u << (2 * q.m)) - 1u);
    const uint32_t mshift = 64 - 2 * q.m;
    const uint32_t ng = (q.nh + 7) >> 3;

    uint32_t tile = blockIdx.x;
    if (tile < p.n_tiles) issue_load(tile, 0);

    for (; tile < p.n_tiles; tile += gridDim.x) {
        const uint32_t next = tile + gridDim.x;
        if (next < p.n_tiles) issue_load(next, stage ^ 1);
        const uint32_t nreads = tile_reads_of(tile);
        if (((nreads * p.L) & 15u) == 0) {
            mbar_wait(&bars[stage], (phase_bits >> stage) & 1u);
            phase_bits ^= 1u << stage;
        } else {
            __syncthreads();
        }
        const uint8_t *src_tile = stage0 + stage * stage_bytes;

        // ---- A: 2-bit encode
        encode_tile(p, src_tile, nreads, enc_b, bad4, flag);
        __syncthreads();
        if (tid == 0) s_nstart = 0;                      // (read by D2 of the previous tile two barriers ago)

        // ---- B: hash of the m-mer starting at every code position j < nh; a thread takes 8
        // consecutive positions out of one 64-bit funnel of the encoded words
        for (uint32_t g = tid; g < nreads * ng; g += kSwThreads) {
            const uint32_t r = g / ng, j0 = (g - r * ng) * 8;
            const uint32_t wi = j0 >> 5, sh = (j0 & 31u) * 2u;
            const uint64_t *e = enc + r * enc_row;
            const uint64_t a = wi <= p.nw ? e[wi] : 0ull;
            const uint64_t b = wi + 1 <= p.nw ? e[wi + 1] : 0ull;
            const uint64_t x = sh ? ((a << sh) | (b >> (64 - sh))) : a;
            uint32_t *row = hh + r * q.nh_stride + j0;
            if constexpr (CANON) {
                // canonical m-mer min(mm, rc(mm)): the m-mers of rc(x) are the reverse complements of
                // x's, so the window's minimizer (its bin, its owner rank) is the same on both strands
#pragma unroll
                for (uint32_t i = 0; i < 8; i++) {
                    const uint32_t mm = (uint32_t)(x >> (mshift - 2 * i)) & mmask;
                    uint32_t r = __brev(mm);
                    r = ((r >> 1) & 0x55555555u) | ((r & 0x55555555u) << 1);
                    if (j0 + i < q.nh) row[i] = mmer_hash(min(mm, (r >> (32 - 2 * q.m)) ^ mmask));
                }
            } else {
#pragma unroll
                for (uint32_t i = 0; i < 8; i++)
                    if (j0 + i < q.nh) row[i] = mmer_hash((uint32_t)(x >> (mshift - 2 * i)) & mmask);
            }
        }
        __syncthreads();

        // ---- C: minimum over the w m-mers of each window -> bin of the window. A thread takes a
        // segment of s <= 17 consecutive windows plus, as a look-behind, the window before them.
        // All of those windows contain the m-mers [s'-1, w) counted from the first one (the core);
        // window i adds a suffix of [i, s'-1) and a prefix of [w, w+i). With the bins in registers
        // the thread also finds where runs of equal bins start inside its segment: bit i of
        // seg_st = window i starts a run, bit i of seg_bd = it starts one or holds no k-mer.
        const uint32_t n_seg = nreads * q.segs_per_read;
        for (uint32_t sg = tid; sg < n_seg; sg += kSwThreads) {
            const uint32_t r = sg / q.segs_per_read;
            const uint32_t p0 = (sg - r * q.segs_per_read) * q.seg_len;
            if (p0 >= p.nk) { seg_st[sg] = 0; seg_bd[sg] = 0; continue; }
            const uint32_t s = min(q.seg_len, p.nk - p0);
            const uint32_t lb = p0 > 0 ? 1u : 0u;                  // look-behind window
            const uint32_t se = s + lb;                            // windows whose bin this thread derives
            const uint32_t *g = hh + r * q.nh_stride + p0 - lb;
            uint32_t S[kSwMaxSeg];
            S[kSwMaxSeg - 1] = 0xffffffffu;
#pragma unroll
            for (int i = kSwMaxSeg - 2; i >= 0; i--) {
                const uint32_t v = (uint32_t)i + 1 < se ? g[i] : 0xffffffffu;
                S[i] = min(v, S[i + 1]);
            }
            uint32_t core = 0xffffffffu;
            for (uint32_t t = se - 1; t < q.w; t++) core = min(core, g[t]);
            uint32_t pm = 0xffffffffu;
            const bool check = flag[r] != 0;
            uint32_t *brow = bid + r * p.nk + p0 - lb;
            uint32_t prev = kNoBin, stm = 0, bdm = 0;
#pragma unroll
            for (uint32_t i = 0; i < (uint32_t)kSwMaxSeg; i++) {
                if (i < se) {
                    const uint32_t mn = min(min(S[i], core), pm);
                    const bool valid = check ? kmer_window_valid(bad4 + r * p.nb4, p0 - lb + i, p.k) : true;
                    const uint32_t b = valid ? bin_of_min(mn, q.n_bins) : kNoBin;
                    if (i >= lb) {                                 // an owned window
                        if (!valid) invalid_local++;
                        brow[i] = b;
                        const uint32_t st = (valid && b != prev) ? 1u : 0u;
                        stm |= st << (i - lb);
                        bdm |= (st | (valid ? 0u : 1u)) << (i - lb);
                    }
                    prev = b;
                    if (i + 1 < se) pm = min(pm, g[q.w + i]);
                }
            }
            seg_st[sg] = stm;
            seg_bd[sg] = bdm;
        }
        __syncthreads();

        // ---- D: a run of equal bins becomes records of at most cmax windows: 64W bases from the
        // run's first base (the first key and the bases that follow it), the window count in the
        // low byte of the last word.
        // D1: compact list of the run starts, entry = segment << 5 | window inside the segment
        // (the m-mer hashes are dead: the list lives in their place).
        uint32_t *list = hh;
        for (uint32_t base = 0; base < n_seg; base += kSwThreads) {
            const uint32_t sg = base + tid;
            uint32_t stm = sg < n_seg ? seg_st[sg] : 0u;
            const uint32_t cnt = __popc(stm);
            uint32_t incl = cnt;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= (uint32_t)o) incl += t;
            }
            uint32_t off = 0;
            if (lane == 31 && incl) off = atomicAdd(&s_nstart, incl);
            off = __shfl_sync(0xffffffffu, off, 31) + incl - cnt;
            while (stm) {
                const uint32_t i = __ffs(stm) - 1;
                stm &= stm - 1;
                list[off++] = (sg << 5) | i;
            }
        }
        __syncthreads();
        // D2: one thread per run. The run ends at the next boundary bit (this segment's or a later
        // one's of the same read) or at the end of the read. The bin's cursor is bumped first; the
        // record is assembled while that atomic is in flight.
        const uint32_t n_start = s_nstart;
        for (uint32_t en = tid; en < n_start; en += kSwThreads) {
            const uint32_t ent = list[en];
            const uint32_t sg = ent >> 5, wi0 = ent & 31u;
            const uint32_t r = sg / q.segs_per_read, si = sg - r * q.segs_per_read;
            const uint32_t pos = si * q.seg_len + wi0;
            uint32_t end = p.nk;
            {
                uint32_t mk = seg_bd[sg] & ~(0xffffffffu >> (31 - wi0));          // boundaries after this window
                uint32_t sj = si;
                while (mk == 0 && ++sj < q.segs_per_read) mk = seg_bd[r * q.segs_per_read + sj];
                if (mk) end = min(p.nk, sj * q.seg_len + (uint32_t)__ffs(mk) - 1);
            }
            const uint32_t len = end - pos;
            const uint32_t b = bid[r * p.nk + pos];
            const uint64_t *e = enc + r * enc_row;
            for (uint32_t q0 = 0; q0 < len; q0 += q.cmax) {
                const uint32_t idx = atomicAdd(&q.cursor[b], 1u);
                const uint32_t c = min(q.cmax, len - q0);
                const uint32_t wi = (pos + q0) >> 5, sh = ((pos + q0) & 31u) * 2u;
                uint64_t ew[2 * W + 1];
#pragma unroll
                for (int t = 0; t < 2 * W + 1; t++) ew[t] = wi + t <= p.nw ? e[wi + t] : 0ull;
                uint64_t rec[2 * W];
#pragma unroll
                for (int t = 0; t < 2 * W; t++) rec[t] = sh ? ((ew[t] << sh) | (ew[t + 1] >> (64 - sh))) : ew[t];
                // bases behind the last window are whatever follows in the read: zeroed, so that the same
                // run of the same locus gives the same record in every read (S2 counts equal records once)
                const uint32_t nbases = q.span + c - 1;
#pragma unroll
                for (int t = 0; t < 2 * W; t++) {
                    const int keep = (int)nbases - 32 * t;
                    if (keep <= 0) rec[t] = 0;
                    else if (keep < 32) rec[t] &= ~0ull << (64 - 2 * keep);
                }
                rec[2 * W - 1] = (rec[2 * W - 1] & ~0xffull) | c;
                ulonglong2 *dst = nullptr;
                if (idx < q.bin_cap) {
                    dst = reinterpret_cast<ulonglong2 *>(q.bins) + ((uint64_t)b * q.bin_cap + idx) * W;
                } else {
                    const unsigned long long oi = atomicAdd(&q.sc[SW_OVF], 1ull);
                    if (oi < q.ovf_cap) dst = reinterpret_cast<ulonglong2 *>(q.ovf) + oi * W;
                    else atomicOr(&q.sc[SW_FAIL], 1ull);
                }
                if (dst) {
#pragma unroll
                    for (int t = 0; t < W; t++) dst[t] = make_ulonglong2(rec[2 * t], rec[2 * t + 1]);
                }
                windows_local += c;
                records_local++;
            }
        }
        for (uint32_t i = tid; i < nreads; i += kSwThreads) flag[i] = 0;
        __syncthreads();
        stage ^= 1;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        invalid_local += __shfl_xor_sync(0xffffffffu, invalid_local, o);
        windows_local += __shfl_xor_sync(0xffffffffu, windows_local, o);
        records_local += __shfl_xor_sync(0xffffffffu, records_local, o);
    }
    if (lane == 0) {
        if (invalid_local) atomicAdd(&q.sc[SW_INVALID], invalid_local);
        if (windows_local) atomicAdd(&q.sc[SW_WINDOWS], windows_local);
        if (records_local) atomicAdd(&q.sc[SW_RECORDS], records_local);
    }
}

// ======================================================================= S2: count
// a second, independent hash: which of the 2^bits passes over a bin a key belongs to
__device__ __forceinline__ uint32_t pass_hash(uint32_t h) { return (h ^ (h >> 15)) * 0x2C1B3C6Du; }

// KC_SW_PROFILE (off by default; tools/s2_profile.py builds with it): every warp of sw_count_kernel
// adds clock64() deltas per phase into g_sw_prof, plus a few counters of the insert path. Lane 0
// takes the time at phase boundaries, most of which are barriers, so a phase's share includes the
// warp's wait for the CTA's slowest warp in that phase. Without the switch the macros are empty.
enum {
    SWP_UNIT = 0,       // unit hand-over, descriptors, phantom key, first round's records
    SWP_DEDUP,          // record table claims
    SWP_SCAN,           // scan of the surviving records' windows, placement in shared memory, slots handed back
    SWP_OPEN,           // next round's prefetch, opening the thread's first record
    SWP_INSERT,         // the insert loop, drains excluded
    SWP_DRAIN,          // draining the per-warp collision queue
    SWP_ROUND_END,      // distinct-key count and the barrier that closes a round
    SWP_EMIT,           // emit of the pass with its table clear, abort handling
    SWP_PHASES,
    SWP_QUEUED = SWP_PHASES,    // occurrences sent to the collision queue
    SWP_DRAIN_PROBES,           // buckets probed by the drains
    SWP_WARPS,                  // warps that ran
    SWP_TOTAL,                  // cycles of those warps, start to end
    SWP_SLOTS
};
#ifdef KC_SW_PROFILE
__device__ unsigned long long g_sw_prof[SWP_SLOTS];
// the sums live in shared memory (lane 0 of each warp adds), so that the timer costs S2 two registers
// and leaves it at the default build's occupancy
#define SWP_DECL                                                                                      \
    __shared__ unsigned long long s_prof[THREADS / 32][SWP_SLOTS];                                    \
    if (lane == 0)                                                                                    \
        for (int i_ = 0; i_ < SWP_SLOTS; i_++) s_prof[warp][i_] = 0;                                  \
    const long long swp_t0 = clock64();                                                               \
    long long swp_t = swp_t0
#define SWP_MARK(ph)                                                                                  \
    do {                                                                                              \
        const long long t_ = clock64();                                                               \
        if (lane == 0) s_prof[warp][ph] += (unsigned long long)(t_ - swp_t);                          \
        swp_t = t_;                                                                                   \
    } while (0)
#define SWP_ADD(c, v) atomicAdd(&s_prof[warp][c], (unsigned long long)(v))
#define SWP_ADD_ACTIVE(c)                                                                             \
    do {                                                                                              \
        const uint32_t am_ = __activemask();                                                          \
        if (lane == (uint32_t)__ffs(am_) - 1) SWP_ADD(c, __popc(am_));                                \
    } while (0)
#define SWP_FLUSH()                                                                                   \
    do {                                                                                              \
        __syncwarp();                                                                                 \
        if (lane == 0) {                                                                              \
            s_prof[warp][SWP_WARPS] = 1;                                                              \
            s_prof[warp][SWP_TOTAL] = (unsigned long long)(clock64() - swp_t0);                       \
            for (int i_ = 0; i_ < SWP_SLOTS; i_++) atomicAdd(&g_sw_prof[i_], s_prof[warp][i_]);       \
        }                                                                                             \
    } while (0)
#else
#define SWP_DECL do {} while (0)
#define SWP_MARK(ph) do {} while (0)
#define SWP_ADD(c, v) do {} while (0)
#define SWP_ADD_ACTIVE(c) do {} while (0)
#define SWP_FLUSH() do {} while (0)
#endif

struct SwCountParams {
    // bins [bin_begin, bin_begin + n_bins) are counted here; the records of a bin are what every
    // source put there (one source on one GPU; with several GPUs the peers' bins are read in place,
    // over NVLink -- the exchange of super-window records is the load side of this kernel)
    uint32_t n_src;
    const uint32_t *src_cursor[8];
    const uint8_t *src_bins[8];
    const unsigned long long *src_sc[8];
    uint32_t bin_begin;
    const uint8_t *ovf;
    uint32_t n_bins, bin_cap, ovf_slice;
    uint64_t ovf_cap;
    uint64_t last_mask;
    uint64_t *d_keys;
    uint32_t *d_counts;
    uint64_t d_cap;
    uint32_t *hist1;
    int shift1, nb1;
    int add_phantom;
    unsigned long long *sc;
};

// S2's CTA and table shape, the one instantiated for each key width: 512 threads and a 4096-slot
// table, with rounds of 2 records per thread for 64-bit keys (whole bins per round: 5.06 ms at C2
// against 6.06 ms with 1) and 1 for 128-bit keys. Picked by a sweep over CTA sizes (128 to 512),
// table sizes (2048 to 8192 slots) and records per thread (1 to 4); see DESIGN §4.1.
template <int W> struct SwCountCfg {
    static constexpr int THREADS = 512, TSLOTS = 4096, RPT = W == 1 ? 2 : 1;
};

// One work unit = one bin, or one slice of the overflow list. The CTA stages RPT * THREADS records
// at a time, splits their windows evenly over its threads (a thread takes a contiguous range of
// the flattened window sequence, so it slides the window inside a record and every lane has the
// same number of keys), and counts them in a shared-memory table. The insert loop is a per-lane
// state machine -- one probe of the lane's current key per iteration, a lane that is done with a
// key fetches its next one in the same loop -- so lanes with short and long probe sequences do not
// wait for each other. A unit with more distinct keys than the table takes is redone in 2, 4, ...
// passes, pass v counting the keys whose pass hash starts with v: the records a unit emits are
// always key-distinct.
// CANON: every window's key is min(forward, rc) (the records still hold forward bases).
template <int W, int THREADS, int TSLOTS, int RPT, bool CANON>
__global__ void __launch_bounds__(THREADS) sw_count_kernel(SwCountParams p) {
    constexpr int RB = THREADS * RPT;                                       // records per round
    extern __shared__ __align__(16) uint8_t cs_smem[];
    Key<W> *tk = reinterpret_cast<Key<W> *>(cs_smem);                       // [TSLOTS]
    ulonglong2 *recs = reinterpret_cast<ulonglong2 *>(tk + TSLOTS);         // [RB * W]
    uint32_t *tc = reinterpret_cast<uint32_t *>(recs + RB * W);             // [TSLOTS]
    uint32_t *s_start = tc + TSLOTS;                                        // [THREADS] thread t's first record << 8 | window in it
    uint32_t *s_hist = s_start + THREADS;                                   // [kNb1Max]
    constexpr int kQueue = RPT > 1 ? 64 : 96;                               // collided keys a warp parks before it drains them
    Key<W> *queue = reinterpret_cast<Key<W> *>(s_hist + kNb1Max);           // [THREADS / 32][kQueue]
    uint32_t *queue_m = reinterpret_cast<uint32_t *>(queue + (THREADS / 32) * kQueue);   // their weights
    // record-level table (DEDUP): equal records of a round are counted once, with a multiplicity
    constexpr bool DEDUP = (W == 1);
    constexpr int RT = DEDUP ? RB : 1;                                      // (whole-bin rounds: records are ~40% distinct)
    ulonglong2 *rt_keys = reinterpret_cast<ulonglong2 *>(queue_m + (THREADS / 32) * kQueue);   // [RT]
    uint32_t *rt_mult = reinterpret_cast<uint32_t *>(rt_keys + RT);         // [RT]
    uint32_t *rec_mult = rt_mult + RT;                                      // [RB] weight of staged record i (0: a duplicate)
    __shared__ uint32_t s_unit, s_m, s_ones, s_abort;
    __shared__ unsigned long long s_base;
    __shared__ uint32_t s_warp[THREADS / 32];
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr uint32_t kLimit = TSLOTS / 4 * 3;
    constexpr uint32_t hshift = 32 - ILog2<(uint32_t)TSLOTS>::v;
    [[maybe_unused]] const uint32_t rc_sh = CANON ? rc_shift_of(p.last_mask) : 0u;

    {
        Key<W> empty;
        key_set_ones<W>(empty);
        for (uint32_t i = tid; i < (uint32_t)TSLOTS; i += THREADS) { tk[i] = empty; tc[i] = 0; }
        for (uint32_t i = tid; i < (uint32_t)p.nb1; i += THREADS) s_hist[i] = 0;
        if constexpr (DEDUP)
            for (uint32_t i = tid; i < (uint32_t)RT; i += THREADS) { rt_keys[i] = make_ulonglong2(~0ull, ~0ull); rt_mult[i] = 0; }
        if (tid == 0) { s_m = 0; s_ones = 0; s_abort = 0; }
    }
    unsigned long long n_ovf = p.sc[SW_OVF];
    if (n_ovf > p.ovf_cap) n_ovf = p.ovf_cap;
    const uint32_t n_ovf_units = (uint32_t)((n_ovf + p.ovf_slice - 1) / p.ovf_slice);
    const uint32_t n_units = p.n_bins + n_ovf_units;
    unsigned long long occ_local = 0;
    uint32_t aborts_local = 0, multi_local = 0, dedup_local = 0;
    SWP_DECL;
    // Work units are drawn from an atomic ticket two units ahead, so that a CTA knows its next unit
    // while it counts the current one: the next unit's record counts and its first round of
    // records are fetched in the shadow of the current unit's inserts (with several GPUs those
    // are loads from a peer's HBM, several microseconds each). Unit descriptors live in shared
    // memory, double-buffered: [0..7] records of sources 0..s-1 come before source s's, [8] records.
    __shared__ uint32_t s_desc[2][10];
    __shared__ uint32_t s_next;
    __shared__ const uint8_t *s_bins[8];
    if (tid < 8) s_bins[tid] = tid < p.n_src ? p.src_bins[tid] : p.src_bins[0];
    auto setup = [&](uint32_t u, uint32_t buf) {         // warp 0
        if (warp != 0) return;
        uint32_t c = 0;
        if (u < p.n_bins && lane < p.n_src) {
            c = p.src_cursor[lane][p.bin_begin + u];
            c = c < p.bin_cap ? c : p.bin_cap;
        }
        uint32_t incl = c;
#pragma unroll
        for (int o = 1; o < 8; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= (uint32_t)o) incl += t;
        }
        if (lane < 8) s_desc[buf][lane] = incl - c;
        if (lane == 7) {
            uint32_t n = incl;
            if (u >= p.n_bins) {
                n = 0;
                if (u < n_units) n = (uint32_t)min((unsigned long long)p.ovf_slice, n_ovf - (uint64_t)(u - p.n_bins) * p.ovf_slice);
            }
            s_desc[buf][8] = n;
        }
    };
    // where record i of unit u (descriptor in buffer buf) lives
    auto rec_of = [&](uint32_t u, uint32_t buf, uint32_t i) -> const ulonglong2 * {
        if (u >= p.n_bins)
            return reinterpret_cast<const ulonglong2 *>(p.ovf) + ((uint64_t)(u - p.n_bins) * p.ovf_slice + i) * W;
        uint32_t off = i, q_src = 0;
        for (uint32_t q = 1; q < p.n_src; q++)
            if (i >= s_desc[buf][q]) { off = i - s_desc[buf][q]; q_src = q; }
        return reinterpret_cast<const ulonglong2 *>(s_bins[q_src]) + ((uint64_t)(p.bin_begin + u) * p.bin_cap + off) * W;
    };
    uint32_t t_c = 0;                                // thread 0: the ticket after the next one (its atomic is in flight for a whole unit)
    if (tid == 0) {
        const uint32_t t_a = (uint32_t)atomicAdd(&p.sc[SW_TICKET], 1ull);
        const uint32_t t_b = (uint32_t)atomicAdd(&p.sc[SW_TICKET], 1ull);
        s_unit = t_a;
        s_next = t_b;
        t_c = t_b < n_units ? (uint32_t)atomicAdd(&p.sc[SW_TICKET], 1ull) : t_b;
    }
    __syncthreads();
    setup(s_unit, 0);
    uint32_t par = 0;                                // descriptor buffer of the current unit
    uint32_t pf_id = 0xffffffffu;                    // unit whose first round sits in pf[]
    ulonglong2 pf[RPT][W];
    bool first_iter = true;

    while (true) {
        if (!first_iter) {
            // (the previous unit ended with a barrier) hand over to the next unit
            if (tid == 0) {
                s_unit = s_next;
                s_next = t_c;
                if (t_c < n_units) t_c = (uint32_t)atomicAdd(&p.sc[SW_TICKET], 1ull);
            }
            par ^= 1;
        }
        first_iter = false;
        __syncthreads();
        const uint32_t u = s_unit, un = s_next;
        if (u >= n_units) break;
        setup(un, par ^ 1);                          // (consumed after later barriers)
        const uint32_t n_rec = s_desc[par][8];
        auto rec_at = [&](uint32_t i) -> const ulonglong2 * { return rec_of(u, par, i); };
        // key 0 joins with count += 0 whenever a slot held no k-mer on any rank (SURVEY F7): its bin is bin 0
        bool phantom = false;
        if (u == 0 && p.bin_begin == 0 && p.add_phantom) {
#pragma unroll
            for (int q = 0; q < 8; q++)
                if ((uint32_t)q < p.n_src && p.src_sc[q][SW_INVALID] != 0) phantom = true;
        }
        if (n_rec == 0 && !phantom) { __syncthreads(); continue; }
        if (tid == 0 && n_rec > (uint32_t)RB) multi_local++;

        uint32_t bits = 0, val = 0;
        while (true) {                                   // passes over the unit
            uint32_t claims = 0;
            auto in_pass = [&](uint32_t h) -> bool { return bits == 0 || (pass_hash(h) >> (32 - bits)) == val; };
            if (phantom && tid == 0) {
                Key<W> zero;
#pragma unroll
                for (int i = 0; i < W; i++) zero.w[i] = 0;
                const uint32_t hv = key_hash<W>(zero);
                if (in_pass(hv)) {
                    uint32_t hb = hv >> (hshift + 1);
                    bool done = false;
#pragma unroll 1
                    for (uint32_t probes = 0; probes < 64u && !done; probes++) {
#pragma unroll 1
                        for (uint32_t sl = 0; sl < 2 && !done; sl++) {
                            Key<W> cur = tk[2 * hb + sl];
                            if (key_any_word_ones<W>(cur)) {
                                cur = slot_claim(&tk[2 * hb + sl], zero);
                                if (key_all_ones<W>(cur)) { claims++; done = true; }
                            }
                            if (key_eq<W>(cur, zero)) done = true;
                        }
                        hb = (hb + 1) & (TSLOTS / 2 - 1);
                    }
                    if (!done) s_abort = 1;
                }
            }
            bool aborted = false;
            // the first round's records: prefetched while the previous unit was counted, or fetched now
            if (pf_id != u) {
#pragma unroll
                for (int u2 = 0; u2 < RPT; u2++) {
                    const uint32_t i = u2 * THREADS + tid;
                    if (i < n_rec) {
                        const ulonglong2 *rp = rec_at(i);
#pragma unroll
                        for (int t = 0; t < W; t++) pf[u2][t] = rp[t];
                    }
                }
            }
            pf_id = 0xffffffffu;
            SWP_MARK(SWP_UNIT);
            for (uint32_t r0 = 0; r0 < n_rec; r0 += RB) {
                const uint32_t nr = min((uint32_t)RB, n_rec - r0);
                // The round's records sit in registers (fetched with a stride of THREADS: coalesced).
                // Equal records of the round (the same run of the same locus, seen by several reads) are
                // counted once: the first copy claims a slot of the record table and carries the
                // multiplicity, the others drop out. The table is empty at the start of every round: a
                // claimed slot is handed back by its owner once the multiplicity has been read.
                uint32_t c[RPT], rslot[RPT];
                bool live[RPT];
#pragma unroll
                for (int u2 = 0; u2 < RPT; u2++) {
                    const uint32_t i = u2 * THREADS + tid;
                    c[u2] = i < nr ? (uint32_t)(pf[u2][W - 1].y & 0xffull) : 0u;
                    live[u2] = i < nr;
                    rslot[u2] = 0xffffffffu;
                }
                if constexpr (DEDUP) {
#pragma unroll
                    for (int u2 = 0; u2 < RPT; u2++) {
                        if (live[u2]) {
                            const ulonglong2 rec = pf[u2][0];
                            uint32_t h = ((uint32_t)rec.x ^ (uint32_t)(rec.x >> 32) * 0x85EBCA6Bu ^ (uint32_t)(rec.y >> 8) * 0xC2B2AE35u ^
                                          (uint32_t)(rec.y >> 40)) * 0x9E3779B1u >> (32 - ILog2<(uint32_t)RT>::v);
                            while (true) {                       // the table holds at least the records of a round: never full
                                ulonglong2 cur = rt_keys[h];
                                if (cur.x == ~0ull || cur.y == ~0ull) {        // looks empty (a record is never all ones): settled by the CAS
                                    const uint32_t a = smem_u32(&rt_keys[h]);
                                    asm volatile(
                                        "{\n"
                                        ".reg .b128 c, n, o;\n"
                                        "mov.b128 c, {%3, %3};\n"
                                        "mov.b128 n, {%4, %5};\n"
                                        "atom.shared.cas.b128 o, [%2], c, n;\n"
                                        "mov.b128 {%0, %1}, o;\n"
                                        "}\n"
                                        : "=l"(cur.x), "=l"(cur.y)
                                        : "r"(a), "l"(~0ull), "l"(rec.x), "l"(rec.y)
                                        : "memory");
                                    if (cur.x == ~0ull && cur.y == ~0ull) { rslot[u2] = h; atomicAdd(&rt_mult[h], 1u); break; }
                                }
                                if (cur.x == rec.x && cur.y == rec.y) { atomicAdd(&rt_mult[h], 1u); break; }
                                h = (h + 1) & (RT - 1);
                            }
                            live[u2] = rslot[u2] != 0xffffffffu;
                            dedup_local += live[u2] ? 0u : 1u;
                        }
                    }
                }
                SWP_MARK(SWP_DEDUP);
                // One block scan gives every surviving record its place in the compacted round (high
                // half) and the index of its first window in the flattened window sequence (low half: a
                // round has fewer than 65536 windows). A thread's records are adjacent in that order. The
                // scan's barrier also completes the record table's multiplicities.
                uint32_t vsum = 0;
#pragma unroll
                for (int u2 = 0; u2 < RPT; u2++) vsum += live[u2] ? ((1u << 16) | c[u2]) : 0u;
                uint32_t incl = vsum;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
                    if (lane >= (uint32_t)o) incl += t;
                }
                if (lane == 31) s_warp[warp] = incl;
                __syncthreads();
                uint32_t excl = incl - vsum, all = 0;
#pragma unroll
                for (int wq = 0; wq < THREADS / 32; wq++) {
                    const uint32_t t = s_warp[wq];
                    if ((uint32_t)wq < warp) excl += t;
                    all += t;
                }
                const uint32_t tot = all & 0xffffu;
                // this thread's share of the tot windows: [f0, f1)
                const uint32_t per = (tot + THREADS - 1) / THREADS;
#pragma unroll
                for (int u2 = 0; u2 < RPT; u2++) {
                    if (live[u2]) {
                        const uint32_t ci = excl >> 16, w0 = excl & 0xffffu;
#pragma unroll
                        for (int t = 0; t < W; t++) recs[ci * W + t] = pf[u2][t];
                        uint32_t m = 1;
                        if constexpr (DEDUP) {
                            m = rt_mult[rslot[u2]];
                            rt_keys[rslot[u2]] = make_ulonglong2(~0ull, ~0ull);
                            rt_mult[rslot[u2]] = 0;
                        }
                        rec_mult[ci] = m;
                        // the threads whose first window lies in this record start here (a record has at
                        // least one window, so per > 0; t * per < tot keeps t < THREADS)
                        for (uint32_t t = (w0 + per - 1) / per; t * per < w0 + c[u2]; t++) s_start[t] = ci << 8 | (t * per - w0);
                        excl += (1u << 16) | c[u2];
                    }
                }
                __syncthreads();
                SWP_MARK(SWP_SCAN);
                // prefetch the next round
#pragma unroll
                for (int u2 = 0; u2 < RPT; u2++) {
                    const uint32_t i = r0 + RB + u2 * THREADS + tid;
                    if (i < n_rec) {
                        const ulonglong2 *rp = rec_at(i);
#pragma unroll
                        for (int t = 0; t < W; t++) pf[u2][t] = rp[t];
                    }
                }
                if (r0 + RB >= n_rec && bits == 0 && un < n_units) {     // last round of the unit's first pass: the next unit's first round
                    const uint32_t n_next = s_desc[par ^ 1][8];
#pragma unroll
                    for (int u2 = 0; u2 < RPT; u2++) {
                        const uint32_t i = u2 * THREADS + tid;
                        if (i < n_next) {
                            const ulonglong2 *rp = rec_of(un, par ^ 1, i);
#pragma unroll
                            for (int t = 0; t < W; t++) pf[u2][t] = rp[t];
                        }
                    }
                    pf_id = un;
                }
                const uint32_t f0 = min(tid * per, tot), f1 = min(f0 + per, tot);
                {
                    uint32_t rem = f1 - f0;                        // windows this lane still has to fetch
                    occ_local += rem;
                    uint32_t ri = 0;                               // next record to open
                    uint64_t rw[2 * W];
#pragma unroll
                    for (int t = 0; t < 2 * W; t++) rw[t] = 0;
                    uint32_t in_rec = 0;                           // windows left in the open record
                    uint32_t wgt = 1;                              // how many equal records the open one stands for
                    if (rem) {   // open the first record at window j
                        const uint32_t st = s_start[tid];
                        ri = st >> 8;
                        const uint32_t j = st & 0xffu;
                        wgt = rec_mult[ri];
#pragma unroll
                        for (int t = 0; t < W; t++) { const ulonglong2 v = recs[ri * W + t]; rw[2 * t] = v.x; rw[2 * t + 1] = v.y; }
                        const uint32_t cnt = (uint32_t)(rw[2 * W - 1] & 0xffull);
                        uint32_t sh = 2 * j;
                        if constexpr (W > 1) {
                            while (sh >= 64) {
#pragma unroll
                                for (int t = 0; t < 2 * W - 1; t++) rw[t] = rw[t + 1];
                                rw[2 * W - 1] = 0;
                                sh -= 64;
                            }
                        }
                        if (sh) {
#pragma unroll
                            for (int t = 0; t < 2 * W - 1; t++) rw[t] = (rw[t] << sh) | (rw[t + 1] >> (64 - sh));
                            rw[2 * W - 1] <<= sh;
                        }
                        in_rec = min(rem, cnt - j);
                        ri++;
                    }
                    SWP_MARK(SWP_OPEN);
                    // Pass 1: every lane gives each of its keys ONE probe at its home bucket (two
                    // adjacent slots, one 16-byte load for 64-bit keys) -- no loop, so no lane waits for
                    // another's probe sequence. A key whose bucket is taken by two other keys goes to
                    // the warp's queue; the queue is drained with the usual bucket-by-bucket probing
                    // whenever it fills up, and after the last key.
                    Key<W> *wq = queue + warp * kQueue;
                    uint32_t *wqm = queue_m + warp * kQueue;
                    uint32_t qn = 0;                               // keys queued (uniform across the warp)
                    // found or placed in bucket hb (count += kw): true; both slots hold other keys: false
                    auto try_bucket = [&](uint32_t hb, const Key<W> &key, uint32_t kw, bool act) -> bool {
                        Key<W> k0, k1;
                        if constexpr (W == 1) {
                            const ulonglong2 v = *reinterpret_cast<const ulonglong2 *>(tk + 2 * hb);
                            k0.w[0] = v.x; k1.w[0] = v.y;
                        } else {
                            k0 = tk[2 * hb]; k1 = tk[2 * hb + 1];
                        }
                        // a slot that looks (even partly: a 128-bit read may tear) empty is settled by a CAS
                        const bool e0 = key_any_word_ones<W>(k0), e1 = key_any_word_ones<W>(k1);
                        const bool h1 = !e1 && key_eq<W>(k1, key);
                        bool hit = h1 || (!e0 && key_eq<W>(k0, key));
                        uint32_t slot = 2 * hb + (h1 ? 1u : 0u);
                        if (act && !hit && (e0 || e1)) {           // only these lanes branch off
                            slot = 2 * hb + (e0 ? 0u : 1u);
                            Key<W> old = slot_claim(&tk[slot], key);
                            bool claimed = key_all_ones<W>(old);
                            hit = claimed || key_eq<W>(old, key);
                            if (!hit && e0 && e1) {                // slot 0 went to another key; slot 1 looked empty too
                                slot = 2 * hb + 1;
                                old = slot_claim(&tk[slot], key);
                                claimed = key_all_ones<W>(old);
                                hit = claimed || key_eq<W>(old, key);
                            }
                            claims += claimed ? 1u : 0u;
                        }
                        if (act && hit) atomicAdd(&tc[slot], kw);
                        return hit;
                    };
                    auto drain = [&]() {
                        SWP_MARK(SWP_INSERT);
                        __syncwarp();
                        for (uint32_t en = lane; en < qn; en += 32) {
                            const Key<W> k = wq[en];
                            const uint32_t kw = wqm[en];
                            uint32_t hb = key_hash<W>(k) >> (hshift + 1);
                            bool done = false;
#pragma unroll 1
                            for (uint32_t probes = 0; probes < 64u && !done; probes++) {
                                done = try_bucket(hb, k, kw, true);
                                SWP_ADD_ACTIVE(SWP_DRAIN_PROBES);
                                hb = (hb + 1) & (TSLOTS / 2 - 1);
                            }
                            if (!done) s_abort = 1;                // table (nearly) full: the pass is abandoned
                        }
                        __syncwarp();
                        qn = 0;
                        SWP_MARK(SWP_DRAIN);
                    };
#pragma unroll 1
                    for (uint32_t it = 0; it < per; it++) {
                        bool act = rem != 0;
                        Key<W> key;
#pragma unroll
                        for (int t = 0; t < W; t++) key.w[t] = 0;
                        uint32_t hb = 0;
                        if (act) {
                            if (in_rec == 0) {
                                wgt = rec_mult[ri];
#pragma unroll
                                for (int t = 0; t < W; t++) { const ulonglong2 v = recs[ri * W + t]; rw[2 * t] = v.x; rw[2 * t + 1] = v.y; }
                                in_rec = min(rem, (uint32_t)(rw[2 * W - 1] & 0xffull));
                                ri++;
                            }
#pragma unroll
                            for (int t = 0; t < W; t++) key.w[t] = rw[t];
                            key.w[W - 1] &= p.last_mask;
                            if constexpr (CANON) key = key_canonical<W>(key, rc_sh);
                            in_rec--;
                            rem--;
#pragma unroll
                            for (int t = 0; t < 2 * W - 1; t++) rw[t] = (rw[t] << 2) | (rw[t + 1] >> 62);
                            rw[2 * W - 1] <<= 2;
                            if (key_all_ones<W>(key)) {            // the table's empty marker: counted on the side
                                if (in_pass(0x9E3779B1u)) atomicAdd(&s_ones, wgt);
                                act = false;
                            } else {
                                const uint32_t hv = key_hash<W>(key);
                                hb = hv >> (hshift + 1);
                                act = in_pass(hv);
                            }
                        }
                        const bool hit = try_bucket(hb, key, wgt, act);       // (inactive lanes read bucket 0: harmless)
                        const bool coll = act && !hit;
                        const uint32_t cm = __ballot_sync(0xffffffffu, coll);
                        if (cm) {
                            if (coll) {
                                const uint32_t qi = qn + __popc(cm & lanemask_lt());
                                wq[qi] = key;
                                wqm[qi] = wgt;
                            }
                            qn += __popc(cm);
                            if (lane == 0) SWP_ADD(SWP_QUEUED, __popc(cm));
                            if (qn > (uint32_t)kQueue - 32u) drain();
                        }
                    }
                    if (qn) drain();
                    SWP_MARK(SWP_INSERT);
                }
                // distinct keys so far
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) claims += __shfl_xor_sync(0xffffffffu, claims, o);
                if (lane == 0 && claims) atomicAdd(&s_m, claims);
                claims = 0;
                __syncthreads();
                SWP_MARK(SWP_ROUND_END);
                if (s_abort || s_m > kLimit) { aborted = true; break; }
            }
            if (!aborted && n_rec == 0) {                // the phantom alone: no round ran (a round's end counted the claims)
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) claims += __shfl_xor_sync(0xffffffffu, claims, o);
                if (lane == 0 && claims) atomicAdd(&s_m, claims);
                __syncthreads();
                if (s_abort) aborted = true;
            }
            if (aborted) {
                // occurrences of this pass are counted again by its two halves
                Key<W> empty;
                key_set_ones<W>(empty);
                __syncthreads();
                for (uint32_t i = tid; i < (uint32_t)TSLOTS; i += THREADS) { tk[i] = empty; tc[i] = 0; }
                if (tid == 0) { s_m = 0; s_ones = 0; s_abort = 0; }
                aborts_local++;
                bits++;                                   // left half first
                if (bits > 24) {
                    if (tid == 0) atomicOr(&p.sc[SW_FAIL], 4ull);
                    __syncthreads();
                    break;
                }
                val <<= 1;
                __syncthreads();
                SWP_MARK(SWP_EMIT);
                continue;
            }
            // ---- emit the pass: distinct (key, count) records appended to D, table cleared. Warp w
            // takes the slots [w * SPW, (w + 1) * SPW): it counts its live slots while thread 0's
            // atomic on |D| is in flight, and one scan of the warps' counts places every record.
            constexpr uint32_t SPW = TSLOTS / (THREADS / 32);
            const uint32_t m = s_m, ones = s_ones;
            const uint32_t m_tot = m + (ones ? 1u : 0u);
            if (tid == 0) s_base = m_tot ? atomicAdd(&p.sc[SW_D], (unsigned long long)m_tot) : 0ull;
            const Key<W> *wtk = tk + warp * SPW;
            uint32_t wlive = 0;
#pragma unroll
            for (uint32_t i0 = 0; i0 < SPW; i0 += 32) wlive += __popc(__ballot_sync(0xffffffffu, !key_all_ones<W>(wtk[i0 + lane])));
            if (lane == 0) s_warp[warp] = wlive;
            __syncthreads();
            const unsigned long long base = s_base;
            if (base + m_tot > p.d_cap) {
                if (tid == 0) atomicOr(&p.sc[SW_FAIL], 2ull);
            }
            unsigned long long o_run = base;
#pragma unroll
            for (int wq = 0; wq < THREADS / 32; wq++) o_run += (uint32_t)wq < warp ? s_warp[wq] : 0u;
            Key<W> empty;
            key_set_ones<W>(empty);
#pragma unroll 1
            for (uint32_t i0 = 0; i0 < SPW; i0 += 32) {
                const uint32_t i = warp * SPW + i0 + lane;
                const Key<W> k = tk[i];
                const bool live = !key_all_ones<W>(k);
                const uint32_t bal = __ballot_sync(0xffffffffu, live);
                if (live) {
                    const unsigned long long o = o_run + __popc(bal & lanemask_lt());
                    if (o < p.d_cap) {
                        st_key<W>(p.d_keys, o, k);
                        p.d_counts[o] = tc[i];
                    }
                    atomicAdd(&s_hist[k.w[0] >> p.shift1], 1u);
                    tk[i] = empty;
                    tc[i] = 0;
                }
                o_run += __popc(bal);
            }
            if (ones && tid == 0) {
                const unsigned long long o = base + m;
                if (o < p.d_cap) {
                    st_key<W>(p.d_keys, o, empty);
                    p.d_counts[o] = ones;
                }
                atomicAdd(&s_hist[p.nb1 - 1], 1u);
            }
            __syncthreads();
            if (tid == 0) { s_m = 0; s_ones = 0; }
            // next pass: climb while this was a right half, then step to the right sibling
            // (pass ids are prefixes of the pass hash, most significant bit first)
            while (bits > 0 && (val & 1u)) { val >>= 1; bits--; }
            if (bits == 0) { SWP_MARK(SWP_EMIT); break; }      // (the next unit starts with a barrier)
            val |= 1u;
            __syncthreads();
            SWP_MARK(SWP_EMIT);
        }
    }
    __syncthreads();
    for (uint32_t i = tid; i < (uint32_t)p.nb1; i += THREADS) {
        const uint32_t c = s_hist[i];
        if (c) atomicAdd(&p.hist1[i], c);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) occ_local += __shfl_xor_sync(0xffffffffu, occ_local, o);
    for (int o = 16; o > 0; o >>= 1) dedup_local += __shfl_xor_sync(0xffffffffu, dedup_local, o);
    if (lane == 0 && occ_local) atomicAdd(&p.sc[SW_OCC], occ_local);
    if (lane == 0 && dedup_local) atomicAdd(&p.sc[SW_DEDUP], (unsigned long long)dedup_local);
    if (tid == 0 && aborts_local) atomicAdd(&p.sc[SW_ABORTS], (unsigned long long)aborts_local);
    if (tid == 0 && multi_local) atomicAdd(&p.sc[SW_MULTI], (unsigned long long)multi_local);
    SWP_FLUSH();
}

// ============================================================ S3: ordering the records
// per-bin counters of the record scatter and of S3c's counting sort are indexed through pad32
constexpr int kRsBinsPadded = kRsBins + kRsBins / 32;

// One block. S2 left a histogram of the records' leading b1_max bits; the plan picks the two
// digit widths from the number of records actually there -- B = b1 + b2 bits so that a sub-bucket
// holds about sub_target records, level 1 as narrow as level 2's limit of 9 bits allows (long
// runs per bin in the unordered first scatter) -- folds the histogram to b1 bits and scans it.
__global__ void __launch_bounds__(1024) sw_plan_kernel(const uint32_t *__restrict__ hist1, int b1_max, uint64_t d_cap,
                                                       uint32_t sub_target, int sig_bits, uint32_t *__restrict__ base1,
                                                       uint32_t *__restrict__ cursor1, SuperPlanDev *__restrict__ plan,
                                                       const unsigned long long *__restrict__ sc) {
    __shared__ uint32_t s_a[32];
    unsigned long long nd = sc[SW_D];
    if (nd > d_cap) nd = d_cap;
    int B = 1;
    while (B < b1_max + 10 && B < sig_bits && (nd >> B) > sub_target) B++;
    int b1 = B - 9 > (B < 16 ? B / 2 : 8) ? B - 9 : (B < 16 ? B / 2 : 8);       // (level 2 takes a 10th bit only when level 1 is at its 10)
    if (b1 > b1_max) b1 = b1_max;
    if (b1 < 1) b1 = 1;
    const int b2 = B - b1 > 0 ? B - b1 : 0;
    const int nb1 = 1 << b1, group = 1 << (b1_max - b1);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    uint32_t c = 0;
    if (tid < nb1)
        for (int j = 0; j < group; j++) c += hist1[tid * group + j];
    uint32_t ia = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t xa = __shfl_up_sync(0xffffffffu, ia, o);
        if (lane >= o) ia += xa;
    }
    if (lane == 31) s_a[warp] = ia;
    __syncthreads();
    uint32_t oa = 0;
    for (int w = 0; w < warp; w++) oa += s_a[w];
    if (tid < nb1) {
        base1[tid] = oa + ia - c;
        cursor1[tid] = oa + ia - c;
        if (tid == nb1 - 1) base1[nb1] = oa + ia;
    }
    if (tid == 0) {
        plan->n_d = (uint32_t)nd;
        plan->b1 = (uint32_t)b1;
        plan->b2 = (uint32_t)b2;
        plan->shift2 = 64 - b1 - b2;
        plan->n_sub = (uint32_t)nb1 << b2;
        plan->prefix_bits = b1 + b2;
        plan->sub0 = 0;
    }
}

// ------------------------------------------------------------- multi-GPU exchange
// Every rank has counted its own reads (S2) and holds the histogram of its records' leading
// kXB1 bits; the histograms of all ranks were all-gathered. One block derives, identically on
// every rank: the owner of each level-1 bucket (contiguous bucket ranges with about equal record
// totals: rank o owns keys whose leading bits lie in [lo[o], lo[o+1])) and the level-2 digit width
// (from the global total, so that every rank cuts the same sub-buckets); and for this rank: its own
// level-1 bases (the local scatter), where its key range starts and ends inside every source's
// grouped array, and the plan of its part of the key space.
constexpr int kXB1 = 10;                // bits of the histogram the ranks exchange
constexpr int kXB2Max = 11;             // most level-2 bits of an exchange (2^21 sub-buckets over all ranks)
typedef SuperXInfo XDev;
struct XScalars { const unsigned long long *sc[8]; };

__global__ void __launch_bounds__(1024) x_plan_kernel(const uint32_t *__restrict__ all_hist, uint32_t rank, uint32_t P,
                                                      int keep_ranges, uint64_t d_cap, uint32_t sub_target, int large_plan, int sig_bits,
                                                      uint32_t *__restrict__ base1, uint32_t *__restrict__ cursor1,
                                                      SuperPlanDev *__restrict__ plan, XDev *__restrict__ x,
                                                      unsigned long long *__restrict__ sc, XScalars peers) {
    constexpr int NB = 1 << kXB1;
    __shared__ unsigned long long s_scan[32];
    __shared__ uint32_t s_lo[17];
    __shared__ unsigned long long s_total, s_b, s_e;
    __shared__ int s_b1, s_b2, s_large;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // block-wide inclusive scan of 64-bit values (1024 threads)
    auto block_incl = [&](unsigned long long v) -> unsigned long long {
        unsigned long long incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        __syncthreads();
        if (lane == 31) s_scan[warp] = incl;
        __syncthreads();
        unsigned long long off = 0;
        for (int w = 0; w < warp; w++) off += s_scan[w];
        return off + incl;
    };
    unsigned long long tot = 0;
    for (uint32_t s2 = 0; s2 < P; s2++) tot += all_hist[s2 * NB + tid];
    const unsigned long long cum = block_incl(tot);
    if (tid == NB - 1) s_total = cum;
    if (tid <= 16) s_lo[tid] = NB;
    __syncthreads();
    const unsigned long long total = s_total;
    if (tid == 0) {
        // digit widths from the job's record total: B bits so that a sub-bucket holds about sub_target
        // records, level 1 as narrow as level 2's limit of 10 bits allows but not below 8 (the key
        // ranges of up to 8 ranks are cut at level-1 buckets)
        // A job too large for 2^20 sub-buckets of sub_target records takes an 11th level-2 bit (a rank
        // holds 1/P of the sub-buckets, so its own arrays stay within kSuperMaxSub) and, if the
        // sub-buckets are still too large for the small S3c variant, the large one (x->fin_large).
        int B = 8;
        while (B < kXB1 + kXB2Max && B < sig_bits && (total >> B) > sub_target) B++;
        int b1 = B - 10 > 8 ? B - 10 : 8;
        if (b1 > kXB1 || keep_ranges) b1 = kXB1;     // kept ranges may have been cut at any histogram bin
        if (b1 > sig_bits) b1 = sig_bits;
        s_b1 = b1;
        s_b2 = B - b1 > 0 ? B - b1 : 0;
    }
    __syncthreads();
    const int b1 = s_b1, fold = kXB1 - b1;                     // 2^fold histogram bins per level-1 bucket
    // owner of histogram bin tid = owner of its level-1 bucket: where the middle of the BUCKET falls in
    // P equal shares of the total (all bins of a bucket get the same owner)
    const uint32_t bk0 = ((uint32_t)tid >> fold) << fold;      // first bin of this bin's bucket
    __shared__ unsigned long long s_cum[NB + 1];
    s_cum[tid + 1] = cum;
    if (tid == 0) s_cum[0] = 0;
    __syncthreads();
    const unsigned long long bk_lo = s_cum[bk0], bk_hi = s_cum[bk0 + (1u << fold)];
    uint32_t owner = 0;
    if (total) owner = (uint32_t)((bk_lo + (bk_hi - bk_lo) / 2) * P / total);
    if (owner >= P) owner = P - 1;
    atomicMin(&s_lo[owner], bk0);
    __syncthreads();
    if (tid == 0) {                                   // owners without a bucket start where the next one does
        s_lo[P] = NB;
        for (int o = (int)P - 1; o >= 0; o--)
            if (s_lo[o] > s_lo[o + 1]) s_lo[o] = s_lo[o + 1];
        s_lo[0] = 0;
        if (keep_ranges)                              // the ranges of the previous exchange (runs that will be merged)
            for (uint32_t o = 0; o <= P; o++) s_lo[o] = x->lo[o];
        for (uint32_t o = 0; o <= P; o++) x->lo[o] = s_lo[o];
        // no rank may end up with more than kSuperMaxSub sub-buckets (its arrays): the widest key range decides
        uint32_t widest = 1;
        for (uint32_t o = 0; o < P; o++) {
            const uint32_t wd = ((s_lo[o + 1] + (1u << fold) - 1) >> fold) - (s_lo[o] >> fold);
            widest = wd > widest ? wd : widest;
        }
        while (s_b2 > 0 && ((unsigned long long)widest << s_b2) > kSuperMaxSub) s_b2--;
        // sub-buckets beyond the small S3c variant's reach: every rank sorts with the large one
        s_large = (large_plan || (total >> (b1 + s_b2)) > sub_target) ? 1 : 0;
    }
    __syncthreads();
    const uint32_t my_lo = s_lo[rank], my_hi = s_lo[rank + 1];      // in histogram bins (multiples of 2^fold unless kept)
    // this rank's key range inside every source's grouped array
    unsigned long long n_recv = 0;
    for (uint32_t s2 = 0; s2 < P; s2++) {
        const unsigned long long incl = block_incl(all_hist[s2 * NB + tid]);
        if (tid == 0) { s_b = 0; s_e = 0; }
        __syncthreads();
        if (my_lo > 0 && tid == (int)my_lo - 1) s_b = incl;
        if (my_hi > 0 && tid == (int)my_hi - 1) s_e = incl;
        __syncthreads();
        if (tid == 0) { x->src_range[s2][0] = (uint32_t)s_b; x->src_range[s2][1] = (uint32_t)s_e; }
        n_recv += s_e - s_b;
        __syncthreads();
    }
    // own level-1 bases: the local scatter groups this rank's records by their leading b1 bits
    {
        const uint32_t nb1 = 1u << b1;
        uint32_t c = 0;
        if ((uint32_t)tid < nb1)
            for (int j = 0; j < (1 << fold); j++) c += all_hist[rank * NB + ((uint32_t)tid << fold) + j];
        const unsigned long long incl = block_incl(c);
        if ((uint32_t)tid < nb1) {
            base1[tid] = (uint32_t)(incl - c);
            cursor1[tid] = (uint32_t)(incl - c);
            if ((uint32_t)tid == nb1 - 1) base1[nb1] = (uint32_t)incl;
        }
    }
    if (tid == 0) {
        const int b2 = s_b2;                                   // (as settled above)
        unsigned long long nd = sc[SW_D];
        if (nd > d_cap) nd = d_cap;
        uint32_t any_ovf = 0;
        for (uint32_t s2 = 0; s2 < P; s2++)
            if (peers.sc[s2][SW_OVF] != 0) any_ovf = 1;
        plan->n_d = (uint32_t)nd;
        plan->b1 = (uint32_t)b1;
        plan->b2 = (uint32_t)b2;
        plan->shift2 = 64 - b1 - b2;
        // this rank's sub-buckets: the (b1+b2)-bit prefixes inside its key range
        plan->sub0 = (my_lo >> fold) << b2;
        plan->n_sub = (((my_hi + (1u << fold) - 1) >> fold) << b2) - plan->sub0;
        plan->prefix_bits = b1 + b2;
        x->n_recv = (uint32_t)(n_recv > 0xffffffffull ? 0xffffffffull : n_recv);
        x->any_ovf = any_ovf;
        x->fin_large = (uint32_t)s_large;
        if (n_recv > d_cap) atomicOr(&sc[SW_FAIL], 16ull);       // this rank's share does not fit its buffers
    }
}

// level-2 counters of this rank's sub-buckets = sum over the sources' own histograms (peer loads)
struct XPeers {
    const uint64_t *keys[8];
    const uint32_t *counts[8];
    const uint32_t *hist2[8];
};
__global__ void __launch_bounds__(256) x_merge_hist_kernel(XPeers peers, uint32_t P, const SuperPlanDev *__restrict__ plan,
                                                           uint32_t *__restrict__ out) {
    const uint32_t n = plan->n_sub, sub0 = plan->sub0;
    for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x) {
        uint32_t c = 0;
        for (uint32_t s2 = 0; s2 < P; s2++) c += peers.hist2[s2][sub0 + j];
        out[j] = c;
    }
}

constexpr int kRsThreads = 256;
template <int W> struct RsCfg { static constexpr int ITEMS = 16 / W, TILE = kRsThreads * ITEMS; };

// Scatter of (key, count) records by a digit of the key, over flat tiles of the input.
// LEVEL 1: digit = leading b1 bits, any bin may occur in a tile.
// LEVEL 2: the input is grouped by the level-1 digit, so a tile's keys name (almost always) one
// or two level-1 buckets: bins are relative to the first key's bucket, two buckets wide when the
// tile straddles a boundary; a key further away is placed on its own.
template <int W, int LEVEL>
__global__ void __launch_bounds__(kRsThreads) rec_scatter_kernel(const uint64_t *__restrict__ in_keys,
                                                                 const uint32_t *__restrict__ in_counts,
                                                                 uint64_t *__restrict__ out_keys,
                                                                 uint32_t *__restrict__ out_counts,
                                                                 const SuperPlanDev *__restrict__ plan, int b1,
                                                                 const unsigned long long *__restrict__ n_ptr, uint64_t cap,
                                                                 uint32_t *__restrict__ g_cursor,
                                                                 const uint32_t *__restrict__ range) {
    constexpr int ITEMS = RsCfg<W>::ITEMS, TILE = RsCfg<W>::TILE;
    extern __shared__ __align__(16) uint8_t rs_smem[];
    Key<W> *stg_k = reinterpret_cast<Key<W> *>(rs_smem);                    // [TILE]
    uint32_t *stg_c = reinterpret_cast<uint32_t *>(stg_k + TILE);           // [TILE]
    uint32_t *cnt = stg_c + TILE, *start = cnt + kRsBinsPadded, *gbase = start + kRsBinsPadded;   // indexed through pad32
    __shared__ uint32_t s_warp[kRsThreads / 32];
    uint32_t n, first = 0;
    if (LEVEL == 1) {
        unsigned long long nn = *n_ptr;
        n = (uint32_t)(nn > cap ? cap : nn);
    } else if (range) {                          // a slice of a (peer's) grouped array: records [range[0], range[1])
        first = range[0];
        n = range[1];
    } else {
        n = plan->n_d;
    }
    const int b2 = LEVEL == 1 ? 0 : (int)plan->b2;
    if (LEVEL == 1) b1 = (int)plan->b1;
    const int shift = LEVEL == 1 ? 64 - b1 : (int)plan->shift2;
    const uint32_t nb2 = 1u << b2;
    const uint32_t sub0 = LEVEL == 1 ? 0u : plan->sub0;     // cursors are indexed relative to this rank's first sub-bucket
    for (uint32_t begin = first + blockIdx.x * (uint32_t)TILE; begin < n; begin += gridDim.x * (uint32_t)TILE) {
        const uint32_t end = begin + TILE < n ? begin + TILE : n;
        Key<W> key[ITEMS];
        uint32_t val[ITEMS];
        uint16_t rank[ITEMS];
#pragma unroll
        for (int i = 0; i < ITEMS; i++) {
            const uint32_t idx = begin + i * kRsThreads + threadIdx.x;
            if (idx < end) { key[i] = ld_key<W>(in_keys, idx); val[i] = in_counts[idx]; }
            else { key[i].w[0] = 0; val[i] = 0; }
        }
        uint32_t p0 = 0, nb;
        if (LEVEL == 1) {
            nb = 1u << b1;
        } else {
            p0 = ((uint32_t)(in_keys[(size_t)begin * W] >> shift) >> b2) << b2;       // first sub-bucket of the first key's bucket
            const uint32_t pl = (uint32_t)(in_keys[(size_t)(end - 1) * W] >> shift);
            // (b2 = 11: the counters hold one bucket; the keys of a tile's second bucket are placed one by one)
            nb = (pl >> b2) == (p0 >> b2) || 2 * nb2 > (uint32_t)kRsBins ? nb2 : 2 * nb2;
        }
        for (uint32_t i = threadIdx.x; i < nb; i += kRsThreads) cnt[pad32(i)] = 0;
        __syncthreads();
#pragma unroll
        for (int i = 0; i < ITEMS; i++) {
            const uint32_t idx = begin + i * kRsThreads + threadIdx.x;
            rank[i] = 0xffffu;
            if (idx < end) {
                const uint32_t pfx = (uint32_t)(key[i].w[0] >> shift);
                const uint32_t rel = pfx - p0;
                if (rel < nb) rank[i] = (uint16_t)atomicAdd(&cnt[pad32(rel)], 1u);
                else {
                    const uint32_t o = atomicAdd(&g_cursor[pfx - sub0], 1u);
                    st_key<W>(out_keys, o, key[i]);
                    out_counts[o] = val[i];
                }
            }
        }
        __syncthreads();
        const uint32_t total = block_scan_bins<kRsThreads, kRsBins, true>(cnt, start, (int)nb, s_warp);
        // reserve the bins' ranges, stage the records while the atomics are in flight, then look at the answers
        uint32_t reserved[kRsBins / kRsThreads];
#pragma unroll
        for (int u = 0; u < kRsBins / kRsThreads; u++) {
            const uint32_t b = u * kRsThreads + threadIdx.x;
            reserved[u] = 0;
            if (b < nb) {
                const uint32_t c = cnt[pad32(b)];
                if (c) reserved[u] = atomicAdd(&g_cursor[p0 - sub0 + b], c);
            }
        }
#pragma unroll
        for (int i = 0; i < ITEMS; i++)
            if (rank[i] != 0xffffu) {
                const uint32_t o = start[pad32((uint32_t)(key[i].w[0] >> shift) - p0)] + rank[i];
                stg_k[o] = key[i];
                stg_c[o] = val[i];
            }
#pragma unroll
        for (int u = 0; u < kRsBins / kRsThreads; u++) {
            const uint32_t b = u * kRsThreads + threadIdx.x;
            if (b < nb) gbase[pad32(b)] = reserved[u] - start[pad32(b)];
        }
        __syncthreads();
        for (uint32_t i = threadIdx.x; i < total; i += kRsThreads) {
            const Key<W> k = stg_k[i];
            const uint32_t o = gbase[pad32((uint32_t)(k.w[0] >> shift) - p0)] + i;
            st_key<W>(out_keys, o, k);
            out_counts[o] = stg_c[i];
        }
        __syncthreads();
    }
}

// Key-placement path: D's keys were written by the extraction (one per k-mer slot, key 0 where a
// slot holds no k-mer). Every record gets count 1; the histogram of the leading b1 bits that S2
// would have kept is built here; sc[SW_D] = n.
template <int W>
__global__ void __launch_bounds__(256) place_init_kernel(const uint64_t *__restrict__ keys, uint32_t *__restrict__ counts,
                                                         uint64_t n, int shift1, uint32_t *__restrict__ hist1,
                                                         unsigned long long *__restrict__ sc) {
    __shared__ uint32_t sh[kNb1Max];
    for (uint32_t i = threadIdx.x; i < kNb1Max; i += 256) sh[i] = 0;
    __syncthreads();
    for (uint64_t i = blockIdx.x * 256ull + threadIdx.x; i < n; i += gridDim.x * 256ull) {
        counts[i] = 1u;
        atomicAdd(&sh[(uint32_t)(keys[i * W] >> shift1)], 1u);
    }
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < kNb1Max; i += 256) {
        const uint32_t c = sh[i];
        if (c) atomicAdd(&hist1[i], c);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) sc[SW_D] = n;
}

// the run's first record loses the empty slots that were counted as key 0 (SURVEY F7: the record
// itself stays, with whatever real occurrences key 0 has)
template <int W>
__global__ void place_fix_zero_kernel(const uint64_t *__restrict__ keys, uint32_t *__restrict__ counts,
                                      const unsigned long long *__restrict__ n_invalid) {
    bool zero = true;
    for (int w = 0; w < W; w++) zero = zero && keys[w] == 0;
    if (zero) counts[0] -= (uint32_t)*n_invalid;
}

// Level-2 histogram of the level-1-grouped keys (flat chunks; counters of the chunk's first
// bucket in shared memory, stragglers straight to the global counter).
constexpr uint32_t kH2Chunk = 16384;
template <int W>
__global__ void __launch_bounds__(256) rec_hist2_kernel(const uint64_t *__restrict__ keys,
                                                        const SuperPlanDev *__restrict__ plan,
                                                        uint32_t *__restrict__ g_hist2) {
    __shared__ uint32_t sh[kRsBins];             // nb2 <= 2048 (b2 <= kXB2Max)
    const uint32_t n = plan->n_d;
    const int b2 = (int)plan->b2, shift2 = (int)plan->shift2;
    const uint32_t nb2 = 1u << b2, m2 = nb2 - 1;
    for (uint32_t begin = blockIdx.x * kH2Chunk; begin < n; begin += gridDim.x * kH2Chunk) {
        const uint32_t end = begin + kH2Chunk < n ? begin + kH2Chunk : n;
        for (uint32_t i = threadIdx.x; i < nb2; i += 256) sh[i] = 0;
        const uint32_t b0 = (uint32_t)(keys[(size_t)begin * W] >> shift2) >> b2;
        __syncthreads();
#pragma unroll 4
        for (uint32_t i = begin + threadIdx.x; i < end; i += 256) {
            const uint32_t pfx = (uint32_t)(keys[(size_t)i * W] >> shift2);
            if ((pfx >> b2) == b0) atomicAdd(&sh[pfx & m2], 1u);
            else atomicAdd(&g_hist2[pfx], 1u);
        }
        __syncthreads();
        for (uint32_t i = threadIdx.x; i < nb2; i += 256) {
            const uint32_t c = sh[i];
            if (c) atomicAdd(&g_hist2[(size_t)b0 * nb2 + i], c);
        }
        __syncthreads();
    }
}

struct FinishParams {
    const uint64_t *in_keys;
    const uint32_t *in_counts;
    const uint32_t *base2;          // [n_sub + 1]
    const SuperPlanDev *plan;
    uint64_t *out_keys;             // records of sub-bucket j at out[base2[j] ...)
    uint32_t *out_counts;
    uint32_t *m_out;                // DUP: records sub-bucket j kept
    uint32_t *big;                  // records of sub-bucket j if it is too large for this kernel, else 0
    unsigned long long *sc;
};

// S3c: one CTA per sub-bucket (at most CAP records, all sharing their leading prefix_bits). The
// records go from global memory into registers, are grouped by a counting sort on the next key
// bits (about two bins per record) in shared memory, and every record then finds its final place
// by comparing itself with the few records of its own bin -- no serial insertion sort, every lane
// busy. A bitonic network takes over when some bin is crowded (keys sharing their next bits, many
// copies of one key). DUP: equal keys are folded (counts added, uint32 wrap), survivors compacted.
// The records are written once, in key order.
template <int W, int THREADS, int CAP, bool DUP>
__global__ void __launch_bounds__(THREADS) rec_finish_kernel(FinishParams p) {
    constexpr int kPer = CAP / THREADS;
    extern __shared__ __align__(16) uint8_t fs_smem[];
    Key<W> *sk = reinterpret_cast<Key<W> *>(fs_smem);                  // grouped by bin [CAP]
    Key<W> *fk = sk + (DUP ? CAP : 0);                                 // DUP: in final order [CAP]
    uint32_t *scn = reinterpret_cast<uint32_t *>(fk + CAP);            // [CAP]
    uint32_t *fc = scn + (DUP ? CAP : 0);                              // DUP [CAP]
    uint32_t *c3 = fc + CAP;                                           // counting-sort bins [CAP], indexed through pad32
    uint32_t *s3 = c3 + CAP + CAP / 32;                                // their starts       [CAP], likewise
    __shared__ uint32_t s_maxbin, s_cnt, s_j, s_b, s_e;
    __shared__ uint32_t s_warp[THREADS / 32];
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t n_sub = p.plan->n_sub;
    const int prefix_bits = (int)p.plan->prefix_bits;
    unsigned long long folded_local = 0;
    // Work tickets are drawn two ahead by thread 0: the ticket after next is in flight while the next
    // sub-bucket's bounds are being loaded, so neither the atomic's nor the loads' round trip is waited
    // for at the top of the loop (they cost ~9 % of the kernel's samples when fetched on demand).
    uint32_t t1 = 0, t2 = 0, b1 = 0, e1 = 0;
    if (tid == 0) {
        t1 = (uint32_t)atomicAdd(&p.sc[SW_TICKET2], 1ull);
        t2 = t1 < n_sub ? (uint32_t)atomicAdd(&p.sc[SW_TICKET2], 1ull) : n_sub;
        if (t1 < n_sub) { b1 = p.base2[t1]; e1 = p.base2[t1 + 1]; }
    }

    while (true) {
        if (tid == 0) {
            s_j = t1; s_b = b1; s_e = e1;
            t1 = t2;
            if (t1 < n_sub) {
                b1 = p.base2[t1]; e1 = p.base2[t1 + 1];
                t2 = (uint32_t)atomicAdd(&p.sc[SW_TICKET2], 1ull);
            }
        }
        __syncthreads();
        const uint32_t j = s_j;
        if (j >= n_sub) break;
        const uint32_t b = s_b, n = s_e - b;
        if (n == 0) {
            if (tid == 0) { p.big[j] = 0; if (DUP) p.m_out[j] = 0; }
            __syncthreads();
            continue;
        }
        if (n > (uint32_t)CAP) {                     // does not fit: left to the radix sorter (super_big_*)
            if (tid == 0) {
                p.big[j] = n;
                atomicAdd(&p.sc[SW_BIG], 1ull);
                atomicAdd(&p.sc[SW_BIG_RECORDS], (unsigned long long)n);
                if (DUP) p.m_out[j] = 0;
            }
            __syncthreads();
            continue;
        }
        if (tid == 0) p.big[j] = 0;
        // the loads are issued first; their latency overlaps the clearing of the bins
        Key<W> rk[kPer];
        uint32_t rc[kPer], rr[kPer];
#pragma unroll
        for (int u = 0; u < kPer; u++) {
            const uint32_t i = u * THREADS + tid;
            if (u * THREADS >= n) break;
            if (i < n) { rk[u] = ld_key<W>(p.in_keys, b + i); rc[u] = p.in_counts[b + i]; }
        }
        uint32_t nb3 = 2 * pow2_ceil_u32(n);
        nb3 = nb3 < 64 ? 64 : (nb3 > (uint32_t)CAP ? (uint32_t)CAP : nb3);
        int shift3 = 64 - prefix_bits - (31 - __clz(nb3));
        if (shift3 < 0) shift3 = 0;
        for (uint32_t i = tid; i < nb3; i += THREADS) c3[pad32(i)] = 0;
        if (tid == 0) { s_maxbin = 0; s_cnt = 0; }
        __syncthreads();
#pragma unroll
        for (int u = 0; u < kPer; u++) {
            const uint32_t i = u * THREADS + tid;
            if (u * THREADS >= n) break;
            if (i < n) rr[u] = atomicAdd(&c3[pad32((uint32_t)(rk[u].w[0] >> shift3) & (nb3 - 1))], 1u);
        }
        __syncthreads();
        // exclusive scan of the nb3 bins: thread t owns bins [t * per3, (t + 1) * per3)
        {
            const uint32_t per3 = nb3 >= (uint32_t)THREADS ? nb3 / THREADS : 1u;
            const uint32_t b0 = tid * per3;
            uint32_t sum = 0, mx = 0;
            if (b0 < nb3)
                for (uint32_t q = 0; q < per3; q++) { const uint32_t v = c3[pad32(b0 + q)]; sum += v; mx = max(mx, v); }
            if (mx > 2) atomicMax(&s_maxbin, mx);
            uint32_t incl = sum;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= (uint32_t)o) incl += t;
            }
            if (lane == 31) s_warp[warp] = incl;
            __syncthreads();
            uint32_t off = 0;
#pragma unroll
            for (int w = 0; w < THREADS / 32; w++) if ((uint32_t)w < warp) off += s_warp[w];
            uint32_t run = off + incl - sum;
            if (b0 < nb3)
                for (uint32_t q = 0; q < per3; q++) { s3[pad32(b0 + q)] = run; run += c3[pad32(b0 + q)]; }
            __syncthreads();
        }
        const uint32_t maxbin = s_maxbin;
#pragma unroll
        for (int u = 0; u < kPer; u++) {
            const uint32_t i = u * THREADS + tid;
            if (u * THREADS >= n) break;
            if (i < n) {
                const uint32_t o = s3[pad32((uint32_t)(rk[u].w[0] >> shift3) & (nb3 - 1))] + rr[u];
                sk[o] = rk[u];
                scn[o] = rc[u];
            }
        }
        __syncthreads();
        const Key<W> *srt_k = fk;           // DUP: where the sorted sequence ends up in shared memory
        uint32_t *srt_c = fc;
        if (maxbin <= 32) {
            // position inside the bin = records of the bin that sort before this one
            for (uint32_t i = tid; i < n; i += THREADS) {
                const Key<W> k = sk[i];
                const uint32_t d = (uint32_t)(k.w[0] >> shift3) & (nb3 - 1);
                const uint32_t s0 = s3[pad32(d)], cn = c3[pad32(d)];
                uint32_t less = 0;
                for (uint32_t q = 0; q < cn; q++) {
                    const Key<W> o = sk[s0 + q];
                    less += (key_lt<W>(o, k) || (DUP && s0 + q < i && key_eq<W>(o, k))) ? 1u : 0u;
                }
                if (!DUP) {
                    st_key<W>(p.out_keys, b + s0 + less, k);
                    p.out_counts[b + s0 + less] = scn[i];
                } else {
                    fk[s0 + less] = k;
                    fc[s0 + less] = scn[i];
                }
            }
        } else {
            // crowded bins: bitonic network over the grouped arrays; pads are all-ones keys that
            // sort behind a real all-ones key
            srt_k = sk;
            srt_c = scn;
            const uint32_t p2 = pow2_ceil_u32(n);
            Key<W> pad;
            key_set_ones<W>(pad);
            for (uint32_t i = n + tid; i < p2; i += THREADS) { sk[i] = pad; scn[i] = 0; }
            __syncthreads();
            for (uint32_t size = 2; size <= p2; size <<= 1) {
                for (uint32_t stride = size >> 1; stride > 0; stride >>= 1) {
                    for (uint32_t t = tid; t < (p2 >> 1); t += THREADS) {
                        const uint32_t lo = 2 * t - (t & (stride - 1));
                        const uint32_t hi = lo + stride;
                        const bool up = (lo & size) == 0;
                        const Key<W> a = sk[lo], bq = sk[hi];
                        const uint32_t ca = scn[lo], cb = scn[hi];
                        // order: key ascending, then count descending (real records before pads)
                        const bool b_lt_a = key_lt<W>(bq, a) || (key_eq<W>(bq, a) && cb > ca);
                        if (b_lt_a == up) {
                            sk[lo] = bq; sk[hi] = a;
                            scn[lo] = cb; scn[hi] = ca;
                        }
                    }
                    __syncthreads();
                }
            }
            if (!DUP) {
                for (uint32_t i = tid; i < n; i += THREADS) {
                    st_key<W>(p.out_keys, b + i, sk[i]);
                    p.out_counts[b + i] = scn[i];
                }
            }
        }
        if (DUP) {
            __syncthreads();
            // fold: every record that equals its predecessor adds its count to the head of its group
            for (uint32_t i = tid; i < n; i += THREADS) {
                if (i > 0 && key_eq<W>(srt_k[i], srt_k[i - 1])) {
                    uint32_t hd = i - 1;
                    while (hd > 0 && key_eq<W>(srt_k[hd], srt_k[hd - 1])) hd--;
                    atomicAdd(&srt_c[hd], srt_c[i]);
                }
            }
            __syncthreads();
            // compaction of the heads, in order: warp ballots + running offset
            for (uint32_t i0 = 0; i0 < n; i0 += THREADS) {
                const uint32_t i = i0 + tid;
                const bool head = i < n && (i == 0 || !key_eq<W>(srt_k[i], srt_k[i - 1]));
                const uint32_t bal = __ballot_sync(0xffffffffu, head);
                if (lane == 0) s_warp[warp] = __popc(bal);
                __syncthreads();
                uint32_t off = s_cnt;
                for (uint32_t w = 0; w < warp; w++) off += s_warp[w];
                if (head) {
                    const uint32_t o = b + off + __popc(bal & lanemask_lt());
                    st_key<W>(p.out_keys, o, srt_k[i]);
                    p.out_counts[o] = srt_c[i];
                }
                __syncthreads();
                if (tid == 0) {
                    uint32_t t = 0;
                    for (int w = 0; w < THREADS / 32; w++) t += s_warp[w];
                    s_cnt += t;
                }
                __syncthreads();
            }
            if (tid == 0) {
                p.m_out[j] = s_cnt;
                folded_local += n - s_cnt;
            }
        }
        __syncthreads();
    }
    if (DUP && tid == 0 && folded_local) atomicAdd(&p.sc[SW_FOLDED], folded_local);
}

// ---- sub-buckets too large for S3c (see kc_super.cuh): records of sub-bucket j are
// D[base2[j] .. base2[j] + big[j]); in the gathered / sorted array they sit at bigoff[j].
template <int W>
__global__ void __launch_bounds__(256) big_gather_kernel(const uint64_t *__restrict__ in_keys,
                                                         const uint32_t *__restrict__ in_counts,
                                                         const uint32_t *__restrict__ base2,
                                                         const uint32_t *__restrict__ big,
                                                         const uint32_t *__restrict__ bigoff,
                                                         const SuperPlanDev *__restrict__ plan,
                                                         uint64_t *__restrict__ tk, uint32_t *__restrict__ tc) {
    const uint32_t n_sub = plan->n_sub;
    for (uint32_t j = blockIdx.x; j < n_sub; j += gridDim.x) {
        const uint32_t n = big[j];
        if (n == 0) continue;
        const uint32_t b = base2[j], o = bigoff[j];
        for (uint32_t i = threadIdx.x; i < n; i += 256) {
            st_key<W>(tk, o + i, ld_key<W>(in_keys, b + i));
            tc[o + i] = in_counts[b + i];
        }
    }
}

// Sorted records of every large sub-bucket -> its place in S3c's output. DUP: equal keys are
// adjacent; the first of a group keeps the key, the counts are added up (uint32 wrap), the heads are
// compacted and m_out[j] says how many there are.
template <int W, bool DUP>
__global__ void __launch_bounds__(256) big_place_kernel(const uint64_t *__restrict__ sk, const uint32_t *__restrict__ sc_counts,
                                                        const uint32_t *__restrict__ base2,
                                                        const uint32_t *__restrict__ big,
                                                        const uint32_t *__restrict__ bigoff,
                                                        const SuperPlanDev *__restrict__ plan,
                                                        uint64_t *__restrict__ out_keys, uint32_t *__restrict__ out_counts,
                                                        uint32_t *__restrict__ m_out, unsigned long long *__restrict__ sc) {
    __shared__ uint32_t s_warp[8];
    __shared__ uint32_t s_run;
    const uint32_t n_sub = plan->n_sub;
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (uint32_t j = blockIdx.x; j < n_sub; j += gridDim.x) {
        const uint32_t n = big[j];
        if (n == 0) continue;
        const uint32_t b = base2[j], o = bigoff[j];
        if constexpr (!DUP) {
            for (uint32_t i = tid; i < n; i += 256) {
                st_key<W>(out_keys, b + i, ld_key<W>(sk, o + i));
                out_counts[b + i] = sc_counts[o + i];
            }
        } else {
        // two sweeps over the segment: heads take their place (key + own count), then the others add
        // their counts to the head of their group; a record's group index = heads up to and including it - 1
        for (int sweep = 0; sweep < 2; sweep++) {
            if (tid == 0) s_run = 0;
            __syncthreads();
            for (uint32_t i0 = 0; i0 < n; i0 += 256) {
                const uint32_t i = i0 + tid;
                bool head = false;
                Key<W> k;
                if (i < n) {
                    k = ld_key<W>(sk, o + i);
                    head = i == 0 || !key_eq<W>(k, ld_key<W>(sk, o + i - 1));
                }
                const uint32_t bal = __ballot_sync(0xffffffffu, head);
                if (lane == 0) s_warp[warp] = __popc(bal);
                __syncthreads();
                uint32_t before = s_run;
                for (uint32_t w = 0; w < warp; w++) before += s_warp[w];
                const uint32_t incl = before + __popc(bal & (lanemask_lt() | (1u << lane)));   // heads in [0, i]
                if (i < n) {
                    if (sweep == 0 && head) {
                        st_key<W>(out_keys, b + incl - 1, k);
                        out_counts[b + incl - 1] = sc_counts[o + i];
                    } else if (sweep == 1 && !head) {
                        atomicAdd(&out_counts[b + incl - 1], sc_counts[o + i]);
                    }
                }
                __syncthreads();
                if (tid == 0) {
                    uint32_t t = 0;
                    for (int w = 0; w < 8; w++) t += s_warp[w];
                    s_run += t;
                }
                __syncthreads();
            }
            __threadfence();
            __syncthreads();
        }
        if (tid == 0) {
            m_out[j] = s_run;
            if (n > s_run) atomicAdd(&sc[SW_FOLDED], (unsigned long long)(n - s_run));
        }
        __syncthreads();
        }
    }
}

inline uint64_t round512(uint64_t b) { return (b + 511) & ~511ull; }

constexpr int kFinCapSmall = 2048, kFinCapLarge = 4096;     // records a sub-bucket may hold (S3c variants)
constexpr int kFinCapWide = 1024;                           // ... of 192/256-bit keys (folding variant, 2-3 CTAs per SM)

}  // namespace

// ------------------------------------------------------------------------ host
static void plan_layout(SuperPlan &pl, bool ext_e);

namespace {
constexpr uint32_t kS1TileBytes = 4800;         // bytes of reads per S1 tile (3200: 3.82 ms, 4800: 3.60, 6400: 4.0, 9600: 4.28 at C2)
constexpr uint32_t kS1MaxSmem = 200 * 1024;     // S1's dynamic shared memory at most

// S1's dynamic shared memory: the extraction's tile (ep: extract_plan with kS1TileBytes), then per
// read of the tile the m-mer hashes, the windows' bins and two words per segment
struct S1Smem { uint32_t h_off, bin_off, bits_off, total; };
S1Smem s1_smem(const SuperPlan &pl, const ExtractParams &ep) {
    S1Smem r;
    r.h_off = (ep.smem_total + 15u) & ~15u;
    r.bin_off = r.h_off + ep.tile_reads * pl.nh_stride * 4;
    r.bits_off = r.bin_off + ep.tile_reads * pl.nk * 4;
    r.total = r.bits_off + 2 * ep.tile_reads * pl.segs_per_read * 4;
    return r;
}

// minimizer length m and what follows from it: window of w m-mers, rows of m-mer hashes, segments
void set_minimizer(SuperPlan &pl, uint32_t m) {
    pl.m = m;
    pl.w = pl.span - pl.m + 1;
    pl.nh = pl.nk + pl.w - 1;
    pl.nh_stride = (pl.nh + 8) | 1u;                                   // odd stride: rows start in different banks
    pl.seg_len = pl.w - 1 < (uint32_t)kSwMaxSeg - 1 ? pl.w - 1 : (uint32_t)kSwMaxSeg - 1;   // + the look-behind window
    pl.segs_per_read = (pl.nk + pl.seg_len - 1) / pl.seg_len;
    pl.seg_len = (pl.nk + pl.segs_per_read - 1) / pl.segs_per_read;    // even the segments out
}

// records per sub-bucket the device plan aims for: 70 % of S3c's capacity. KC_SW_SUB_TARGET (tests)
// forces deep level-2 plans on small inputs.
uint32_t plan_sub_target(uint32_t fin_cap) {
    if (const char *v = getenv("KC_SW_SUB_TARGET")) {
        const int t = atoi(v);
        if (t > 0) return (uint32_t)t;
    }
    return fin_cap * 7 / 10;
}
}  // namespace

bool super_plan(uint32_t k, uint32_t L, uint32_t flags, uint64_t max_windows, uint32_t occ_per_bin, SuperPlan *out,
                double record_headroom, uint64_t distinct_hint, bool ext_e) {
    if (k == 0 || k > 64 || L < k || L > 4096) return false;
    if (flags & kPlanCanonical) flags |= kPlanStrict;                  // a canonical key is exactly k bases
    const bool strict = (flags & kPlanStrict) != 0;
    SuperPlan pl{};
    pl.flags = flags & (kPlanStrict | kPlanCanonical);
    pl.W = (int)((k + 31) / 32);
    pl.k = k;
    pl.L = L;
    pl.last_mask = key_last_mask(k, strict);
    pl.span = pl.last_mask != ~0ull ? k : 32u * pl.W;
    if (pl.span < 22) return false;
    pl.nk = L - k + 1;
    pl.cmax = 32u * pl.W - 3;
    if (max_windows == 0) max_windows = 1;
    if (occ_per_bin == 0) {
        // a bin's distinct keys should fit S2's table in one pass (3072 of its 4096 slots, bins vary by
        // ~20%): 8192 occurrences at the 5x redundancy of config 2, fewer when the caller expects
        // fewer repeats
        occ_per_bin = 8192;
        if (distinct_hint && distinct_hint < max_windows) {
            const double per_key = (double)max_windows / (double)distinct_hint;
            const double occ = 2200.0 * per_key;
            if (occ < 8192.0) occ_per_bin = occ < 1024.0 ? 1024u : ((uint32_t)occ + 255u) & ~255u;
        }
    }
    uint64_t nb = (max_windows + occ_per_bin - 1) / occ_per_bin;
    if (nb < 8) nb = 8;
    if (nb > (1ull << 24)) nb = 1ull << 24;
    pl.n_bins = (uint32_t)nb;
    // Minimizer length: a bin's load is the sum of the weights of the m-mers hashed into it, and those
    // weights are very uneven (an m-mer with a small hash is the minimizer of many windows). With
    // ~190 m-mers per bin the load's sd is ~20% of the mean; with 16 it is 70% and half the bins
    // overflow (seen at 1e6 bins with m = 12). So m grows with the bin count: 12 up to 87k bins
    // (config 2), 13 up to 350k, 14 up to 1.4M, ... -- longer minimizers change more often
    // (2 / (w + 1) records per window), which costs a few percent more records.
    // A longer minimizer also means shorter segments, so more of S1's shared memory per read: near
    // the longest reads the path takes, m stops growing where S1 would no longer fit (uneven bins
    // then only send more records to the overflow list). Reads too long for S1 even at m = 12 are
    // not for this path, whatever the plan's size.
    ExtractParams ep;
    if (!extract_plan(nullptr, 16, L, k, pl.flags, nullptr, &ep, kS1TileBytes)) return false;
    set_minimizer(pl, 12);
    if (s1_smem(pl, ep).total > kS1MaxSmem) return false;
    while (pl.m < 16 && pl.m + 8 < pl.span && (1ull << (2 * pl.m)) < 192ull * pl.n_bins) {
        SuperPlan longer = pl;
        set_minimizer(longer, pl.m + 1);
        if (s1_smem(longer, ep).total > kS1MaxSmem) break;
        pl = longer;
    }
    // records per window: a new record whenever the minimizer changes (2 / (w + 1) of the windows for a
    // random order), at every read start, and every cmax windows
    const double rho = 2.0 / (pl.w + 1) + 1.2 / pl.nk + 1.0 / pl.cmax * 0.25;
    const double est_total = (double)max_windows * rho;
    const double per_bin = est_total / (double)pl.n_bins;
    // minimizer weights make bins uneven: sd ~20% of the mean at 8192 occurrences per bin, growing as
    // bins shrink (fewer minimizers each). Five sigma of room, so that only skewed input overflows.
    pl.bin_cap = (uint32_t)(per_bin * (1.0 + 90.0 / sqrt((double)occ_per_bin))) + 64;
    pl.bin_cap = (pl.bin_cap + 3) & ~3u;
    // (also what bounds the pieces device-resident input is accumulated in: 1/32 of the plan's windows each)
    pl.ovf_cap = (uint64_t)(est_total * 0.6) + 8192;
    if (pl.ovf_cap < max_windows / 16) pl.ovf_cap = max_windows / 16;
    pl.ovf_slice = 4096;
    // records the dense / grouped arrays hold: every k-mer distinct unless the caller knows better
    const uint64_t d_base = distinct_hint && distinct_hint < max_windows ? distinct_hint + distinct_hint / 8 + 4096 : max_windows;
    pl.d_cap = d_base + (uint64_t)((double)d_base * record_headroom) + (record_headroom > 0 ? 8192 : 0);
    if (pl.d_cap > (1ull << 32) - 2) pl.d_cap = (1ull << 32) - 2;
    if (pl.d_cap < 1024) pl.d_cap = 1024;
    // S2 keeps a histogram of the leading b1 bits; the device plan picks the digits from it
    // sub-buckets of 2048 records unless the 2^20 sub-buckets two levels can cut would be too few
    pl.fin_cap = pl.d_cap > (uint64_t)kSuperMaxSub * (kFinCapSmall * 7 / 10) ? kFinCapLarge : kFinCapSmall;
    pl.sub_target = plan_sub_target(pl.fin_cap);
    const int sig = key_sig_bits(pl.W, pl.last_mask);
    pl.b1 = sig < 10 ? sig : 10;
    plan_layout(pl, ext_e);
    *out = pl;
    return true;
}

// workspace layout of a plan whose sizes are set
static void plan_layout(SuperPlan &pl, bool ext_e) {
    uint64_t o = 0;
    auto take = [&](uint64_t bytes) { uint64_t r = o; o += round512(bytes); return r; };
    const uint64_t rec_bytes = 16ull * pl.W;
    pl.off_cursor = take((uint64_t)pl.n_bins * 4);
    pl.off_hist1 = take((kNb1Max + 8) * 4);
    pl.off_hist2 = take((uint64_t)(2 * kSuperMaxSub + 8) * 4);          // exchange: sub-buckets of ALL ranks (up to 2^21)
    pl.off_base1 = take((kNb1Max + 8) * 4);
    pl.off_cur1 = take((kNb1Max + 8) * 4);
    pl.off_base2 = take((uint64_t)(kSuperMaxSub + 8) * 4);
    pl.off_cur2 = take((uint64_t)(kSuperMaxSub + 8) * 4);
    pl.off_mout = take((uint64_t)(kSuperMaxSub + 8) * 4);
    pl.off_off = take((uint64_t)(kSuperMaxSub + 8) * 4);
    pl.off_plan = take(sizeof(SuperPlanDev));
    pl.off_x = take(sizeof(XDev));
    pl.off_sc = take(SW_COUNT * 8);
    pl.off_h2m = take((uint64_t)(kSuperMaxSub + 8) * 4);
    pl.off_big = take((uint64_t)(kSuperMaxSub + 8) * 4);
    pl.off_bigoff = take((uint64_t)(kSuperMaxSub + 8) * 4);
    pl.off_bins = take((uint64_t)pl.n_bins * pl.bin_cap * rec_bytes);
    pl.off_ovf = take(pl.ovf_cap * rec_bytes);
    pl.off_dk = take(pl.d_cap * 8 * pl.W + 64);
    pl.off_dc = take(pl.d_cap * 4 + 64);
    pl.ext_e = ext_e;
    pl.ext_ek = nullptr;
    pl.ext_ec = nullptr;
    pl.off_ek = pl.off_ec = o;
    if (!ext_e) {
        pl.off_ek = take(pl.d_cap * 8 * pl.W + 64);
        pl.off_ec = take(pl.d_cap * 4 + 64);
    }
    pl.ws_bytes = o;
}

// Plan of the key-placement path (see kc_super.cuh): no bins, no S1/S2 -- D is filled with one
// (key, 1) record per k-mer slot by the caller, S3a..S3c place, sort and FOLD them. Any key width.
bool place_plan(uint32_t k, bool strict, uint64_t n_records, SuperPlan *out) {
    if (k == 0 || k > 128 || n_records == 0 || n_records > (1ull << 32) - 2) return false;
    SuperPlan pl{};
    pl.W = (int)((k + 31) / 32);
    pl.k = k;
    pl.last_mask = key_last_mask(k, strict);
    pl.span = pl.last_mask != ~0ull ? k : 32u * pl.W;
    pl.n_bins = 8;                                  // (unused: the arrays just exist)
    pl.d_cap = n_records < 1024 ? 1024 : n_records;
    // occurrences, not distinct keys, fill the sub-buckets; the folding S3c holds two copies of a
    // sub-bucket, so only its 2048-record variant fits shared memory for every key width
    // (192/256-bit keys: 1024-record sub-buckets keep two or three CTAs on an SM, as long as 2^20 of them are enough)
    pl.fin_cap = pl.W >= 3 && n_records <= (uint64_t)kSuperMaxSub * (kFinCapWide * 7 / 10) ? kFinCapWide : kFinCapSmall;
    pl.sub_target = plan_sub_target(pl.fin_cap);
    const int sig = key_sig_bits(pl.W, pl.last_mask);
    pl.b1 = sig < 10 ? sig : 10;
    plan_layout(pl, false);
    *out = pl;
    return true;
}

namespace {
template <class T> T *at(void *ws, uint64_t off) { return reinterpret_cast<T *>(static_cast<uint8_t *>(ws) + off); }
// the second record buffer: inside the workspace, or the caller's (SuperPlan::ext_e)
uint64_t *ek_of(const SuperPlan &pl, void *ws) { return pl.ext_e ? pl.ext_ek : at<uint64_t>(ws, pl.off_ek); }
uint32_t *ec_of(const SuperPlan &pl, void *ws) { return pl.ext_e ? pl.ext_ec : at<uint32_t>(ws, pl.off_ec); }
}  // namespace

cudaError_t super_reset(const SuperPlan &pl, void *ws, unsigned long long *d_sc, cudaStream_t s) {
    cudaError_t e;
    // cursor, hist1, hist2 are contiguous at the start of the workspace
    if ((e = cudaMemsetAsync(ws, 0, pl.off_base1, s)) != cudaSuccess) return e;
    return cudaMemsetAsync(d_sc, 0, SW_COUNT * 8, s);
}

template <int W>
static cudaError_t super_scatter_w(const SuperPlan &pl, const void *d_reads, uint64_t n_reads, void *ws,
                                   unsigned long long *d_sc, int n_sms, cudaStream_t s) {
    SwScatterParams q{};
    if (!extract_plan(d_reads, n_reads, pl.L, pl.k, pl.flags, &d_sc[SW_INVALID], &q.ep, kS1TileBytes))
        return cudaErrorInvalidValue;
    if (q.ep.n_tiles == 0) return cudaSuccess;
    q.m = pl.m; q.w = pl.w; q.nh = pl.nh; q.nh_stride = pl.nh_stride;
    q.seg_len = pl.seg_len; q.segs_per_read = pl.segs_per_read; q.cmax = pl.cmax; q.span = pl.span;
    const S1Smem lay = s1_smem(pl, q.ep);           // (super_plan only makes plans that fit)
    q.h_off = lay.h_off;
    q.bin_off = lay.bin_off;
    q.bits_off = lay.bits_off;
    const uint32_t smem = lay.total;
    if (smem > kS1MaxSmem) return cudaErrorInvalidValue;
    q.n_bins = pl.n_bins; q.bin_cap = pl.bin_cap; q.ovf_cap = pl.ovf_cap;
    q.cursor = at<uint32_t>(ws, pl.off_cursor);
    q.bins = at<uint8_t>(ws, pl.off_bins);
    q.ovf = at<uint8_t>(ws, pl.off_ovf);
    q.sc = d_sc;
    auto kern = (pl.flags & kPlanCanonical) ? sw_scatter_kernel<W, true> : sw_scatter_kernel<W, false>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    int per_sm = 1;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kSwThreads, smem);
    per_sm = per_sm < 1 ? 1 : (per_sm > 6 ? 6 : per_sm);
    uint32_t grid = (uint32_t)n_sms * per_sm;
    if (grid > q.ep.n_tiles) grid = q.ep.n_tiles;
    kern<<<grid, kSwThreads, smem, s>>>(q);
    return cudaGetLastError();
}

cudaError_t super_scatter(const SuperPlan &pl, const void *d_reads, uint64_t n_reads, void *ws,
                          unsigned long long *d_sc, int n_sms, cudaStream_t s) {
    if (pl.W == 1) return super_scatter_w<1>(pl, d_reads, n_reads, ws, d_sc, n_sms, s);
    if (pl.W == 2) return super_scatter_w<2>(pl, d_reads, n_reads, ws, d_sc, n_sms, s);
    return cudaErrorInvalidValue;
}

template <int W, bool CANON>
static cudaError_t launch_count(const SwCountParams &cp, int n_sms, cudaStream_t s) {
    constexpr uint32_t THREADS = SwCountCfg<W>::THREADS, TSLOTS = SwCountCfg<W>::TSLOTS, RPT = SwCountCfg<W>::RPT;
    const uint32_t RB = THREADS * RPT, RT = W == 1 ? RB : 1;
    const uint32_t smem = TSLOTS * (8 * W + 4) + RB * 16 * W + THREADS * 4 + kNb1Max * 4 +
                          (THREADS / 32) * (RPT > 1 ? 64 : 96) * (8 * W + 4) + RT * 20 + RB * 4 + 64;
    auto kern = sw_count_kernel<W, THREADS, TSLOTS, RPT, CANON>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    int per_sm = 1;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, THREADS, smem);
    if (per_sm < 1) per_sm = 1;
    kern<<<(uint32_t)n_sms * per_sm, THREADS, smem, s>>>(cp);
    return cudaGetLastError();
}

template <int W>
static cudaError_t super_count_bins_w(const SuperPlan &pl, bool add_phantom, void *ws, unsigned long long *d_sc, int n_sms,
                                      cudaStream_t s, void *const *peer_ws = nullptr, uint32_t rank = 0,
                                      uint32_t n_ranks = 1) {
    SwCountParams cp{};
    const uint32_t n_src = peer_ws ? n_ranks : 1u;
    cp.n_src = n_src;
    for (uint32_t i = 0; i < n_src; i++) {
        void *w = peer_ws ? peer_ws[i] : ws;
        cp.src_cursor[i] = at<uint32_t>(w, pl.off_cursor);
        cp.src_bins[i] = at<uint8_t>(w, pl.off_bins);
        cp.src_sc[i] = peer_ws ? at<unsigned long long>(w, pl.off_sc) : d_sc;
    }
    // rank r counts the bins [r * n_bins / P, (r + 1) * n_bins / P): bins are hash values, so the split is even
    cp.bin_begin = peer_ws ? (uint32_t)((uint64_t)pl.n_bins * rank / n_ranks) : 0u;
    cp.n_bins = peer_ws ? (uint32_t)((uint64_t)pl.n_bins * (rank + 1) / n_ranks) - cp.bin_begin : pl.n_bins;
    cp.ovf = at<uint8_t>(ws, pl.off_ovf);
    cp.bin_cap = pl.bin_cap; cp.ovf_slice = pl.ovf_slice; cp.ovf_cap = pl.ovf_cap;
    cp.last_mask = pl.last_mask;
    cp.d_keys = at<uint64_t>(ws, pl.off_dk); cp.d_counts = at<uint32_t>(ws, pl.off_dc); cp.d_cap = pl.d_cap;
    cp.hist1 = at<uint32_t>(ws, pl.off_hist1); cp.shift1 = 64 - pl.b1; cp.nb1 = 1 << pl.b1;
    cp.add_phantom = add_phantom ? 1 : 0;
    cp.sc = d_sc;
    return (pl.flags & kPlanCanonical) ? launch_count<W, true>(cp, n_sms, s) : launch_count<W, false>(cp, n_sms, s);
}

cudaError_t super_count_bins(const SuperPlan &pl, bool add_phantom, void *ws, unsigned long long *d_sc, int n_sms,
                             cudaStream_t s, void *const *peer_ws, uint32_t rank, uint32_t n_ranks) {
    if (peer_ws && (n_ranks == 0 || n_ranks > 8 || rank >= n_ranks)) return cudaErrorInvalidValue;
    if (pl.W == 1) return super_count_bins_w<1>(pl, add_phantom, ws, d_sc, n_sms, s, peer_ws, rank, n_ranks);
    if (pl.W == 2) return super_count_bins_w<2>(pl, add_phantom, ws, d_sc, n_sms, s, peer_ws, rank, n_ranks);
    return cudaErrorInvalidValue;
}

// S3a / S3b / the exchange's pull: in -> out by the plan's level-1 or level-2 digit (range: see rec_scatter_kernel)
template <int W, int LEVEL>
static cudaError_t launch_rec_scatter(const SuperPlan &pl, const uint64_t *in_keys, const uint32_t *in_counts,
                                      uint64_t *out_keys, uint32_t *out_counts, const SuperPlanDev *plan,
                                      unsigned long long *d_sc, uint32_t *cursor, const uint32_t *range, int n_sms,
                                      cudaStream_t s) {
    const uint32_t smem = RsCfg<W>::TILE * (8 * W + 4) + 3 * kRsBinsPadded * 4;
    auto kern = rec_scatter_kernel<W, LEVEL>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    int per_sm = 1;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kRsThreads, smem);
    if (per_sm < 1) per_sm = 1;
    kern<<<(uint32_t)n_sms * per_sm, kRsThreads, smem, s>>>(in_keys, in_counts, out_keys, out_counts, plan, pl.b1,
                                                           &d_sc[SW_D], pl.d_cap, cursor, range);
    return cudaGetLastError();
}

template <int W>
static cudaError_t super_place_w(const SuperPlan &pl, void *ws, unsigned long long *d_sc, int n_sms, cudaStream_t s,
                                 cudaEvent_t *evs) {
    cudaError_t e;
    uint64_t *dk = at<uint64_t>(ws, pl.off_dk), *ek = ek_of(pl, ws);
    uint32_t *dc = at<uint32_t>(ws, pl.off_dc), *ec = ec_of(pl, ws);
    if (!ek || !ec) return cudaErrorInvalidValue;
    uint32_t *hist1 = at<uint32_t>(ws, pl.off_hist1), *base1 = at<uint32_t>(ws, pl.off_base1),
             *cur1 = at<uint32_t>(ws, pl.off_cur1), *hist2 = at<uint32_t>(ws, pl.off_hist2),
             *base2 = at<uint32_t>(ws, pl.off_base2), *cur2 = at<uint32_t>(ws, pl.off_cur2);
    SuperPlanDev *plan = at<SuperPlanDev>(ws, pl.off_plan);
    // ---- S3a: level-1 bases + device plan, scatter D -> E
    sw_plan_kernel<<<1, 1024, 0, s>>>(hist1, pl.b1, pl.d_cap, pl.sub_target, key_sig_bits(pl.W, pl.last_mask), base1, cur1,
                                      plan, d_sc);
    if ((e = launch_rec_scatter<W, 1>(pl, dk, dc, ek, ec, plan, d_sc, cur1, nullptr, n_sms, s)) != cudaSuccess) return e;
    if (evs) cudaEventRecord(evs[0], s);
    // ---- level-2 histogram + scan (b2 == 0: one counter per level-1 bucket)
    rec_hist2_kernel<W><<<(uint32_t)n_sms * 8, 256, 0, s>>>(ek, plan, hist2);
    if ((e = exclusive_scan(hist2, &plan->n_sub, kSuperMaxSub, base2, cur2, nullptr, s)) != cudaSuccess) return e;
    if (evs) cudaEventRecord(evs[1], s);
    // ---- S3b: scatter E -> D by the level-2 digit
    if ((e = launch_rec_scatter<W, 2>(pl, ek, ec, dk, dc, plan, d_sc, cur2, nullptr, n_sms, s)) != cudaSuccess) return e;
    if (evs) cudaEventRecord(evs[2], s);
    return cudaSuccess;
}

cudaError_t super_place(const SuperPlan &pl, void *ws, unsigned long long *d_sc, int n_sms, cudaStream_t s, cudaEvent_t *evs) {
    if (pl.W == 1) return super_place_w<1>(pl, ws, d_sc, n_sms, s, evs);
    if (pl.W == 2) return super_place_w<2>(pl, ws, d_sc, n_sms, s, evs);
    if (pl.W == 3) return super_place_w<3>(pl, ws, d_sc, n_sms, s, evs);
    if (pl.W == 4) return super_place_w<4>(pl, ws, d_sc, n_sms, s, evs);
    return cudaErrorInvalidValue;
}

// ---- key-placement path
cudaError_t place_init(const SuperPlan &pl, void *ws, unsigned long long *d_sc, uint64_t n, int n_sms, cudaStream_t s) {
    cudaError_t e;
    if (n > pl.d_cap) return cudaErrorInvalidValue;
    // cursor, hist1, hist2 are contiguous at the start of the workspace
    if ((e = cudaMemsetAsync(ws, 0, pl.off_base1, s)) != cudaSuccess) return e;
    const uint64_t *dk = at<uint64_t>(ws, pl.off_dk);
    uint32_t *dc = at<uint32_t>(ws, pl.off_dc), *hist1 = at<uint32_t>(ws, pl.off_hist1);
    const uint32_t grid = (uint32_t)n_sms * 8;
    const int shift1 = 64 - pl.b1;
    switch (pl.W) {
        case 1: place_init_kernel<1><<<grid, 256, 0, s>>>(dk, dc, n, shift1, hist1, d_sc); break;
        case 2: place_init_kernel<2><<<grid, 256, 0, s>>>(dk, dc, n, shift1, hist1, d_sc); break;
        case 3: place_init_kernel<3><<<grid, 256, 0, s>>>(dk, dc, n, shift1, hist1, d_sc); break;
        case 4: place_init_kernel<4><<<grid, 256, 0, s>>>(dk, dc, n, shift1, hist1, d_sc); break;
        default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

uint64_t *place_keys(const SuperPlan &pl, void *ws) { return at<uint64_t>(ws, pl.off_dk); }

cudaError_t place_fix_zero(int W, const uint64_t *run_keys, uint32_t *run_counts, const unsigned long long *d_n_invalid,
                           cudaStream_t s) {
    switch (W) {
        case 1: place_fix_zero_kernel<1><<<1, 1, 0, s>>>(run_keys, run_counts, d_n_invalid); break;
        case 2: place_fix_zero_kernel<2><<<1, 1, 0, s>>>(run_keys, run_counts, d_n_invalid); break;
        case 3: place_fix_zero_kernel<3><<<1, 1, 0, s>>>(run_keys, run_counts, d_n_invalid); break;
        case 4: place_fix_zero_kernel<4><<<1, 1, 0, s>>>(run_keys, run_counts, d_n_invalid); break;
        default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

cudaError_t super_count(const SuperPlan &pl, bool add_phantom, void *ws, unsigned long long *d_sc, int n_sms,
                        cudaStream_t s, cudaEvent_t *evs) {
    cudaError_t e = super_count_bins(pl, add_phantom, ws, d_sc, n_sms, s);
    if (e != cudaSuccess) return e;
    if (evs) cudaEventRecord(evs[0], s);
    return super_place(pl, ws, d_sc, n_sms, s, evs ? evs + 1 : nullptr);
}

void super_tmp_buffers(const SuperPlan &pl, void *ws, uint64_t **tmp_keys, uint32_t **tmp_counts) {
    *tmp_keys = ek_of(pl, ws);
    *tmp_counts = ec_of(pl, ws);
}

template <int W, bool DUP, int THREADS, int CAP>
static cudaError_t super_finish_w(const SuperPlan &pl, void *ws, unsigned long long *d_sc, uint64_t *out_keys,
                                  uint32_t *out_counts, int n_sms, cudaStream_t s) {
    FinishParams fp{};
    fp.in_keys = at<uint64_t>(ws, pl.off_dk);
    fp.in_counts = at<uint32_t>(ws, pl.off_dc);
    fp.base2 = at<uint32_t>(ws, pl.off_base2);
    fp.plan = at<SuperPlanDev>(ws, pl.off_plan);
    fp.out_keys = out_keys;
    fp.out_counts = out_counts;
    fp.m_out = at<uint32_t>(ws, pl.off_mout);
    fp.big = at<uint32_t>(ws, pl.off_big);
    fp.sc = d_sc;
    const uint32_t smem = (DUP ? 2 : 1) * CAP * (8 * W + 4) + 2 * (CAP + CAP / 32) * 4;
    auto kern = rec_finish_kernel<W, THREADS, CAP, DUP>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    int per_sm = 1;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, THREADS, smem);
    if (per_sm < 1) per_sm = 1;
    kern<<<(uint32_t)n_sms * per_sm, THREADS, smem, s>>>(fp);
    return cudaGetLastError();
}

template <int W>
static cudaError_t super_finish_d(const SuperPlan &pl, bool dup, void *ws, unsigned long long *d_sc, uint64_t *out_keys,
                                  uint32_t *out_counts, int n_sms, cudaStream_t s) {
    if (pl.fin_cap == kFinCapLarge)
        return dup ? super_finish_w<W, true, 512, kFinCapLarge>(pl, ws, d_sc, out_keys, out_counts, n_sms, s)
                   : super_finish_w<W, false, 512, kFinCapLarge>(pl, ws, d_sc, out_keys, out_counts, n_sms, s);
    return dup ? super_finish_w<W, true, 256, kFinCapSmall>(pl, ws, d_sc, out_keys, out_counts, n_sms, s)
               : super_finish_w<W, false, 256, kFinCapSmall>(pl, ws, d_sc, out_keys, out_counts, n_sms, s);
}

cudaError_t super_finish(const SuperPlan &pl, bool dup, void *ws, unsigned long long *d_sc, uint64_t *out_keys,
                         uint32_t *out_counts, int n_sms, cudaStream_t s) {
    if (pl.W == 1) return super_finish_d<1>(pl, dup, ws, d_sc, out_keys, out_counts, n_sms, s);
    if (pl.W == 2) return super_finish_d<2>(pl, dup, ws, d_sc, out_keys, out_counts, n_sms, s);
    // 192/256-bit keys (key-placement path): the folding variant over 2048-record sub-buckets only
    if (!dup || (pl.fin_cap != kFinCapSmall && pl.fin_cap != kFinCapWide)) return cudaErrorInvalidValue;
    if (pl.fin_cap == kFinCapWide) {
        if (pl.W == 3) return super_finish_w<3, true, 256, kFinCapWide>(pl, ws, d_sc, out_keys, out_counts, n_sms, s);
        if (pl.W == 4) return super_finish_w<4, true, 256, kFinCapWide>(pl, ws, d_sc, out_keys, out_counts, n_sms, s);
    } else {
        if (pl.W == 3) return super_finish_w<3, true, 512, kFinCapSmall>(pl, ws, d_sc, out_keys, out_counts, n_sms, s);
        if (pl.W == 4) return super_finish_w<4, true, 512, kFinCapSmall>(pl, ws, d_sc, out_keys, out_counts, n_sms, s);
    }
    return cudaErrorInvalidValue;
}

cudaError_t super_big_gather(const SuperPlan &pl, void *ws, uint64_t *tk, uint32_t *tc, int n_sms, cudaStream_t s) {
    SuperPlanDev *plan = at<SuperPlanDev>(ws, pl.off_plan);
    uint32_t *big = at<uint32_t>(ws, pl.off_big), *bigoff = at<uint32_t>(ws, pl.off_bigoff), *base2 = at<uint32_t>(ws, pl.off_base2);
    cudaError_t e = exclusive_scan(big, &plan->n_sub, kSuperMaxSub, bigoff, nullptr, nullptr, s);
    if (e != cudaSuccess) return e;
    const uint64_t *dk = at<uint64_t>(ws, pl.off_dk);
    const uint32_t *dc = at<uint32_t>(ws, pl.off_dc);
    if (pl.W == 1) big_gather_kernel<1><<<(uint32_t)n_sms * 8, 256, 0, s>>>(dk, dc, base2, big, bigoff, plan, tk, tc);
    else if (pl.W == 2) big_gather_kernel<2><<<(uint32_t)n_sms * 8, 256, 0, s>>>(dk, dc, base2, big, bigoff, plan, tk, tc);
    else if (pl.W == 3) big_gather_kernel<3><<<(uint32_t)n_sms * 8, 256, 0, s>>>(dk, dc, base2, big, bigoff, plan, tk, tc);
    else big_gather_kernel<4><<<(uint32_t)n_sms * 8, 256, 0, s>>>(dk, dc, base2, big, bigoff, plan, tk, tc);
    return cudaGetLastError();
}

cudaError_t super_big_place(const SuperPlan &pl, bool dup, void *ws, unsigned long long *d_sc, const uint64_t *sk,
                            const uint32_t *sc_counts, uint64_t *out_keys, uint32_t *out_counts, int n_sms, cudaStream_t s) {
    const SuperPlanDev *plan = at<SuperPlanDev>(ws, pl.off_plan);
    const uint32_t *big = at<uint32_t>(ws, pl.off_big), *bigoff = at<uint32_t>(ws, pl.off_bigoff), *base2 = at<uint32_t>(ws, pl.off_base2);
    uint32_t *m_out = at<uint32_t>(ws, pl.off_mout);
    const uint32_t grid = (uint32_t)n_sms * 8;
    if (pl.W == 1) {
        if (dup) big_place_kernel<1, true><<<grid, 256, 0, s>>>(sk, sc_counts, base2, big, bigoff, plan, out_keys, out_counts, m_out, d_sc);
        else big_place_kernel<1, false><<<grid, 256, 0, s>>>(sk, sc_counts, base2, big, bigoff, plan, out_keys, out_counts, m_out, d_sc);
    } else if (pl.W == 2) {
        if (dup) big_place_kernel<2, true><<<grid, 256, 0, s>>>(sk, sc_counts, base2, big, bigoff, plan, out_keys, out_counts, m_out, d_sc);
        else big_place_kernel<2, false><<<grid, 256, 0, s>>>(sk, sc_counts, base2, big, bigoff, plan, out_keys, out_counts, m_out, d_sc);
    } else if (pl.W == 3 && dup) {
        big_place_kernel<3, true><<<grid, 256, 0, s>>>(sk, sc_counts, base2, big, bigoff, plan, out_keys, out_counts, m_out, d_sc);
    } else if (pl.W == 4 && dup) {
        big_place_kernel<4, true><<<grid, 256, 0, s>>>(sk, sc_counts, base2, big, bigoff, plan, out_keys, out_counts, m_out, d_sc);
    } else {
        return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

cudaError_t super_fold_offsets(const SuperPlan &pl, void *ws, unsigned long long *d_sc, cudaStream_t s) {
    SuperPlanDev *plan = at<SuperPlanDev>(ws, pl.off_plan);
    return exclusive_scan(at<uint32_t>(ws, pl.off_mout), &plan->n_sub, kSuperMaxSub, at<uint32_t>(ws, pl.off_off), nullptr,
                          &d_sc[SW_OUT], s);
}

cudaError_t super_gather(const SuperPlan &pl, void *ws, const uint64_t *tmp_keys, const uint32_t *tmp_counts,
                         uint64_t *out_keys, uint32_t *out_counts, int n_sms, cudaStream_t s) {
    const SuperPlanDev *plan = at<SuperPlanDev>(ws, pl.off_plan);
    const uint32_t *src = at<uint32_t>(ws, pl.off_base2), *off = at<uint32_t>(ws, pl.off_off);
    return gather_records(pl.W, tmp_keys, tmp_counts, src, off, &plan->n_sub, kSuperMaxSub, out_keys, out_counts, n_sms, s);
}

void super_use_large_finish(SuperPlan *pl) { pl->fin_cap = kFinCapLarge; }

// ---- multi-GPU exchange (see x_plan_kernel). Every rank's workspace has the same layout, so a
// peer's buffers are found from its workspace base.
template <int W>
static cudaError_t super_x_local_w(const SuperPlan &pl, void *ws, unsigned long long *d_sc, const uint32_t *d_all_hist,
                                   uint32_t rank, uint32_t n_ranks, bool keep_ranges, void *const *peer_ws, int n_sms,
                                   cudaStream_t s) {
    if (pl.ext_e) return cudaErrorInvalidValue;      // the peers find E through the workspace mapping
    uint64_t *dk = at<uint64_t>(ws, pl.off_dk), *ek = at<uint64_t>(ws, pl.off_ek);
    uint32_t *dc = at<uint32_t>(ws, pl.off_dc), *ec = at<uint32_t>(ws, pl.off_ec);
    SuperPlanDev *plan = at<SuperPlanDev>(ws, pl.off_plan);
    XScalars xs{};
    for (uint32_t i = 0; i < n_ranks; i++) xs.sc[i] = peer_ws ? at<unsigned long long>(peer_ws[i], pl.off_sc) : d_sc;
    x_plan_kernel<<<1, 1024, 0, s>>>(d_all_hist, rank, n_ranks, keep_ranges ? 1 : 0, pl.d_cap, pl.sub_target,
                                     pl.fin_cap == kFinCapLarge ? 1 : 0, key_sig_bits(pl.W, pl.last_mask),
                                     at<uint32_t>(ws, pl.off_base1), at<uint32_t>(ws, pl.off_cur1), plan,
                                     at<XDev>(ws, pl.off_x), d_sc, xs);
    cudaError_t e = launch_rec_scatter<W, 1>(pl, dk, dc, ek, ec, plan, d_sc, at<uint32_t>(ws, pl.off_cur1), nullptr, n_sms, s);
    if (e != cudaSuccess) return e;
    rec_hist2_kernel<W><<<(uint32_t)n_sms * 8, 256, 0, s>>>(ek, plan, at<uint32_t>(ws, pl.off_hist2));
    return cudaGetLastError();
}

cudaError_t super_x_local(const SuperPlan &pl, void *ws, unsigned long long *d_sc, const uint32_t *d_all_hist,
                          uint32_t rank, uint32_t n_ranks, bool keep_ranges, void *const *peer_ws, int n_sms, cudaStream_t s) {
    if (pl.b1 != kXB1 || n_ranks == 0 || n_ranks > 8 || rank >= n_ranks) return cudaErrorInvalidValue;
    if (pl.W == 1) return super_x_local_w<1>(pl, ws, d_sc, d_all_hist, rank, n_ranks, keep_ranges, peer_ws, n_sms, s);
    if (pl.W == 2) return super_x_local_w<2>(pl, ws, d_sc, d_all_hist, rank, n_ranks, keep_ranges, peer_ws, n_sms, s);
    return cudaErrorInvalidValue;
}

template <int W>
static cudaError_t super_x_pull_w(const SuperPlan &pl, void *ws, unsigned long long *d_sc, void *const *peer_ws,
                                  uint32_t rank, uint32_t n_ranks, int n_sms, cudaStream_t s) {
    SuperPlanDev *plan = at<SuperPlanDev>(ws, pl.off_plan);
    XDev *x = at<XDev>(ws, pl.off_x);
    XPeers peers{};
    for (uint32_t i = 0; i < n_ranks; i++) {
        peers.keys[i] = at<uint64_t>(peer_ws[i], pl.off_ek);
        peers.counts[i] = at<uint32_t>(peer_ws[i], pl.off_ec);
        peers.hist2[i] = at<uint32_t>(peer_ws[i], pl.off_hist2);
    }
    uint32_t *h2m = at<uint32_t>(ws, pl.off_h2m), *base2 = at<uint32_t>(ws, pl.off_base2), *cur2 = at<uint32_t>(ws, pl.off_cur2);
    x_merge_hist_kernel<<<(uint32_t)n_sms * 4, 256, 0, s>>>(peers, n_ranks, plan, h2m);
    cudaError_t e = exclusive_scan(h2m, &plan->n_sub, kSuperMaxSub, base2, cur2, nullptr, s);
    if (e != cudaSuccess) return e;
    // the level-2 scatter reads this rank's key range straight out of every source's grouped array:
    // the exchange happens inside the kernel's loads (NVLink / NVSwitch for the peers). Rank r starts
    // with source r + 1 and ends with its own records: at any time every source is read by one peer,
    // not by all of them (the ranks enter this step together), so no GPU's outgoing links are the
    // bottleneck of a round while the others idle.
    for (uint32_t j = 1; j <= n_ranks; j++) {
        const uint32_t i = (rank + j) % n_ranks;
        e = launch_rec_scatter<W, 2>(pl, peers.keys[i], peers.counts[i], at<uint64_t>(ws, pl.off_dk),
                                     at<uint32_t>(ws, pl.off_dc), plan, d_sc, cur2, &x->src_range[i][0], n_sms, s);
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

cudaError_t super_x_pull(const SuperPlan &pl, void *ws, unsigned long long *d_sc, void *const *peer_ws, uint32_t rank,
                         uint32_t n_ranks, int n_sms, cudaStream_t s) {
    if (n_ranks == 0 || n_ranks > 8 || rank >= n_ranks) return cudaErrorInvalidValue;
    if (pl.W == 1) return super_x_pull_w<1>(pl, ws, d_sc, peer_ws, rank, n_ranks, n_sms, s);
    if (pl.W == 2) return super_x_pull_w<2>(pl, ws, d_sc, peer_ws, rank, n_ranks, n_sms, s);
    return cudaErrorInvalidValue;
}

uint32_t *super_hist1(const SuperPlan &pl, void *ws) { return at<uint32_t>(ws, pl.off_hist1); }
const SuperXInfo *super_x_info(const SuperPlan &pl, void *ws) { return at<XDev>(ws, pl.off_x); }

}  // namespace kc

#ifdef KC_SW_PROFILE
// S2's phase timer (KC_SW_PROFILE builds only): copies the SWP_SLOTS sums out, then zeroes them when reset != 0
extern "C" int kc_sw_profile_read(unsigned long long *out, int reset) {
    cudaError_t e = cudaMemcpyFromSymbol(out, kc::g_sw_prof, sizeof(kc::g_sw_prof));
    if (e == cudaSuccess && reset) {
        static const unsigned long long zero[kc::SWP_SLOTS] = {};
        e = cudaMemcpyToSymbol(kc::g_sw_prof, zero, sizeof(zero));
    }
    return e == cudaSuccess ? 0 : -1;
}
#endif
