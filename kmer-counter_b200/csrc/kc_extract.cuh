// kc_extract.cuh -- fused 2-bit encode + k-mer window extraction (sm_100a).
//
// Replaces bitEncode (GPUHandler.cu:10-111) and extractKMers (:129-233): the
// encoded reads never travel through HBM.  A persistent CTA streams tiles of
// whole reads into shared memory with TMA bulk copies (double-buffered behind
// mbarriers), encodes each read once into 2-bit words, and then every thread
// assembles one key per output slot with a 64-bit funnel shift and hands it to a
// Sink (store to the slot array, hash-table insert, ...).
//
// Key semantics (SURVEY.md Appendix A.2, verified against the reference's own
// kernels by tests/): the key for position p is the 2-bit codes of the bases
// s[p .. p+span), MSB first, where span = 32*W when k%32 is 0/29/30/31 (the
// reference's missing tail mask, F4) and k otherwise; positions past the read end
// contribute 0; non-ACGT letters contribute 3 and invalidate every k-mer [p,p+k)
// that contains them.  The span is carried by Params::last_mask.
//
// Canonical keys (KC_CANONICAL, always with the strict span k): the key handed to the sink is
// min(x, rc(x)) in record order, rc = the complemented bases of x in reverse order, left-aligned.
// It is a template parameter of the kernel, so the forward instantiations are untouched.
#pragma once

#include "kc_common.cuh"

namespace kc {

struct ExtractParams {
    const uint8_t *reads;    // packed lines, stride L, 16-byte aligned
    uint64_t n_reads;
    uint32_t L, k;
    uint32_t nk;             // L - k + 1 slots per read
    uint32_t nw;             // ceil(L/32) encoded words per read (+1 zero pad word in smem)
    uint32_t nb4;            // ceil(L/4) bytes of bad-nibbles per read
    uint32_t tile_reads;     // reads per tile, multiple of 16 -> tile bytes % 16 == 0
    uint32_t n_tiles;
    uint32_t nk_magic;       // floor(2^32 / nk) + 1
    uint32_t nb4_magic;      // floor(2^32 / nb4) + 1
    uint32_t segs_per_read, seg_len;   // rolling walk: a read's nk positions in segs_per_read runs of seg_len
    uint64_t last_mask;      // applied to key word W-1
    uint32_t plan_flags;     // kPlanStrict | kPlanCanonical the plan was made for (kept so that a plan can be re-made)
    unsigned long long *n_invalid;  // += slots that hold no k-mer (the phantom of SURVEY F7)
    uint32_t stage_bytes, enc_off, bad_off, flag_off, bar_off, smem_total;  // shared-memory layout
};

inline void extract_smem_layout(ExtractParams &p) {
    p.stage_bytes = (p.tile_reads * p.L + 127u) & ~127u;
    p.enc_off = 2 * p.stage_bytes;
    p.bad_off = p.enc_off + p.tile_reads * (p.nw + 1) * 8;
    p.flag_off = p.bad_off + ((p.tile_reads * p.nb4 + 15u) & ~15u);
    p.bar_off = (p.flag_off + p.tile_reads + 15u) & ~15u;
    p.smem_total = p.bar_off + 16;
}

// extract_plan's flags: the KC_COMPAT_STRICT and KC_CANONICAL bits of kc_config.flags
constexpr uint32_t kPlanStrict = 0x1u, kPlanCanonical = 0x2u;

constexpr int kExtractThreads = 256;
constexpr uint32_t kMaxSegLen = 18;      // positions a thread walks in the sliding-window mode (plan: seg_len <= 18)

// Sink protocol (all members __device__; every thread of the CTA calls every hook):
//   static constexpr int kSweeps      phase-B sweeps over a tile's slots (1, or 2 for rank-then-place)
//   void begin(uint8_t *extra_smem)   once per CTA; the kernel syncs afterwards
//   void sweep_begin(int sw, uint32_t n_slots) / void sweep_end(int sw)
//                                     around each sweep; may __syncthreads(); the kernel syncs
//                                     between the slot loop and sweep_end
//   void operator()(int sw, uint64_t slot, const Key<W>&, bool valid)
//   void finish()                     once per CTA after the last tile
// extra_smem starts at ExtractParams::smem_total (16-byte aligned); launch with that many more bytes.
struct SinkBase {
    static constexpr int kSweeps = 1;
    static constexpr bool kRolling = false;   // true: slot order is irrelevant, use the sliding-window walk
    static constexpr bool kTopOnlySweep0 = false;   // true: sweep 0 only needs the top 32 bits of key word 0 (top())
    __device__ __forceinline__ void begin(uint8_t *) {}
    __device__ __forceinline__ void top(uint32_t, bool) {}
    __device__ __forceinline__ void sweep_begin(int, uint32_t) {}
    __device__ __forceinline__ void sweep_end(int) {}
    __device__ __forceinline__ void finish() {}
};

// code: A0 C1 G2 T3, anything else 3 + bad (GPUHandler.cu:42-88)
__device__ __forceinline__ uint32_t base_code(uint32_t c, uint32_t &bad) {
    uint32_t code = ((c >> 1) ^ (c >> 2)) & 3u;
    bool ok = (c == 'A') | (c == 'C') | (c == 'G') | (c == 'T');
    bad = ok ? 0u : 1u;
    return ok ? code : 3u;
}

// Phase A of every extraction kernel: the CTA turns the ASCII reads of one tile (shared
// memory, stride L) into 2-bit codes. Every thread takes groups of 4 bases (one 32-bit shared
// load) and produces one byte of codes with SIMD-in-register arithmetic; the (read, group)
// pairs of the tile are spread over the whole CTA. enc_b = rows of (nw + 1) 64-bit words per
// read whose pad bytes were zeroed once; bad4 = one nibble of "not ACGT" bits per group;
// flag[r] != 0 if read r has any such base. Follows bitEncode (GPUHandler.cu:42-101).
__device__ __forceinline__ void encode_tile(const ExtractParams &p, const uint8_t *src_tile, uint32_t nreads,
                                            uint8_t *enc_b, uint8_t *bad4, uint8_t *flag) {
    const uint32_t enc_row = p.nw + 1;
    const uint32_t *src32 = reinterpret_cast<const uint32_t *>(src_tile);
    const uint32_t n_groups = nreads * p.nb4;
    for (uint32_t g = threadIdx.x; g < n_groups; g += blockDim.x) {
        uint32_t r = p.nb4 == 1 ? g : __umulhi(g, p.nb4_magic);
        if (r * p.nb4 > g) r--;
        const uint32_t q = g - r * p.nb4;                                   // byte q of the read's bit string
        const uint32_t j0 = q * 4;
        const uint32_t addr = r * p.L + j0;
        const uint32_t w0 = src32[addr >> 2], w1 = src32[(addr >> 2) + 1];
        uint32_t x = __funnelshift_r(w0, w1, (addr & 3u) * 8u);             // bytes addr .. addr+3
        const uint32_t left = p.L - j0;                                      // bases of this read in x
        if (left < 4) x = (x & (0xffffffffu >> (32 - 8 * left))) | (0x41414141u << (8 * left));   // pad with 'A'
        // code = ((c >> 1) ^ (c >> 2)) & 3 for A,C,G,T = 0,1,2,3 (GPUHandler.cu:42-78)
        uint32_t t = ((x >> 1) ^ (x >> 2)) & 0x03030303u;
        // letter each byte should be, picked by (c >> 1) & 3 out of "ACTG": equal <=> valid
        const uint32_t i4 = (x >> 1) & 0x03030303u;
        const uint32_t sel = __byte_perm(i4 | (i4 >> 4), 0u, 0x4420u);      // nibble i = index of byte i
        const uint32_t diff = x ^ __byte_perm(0x47544341u, 0u, sel);
        uint32_t badn = 0;
        if (diff) {                                                          // rare: some byte is not ACGT
#pragma unroll
            for (uint32_t b = 0; b < 4; b++)
                if ((diff >> (8 * b)) & 0xffu) { badn |= 1u << b; t |= 3u << (8 * b); }   // code 3 + filter bit (:79-87)
            flag[r] = 1;
        }
        // byte q of the big-endian bit string -> little-endian byte inside its word
        enc_b[(r * enc_row + (q >> 3)) * 8 + (7 - (q & 7))] = (uint8_t)((t * 0x40100401u) >> 24);   // b0<<6|b1<<4|b2<<2|b3
        bad4[r * p.nb4 + q] = (uint8_t)badn;
    }
}

// Reverse complement of a 64-bit word of 32 bases: base order reversed, code ^ 3 (A0 C1 G2 T3).
__device__ __forceinline__ uint64_t word_revcomp(uint64_t x) {
    x = __brevll(x);                                                         // bits reversed ...
    x = ((x >> 1) & 0x5555555555555555ull) | ((x & 0x5555555555555555ull) << 1);   // ... bases back in bit order
    return ~x;
}
// The canonical key of a strict key x (k bases left-aligned, low bits zero): min(x, rc(x)) in record
// order. rc_sh = 2 (32 W - k) = the zero tail of word W-1, always < 64.
template <int W>
__device__ __forceinline__ Key<W> key_canonical(const Key<W> &x, uint32_t rc_sh) {
    uint64_t r[W + 1];
#pragma unroll
    for (int q = 0; q < W; q++) r[q] = word_revcomp(x.w[W - 1 - q]);
    r[W] = 0;
    Key<W> rc;
#pragma unroll
    for (int q = 0; q < W; q++) rc.w[q] = rc_sh ? ((r[q] << rc_sh) | (r[q + 1] >> (64 - rc_sh))) : r[q];
    return key_lt<W>(rc, x) ? rc : x;
}
// rc_sh of a plan: the bits last_mask clears
__device__ __forceinline__ uint32_t rc_shift_of(uint64_t last_mask) { return (uint32_t)__ffsll((long long)last_mask) - 1u; }

// rare path: any bad base inside [pos, pos+k) kills the k-mer (bad4 row of the read)
__device__ __forceinline__ bool kmer_window_valid(const uint8_t *bn, uint32_t pos, uint32_t k) {
    const uint32_t lo = pos, hi = pos + k;  // [lo, hi)
    for (uint32_t q = lo >> 2; q <= (hi - 1) >> 2; q++) {
        uint32_t m = bn[q];
        const uint32_t b0 = q * 4;
        if (b0 < lo) m &= 0xFu << (lo - b0);
        if (b0 + 4 > hi) m &= 0xFu >> (b0 + 4 - hi);
        if (m & 0xFu) return false;
    }
    return true;
}

template <int W, class Sink, bool CANON = false>
__global__ void __launch_bounds__(kExtractThreads) extract_kernel(ExtractParams p, Sink sink) {
    extern __shared__ __align__(128) uint8_t smem[];
    const uint32_t stage_bytes = p.stage_bytes;
    uint8_t *stage0 = smem;
    uint64_t *enc = reinterpret_cast<uint64_t *>(smem + p.enc_off);
    uint8_t *enc_b = reinterpret_cast<uint8_t *>(enc);
    const uint32_t enc_row = p.nw + 1;
    uint8_t *bad4 = smem + p.bad_off;
    uint8_t *flag = smem + p.flag_off;
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem + p.bar_off);
    const uint32_t tid = threadIdx.x, lane = tid & 31;
    [[maybe_unused]] const uint32_t rc_sh = CANON ? rc_shift_of(p.last_mask) : 0u;

    if (tid == 0) {
        mbar_init(&bars[0], 1);
        mbar_init(&bars[1], 1);
        mbar_fence_init();
    }
    for (uint32_t i = tid; i < p.tile_reads * enc_row; i += kExtractThreads) enc[i] = 0;
    for (uint32_t i = tid; i < p.tile_reads; i += kExtractThreads) flag[i] = 0;
    sink.begin(smem + p.smem_total);
    __syncthreads();

    auto tile_reads_of = [&](uint32_t t) -> uint32_t {
        uint64_t first = (uint64_t)t * p.tile_reads;
        uint64_t left = p.n_reads - first;
        return left < p.tile_reads ? (uint32_t)left : p.tile_reads;
    };
    // Full tiles go through the TMA unit; a ragged last tile whose byte count is
    // not a multiple of 16 is copied with plain loads by the whole CTA.
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
            for (uint32_t i = tid; i < bytes; i += kExtractThreads) dst[i] = src[i];
        }
    };

    uint32_t phase_bits = 0;  // bit s = parity to wait for on stage s
    uint32_t stage = 0;
    unsigned long long invalid_local = 0;

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

        // ---- phase A: 2-bit encode of the tile's reads (encode_tile, above) ----
        encode_tile(p, src_tile, nreads, enc_b, bad4, flag);
        __syncthreads();

        // ---- phase B ----
        const uint32_t total = nreads * p.nk;
        const uint64_t slot0 = (uint64_t)tile * p.tile_reads * p.nk;
        // rare path: any bad base inside [pos, pos+k) kills the k-mer
        auto kmer_valid = [&](uint32_t r, uint32_t pos) -> bool {
            const uint8_t *bn = bad4 + r * p.nb4;
            const uint32_t lo = pos, hi = pos + p.k;  // [lo, hi)
            for (uint32_t q = lo >> 2; q <= (hi - 1) >> 2; q++) {
                uint32_t m = bn[q];
                const uint32_t b0 = q * 4;
                if (b0 < lo) m &= 0xFu << (lo - b0);
                if (b0 + 4 > hi) m &= 0xFu >> (b0 + 4 - hi);
                if (m & 0xFu) return false;
            }
            return true;
        };
#pragma unroll
        for (int sw = 0; sw < Sink::kSweeps; sw++) {
            sink.sweep_begin(sw, total);
            if constexpr (Sink::kRolling) {
                // Sinks that ignore the slot index: a thread walks a segment of consecutive
                // positions of one read and slides the 32W-base window by one base per key
                // (funnel shifts) instead of rebuilding it from the encoded words.
                const uint32_t n_seg = nreads * p.segs_per_read;
                for (uint32_t sg = tid; sg < n_seg; sg += kExtractThreads) {
                    const uint32_t r = sg / p.segs_per_read;
                    const uint32_t p0 = (sg - r * p.segs_per_read) * p.seg_len;
                    const uint32_t p1 = min(p0 + p.seg_len, p.nk);
                    const uint32_t wi = p0 >> 5;
                    const uint64_t *e = enc + r * enc_row + wi;
                    const uint32_t sh = (p0 & 31u) * 2u;
                    uint64_t ew[W + 2];
#pragma unroll
                    for (int q = 0; q < W + 2; q++) ew[q] = (wi + q <= p.nw) ? e[q] : 0ull;
                    uint64_t win[W + 1];                                           // win[W] = lookahead word
#pragma unroll
                    for (int q = 0; q <= W; q++) win[q] = sh ? ((ew[q] << sh) | (ew[q + 1] >> (64 - sh))) : ew[q];
                    const bool check = flag[r] != 0;
                    if (Sink::kTopOnlySweep0 && !CANON && sw == 0) {
                        // the sink only wants leading key bits here (a digit histogram): they all come
                        // from the 64-bit window at p0, one constant funnel shift per position (not so for
                        // canonical keys, whose leading bits depend on the whole k-mer)
                        const uint64_t x = win[0];
#pragma unroll
                        for (uint32_t i = 0; i < kMaxSegLen; i++) {
                            const uint32_t pos = p0 + i;
                            if (pos < p1) {
                                const bool valid = check ? kmer_valid(r, pos) : true;
                                if (!valid) invalid_local++;
                                sink.top((uint32_t)((x << (2 * i)) >> 32), valid);
                            }
                        }
                        continue;
                    }
                    for (uint32_t pos = p0; pos < p1; pos++) {
                        Key<W> key;
#pragma unroll
                        for (int q = 0; q < W; q++) key.w[q] = win[q];
                        key.w[W - 1] &= p.last_mask;
                        if constexpr (CANON) key = key_canonical<W>(key, rc_sh);
                        const bool valid = check ? kmer_valid(r, pos) : true;
                        if (sw == 0 && !valid) invalid_local++;
                        sink(sw, slot0 + r * p.nk + pos, key, valid);
#pragma unroll
                        for (int q = 0; q < W; q++) win[q] = (win[q] << 2) | (win[q + 1] >> 62);
                        win[W] <<= 2;
                    }
                }
            } else {
                // one key per thread per step, slots are contiguous in the output
                for (uint32_t s = tid; s < total; s += kExtractThreads) {
                    uint32_t r = p.nk == 1 ? s : __umulhi(s, p.nk_magic);
                    if (r * p.nk > s) r--;
                    const uint32_t pos = s - r * p.nk;
                    const uint64_t *e = enc + r * enc_row + (pos >> 5);
                    const uint32_t sh = (pos & 31u) * 2u;
                    Key<W> key;
                    uint64_t a = e[0];
#pragma unroll
                    for (int q = 0; q < W; q++) {
                        uint64_t b = e[q + 1];
                        key.w[q] = sh ? ((a << sh) | (b >> (64 - sh))) : a;
                        a = b;
                    }
                    key.w[W - 1] &= p.last_mask;
                    if constexpr (CANON) key = key_canonical<W>(key, rc_sh);
                    const bool valid = flag[r] ? kmer_valid(r, pos) : true;
                    if (sw == 0 && !valid) invalid_local++;
                    sink(sw, slot0 + s, key, valid);
                }
            }
            __syncthreads();
            sink.sweep_end(sw);
        }
        for (uint32_t i = tid; i < nreads; i += kExtractThreads) flag[i] = 0;       // for the next tile's phase A
        __syncthreads();
        stage ^= 1;
    }

    // one atomic per warp
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) invalid_local += __shfl_xor_sync(0xffffffffu, invalid_local, o);
    if (lane == 0 && invalid_local) atomicAdd(p.n_invalid, invalid_local);
    sink.finish();
}

// the instantiation a plan asks for (kPlanCanonical: canonical keys)
template <int W, class Sink>
inline auto extract_kernel_for(const ExtractParams &p) {
    return (p.plan_flags & kPlanCanonical) ? extract_kernel<W, Sink, true> : extract_kernel<W, Sink, false>;
}

}  // namespace kc
