// kc_super.cuh -- plan and launchers of the super-window counting path (kc_super.cu).
//
// The path replaces extractKMers + the TBB accumulate + sortKmers + reduceKMers
// (GPUHandler.cu:129-360, KMerCounter.cpp:61-82) for one chunk -- or for many chunks
// accumulated into the same bins -- without ever writing a key per k-mer occurrence to
// HBM:
//
//   S1  reads -> 2-bit "super-window" records.  Consecutive k-mer windows of a read whose
//       minimizer (smallest hashed m-mer inside the window) falls into the same bin are
//       packed into ONE 16W-byte record (first window + following bases + window count);
//       a record is appended to its bin.  ~1.6 bytes per k-mer occurrence instead of 8W.
//   S2  one CTA per bin: the records are expanded in shared memory and every window is
//       inserted into a shared-memory open-addressing table (equal keys always share a bin,
//       because the bin is a function of the key).  The distinct (key, count) records of the
//       bin are appended to a dense array D.
//   S3  D (U records, not N occurrences) is put into key order: two most-significant-digit
//       scatter passes and a shared-memory sort per sub-bucket, written straight into the run.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "kc_extract.cuh"

namespace kc {

// device scalars of one super-window pipeline (unsigned long long each)
enum {
    SW_INVALID = 0,     // k-mer slots without a k-mer (SURVEY F7)
    SW_OVF = 1,         // records appended to the overflow list (may exceed its capacity)
    SW_D = 2,           // records appended to D (may exceed its capacity)
    SW_FAIL = 3,        // bit 0: overflow list full, bit 1: D full, bit 2: a bin could not be split,
                        // bit 3: a sub-bucket does not fit shared memory
    SW_TICKET = 4,      // S2 work ticket
    SW_WINDOWS = 5,     // windows packed into records by S1 (debug invariant: == slots - invalid)
    SW_OCC = 6,         // occurrences counted by S2 (debug invariant)
    SW_ABORTS = 7,      // bin passes S2 had to split
    SW_FOLDED = 8,      // duplicate records folded by S3c
    SW_OUT = 9,         // records in the run (DUP mode: after folding)
    SW_RECORDS = 10,    // records S1 wrote (bins + overflow)
    SW_TICKET2 = 11,    // S3c work ticket
    SW_BIG = 12,        // sub-buckets too large for S3c's shared memory (sorted by the radix sorter instead)
    SW_BIG_RECORDS = 13,// records in them
    SW_DEDUP = 14,      // records S2 counted through an equal record instead of expanding them (every pass)
    SW_MULTI = 15,      // S2 work units whose records took more than one round
    SW_COUNT = 16
};

struct SuperPlanDev {           // level-2 plan, decided on the device once |D| is known
    uint32_t n_d;               // records in D (clamped to capacity)
    uint32_t b2, shift2, n_sub; // level-2 digit bits, key shift of the (b1+b2)-bit prefix, sub-buckets
    uint32_t prefix_bits;
    uint32_t b1;                // level-1 digit bits actually used (<= SuperPlan::b1)
    uint32_t sub0;              // first (absolute) sub-bucket of this rank's key range; 0 on one GPU
    uint32_t pad[1];
};

struct SuperXInfo {             // multi-GPU exchange: what the device plan decided (kc_xchg_info)
    uint32_t lo[16];            // rank o owns the keys whose leading 10 bits lie in [lo[o], lo[o + 1])
    uint32_t src_range[8][2];   // records of this rank's key range inside rank s's grouped array
    uint32_t n_recv;            // records this rank pulls (its own included)
    uint32_t any_ovf;           // some rank's overflow list is in use: records may repeat across ranks
    uint32_t fin_large;         // the job's sub-buckets need S3c's large variant (more than 2^21 x sub_target records)
    uint32_t pad[1];
};

struct SuperPlan {
    int W;
    uint32_t k, L, span;        // span = bases that make up a key (32W or k, SURVEY F4)
    uint32_t m, w;              // minimizer length, m-mers per window (span - m + 1)
    uint32_t nk, nh, nh_stride; // windows per read, m-mer positions per read (nk + w - 1), smem row stride
    uint32_t seg_len, segs_per_read;
    uint32_t cmax;              // most windows one record holds (32W - 3)
    uint32_t n_bins, bin_cap;   // bins and records per bin
    uint64_t ovf_cap;           // records of the shared overflow list
    uint32_t ovf_slice;         // overflow records per S2 work unit
    uint64_t d_cap;             // records D / the level buffers hold
    int b1;                     // bits of the histogram S2 keeps (most level-1 digit bits; 1 << b1 <= 1024)
    uint32_t sub_target;        // records per sub-bucket the level-2 plan aims for
    int fin_cap;                // records a sub-bucket may hold (the S3c variant: 2048 or 4096)
    uint64_t last_mask;
    // workspace layout (bytes from the workspace base)
    uint64_t off_cursor, off_bins, off_ovf, off_hist1, off_base1, off_cur1, off_hist2, off_base2, off_cur2,
        off_mout, off_off, off_plan, off_x, off_sc, off_h2m, off_big, off_bigoff, off_dk, off_dc, off_ek, off_ec, ws_bytes;
    // The second record buffer (E: level-1 grouped records, later S3c's output) may live outside
    // the workspace (ext_e): the accumulating mode makes it the run itself, sized once |D| is
    // known, so a flush holds D and the run and nothing else of that size.
    bool ext_e;
    uint64_t *ext_ek;
    uint32_t *ext_ec;
    uint32_t flags;             // kPlanStrict | kPlanCanonical; canonical: keys are min(x, rc(x)), S1 bins
                                // windows by their canonical minimizer so that x and rc(x) share a bin
};

constexpr uint32_t kSuperMaxSub = 1u << 20;

// Plans a pipeline for up to max_windows k-mer slots (one chunk, or everything that will be
// accumulated before the count). flags: kPlanStrict / kPlanCanonical (as extract_plan).
// occ_per_bin = 0 -> default. Returns false for shapes the path does not take (W > 2, span < 22,
// reads too long for S1's shared memory). Every plan it makes fits S1: whether the path takes a
// shape does not depend on max_windows or occ_per_bin.
bool super_plan(uint32_t k, uint32_t L, uint32_t flags, uint64_t max_windows, uint32_t occ_per_bin, SuperPlan *out,
                double record_headroom = 0.0, uint64_t distinct_hint = 0, bool ext_e = false);

// zero cursors, histograms and scalars: once before the first super_scatter of a pipeline
cudaError_t super_reset(const SuperPlan &pl, void *ws, unsigned long long *d_sc, cudaStream_t s);
// S1: append the super-window records of (reads, n_reads) to the bins (key semantics of the plan)
cudaError_t super_scatter(const SuperPlan &pl, const void *d_reads, uint64_t n_reads, void *ws,
                          unsigned long long *d_sc, int n_sms, cudaStream_t s);
// S2 .. S3b: count the bins, place the distinct records into sub-buckets. evs (may be NULL):
// events recorded after S2, S3a, H2, S3b.
cudaError_t super_count(const SuperPlan &pl, bool add_phantom, void *ws, unsigned long long *d_sc, int n_sms,
                        cudaStream_t s, cudaEvent_t *evs);
// S3a .. S3b alone (after super_count_bins): evs (may be NULL) recorded after S3a, H2, S3b
cudaError_t super_place(const SuperPlan &pl, void *ws, unsigned long long *d_sc, int n_sms, cudaStream_t s, cudaEvent_t *evs);
// S3c once the host knows |D| (= *d_sc[SW_D]) : sort every sub-bucket into (out_keys, out_counts).
// dup == false: the records are distinct, the output is dense and final (n_d records).
// dup == true : equal keys are folded; the output has gaps, m_out/off describe it; finish with super_gather.
cudaError_t super_finish(const SuperPlan &pl, bool dup, void *ws, unsigned long long *d_sc, uint64_t *out_keys,
                         uint32_t *out_counts, int n_sms, cudaStream_t s);
// Sub-buckets S3c could not take (more than fin_cap records share a (b1+b2)-bit prefix: skewed
// input) are left out by super_finish and counted in d_sc[SW_BIG] / [SW_BIG_RECORDS]. The caller
// then (1) super_big_gather: their records, in sub-bucket order, into (tk, tc) -- room for
// SW_BIG_RECORDS records; (2) sorts that array by key (any sorter: the sub-buckets are key
// ranges, so the sorted array is the concatenation of the sorted sub-buckets); (3) super_big_place:
// the sorted records go to their sub-buckets' places in S3c's output (dup: folded, m_out set).
cudaError_t super_big_gather(const SuperPlan &pl, void *ws, uint64_t *tk, uint32_t *tc, int n_sms, cudaStream_t s);
cudaError_t super_big_place(const SuperPlan &pl, bool dup, void *ws, unsigned long long *d_sc, const uint64_t *sk,
                            const uint32_t *sc_counts, uint64_t *out_keys, uint32_t *out_counts, int n_sms, cudaStream_t s);
// DUP mode: after super_finish, offsets of the survivors (d_sc[SW_OUT] = records) ...
cudaError_t super_fold_offsets(const SuperPlan &pl, void *ws, unsigned long long *d_sc, cudaStream_t s);
// ... and the gather that closes the gaps
cudaError_t super_gather(const SuperPlan &pl, void *ws, const uint64_t *tmp_keys, const uint32_t *tmp_counts,
                         uint64_t *out_keys, uint32_t *out_counts, int n_sms, cudaStream_t s);
// S2 only: count the bins into the dense array D (+ histogram of the records' leading b1 bits).
// With peer_ws (multi-GPU: the ranks' workspaces as mapped here, scalars at off_sc) this rank counts
// its share of the bins and reads what every rank put into them -- the exchange of super-window
// records happens in the kernel's loads.
cudaError_t super_count_bins(const SuperPlan &pl, bool add_phantom, void *ws, unsigned long long *d_sc, int n_sms,
                             cudaStream_t s, void *const *peer_ws = nullptr, uint32_t rank = 0, uint32_t n_ranks = 1);
// ---- multi-GPU (one context per rank, every rank planned alike): after super_count_bins and an
// all-gather of the ranks' histograms (super_hist1: 1024 uint32 each) ...
uint32_t *super_hist1(const SuperPlan &pl, void *ws);
const SuperXInfo *super_x_info(const SuperPlan &pl, void *ws);      // device pointer
// ... the rank groups its own records by their leading 10 bits and counts the global sub-buckets,
// (keep_ranges: cut at the key ranges of the previous exchange instead of balancing anew)
cudaError_t super_x_local(const SuperPlan &pl, void *ws, unsigned long long *d_sc, const uint32_t *d_all_hist,
                          uint32_t rank, uint32_t n_ranks, bool keep_ranges, void *const *peer_ws, int n_sms, cudaStream_t s);
// ... and, once every rank has done that, pulls its key range out of every rank's grouped array
// (peer_ws[i] = rank i's workspace as mapped here) into sub-buckets. Then super_finish(dup = true).
cudaError_t super_x_pull(const SuperPlan &pl, void *ws, unsigned long long *d_sc, void *const *peer_ws, uint32_t rank,
                         uint32_t n_ranks, int n_sms, cudaStream_t s);
// exchange: the device plan found the job's sub-buckets too large for the small S3c variant
// (SuperXInfo::fin_large); super_finish of a plan changed by this sorts with the large one
void super_use_large_finish(SuperPlan *pl);
// ---- key-placement path (KC_COUNT_PLACE): for keys the bins do not take (k > 64: 192/256-bit keys).
// The extraction writes one key per k-mer slot straight into D (place_keys), place_init gives every
// record count 1 and builds the level-1 histogram, and S3a..S3c do the rest: two MSD placement
// passes and a shared-memory sort per sub-bucket that FOLDS equal keys (super_place, then
// super_finish(dup = true), super_fold_offsets, super_gather) -- three passes over the occurrences
// instead of one LSD radix pass per key byte (24..32 for these keys). Sub-buckets crowded by one
// repeated key go through the radix sorter like any oversized sub-bucket (super_big_*).
bool place_plan(uint32_t k, bool strict, uint64_t n_records, SuperPlan *out);
uint64_t *place_keys(const SuperPlan &pl, void *ws);
cudaError_t place_init(const SuperPlan &pl, void *ws, unsigned long long *d_sc, uint64_t n, int n_sms, cudaStream_t s);
// empty slots were placed as key 0: the run's key-0 record (always first) loses *d_n_invalid occurrences
cudaError_t place_fix_zero(int W, const uint64_t *run_keys, uint32_t *run_counts, const unsigned long long *d_n_invalid,
                           cudaStream_t s);
// where S3c's temporary output may live in DUP mode (the level-1 buffer is dead by then)
void super_tmp_buffers(const SuperPlan &pl, void *ws, uint64_t **tmp_keys, uint32_t **tmp_counts);

}  // namespace kc
