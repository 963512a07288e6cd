// kc_internal.h -- launchers shared between the translation units of libkc_b200.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "kc_extract.cuh"
#include "kc_super.cuh"

namespace kc {

// ---- key semantics
// The mask applied to key word W - 1 (SURVEY F4): it keeps the codes of the first k % 32 bases of that
// word when k % 32 != 0 in strict mode, or 1 <= k % 32 <= 28 otherwise; else it is all ones (the key
// spans 32 W bases).
inline uint64_t key_last_mask(uint32_t k, bool strict) {
    const uint32_t m = k % 32;
    const bool masked = strict ? m != 0 : (m >= 1 && m <= 28);
    return masked ? ~0ull << (64 - 2 * m) : ~0ull;
}
// bits of key word 0 that are not zero for every key: the bits a partition or digit plan can split on
inline int key_sig_bits(int W, uint64_t last_mask) { return W == 1 ? 64 - __builtin_ctzll(last_mask) : 64; }

// ---- extraction (kc_extract.cu)
// Fills every field of ExtractParams for (reads, n_reads, L, k); flags: kPlanStrict selects
// KC_COMPAT_STRICT masking, kPlanCanonical canonical keys (implies strict). Returns false for
// unsupported shapes.
bool extract_plan(const void *d_reads, uint64_t n_reads, uint32_t L, uint32_t k, uint32_t flags,
                  unsigned long long *d_n_invalid, ExtractParams *out, uint32_t stage_bytes_target = 12800);
// keys[slot] for every slot r*(L-k+1)+p; slots without a k-mer get key 0
cudaError_t launch_extract_store(const ExtractParams &p, int W, uint64_t *d_keys, int n_sms, cudaStream_t s);

// ---- radix sort (kc_sort.cu)
struct SortWorkspace {          // all device memory, sized by sort_workspace_bytes()
    void *base;
    uint64_t bytes;
};
uint64_t sort_workspace_bytes(uint64_t n, int W);
// LSD radix sort of n keys (W words each, key-major) over the bit range
// [lo_bit, 64*W) counted from the least significant bit of the last word.
// keys_a holds the input; the sorted result lands in *sorted (keys_a or keys_b).
// vals_a/vals_b may be NULL (keys only).  n < 2^30.
cudaError_t radix_sort(uint64_t *keys_a, uint64_t *keys_b, uint32_t *vals_a, uint32_t *vals_b, uint64_t n, int W,
                       int lo_bit, SortWorkspace ws, cudaStream_t s, uint64_t **sorted_keys, uint32_t **sorted_vals,
                       int *n_launches, cudaEvent_t ev_pass_begin, cudaEvent_t ev_pass_end);

// ---- run-length + packing (kc_reduce.cu)
uint64_t rle_workspace_bytes(uint64_t n);
// sorted keys -> unique keys (out_keys, capacity n) + start index of each run
// (out_starts, capacity n+1; out_starts[U] = n is appended); *d_num_unique = U.
cudaError_t rle_unique(const uint64_t *sorted_keys, uint64_t n, int W, uint64_t *out_keys, uint32_t *out_starts,
                       unsigned long long *d_num_unique, void *ws, cudaStream_t s, int *n_launches);
// counts[i] = starts[i+1]-starts[i]; the key-0 record (if first) loses *d_n_invalid occurrences
cudaError_t starts_to_counts(const uint32_t *starts, const uint64_t *keys, int W, uint64_t n_unique,
                             const unsigned long long *d_n_invalid, uint32_t *counts, cudaStream_t s);
// (keys, counts) <-> packed S-byte records
cudaError_t pack_records(const uint64_t *keys, const uint32_t *counts, uint64_t n, int W, void *records,
                         cudaStream_t s);
cudaError_t unpack_records(const void *records, uint64_t n, int W, uint64_t *keys, uint32_t *counts,
                           cudaStream_t s);
// (keys, counts) -> KMerPrinter's text (KMerPrinter.cpp:35-91): 32 W letters, ' ', count, '\n' per record.
// d_text holds print_max_bytes(n, W); *d_bytes = bytes written; ws: print_workspace_bytes(n).
uint64_t print_workspace_bytes(uint64_t n);
uint64_t print_max_bytes(uint64_t n, int W);
cudaError_t print_records_text(const uint64_t *keys, const uint32_t *counts, uint64_t n, int W, char *d_text,
                               unsigned long long *d_bytes, void *ws, cudaStream_t s);
// fold adjacent equal keys of a sorted (keys, counts) sequence, summing counts
cudaError_t fold_sorted_pairs(const uint64_t *keys, const uint32_t *counts, uint64_t n, int W, uint64_t *out_keys,
                              uint32_t *out_counts, unsigned long long *d_num_unique, void *ws, cudaStream_t s,
                              int *n_launches);
// lower_bound of n_q query keys in a sorted unique key array
cudaError_t lower_bounds(const uint64_t *keys, uint64_t n, int W, const uint64_t *d_queries, uint32_t n_q,
                         unsigned long long *d_out, cudaStream_t s);

// ---- count spectrum and count-range filter of a run (kc_spectrum.cu)
// d_hist[min(c, n_bins - 1)] += 1 for every count c (d_hist: n_bins uint64, cleared here); n_bins >= 2
cudaError_t run_histogram(const uint32_t *counts, uint64_t n, uint32_t n_bins, unsigned long long *d_hist, int n_sms,
                          cudaStream_t s, int *n_launches);
// survivors (lo <= count <= hi) per tile, scanned into tile offsets in ws; *d_total = survivors
uint64_t filter_workspace_bytes(uint64_t n);
cudaError_t filter_count(const uint32_t *counts, uint64_t n, uint32_t lo, uint32_t hi, void *ws,
                         unsigned long long *d_total, cudaStream_t s, int *n_launches);
// then the survivors in order into out_keys / out_counts (capacity *d_total), same ws
cudaError_t filter_write(const uint64_t *keys, const uint32_t *counts, uint64_t n, int W, uint32_t lo, uint32_t hi,
                         const void *ws, uint64_t *out_keys, uint32_t *out_counts, cudaStream_t s, int *n_launches);

// ---- merge path (kc_merge.cu)
uint64_t merge_workspace_bytes(uint64_t na, uint64_t nb);
// two sorted unique runs -> one, equal keys summed (uint32 wrap); *d_num_out = records
cudaError_t merge_pair(const uint64_t *ka, const uint32_t *ca, uint64_t na, const uint64_t *kb, const uint32_t *cb,
                       uint64_t nb, int W, uint64_t *out_keys, uint32_t *out_counts,
                       unsigned long long *d_num_out, void *ws, cudaStream_t s, int *n_launches);
// set operations of two sorted unique runs (the KC_SET_* / KC_COUNTS_* values of kc_api.h): op decides
// which keys survive, counts how a key in both runs is counted; union with kCountsSum is merge_pair.
// Same workspace as merge_pair; out_* hold the most records op can give (union na + nb, intersect
// min(na, nb), the subtracts na); *d_num_out = records. A bad op or counts: cudaErrorInvalidValue
enum : uint32_t { kSetUnion = 0, kSetIntersect = 1, kSetSubtract = 2, kSetSubtractCounts = 3 };
enum : uint32_t { kCountsSum = 0, kCountsMin = 1, kCountsMax = 2, kCountsA = 3, kCountsB = 4 };
cudaError_t combine_pair(const uint64_t *ka, const uint32_t *ca, uint64_t na, const uint64_t *kb, const uint32_t *cb,
                         uint64_t nb, int W, uint32_t op, uint32_t counts, uint64_t *out_keys, uint32_t *out_counts,
                         unsigned long long *d_num_out, void *ws, cudaStream_t s, int *n_launches);

// ---- key lookup in a run (kc_query.cu)
// bits of word 0 that select a bucket of the run index of n records: 2^bits + 1 uint64 offsets
int query_index_bits(uint64_t n, int sig_bits);
// offsets[j] = first record of the sorted keys whose top `bits` bits of word 0 are >= j, j = 0 .. 2^bits
cudaError_t query_index(const uint64_t *keys, int W, uint64_t n, int bits, uint64_t *offsets, int n_sms, cudaStream_t s,
                        int *n_launches);
// keys[slot] and valid[slot] (1: the window holds a k-mer) for every slot r*(L-k+1)+p of the plan
cudaError_t query_extract(const ExtractParams &p, int W, uint64_t *d_keys, uint8_t *d_valid, int n_sms, cudaStream_t s);
struct QueryLookup {
    const uint64_t *run_keys;     // the run: n_run sorted unique keys, their counts, its index
    const uint32_t *run_counts;
    const uint64_t *offsets;
    uint32_t shift;               // 64 - index bits
    const uint64_t *keys;         // n query keys (key-major)
    const uint8_t *valid;         // NULL: every key is a query; else keys with valid[i] == 0 get count 0
    uint64_t n;
    uint64_t tail_bits;           // bits of word W-1 a k-mer leaves zero (strict keys); a key with one set gets 0
    bool fold;                    // look up min(x, rc(x)) (canonical context), rc_sh = rc_shift_of(last_mask)
    uint32_t rc_sh;
    uint32_t *counts;             // NULL or counts[i] = the key's count, 0 if absent
    uint32_t *hits;               // NULL or hits[i / nk] += valid keys with lo <= count <= hi (n < 2^32)
    uint32_t nk, lo, hi;
};
cudaError_t query_lookup(const QueryLookup &p, int W, cudaStream_t s);

// ---- hash table (kc_hash.cu), W == 1 only
struct HashTable {
    uint64_t *slots;            // capacity x {key, count|pad} as 2 x uint64
    uint64_t capacity;          // power of two
    unsigned long long *side;   // [0] count of the all-ones key, [1] overflow flag, [3] distinct keys claimed
};
uint64_t hash_table_bytes(uint64_t capacity);
cudaError_t hash_clear(HashTable t, cudaStream_t s);
cudaError_t launch_extract_hash(const ExtractParams &p, HashTable t, int n_sms, cudaStream_t s);
// if *d_n_invalid != 0 make sure key 0 is in the table (with whatever count it has)
cudaError_t hash_touch_zero(HashTable t, const unsigned long long *d_n_invalid, cudaStream_t s);
// occupied slots (+ the all-ones key if seen) -> (keys, counts), unordered; *d_num = records
cudaError_t hash_compact(HashTable t, uint64_t *out_keys, uint32_t *out_counts, unsigned long long *d_num,
                         cudaStream_t s, int *n_launches);

// ---- raw FASTQ text -> packed reads (kc_fastq.cu)
uint64_t fastq_workspace_bytes(uint64_t n_bytes);
cudaError_t fastq_parse(const void *d_text, uint64_t n_bytes, uint32_t L, void *d_reads, uint64_t max_reads,
                        unsigned long long *d_out, void *ws, cudaStream_t s, int *n_launches);

// ---- sub-bucket offsets and gather (kc_partition.cu), for the partitioned hash and the super-window path.
// n entries: *n_ptr (device) or, when n_ptr is NULL, n; with n_ptr set, n is the most *n_ptr can be.
// base[0 .. n] = exclusive scan of counts (base[n] = the total); cursor[0 .. n) and *total get copies when set.
cudaError_t exclusive_scan(const uint32_t *counts, const uint32_t *n_ptr, uint32_t n, uint32_t *base, uint32_t *cursor,
                           unsigned long long *total, cudaStream_t s);
// records of sub-bucket j: tmp[src[j] .. src[j] + off[j + 1] - off[j]) -> out[off[j] ...), for the n sub-buckets
// given as for exclusive_scan. W = 1 .. 4
cudaError_t gather_records(int W, const uint64_t *tmp_keys, const uint32_t *tmp_counts, const uint32_t *src,
                           const uint32_t *off, const uint32_t *n_ptr, uint32_t n, uint64_t *out_keys,
                           uint32_t *out_counts, int n_sms, cudaStream_t s);

// ---- partitioned shared-memory hash counting (kc_partition.cu), W = 1 or 2
uint64_t partition_workspace_bytes(uint64_t n_slots);
// true when out_keys must be keys_a (two partition levels) rather than keys_b
bool partition_two_levels(uint64_t n_slots, int sig_bits, int target_sub);
cudaError_t partition_gather(int W, uint64_t n_slots, int sig_bits, int target_sub, const uint64_t *tmp_keys,
                             const uint32_t *tmp_counts, void *ws, uint64_t *out_keys, uint32_t *out_counts,
                             cudaStream_t s);
void partition_plan_info(uint64_t n_slots, int sig_bits, int target_sub, void *ws, uint32_t *n_sub,
                         uint32_t *prefix_bits, const uint32_t **d_offsets);
uint64_t merge_parts_workspace_bytes(uint32_t n_sub);
cudaError_t merge_parts_count(uint32_t n_src, const uint64_t *const *src_keys, const uint32_t *const *src_counts,
                              const uint32_t *const *src_off, uint32_t n_sub, int prefix_bits, uint64_t *tmp_keys,
                              uint32_t *tmp_counts, unsigned long long *d_num_out, unsigned long long *d_overflow,
                              void *ws, int n_sms, cudaStream_t s, int *n_launches);
cudaError_t merge_parts_gather(uint32_t n_sub, const uint64_t *tmp_keys, const uint32_t *tmp_counts, void *ws,
                               uint64_t *out_keys, uint32_t *out_counts, uint32_t *out_offsets, cudaStream_t s);
// PA's tile: extract_plan with kPaTileBytes of reads (16 reads from L = 201 on)
constexpr uint32_t kPaTileBytes = 6400;
// false when PA cannot take a tile of ep: the extraction's buffers and the tile's keys, staged by level-1
// digit, exceed a CTA's shared memory (long reads: from about 1200 bases for 64-bit keys, 700 for 128-bit)
bool partition_fits(const ExtractParams &ep, int W);
cudaError_t partition_count(int W, const ExtractParams &ep, uint64_t n_slots, int sig_bits, bool add_phantom,
                            uint64_t *keys_a, uint64_t *keys_b, uint64_t *out_keys, uint32_t *out_counts,
                            unsigned long long *d_num_out, unsigned long long *d_overflow,
                            unsigned long long *d_scratch_invalid, void *ws, int n_sms, int target_sub,
                            cudaStream_t s, int *n_launches, cudaEvent_t *evs);

}  // namespace kc
