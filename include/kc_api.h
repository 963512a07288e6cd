/*
 * kc_api.h -- C ABI of the B200-native k-mer counting path (libkc_b200.so).
 *
 * This is the drop-in boundary for the counting path of jsdjayanga/kmer-counter.
 * Plain pointers and sizes only; every call returns an int status (0 = KC_OK,
 * negative = error, message from kc_last_error) and never exits or throws.
 * Citations are file:line into the reference tree.
 *
 * Data contracts
 *   reads    "packed lines": n_bytes of reads back to back at stride read_len,
 *            no separators -- exactly FASTQData::getData() as handed to
 *            processKMers (FASTQFileReader.cpp:63-64, GPUHandler.h:63).  A partial
 *            trailing read is ignored (GPUHandler.cu:13,134).
 *   records  packed, no padding: W = ceil(k/32) little-endian uint64 words (word 0
 *            = most significant bases) + uint32 count; 12/20/28/36 bytes
 *            (KMerSizes.h:10-28 under GPUHandler.h:15's pack(1)).  This is the
 *            run-file / output-file / KMerPrinter format (SortedKMerFile.cpp:22-27).
 *   run      a sorted, key-unique sequence of records, resident on the device.
 *
 * Threading: one kc_ctx may be driven from several host threads as long as each
 * thread uses its own slot (the reference calls processKMers from up to 8
 * threads, one GPUStream each, KMerCounter.cpp:136-138).  Calls that take no slot
 * are serialised internally.
 */
#ifndef KC_API_H
#define KC_API_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KC_OK               0
#define KC_ERR_ARG         -1   /* bad argument / unsupported (k, read_len)            */
#define KC_ERR_CUDA        -2   /* a CUDA call failed                                  */
#define KC_ERR_NOMEM       -3   /* device or pinned allocation failed                  */
#define KC_ERR_CAPACITY    -4   /* destination buffer / slot too small                 */
#define KC_ERR_IO          -5   /* file open / write failed                            */
#define KC_ERR_STATE       -6   /* call out of order (e.g. wait on an idle slot)       */

/* kc_config.flags */
#define KC_COMPAT_REF       0x0u  /* bit-exact with the reference, quirks included (default):
                                     unmasked tail window at k%32 in {29,30,31} and the
                                     zero-count key-0 record (SURVEY.md F4, F7)           */
#define KC_COMPAT_STRICT    0x1u  /* true k-mers: tail always masked to k bases, no phantom */
#define KC_CANONICAL        0x2u  /* canonical k-mers (implies KC_COMPAT_STRICT): a k-mer x and its reverse
                                     complement rc(x) -- the complemented bases (code ^ 3 under A0 C1 G2 T3)
                                     in reverse order, stored like any key -- are counted under one key,
                                     min(x, rc(x)) in record order (words as unsigned 64-bit, word 0 first).
                                     Its count = occurrences of x or rc(x); a palindrome counts once per
                                     occurrence; windows with a non-ACGT byte are dropped. Every method, k
                                     1..128, the accumulating mode and the exchange. The records have the same
                                     format, but a run does not say which keys it holds: never merge canonical
                                     and forward runs, and create every rank of an exchange with the same flags */

/* kc_config.method: how occurrences are counted inside one chunk */
#define KC_COUNT_AUTO       0u
#define KC_COUNT_SORT       1u    /* radix sort + run-length (replaces sortKmers+reduceKMers,
                                     GPUHandler.cu:300-360)                                */
#define KC_COUNT_HASH       2u    /* open-addressing hash tables in shared memory over key-range
                                     partitions (replaces the TBB accumulate, KMerCounter.cpp:61-82);
                                     k <= 64                                                 */
#define KC_COUNT_HASH_GLOBAL 3u   /* one open-addressing table in HBM, then a sort of the distinct
                                     set; kept as the measured baseline for KC_COUNT_HASH      */

#define KC_COUNT_SUPER      4u    /* super-window records (consecutive k-mers of a read that share a
                                     minimizer bin, 2 bits per base) binned by minimizer, counted per bin in
                                     shared-memory tables, distinct records then placed in key order;
                                     k <= 64 with windows of >= 22 bases. What KC_COUNT_AUTO picks there. */

#define KC_COUNT_PLACE      5u    /* one key per k-mer slot, placed by two most-significant-digit passes
                                     into sub-buckets that are sorted and folded in shared memory:
                                     three passes over the occurrences whatever the key width. What
                                     KC_COUNT_AUTO picks for k > 64 (192/256-bit keys, KMerSizes.h:20-28),
                                     where KC_COUNT_SORT needs 24..32 radix passes.            */

typedef struct kc_ctx kc_ctx;
typedef struct kc_run kc_run;

typedef struct kc_config {
    uint32_t struct_size;      /* sizeof(kc_config), for ABI growth                        */
    uint32_t k;                /* kmerLength= (main.cpp:33), 1..128                        */
    uint32_t read_len;         /* lineLength (FASTQFileReader.cpp:30-35), k..4096          */
    int32_t  device;           /* CUDA device ordinal                                      */
    uint32_t flags;            /* KC_COMPAT_* | KC_CANONICAL                               */
    uint32_t method;           /* KC_COUNT_*                                               */
    uint32_t n_slots;          /* pinned input slots (the reference's 8 GPUStreams,
                                  KMerCounter.cpp:117); 0 -> 2                             */
    uint32_t reserved0;
    uint64_t max_chunk_bytes;  /* capacity of each slot = largest chunk submitted;
                                  replaces PrepareGPU's inputSize (GPUHandler.cu:479)      */
    uint64_t table_slots;      /* sizing hint, 0 = default. KC_COUNT_HASH_GLOBAL: table capacity;
                                  KC_COUNT_HASH: k-mer occurrences per sub-bucket; KC_COUNT_SUPER:
                                  k-mer occurrences per minimizer bin                      */
    void    *stream;           /* cudaStream_t to run on, NULL = a stream owned by the ctx */
    uint64_t distinct_hint;    /* accumulating mode: distinct keys expected per flush (sizes the
                                  record buffers); 0 = as many as there are k-mers (always fits) */
} kc_config;

typedef struct kc_stats {
    uint64_t chunks;           /* chunks counted                                           */
    uint64_t reads;            /* reads consumed                                           */
    uint64_t kmer_slots;       /* reads * (L-k+1): the reference's output slots            */
    uint64_t kmers_valid;      /* occurrences actually counted                             */
    uint64_t distinct_last;    /* records in the most recent run                           */
    uint64_t launches;         /* kernels launched by this library so far                  */
    uint64_t h2d_bytes, d2h_bytes;
    /* device time of the most recent chunk, by stage, CUDA events on the ctx stream */
    float ms_extract, ms_count, ms_emit, ms_total;
    /* dominant stage of the most recent chunk = the slowest entry of ms_stage */
    float ms_dominant;         /* summed over its launches                                 */
    uint32_t dominant_launches;
    uint32_t method_used;      /* KC_COUNT_* actually run (a full hash table falls back to sort) */
    uint64_t dominant_bytes;   /* algorithmic bytes moved by those launches                */
    /* per-stage device time and algorithmic bytes of the most recent chunk.
     *   KC_COUNT_SORT : 0 extract, 1 digit histogram, 2 radix scatter passes, 3 run-length, 4 emit
     *   KC_COUNT_HASH : 0 level-1 histogram, 1 extract+scatter1, 2 level-2 histogram, 3 scatter2,
     *                   4 shared-memory count+sort+write, 5 emit
     *   KC_COUNT_HASH_GLOBAL : 0 table clear, 1 extract+insert, 2 compact+sort, 3 emit
     *   KC_COUNT_PLACE : 0 extract, 1 counts + level-1 histogram, 2 record scatter 1, 3 level-2
     *                    histogram, 4 record scatter 2, 5 shared-memory sort + fold + write
     *   KC_COUNT_SUPER : 0 encode+minimizer+record scatter, 1 shared-memory count per bin,
     *                    2 record scatter level 1, 3 level-2 histogram, 4 record scatter level 2,
     *                    5 shared-memory sort + write                                             */
    uint32_t n_stages;
    uint32_t dominant_stage;
    float    ms_stage[8];
    uint64_t stage_bytes[8];
    uint32_t stage_launches[8];
} kc_stats;

/* ---- library ---- */
const char *kc_version(void);
uint32_t kc_key_words(uint32_t k);             /* ceil(k/32)                               */
uint32_t kc_record_size(uint32_t k);           /* 8*W+4 (GPUHandler.cu:235-245)            */
/* R*(L-k+1)*S: the reference's raw output size for a chunk (calculateOutputSize) */
uint64_t kc_output_size(uint64_t n_bytes, uint32_t read_len, uint32_t k);

/* ---- context: replaces PrepareGPU / FreeGPU (GPUHandler.h:61-62, GPUHandler.cu:479-519) ---- */
int  kc_create(const kc_config *cfg, kc_ctx **out);
void kc_destroy(kc_ctx *ctx);
const char *kc_last_error(const kc_ctx *ctx);   /* ctx may be NULL: last create error      */
int  kc_sync(kc_ctx *ctx);                      /* wait for everything queued on the ctx   */
int  kc_stats_get(kc_ctx *ctx, kc_stats *out);

/* the 16 device scalars of the most recent chunk (diagnostics for tests; layout = the SW_* / SC_*
 * enums of the implementation, not a stable interface) */
int  kc_debug_scalars(kc_ctx *ctx, uint64_t *out16);

/* pinned host memory for callers that want zero-copy staging (e2e path) */
int  kc_host_alloc(kc_ctx *ctx, uint64_t bytes, void **out);
int  kc_host_free(kc_ctx *ctx, void *p);

/* ---- counting one chunk: replaces processKMers (GPUHandler.h:63, GPUHandler.cu:397-477) ---- */

/* Synchronous, host in / host out: H2D, extract, count, D2H.  On return
 * records[0..*n_bytes) is the chunk's sorted key-unique run and `reads` may be
 * freed (KMerCounter.cpp:88).  records may be NULL to only learn *n_bytes. */
int  kc_process_chunk(kc_ctx *ctx, uint32_t slot, const char *reads, uint64_t n_bytes,
                      void *records, uint64_t records_cap, uint64_t *out_bytes);

/* Asynchronous, pinned double-buffered: fill the slot's pinned buffer, submit,
 * fill the next slot while this one is copied and counted, then wait. */
int  kc_slot_buffer(kc_ctx *ctx, uint32_t slot, void **ptr, uint64_t *cap);
int  kc_submit(kc_ctx *ctx, uint32_t slot, uint64_t n_bytes);
int  kc_wait(kc_ctx *ctx, uint32_t slot, kc_run **run);   /* caller owns *run (may be NULL
                                                             for an empty chunk)           */

/* Device-resident input (d_reads: device pointer, 16-byte aligned). */
int  kc_count_device(kc_ctx *ctx, const void *d_reads, uint64_t n_bytes, kc_run **run);

/* ---- accumulating mode: many chunks, one count ----
 * The reference turns every chunk into a run file and merges the files (KMerCounter.cpp:51-89 +
 * KMerFileMergeHandler). Here a chunk can instead be packed into 2-bit super-window records that
 * are appended to minimizer bins resident in HBM (about 1.7 bytes per k-mer occurrence); the count
 * happens once, over everything accumulated, in kc_accum_flush. The result is the same artefact as
 * counting the chunks separately and merging their runs. Needs k <= 64 with windows of >= 22 bases.
 *   kc_accum_begin(ctx, expected_reads)   plan + allocate for that many reads (at least one chunk);
 *                                         more reads than planned are handled by counting what has
 *                                         accumulated into a part first (parts are merged by the flush)
 *   kc_accum_add_device / kc_accum_submit / kc_accum_submit_fastq
 *                                         device-resident reads / the slot's pinned buffer / raw FASTQ
 *                                         text (as kc_submit_fastq); asynchronous
 *   kc_accum_wait(ctx, slot)              the slot's buffers may be refilled
 *   kc_accum_flush(ctx, &run)             count -> sorted unique run; the bins are empty again */
int  kc_accum_begin(kc_ctx *ctx, uint64_t expected_reads);
int  kc_accum_add_device(kc_ctx *ctx, const void *d_reads, uint64_t n_bytes);
int  kc_accum_submit(kc_ctx *ctx, uint32_t slot, uint64_t n_bytes);
int  kc_accum_submit_fastq(kc_ctx *ctx, uint32_t slot, const void *host_text, uint64_t n_bytes,
                           uint64_t *consumed, uint32_t *flags);
int  kc_accum_wait(kc_ctx *ctx, uint32_t slot);
int  kc_accum_flush(kc_ctx *ctx, kc_run **run);

/* ---- multi-GPU: hash-partitioned by key range, one context per GPU ("rank") ----
 * The reference has one implicit device (SURVEY.md 5.8). Here up to 8 contexts -- in one process
 * (kc_xchg_run_all, the command line's gpus=N) or one process per GPU (handles exchanged through
 * any host channel) -- each accumulate their share of the reads (kc_accum_add_device /
 * kc_accum_submit after kc_xchg_begin) as super-window records in its own minimizer bins. Two
 * exchanges follow, both fused into the kernel that consumes the data (its loads read the peers'
 * HBM over NVLink / NVSwitch; there is no send/receive step and no staging copy):
 *   1. bins are hash-partitioned: rank r counts bins [r*B/P, (r+1)*B/P) and reads what EVERY rank
 *      put into them (about 1.7 bytes per k-mer occurrence cross the links, not 8), so its distinct
 *      (key, count) records are distinct across the whole job;
 *   2. the key space is cut into P contiguous ranges of about equal record totals (from an
 *      all-gathered 1024-bin histogram), every rank groups its records by their leading bits, and
 *      rank r pulls range r out of all ranks' grouped arrays while placing it into sub-buckets.
 * Rank r ends with the sorted unique records of the r-th key range: the artefact is the
 * concatenation in rank order. Order of calls on every rank, B = a barrier across ranks that the
 * caller provides (stream-ordered is enough: an event wait or a tiny NCCL all-reduce on the
 * context's stream):
 *   [accumulate] -> B -> kc_xchg_count_local -> all-gather of kc_xchg_hist's 1024 uint32 into its
 *   n_ranks x 1024 buffer -> kc_xchg_group_local -> B -> kc_xchg_pull -> B -> kc_xchg_finish. */
int  kc_xchg_begin(kc_ctx *ctx, uint32_t rank, uint32_t n_ranks, uint64_t expected_reads);
int  kc_xchg_export(kc_ctx *ctx, void *handle64);                       /* CUDA IPC handle of this rank's workspace */
/* a peer in another process: every rank must be created with the same k, read_len and flags (the
 * handle carries no plan, so a peer counting other keys is not detected here) */
int  kc_xchg_import(kc_ctx *ctx, uint32_t peer, const void *handle64);
/* a peer in this process: refused (KC_ERR_ARG) if it was planned differently or counts other keys */
int  kc_xchg_set_peer(kc_ctx *ctx, uint32_t peer, kc_ctx *peer_ctx);
int  kc_xchg_count_local(kc_ctx *ctx);
int  kc_xchg_hist(kc_ctx *ctx, void **d_hist, void **d_all_hist);
int  kc_xchg_group_local(kc_ctx *ctx);
int  kc_xchg_pull(kc_ctx *ctx);
int  kc_xchg_finish(kc_ctx *ctx, kc_run **run);
/* on != 0: the following exchanges cut the key space where the previous one did (instead of
 * balancing anew), so that a rank's runs of several exchanges cover one key range and can be merged */
int  kc_xchg_fix_ranges(kc_ctx *ctx, int on);
/* the last exchange: lo[0..n_ranks] = bucket boundaries of the owners' key ranges (of 1024: the
 * leading 10 key bits), records this rank pulled in all, and how many of them came from peers */
int  kc_xchg_info(kc_ctx *ctx, uint32_t *lo, uint64_t *recv_records, uint64_t *remote_records);
/* all ranks in this process: everything above, ordered by events; runs[r] = rank r's key range */
int  kc_xchg_run_all(kc_ctx *const *ctxs, uint32_t n, kc_run **runs);

/* ---- raw FASTQ chunks: replaces FASTQFileReader::readData (FASTQFileReader.cpp:49-89) ----
 * The text must start at a record boundary and be well formed (4 lines per record, the
 * line after the sequence starts with '+', every sequence read_len long); the parse runs
 * on the device.  *consumed = bytes of whole records taken (carry the rest into the next
 * chunk; at end of file terminate the last line with '\n').  *flags != 0 (KC_FASTQ_*) means
 * the text is not of that shape: nothing was counted, use a host parser for this input. */
#define KC_FASTQ_MALFORMED  0x1u   /* a record's third line does not start with '+'   */
#define KC_FASTQ_RAGGED     0x2u   /* a sequence is not read_len long                 */
/* parse only: d_text (16-byte aligned, < 4 GiB) -> d_reads (packed lines) */
int  kc_parse_fastq_device(kc_ctx *ctx, const void *d_text, uint64_t n_bytes, void *d_reads,
                           uint64_t reads_cap_bytes, uint64_t *n_reads, uint64_t *consumed, uint32_t *flags);
/* host text -> H2D -> parse -> count on `slot` (as kc_submit; collect with kc_wait).  The
 * reads parsed must fit the slot (max_chunk_bytes); text beyond that is left unconsumed. */
int  kc_submit_fastq(kc_ctx *ctx, uint32_t slot, const void *host_text, uint64_t n_bytes,
                     uint64_t *consumed, uint32_t *flags);

/* ---- runs: the sorted-run dump (FileDump.cpp:51-58) and its consumers ---- */
uint64_t kc_run_records(const kc_run *run);
int  kc_run_free(kc_ctx *ctx, kc_run *run);
/* Packed records out (D2H), into pageable or pinned memory. Runs on the context's own copy
 * stream and staging buffer, so a consumer thread may read one run back while the producer thread
 * submits and waits for later chunks (calls are serialised among themselves; returns when the bytes
 * are in dst). */
int  kc_run_copy_records(kc_ctx *ctx, const kc_run *run, void *dst, uint64_t cap, uint64_t *out_bytes);
/* The run as text, formatted on the device: replaces KMerPrinter::print (KMerPrinter.cpp:35-91). One
 * line per record -- the 32 letters of every key word (A, C, G, T; most significant base first), a
 * blank, the count in decimal, '\n' -- written to dst (host memory). *out_bytes = the text's size;
 * KC_ERR_CAPACITY (with *out_bytes set) if cap is too small: at most 32 W + 12 bytes per record. */
int  kc_run_print(kc_ctx *ctx, const kc_run *run, char *dst, uint64_t cap, uint64_t *out_bytes);
/* packed records in: a run file's bytes (must be sorted; adjacent equal keys are
 * folded like SortedKMerFile::ReadKmer does, SortedKMerFile.cpp:57-82) */
int  kc_run_upload(kc_ctx *ctx, const void *records, uint64_t n_bytes, kc_run **run);
/* device views for the multi-GPU exchange: keys = n*W uint64 (key-major), counts = n uint32 */
int  kc_run_device(const kc_run *run, void **d_keys, void **d_counts, uint64_t *n);
/* build a run from device arrays holding sorted unique keys (copied) */
int  kc_run_from_device(kc_ctx *ctx, const void *d_keys, const void *d_counts, uint64_t n, kc_run **run);
/* write dumpKmersToFile-style: truncates unless append != 0 */
int  kc_run_write(kc_ctx *ctx, const kc_run *run, const char *path, int append);
/* lower-bound positions of n_splitters keys (each W words, ascending) inside the
 * run: offsets[0]=0, offsets[i+1]=first record >= splitter i, offsets[n_splitters+1]=n */
int  kc_run_split(kc_ctx *ctx, const kc_run *run, const uint64_t *splitters, uint32_t n_splitters,
                  uint64_t *offsets);

/* ---- count spectrum and filtering: what `jellyfish histo` / `kmc_tools histogram` and the count
 * cut-offs of KMC (-ci/-cx) and Jellyfish (-L/-U) give, computed on the device from a finished run ---- */
/* hist[c] = records of the run with count exactly c, for c < n_bins - 1; hist[n_bins - 1] = records
 * with count >= n_bins - 1 (the "high" bin). 2 <= n_bins <= 1 << 24; hist is host memory, overwritten.
 * hist[0] holds zero-count records: under KC_COMPAT_REF the phantom key-0 record (SURVEY F7), and any
 * count that wrapped at 2^32. Records hidden by the run's strict-mode skip are not counted. */
int  kc_run_histogram(kc_ctx *ctx, const kc_run *run, uint64_t *hist, uint32_t n_bins);
/* A new run with the records whose count c satisfies min_count <= c <= max_count, in the same order
 * (so it is sorted and key-unique). The input run is unchanged. The output is sized exactly and has
 * no partition structure (kc_run_parts: n_sub == 0). min_count > max_count -> KC_ERR_ARG.
 * Filter only a run whose counts are final: filtering one chunk's run before it is merged with the
 * others would drop k-mers whose total count is in range. */
int  kc_run_filter(kc_ctx *ctx, const kc_run *run, uint32_t min_count, uint32_t max_count, kc_run **out);

/* Runs produced by KC_COUNT_HASH also carry their partition structure: the key space is cut
 * into n_sub equal ranges on the leading prefix_bits of the key and d_offsets[j] (uint32,
 * n_sub + 1 entries, device memory owned by the run) is the first record of range j. n_sub == 0
 * for runs without it (sort path, uploads, merges). Used by the multi-GPU exchange. */
int  kc_run_parts(const kc_run *run, void **d_offsets, uint32_t *n_sub, uint32_t *prefix_bits);
/* Merge n_src (<= 8) pre-counted parts that cover the same n_sub consecutive key ranges:
 * part s is n_records[s] sorted unique records (d_keys[s], d_counts[s]) with d_offsets[s]
 * (uint32[n_sub + 1], relative to the part) marking the ranges. Equal keys are summed
 * (uint32 wrap). One pass, independent of n_src: each range is combined in a shared-memory table. */
int  kc_merge_parts(kc_ctx *ctx, uint32_t n_src, const void *const *d_keys, const void *const *d_counts,
                    const void *const *d_offsets, const uint64_t *n_records, uint32_t n_sub,
                    uint32_t prefix_bits, kc_run **out);

/* Place the next run: the next run the partitioned path finishes on this context (kc_count_device,
 * kc_wait) is written into caller-owned device arrays -- keys (8W bytes each), counts (uint32) and
 * n_sub + 1 range offsets -- if it has at most cap_records records and cap_ranges offsets;
 * otherwise it is allocated as usual. One-shot; NULL pointers clear it. The run does not own placed
 * arrays (kc_run_free leaves them alone); kc_run_device tells where a run ended up. Used to count
 * straight into peer staging memory. */
int  kc_place_next_run(kc_ctx *ctx, void *d_keys, void *d_counts, void *d_offsets, uint64_t cap_records,
                       uint32_t cap_ranges);

/* Peer staging memory (same node, NVLink / NVSwitch): a rank keeps its run in a kc_peer_alloc'd
 * buffer, its peers map it once with kc_peer_open (the 64-byte handle travels by any host
 * channel) and hand the mapped pointers to kc_merge_parts, whose kernel then loads the parts
 * straight from the peers' HBM: the exchange happens inside the combine kernel.
 * d_offsets[s] may hold absolute record indices into part s's arrays (only differences and the
 * first entry are used), n_records[s] = the records of the n_sub ranges read from it. */
int  kc_peer_alloc(kc_ctx *ctx, uint64_t n_bytes, void **d_ptr, void *handle64);
int  kc_peer_open(kc_ctx *ctx, const void *handle64, void **d_ptr);
int  kc_peer_close(kc_ctx *ctx, void *d_ptr);
int  kc_peer_free(kc_ctx *ctx, void *d_ptr);

/* ---- merge: replaces KMerFileMerger::Merge (KMerFileMerger.cpp:49-96) ---- */
/* Merge n sorted runs into one, adding the counts of equal keys (uint32 wrap).
 * Inputs stay valid and owned by the caller. n may be 0 (empty run) or 1 (copy).
 * Two runs: merge path. More: a pairwise merge-path tree, except that three or more runs of the
 * partitioned path with one plan (chunks of equal size, 64-bit keys) are combined range by range
 * in shared memory, up to 8 per pass (kc_merge_parts). */
int  kc_merge_runs(kc_ctx *ctx, kc_run *const *runs, uint32_t n, kc_run **out);

/* ---- set operations of two runs: what `kmc_tools simple` gives (union, intersect, kmers_subtract,
 * counters_subtract with its -oc count modes), on the device ----
 * For every key x with count a in run A and b in run B:
 *
 *   op                       x in A and B                 x only in A   x only in B
 *   KC_SET_UNION             m(a, b)                      a             b
 *   KC_SET_INTERSECT         m(a, b)                      -             -
 *   KC_SET_SUBTRACT          -                            a             -
 *   KC_SET_SUBTRACT_COUNTS   a - b if a > b, else -       a             -
 *
 * m is the count mode `counts`, for keys in both runs only: KC_COUNTS_SUM (a + b, uint32 wrap, as
 * kc_merge_runs), _MIN, _MAX, _A (A's count), _B (B's count). The subtracts take no mode: they must be
 * given KC_COUNTS_SUM (0). Keys compare as everywhere (words as unsigned 64-bit, word 0 first); a
 * record with count 0 (the KC_COMPAT_REF phantom key-0 record) is an ordinary record; records a run
 * hides with its strict-mode skip are not part of it. The output is a new sorted key-unique run; the
 * inputs are unchanged. Union with KC_COUNTS_SUM is kc_merge_runs of the two runs, byte for byte.
 * Like a merge, the output is allocated for the most records op can give (union nA + nB, intersect
 * min(nA, nB), the subtracts nA) and has no partition structure. Never combine canonical and forward
 * runs: a run does not say which keys it holds.
 * KC_ERR_ARG: a null argument, an unknown op or counts, a mode given to a subtract, or runs whose key
 * width differs from each other or from the context's. On any error *out is NULL. */
#define KC_SET_UNION           0u
#define KC_SET_INTERSECT       1u
#define KC_SET_SUBTRACT        2u
#define KC_SET_SUBTRACT_COUNTS 3u
#define KC_COUNTS_SUM          0u
#define KC_COUNTS_MIN          1u
#define KC_COUNTS_MAX          2u
#define KC_COUNTS_A            3u
#define KC_COUNTS_B            4u
int  kc_run_combine(kc_ctx *ctx, const kc_run *a, const kc_run *b, uint32_t op, uint32_t counts, kc_run **out);

/* ---- measurement support (not a reference interface): deterministic synthetic reads
 * written straight into device memory as packed lines; bit-identical to the host
 * generator used by the tests.  genome_len == 0 -> iid bases; zipf_loci > 0 -> half of
 * the reads start at one of zipf_loci hot loci with P(rank) ~ 1/rank. ---- */
int  kc_synth_reads(void *d_out, uint64_t first_read, uint64_t n_reads, uint32_t read_len,
                    uint64_t genome_len, double sub_rate, double n_rate, uint64_t seed,
                    uint64_t zipf_loci, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* KC_API_H */
