// kc_main.cpp -- command line with the reference's flags (main.cpp:25-89).
//
//   kmer_counter_b200 kmerLength=31 inputFileLocation=<dir> outputFile=<file> [gpuMemoryLimit=..]
//                     [tempFileLocation=..] [noOfMergersAtOnce=..] [noOfMergeThreads=..]
//                     [method=auto|sort|hash] [compat=ref|strict] [canonical=1] [device=N] [keepRuns=1] [parser=gpu|host]
//                     [runBudget=BYTES] [gpus=N] [mode=auto|accumulate|runs] [expectedReads=N]
//                     [minCount=N] [maxCount=N] [histoFile=PATH] [histoMax=N]
//   kmer_counter_b200 print <record file> <ignored> <k>       (KMerPrinter, main.cpp:78-82)
//   kmer_counter_b200 histo <record file> <out|-> <k> [histoMax]
//                     the count spectrum of a record file, computed on the GPU (histoFile's format)
//   kmer_counter_b200 combine <union|intersect|subtract|subtract_counts> <A file> <B file> <out file> <k>
//                     [counts=sum|min|max|a|b] [minCount=N] [maxCount=N] [pieceRecords=N]
//                     a set operation of two record files on the GPU (kc_run_combine; KMC's
//                     `kmc_tools simple`), counts= for keys in both (default: sum for union, min for
//                     intersect), minCount= / maxCount= on the combined counts
//
// minCount= / maxCount= keep only the k-mers whose final count is in range (KMC -ci/-cx, Jellyfish
// -L/-U); histoFile= writes the spectrum of the final counts before that filter: one line "c n" per
// count c = 1..histoMax that n k-mers have, the histoMax line counting every k-mer seen >= histoMax
// times (Jellyfish's histo format). Both run on the device, on the final runs only, so records that
// are filtered out never cross PCIe.
//
// What KMerCounter::Start does (KMerCounter.cpp:108-191), on the B200 path: read fixed
// length reads into pinned chunks, count each chunk on the GPU into a sorted run
// (double-buffered: the next chunk is parsed while the previous one is copied and
// counted), merge the runs on the GPU, write the sorted unique records.
#include <inttypes.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <string>
#include <vector>

#include "../../include/kc_api.h"
#include "FastqChunker.h"
#include "Options.h"
#include "RunMerger.h"

// KMerPrinter::print (KMerPrinter.cpp:35-91): every word as 32 letters, then " count".
static int print_records(const char *path, uint64_t k) {
    FILE *f = fopen(path, "rb");
    if (!f) { fprintf(stderr, "cannot open %s\n", path); return 1; }
    const uint32_t W = kc_key_words((uint32_t)k), S = kc_record_size((uint32_t)k);
    std::vector<unsigned char> buf((size_t)S * 10000);
    std::string line;
    size_t n;
    while ((n = fread(buf.data(), 1, buf.size(), f)) >= S) {
        for (size_t off = 0; off + S <= n; off += S) {
            line.clear();
            for (uint32_t w = 0; w < W; w++) {
                uint64_t v;
                memcpy(&v, &buf[off + 8 * w], 8);
                for (int b = 0; b < 32; b++) line.push_back("ACGT"[(v >> (62 - 2 * b)) & 3]);
            }
            uint32_t c;
            memcpy(&c, &buf[off + 8 * W], 4);
            printf("%s %u\n", line.c_str(), c);
        }
    }
    fclose(f);
    return 0;
}

#include <sys/stat.h>

// "c n" for c = 1..hist.size()-1 with n > 0; the last bin holds every count >= its index
static int write_histo(const char *path, const std::vector<uint64_t> &hist) {
    FILE *f = strcmp(path, "-") == 0 ? stdout : fopen(path, "w");
    if (!f) { fprintf(stderr, "cannot open %s\n", path); return KC_ERR_IO; }
    bool ok = true;
    for (size_t c = 1; c < hist.size() && ok; c++)
        if (hist[c]) ok = fprintf(f, "%zu %" PRIu64 "\n", c, hist[c]) > 0;
    if (f == stdout) ok = fflush(f) == 0 && ok;
    else ok = fclose(f) == 0 && ok;
    if (!ok) { fprintf(stderr, "short write to %s\n", path); return KC_ERR_IO; }
    return KC_OK;
}

// minCount= / maxCount= / histoFile=: applied to every final run just before it is written (every
// rank's key range, the one merged run, or each range of the out-of-core merge); the spectra add up
struct FinalRuns {
    const Options &opt;
    std::vector<uint64_t> hist;                 // histoMax + 1 bins when histoFile= is given
    uint64_t dropped = 0;
    explicit FinalRuns(const Options &o) : opt(o), hist(o.histoFile.empty() ? 0 : (size_t)o.histoMax + 1, 0) {}
    bool active() const { return opt.filtering() || !hist.empty(); }
    int apply(kc_ctx *ctx, kc_run **run) {
        int rc = KC_OK;
        if (!hist.empty()) {
            std::vector<uint64_t> h(hist.size());
            if ((rc = kc_run_histogram(ctx, *run, h.data(), (uint32_t)h.size())) != KC_OK) return rc;
            for (size_t c = 0; c < h.size(); c++) hist[c] += h[c];
        }
        if (opt.filtering()) {
            const auto bound = [](int64_t v, uint32_t none) { return v < 0 ? none : v > 0xffffffffll ? 0xffffffffu : (uint32_t)v; };
            kc_run *kept = nullptr;
            if ((rc = kc_run_filter(ctx, *run, bound(opt.minCount, 0), bound(opt.maxCount, 0xffffffffu), &kept)) != KC_OK) return rc;
            dropped += kc_run_records(*run) - kc_run_records(kept);
            kc_run_free(ctx, *run);
            *run = kept;
        }
        return rc;
    }
};

// `histo <record file> <out|-> <k> [histoMax]`: the file is uploaded piece by piece and each piece's
// spectrum is computed on the GPU; a record file is key-unique, so the pieces' spectra add up
static int histo_records(const char *path, const char *out, uint32_t k, int64_t histo_max) {
    if (histo_max < 1 || histo_max > (1 << 24) - 1) { fprintf(stderr, "histoMax must be 1..%d\n", (1 << 24) - 1); return 2; }
    FILE *f = fopen(path, "rb");
    if (!f) { fprintf(stderr, "cannot open %s\n", path); return 1; }
    kc_config cfg = {};
    cfg.struct_size = sizeof cfg;
    cfg.k = k;
    cfg.read_len = k;
    kc_ctx *ctx = nullptr;
    if (kc_create(&cfg, &ctx) != KC_OK) { fprintf(stderr, "kc_create: %s\n", kc_last_error(nullptr)); fclose(f); return 1; }
    const uint64_t S = kc_record_size(k), piece = ((64ull << 20) / S) * S;
    std::vector<unsigned char> buf(piece);
    std::vector<uint64_t> hist((size_t)histo_max + 1, 0), h(hist.size());
    int rc = KC_OK;
    size_t n;
    while (rc == KC_OK && (n = fread(buf.data(), 1, piece, f)) >= S) {
        kc_run *run = nullptr;
        if ((rc = kc_run_upload(ctx, buf.data(), n, &run)) == KC_OK) rc = kc_run_histogram(ctx, run, h.data(), (uint32_t)h.size());
        if (run) kc_run_free(ctx, run);
        for (size_t c = 0; c < h.size() && rc == KC_OK; c++) hist[c] += h[c];
    }
    fclose(f);
    if (rc != KC_OK) fprintf(stderr, "kmer_counter_b200 histo: %s\n", kc_last_error(ctx));
    kc_destroy(ctx);
    if (rc == KC_OK) rc = write_histo(out, hist);
    return rc == KC_OK ? 0 : 1;
}

// `combine <op> <A file> <B file> <out file> <k> [counts=..] [minCount=N] [maxCount=N] [pieceRecords=N]`:
// files of any size, piece by piece on one context. Each piece fills a buffer of up to pieceRecords
// records from each file and is cut at the smaller of the two buffers' last keys (a file that is
// exhausted does not bound the cut; with both exhausted everything is taken). The records at or below
// the cut go up, are combined (and filtered) on the GPU and appended to the output; the rest of each
// buffer opens the next piece. A key's A and B records so land in the same piece, and the buffer whose
// last key is the cut empties, so every piece makes progress.
struct RecordSource {
    FILE *f = nullptr;
    std::vector<unsigned char> buf;
    uint64_t n = 0, read = 0;       // records in buf, records read in all
    bool eof = false;
    int fill(uint64_t S, uint64_t cap) {
        if (buf.size() < cap * S) buf.resize(cap * S);
        while (!eof && n < cap) {
            const size_t want = (size_t)((cap - n) * S), got = fread(buf.data() + n * S, 1, want, f);
            if (got < want) {
                if (ferror(f)) return KC_ERR_IO;
                eof = true;                         // (a partial record at the end is ignored)
            }
            n += got / S;
            read += got / S;
        }
        return KC_OK;
    }
    const unsigned char *rec(uint64_t i, uint64_t S) const { return buf.data() + i * S; }
};

static int key_cmp(const unsigned char *a, const unsigned char *b, uint32_t W) {
    for (uint32_t w = 0; w < W; w++) {
        uint64_t x, y;
        memcpy(&x, a + 8 * w, 8);
        memcpy(&y, b + 8 * w, 8);
        if (x != y) return x < y ? -1 : 1;
    }
    return 0;
}

// records of src with key <= cut (all of them when cut is null)
static uint64_t upto(const RecordSource &src, const unsigned char *cut, uint64_t S, uint32_t W) {
    if (!cut) return src.n;
    uint64_t lo = 0, hi = src.n;
    while (lo < hi) {
        const uint64_t mid = (lo + hi) / 2;
        if (key_cmp(src.rec(mid, S), cut, W) <= 0) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

static int combine_files(int argc, char **argv) {
    const char *usage = "usage: %s combine <union|intersect|subtract|subtract_counts> <A file> <B file> <out file> <k> "
                        "[counts=sum|min|max|a|b] [minCount=N] [maxCount=N] [pieceRecords=N]\n";
    if (argc < 7) { fprintf(stderr, usage, argv[0]); return 2; }
    const std::string op_name = argv[2];
    const char *ops[] = {"union", "intersect", "subtract", "subtract_counts"};
    const char *modes[] = {"sum", "min", "max", "a", "b"};
    uint32_t op = 4;
    for (uint32_t i = 0; i < 4; i++) if (op_name == ops[i]) op = i;
    const uint32_t k = (uint32_t)strtoul(argv[6], nullptr, 10);
    if (op == 4 || k < 1 || k > 128) { fprintf(stderr, usage, argv[0]); return 2; }
    uint32_t counts = op == KC_SET_INTERSECT ? KC_COUNTS_MIN : KC_COUNTS_SUM;      // KMC's defaults
    int64_t min_count = -1, max_count = -1;
    const uint64_t S = kc_record_size(k), W = kc_key_words(k);
    uint64_t piece = (64ull << 20) / S;
    for (int i = 7; i < argc; i++) {
        const char *eq = strchr(argv[i], '=');
        const std::string key = eq ? std::string(argv[i], eq - argv[i]) : argv[i], val = eq ? eq + 1 : "";
        if (key == "counts") {
            counts = 5;
            for (uint32_t m = 0; m < 5; m++) if (val == modes[m]) counts = m;
            if (counts == 5) { fprintf(stderr, "counts= must be sum, min, max, a or b\n"); return 2; }
        } else if (key == "minCount") min_count = strtoll(val.c_str(), nullptr, 10);
        else if (key == "maxCount") max_count = strtoll(val.c_str(), nullptr, 10);
        else if (key == "pieceRecords") piece = strtoull(val.c_str(), nullptr, 10);
        else { fprintf(stderr, usage, argv[0]); return 2; }
    }
    if (piece < 1 || piece > (1ull << 30)) { fprintf(stderr, "pieceRecords must be 1..%llu\n", 1ull << 30); return 2; }
    const auto bound = [](int64_t v, uint32_t none) { return v < 0 ? none : v > 0xffffffffll ? 0xffffffffu : (uint32_t)v; };
    const bool filtering = min_count >= 0 || max_count >= 0;
    RecordSource src[2];
    src[0].f = fopen(argv[3], "rb");
    src[1].f = fopen(argv[4], "rb");
    FILE *out = fopen(argv[5], "wb");                        // truncated here, appended to piece by piece
    if (!src[0].f || !src[1].f || !out) {
        fprintf(stderr, "cannot open %s\n", !src[0].f ? argv[3] : !src[1].f ? argv[4] : argv[5]);
        for (FILE *f : {src[0].f, src[1].f, out}) if (f) fclose(f);
        return 1;
    }
    fclose(out);
    kc_config cfg = {};
    cfg.struct_size = sizeof cfg;
    cfg.k = k;
    cfg.read_len = k;
    kc_ctx *ctx = nullptr;
    int rc = kc_create(&cfg, &ctx);
    if (rc != KC_OK) fprintf(stderr, "kc_create: %s\n", kc_last_error(nullptr));
    uint64_t written = 0, pieces = 0;
    while (rc == KC_OK) {
        if ((rc = src[0].fill(S, piece)) != KC_OK || (rc = src[1].fill(S, piece)) != KC_OK) {
            fprintf(stderr, "read error\n");
            break;
        }
        if (src[0].n == 0 && src[1].n == 0) break;
        const unsigned char *cut = nullptr;                  // +infinity
        for (const RecordSource &s : src)
            if (!s.eof) {
                const unsigned char *last = s.rec(s.n - 1, S);
                if (!cut || key_cmp(last, cut, (uint32_t)W) < 0) cut = last;
            }
        const uint64_t take[2] = {upto(src[0], cut, S, (uint32_t)W), upto(src[1], cut, S, (uint32_t)W)};
        kc_run *in[2] = {nullptr, nullptr}, *res = nullptr;
        for (int i = 0; i < 2 && rc == KC_OK; i++) rc = kc_run_upload(ctx, src[i].buf.data(), take[i] * S, &in[i]);
        if (rc == KC_OK) rc = kc_run_combine(ctx, in[0], in[1], op, counts, &res);
        if (rc == KC_OK && filtering) {
            kc_run *kept = nullptr;
            rc = kc_run_filter(ctx, res, bound(min_count, 0), bound(max_count, 0xffffffffu), &kept);
            kc_run_free(ctx, res);
            res = kept;
        }
        if (rc == KC_OK) rc = kc_run_write(ctx, res, argv[5], 1);
        if (rc == KC_OK) written += kc_run_records(res);
        for (kc_run *r : {in[0], in[1], res}) if (r) kc_run_free(ctx, r);
        if (rc != KC_OK) { fprintf(stderr, "kmer_counter_b200 combine: %s\n", kc_last_error(ctx)); break; }
        for (int i = 0; i < 2; i++) {                        // the rest opens the next piece
            memmove(src[i].buf.data(), src[i].rec(take[i], S), (size_t)((src[i].n - take[i]) * S));
            src[i].n -= take[i];
        }
        pieces++;
    }
    fclose(src[0].f);
    fclose(src[1].f);
    if (ctx) kc_destroy(ctx);
    if (rc != KC_OK) return 1;
    fprintf(stderr, "combine %s counts=%s a_records=%" PRIu64 " b_records=%" PRIu64 " pieces=%" PRIu64 " records=%" PRIu64 " -> %s\n",
            ops[op], modes[counts], src[0].read, src[1].read, pieces, written, argv[5]);
    return 0;
}

// mode=accumulate: every chunk is only packed into super-window records (kc_accum_*); the count
// happens once, over everything -- on one GPU, or on gpus=N with the two exchanges fused into the
// counting kernels (kc_xchg_*). Returns 1 if this input / shape is not for this mode (the caller
// then counts chunk by chunk into runs), 0 on success, -1 on error.
static int run_accumulate(const Options &opt, FastqChunker &reader, int64_t L, int64_t chunk, uint32_t method,
                          FinalRuns &fin, uint64_t *n_records_out) {
    const int G = opt.gpus;
    // reads to plan for: a FASTQ record is 2L + header + '+' line + newlines
    uint64_t expected = opt.expectedReads > 0 ? (uint64_t)opt.expectedReads : 0;
    if (!expected) {
        uint64_t bytes = 0;
        for (const std::string &f : reader.files()) {
            struct stat st;
            if (stat(f.c_str(), &st) == 0) bytes += (uint64_t)st.st_size;
        }
        expected = bytes / (uint64_t)(2 * L + 6) + 1024;
    }
    const uint64_t per_gpu = (expected + G - 1) / G + (uint64_t)(chunk / L) + 16;
    std::vector<kc_ctx *> ctx(G, nullptr);
    auto destroy_all = [&]() { for (kc_ctx *c : ctx) if (c) kc_destroy(c); };
    for (int g = 0; g < G; g++) {
        kc_config cfg = {};
        cfg.struct_size = sizeof cfg;
        cfg.k = (uint32_t)opt.kmerLength;
        cfg.read_len = (uint32_t)L;
        cfg.device = getenv("KC_CLI_SAME_DEVICE") ? opt.device : opt.device + g;   // (test knob: all ranks on one device)
        cfg.flags = (opt.compat == "strict" ? KC_COMPAT_STRICT : KC_COMPAT_REF) | (opt.canonical ? KC_CANONICAL : 0u);
        cfg.method = method;
        cfg.n_slots = 2;
        cfg.max_chunk_bytes = (uint64_t)chunk;
        if (kc_create(&cfg, &ctx[g]) != KC_OK) { fprintf(stderr, "kc_create(device %d): %s\n", cfg.device, kc_last_error(nullptr)); destroy_all(); return -1; }
        const int rc = G > 1 ? kc_xchg_begin(ctx[g], (uint32_t)g, (uint32_t)G, per_gpu) : kc_accum_begin(ctx[g], per_gpu);
        if (rc == KC_ERR_ARG) { destroy_all(); return 1; }            // k or read length not for the super-window path
        if (rc != KC_OK) { fprintf(stderr, "accumulator: %s\n", kc_last_error(ctx[g])); destroy_all(); return -1; }
    }
    int rc = KC_OK;
    uint64_t n_chunks = 0;
    std::vector<bool> busy(2 * G, false);
    auto settle = [&](uint64_t i) -> int {                          // (gpu, slot) of chunk i is free again
        const int g = (int)(i % G), sl = (int)((i / G) % 2);
        if (!busy[2 * g + sl]) return KC_OK;
        busy[2 * g + sl] = false;
        return kc_accum_wait(ctx[g], (uint32_t)sl);
    };
    bool refused = false;
    if (opt.parser != "host") {
        // FASTQ text goes to the GPUs as it is and is parsed there
        const uint64_t raw_cap = (uint64_t)chunk * 23 / 10 + (1u << 20);
        std::vector<void *> raw(2 * G, nullptr);
        for (int i = 0; i < 2 * G && rc == KC_OK; i++) rc = kc_host_alloc(ctx[i / 2], raw_cap, &raw[i]);
        uint64_t carry = 0;
        std::vector<char> carry_buf;
        for (const std::string &path : reader.files()) {
            if (rc != KC_OK || refused) break;
            FILE *f = fopen(path.c_str(), "rb");
            if (!f) continue;
            carry = 0;
            bool eof = false;
            while (rc == KC_OK && !refused) {
                const int g = (int)(n_chunks % G), sl = (int)((n_chunks / G) % 2);
                if ((rc = settle(n_chunks)) != KC_OK) break;
                char *buf = static_cast<char *>(raw[2 * g + sl]);
                if (carry) memcpy(buf, carry_buf.data(), carry);
                uint64_t total = carry;
                if (!eof) {
                    const size_t n = fread(buf + carry, 1, raw_cap - carry - 1, f);
                    total += n;
                    eof = n < raw_cap - carry - 1;
                }
                if (eof && total > 0 && buf[total - 1] != '\n') buf[total++] = '\n';
                if (total == 0) break;
                uint64_t used = 0;
                uint32_t flags = 0;
                if ((rc = kc_accum_submit_fastq(ctx[g], (uint32_t)sl, buf, total, &used, &flags)) != KC_OK) break;
                if (flags) { refused = true; break; }
                if (used == 0) {
                    if (eof) break;                                 // a truncated last record: ignored
                    rc = KC_ERR_CAPACITY;
                    fprintf(stderr, "a FASTQ record does not fit %llu bytes\n", (unsigned long long)raw_cap);
                    break;
                }
                busy[2 * g + sl] = true;
                n_chunks++;
                carry = total - used;
                carry_buf.assign(buf + used, buf + used + carry);
                if (eof && carry == 0) break;
            }
            fclose(f);
        }
        for (int g = 0; g < G; g++)
            for (int sl = 0; sl < 2; sl++)
                if (busy[2 * g + sl]) { kc_accum_wait(ctx[g], (uint32_t)sl); busy[2 * g + sl] = false; }
        for (int i = 0; i < 2 * G; i++)
            if (raw[i]) kc_host_free(ctx[i / 2], raw[i]);
        if (refused && rc == KC_OK) {
            // what has been accumulated is dropped with the contexts; the caller starts over with the host parser
            fprintf(stderr, "input is not plain 4-line fixed-length FASTQ: parsing on the host instead\n");
            destroy_all();
            Options o2 = opt;
            o2.parser = "host";
            FastqChunker again(opt.inputFileDirectory);
            return run_accumulate(o2, again, L, chunk, method, fin, n_records_out);
        }
    } else {
        while (rc == KC_OK) {
            const int g = (int)(n_chunks % G), sl = (int)((n_chunks / G) % 2);
            if ((rc = settle(n_chunks)) != KC_OK) break;
            void *buf = nullptr;
            uint64_t cap = 0;
            if ((rc = kc_slot_buffer(ctx[g], (uint32_t)sl, &buf, &cap)) != KC_OK) break;
            const int64_t n = reader.read(static_cast<char *>(buf), (int64_t)cap);
            if (n == 0) break;
            if ((rc = kc_accum_submit(ctx[g], (uint32_t)sl, (uint64_t)n)) != KC_OK) break;
            busy[2 * g + sl] = true;
            n_chunks++;
        }
        for (int g = 0; g < G; g++)
            for (int sl = 0; sl < 2; sl++)
                if (busy[2 * g + sl]) { kc_accum_wait(ctx[g], (uint32_t)sl); busy[2 * g + sl] = false; }
    }
    // the count, and the artefact: rank r holds the r-th key range, the file is their concatenation
    std::vector<kc_run *> runs(G, nullptr);
    if (rc == KC_OK) rc = G > 1 ? kc_xchg_run_all(ctx.data(), (uint32_t)G, runs.data()) : kc_accum_flush(ctx[0], &runs[0]);
    uint64_t n_records = 0;
    for (int g = 0; g < G && rc == KC_OK; g++) {
        if (fin.active() && (rc = fin.apply(ctx[g], &runs[g])) != KC_OK) break;
        rc = kc_run_write(ctx[g], runs[g], opt.outputFile.c_str(), g == 0 ? 0 : 1);      // truncates, then appends
        n_records += kc_run_records(runs[g]);
    }
    if (rc != KC_OK) {
        for (int g = 0; g < G; g++) if (kc_last_error(ctx[g])[0]) { fprintf(stderr, "kmer_counter_b200: %s\n", kc_last_error(ctx[g])); break; }
    } else {
        kc_stats st;
        kc_stats_get(ctx[0], &st);
        for (int g = 1; g < G; g++) { kc_stats sg; kc_stats_get(ctx[g], &sg); st.reads += sg.reads; }
        fprintf(stderr, "mode=accumulate gpus=%d parser=%s reads=%llu skipped=%llu chunks=%llu records=%llu", G,
                opt.parser != "host" ? "gpu" : "host", (unsigned long long)(opt.parser != "host" ? st.reads : reader.totalReads()),
                (unsigned long long)reader.skippedReads(), (unsigned long long)n_chunks, (unsigned long long)n_records);
        if (opt.filtering()) fprintf(stderr, " filtered=%llu", (unsigned long long)fin.dropped);
        fprintf(stderr, "\n");
    }
    for (int g = 0; g < G; g++) if (runs[g]) kc_run_free(ctx[g], runs[g]);
    destroy_all();
    if (n_records_out) *n_records_out = n_records;
    return rc == KC_OK ? 0 : -1;
}

static uint32_t method_of(const std::string &m) {
    if (m == "sort") return KC_COUNT_SORT;
    if (m == "hash") return KC_COUNT_HASH;
    if (m == "hash_global") return KC_COUNT_HASH_GLOBAL;
    if (m == "super") return KC_COUNT_SUPER;
    if (m == "place") return KC_COUNT_PLACE;
    return KC_COUNT_AUTO;
}

int main(int argc, char **argv) {
    if (argc == 5 && strncmp(argv[1], "print", 5) == 0) return print_records(argv[2], strtoull(argv[4], nullptr, 10));
    if ((argc == 5 || argc == 6) && strcmp(argv[1], "histo") == 0)
        return histo_records(argv[2], argv[3], (uint32_t)strtoul(argv[4], nullptr, 10), argc == 6 ? strtoll(argv[5], nullptr, 10) : 10000);
    if (argc >= 2 && strcmp(argv[1], "combine") == 0) return combine_files(argc, argv);
    Options opt = Options::parse(argc, argv);
    FinalRuns fin(opt);
    if (opt.inputFileDirectory.empty()) {
        fprintf(stderr, "usage: %s kmerLength=K inputFileLocation=DIR outputFile=FILE [gpuMemoryLimit=BYTES] [canonical=1] ...\n", argv[0]);
        return 2;
    }
    FastqChunker reader(opt.inputFileDirectory);
    if (!reader.ok()) { fprintf(stderr, "no FASTQ input in %s\n", opt.inputFileDirectory.c_str()); return 1; }
    const int64_t L = reader.getLineLength();
    int64_t chunk = opt.chunkSize(L);
    const int64_t max_chunk = (int64_t)((((1ull << 30) - 1) / (uint64_t)(L - opt.kmerLength + 1)) * (uint64_t)L);
    if (chunk > max_chunk) chunk = max_chunk - max_chunk % (16 * L);

    // one count over everything (default where the super-window path applies), unless the reference's
    // run-per-chunk shape is asked for (mode=runs, or its options keepRuns / runBudget)
    const bool want_runs = opt.mode == "runs" || opt.keepRuns || opt.runBudget > 0 ||
                           (opt.mode == "auto" && (method_of(opt.method) != KC_COUNT_AUTO && method_of(opt.method) != KC_COUNT_SUPER));
    if (!want_runs || opt.gpus > 1) {
        uint64_t n_rec = 0;
        const int r = run_accumulate(opt, reader, L, chunk, method_of(opt.method), fin, &n_rec);
        if (r == 0 && !opt.histoFile.empty() && write_histo(opt.histoFile.c_str(), fin.hist) != KC_OK) return 1;
        if (r == 0) { fprintf(stderr, "records=%" PRIu64 " -> %s\n", n_rec, opt.outputFile.c_str()); return 0; }
        if (r < 0) return 1;
        if (opt.gpus > 1) { fprintf(stderr, "gpus=%d needs the super-window path: k <= 64 with windows of at least 22 bases, reads of at most 1140 to 1191 bases by k\n", opt.gpus); return 1; }
        // not a shape for the accumulator: fall through to runs
    }

    kc_config cfg = {};
    cfg.struct_size = sizeof cfg;
    cfg.k = (uint32_t)opt.kmerLength;
    cfg.read_len = (uint32_t)L;
    cfg.device = opt.device;
    cfg.flags = (opt.compat == "strict" ? KC_COMPAT_STRICT : KC_COMPAT_REF) | (opt.canonical ? KC_CANONICAL : 0u);
    cfg.method = method_of(opt.method);
    cfg.n_slots = 2;
    cfg.max_chunk_bytes = (uint64_t)chunk;
    kc_ctx *ctx = nullptr;
    if (kc_create(&cfg, &ctx) != KC_OK) { fprintf(stderr, "kc_create: %s\n", kc_last_error(nullptr)); return 1; }

    int rc = KC_OK;
    uint32_t chunk_id = 0;
    uint64_t gpu_parsed_bytes = 0;
    uint64_t n_records = 0;
    // attempt 0: FASTQ text goes to the GPU as it is and is parsed there (kc_submit_fastq);
    // attempt 1: the host chunker, for input the device parser refuses (or parser=host)
    for (int attempt = opt.parser == "host" ? 1 : 0; attempt < 2; attempt++) {
        RunMerger merger(ctx, opt.noOfMergersAtOnce, (uint32_t)opt.kmerLength, opt.runBudget > 0 ? (uint64_t)opt.runBudget : 0,
                         opt.noOfMergeThreads);
        if (fin.active()) merger.SetFinalHook([&](kc_run **run) { return fin.apply(ctx, run); });
        bool busy[2] = {false, false};
        bool refused = false;
        chunk_id = 0;
        auto collect = [&](uint32_t slot) -> int {
            kc_run *run = nullptr;
            int r = kc_wait(ctx, slot, &run);
            busy[slot] = false;
            if (r != KC_OK) return r;
            if (opt.keepRuns) {                                 // FileDump::dumpKmersToFile naming (FileDump.cpp:51-58)
                std::string path = opt.tempFileLocation + "/" + std::to_string(++chunk_id);
                if ((r = kc_run_write(ctx, run, path.c_str(), 0)) != KC_OK) return r;
            }
            return merger.AddRun(run);
        };
        if (attempt == 0) {
            const uint64_t raw_cap = (uint64_t)chunk * 23 / 10 + (1u << 20);
            void *raw[2] = {nullptr, nullptr};
            if (kc_host_alloc(ctx, raw_cap, &raw[0]) != KC_OK || kc_host_alloc(ctx, raw_cap, &raw[1]) != KC_OK) rc = KC_ERR_NOMEM;
            uint32_t slot = 0;
            for (const std::string &path : reader.files()) {
                if (rc != KC_OK || refused) break;
                FILE *f = fopen(path.c_str(), "rb");
                if (!f) continue;                               // the reference ignores unreadable files too
                uint64_t carry = 0;
                bool eof = false;
                while (rc == KC_OK && !refused) {
                    char *buf = static_cast<char *>(raw[slot]);
                    uint64_t total = carry;
                    if (!eof) {
                        const size_t n = fread(buf + carry, 1, raw_cap - carry - 1, f);
                        total += n;
                        eof = n < raw_cap - carry - 1;
                    }
                    if (eof && total > 0 && buf[total - 1] != '\n') buf[total++] = '\n';
                    if (total == 0) break;
                    if (busy[slot] && (rc = collect(slot)) != KC_OK) break;
                    uint64_t used = 0;
                    uint32_t flags = 0;
                    if ((rc = kc_submit_fastq(ctx, slot, buf, total, &used, &flags)) != KC_OK) break;
                    if (flags) { refused = true; break; }
                    if (used == 0) {
                        // fewer than four lines are left: at end of file that is a truncated record, ignored
                        if (eof) { kc_run *empty = nullptr; rc = kc_wait(ctx, slot, &empty); if (empty) kc_run_free(ctx, empty); break; }
                        rc = KC_ERR_CAPACITY;
                        fprintf(stderr, "a FASTQ record does not fit %llu bytes\n", (unsigned long long)raw_cap);
                        break;
                    }
                    busy[slot] = true;
                    gpu_parsed_bytes += used;
                    carry = total - used;
                    memcpy(raw[slot ^ 1], buf + used, carry);   // the tail opens the next block
                    slot ^= 1;
                    if (eof && carry == 0) break;
                }
                fclose(f);
            }
            for (uint32_t sl = 0; sl < 2 && rc == KC_OK; sl++)
                if (busy[sl]) rc = collect(sl);
            if (raw[0]) kc_host_free(ctx, raw[0]);
            if (raw[1]) kc_host_free(ctx, raw[1]);
            if (refused && rc == KC_OK) {
                for (uint32_t sl = 0; sl < 2; sl++)
                    if (busy[sl]) collect(sl);
                fprintf(stderr, "input is not plain 4-line fixed-length FASTQ: parsing on the host instead\n");
                gpu_parsed_bytes = 0;
                continue;                                       // merger (and its runs) is dropped, start over
            }
        } else {
            for (uint32_t slot = 0; rc == KC_OK; slot ^= 1) {
                if (busy[slot]) rc = collect(slot);             // the other slot keeps the GPU busy meanwhile
                if (rc != KC_OK) break;
                void *buf = nullptr;
                uint64_t cap = 0;
                if ((rc = kc_slot_buffer(ctx, slot, &buf, &cap)) != KC_OK) break;
                const int64_t n = reader.read(static_cast<char *>(buf), (int64_t)cap);
                if (n == 0) break;
                if ((rc = kc_submit(ctx, slot, (uint64_t)n)) != KC_OK) break;
                busy[slot] = true;
            }
            for (uint32_t slot = 0; slot < 2 && rc == KC_OK; slot++)
                if (busy[slot]) rc = collect(slot);
        }
        if (rc == KC_OK) rc = merger.Finish(opt.outputFile.c_str(), &n_records);     // truncates (KMerFileMerger.cpp:129 appends)
        if (rc == KC_OK) {
            kc_stats st;
            kc_stats_get(ctx, &st);
            fprintf(stderr, "parser=%s reads=%" PRIu64 " skipped=%" PRIu64 " kmers=%" PRIu64 " chunks=%" PRIu64
                            " merges=%" PRIu64 " spills=%" PRIu64 " ranges=%" PRIu64,
                    attempt == 0 ? "gpu" : "host", attempt == 0 ? st.reads : reader.totalReads(), reader.skippedReads(),
                    st.kmers_valid, st.chunks, merger.merges(), merger.spills(), merger.ranges());
            if (opt.filtering()) fprintf(stderr, " filtered=%" PRIu64, fin.dropped);
            fprintf(stderr, "\n");
            if (!opt.histoFile.empty()) rc = write_histo(opt.histoFile.c_str(), fin.hist);
        }
        break;
    }
    if (rc != KC_OK) fprintf(stderr, "kmer_counter_b200: %s\n", kc_last_error(ctx));
    else fprintf(stderr, "records=%" PRIu64 " -> %s\n", n_records, opt.outputFile.c_str());
    kc_destroy(ctx);
    return rc == KC_OK ? 0 : 1;
}
