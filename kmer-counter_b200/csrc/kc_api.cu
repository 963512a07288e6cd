// kc_api.cu -- the C ABI (include/kc_api.h) over the kernels of this directory.
//
// Host-side orchestration only: buffer lifetime, stream ordering, stage timing.
// There is no CPU compute path here; if the device cannot run a kernel the call
// fails with KC_ERR_CUDA.
#include <stdarg.h>
#include <stdlib.h>
#include <time.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/kc_api.h"
#include "kc_internal.h"

static_assert(kc::kPlanStrict == KC_COMPAT_STRICT && kc::kPlanCanonical == KC_CANONICAL, "plan flags are kc_config.flags bits");
static_assert(kc::kSetUnion == KC_SET_UNION && kc::kSetIntersect == KC_SET_INTERSECT && kc::kSetSubtract == KC_SET_SUBTRACT &&
                  kc::kSetSubtractCounts == KC_SET_SUBTRACT_COUNTS, "combine_pair takes the KC_SET_* values");
static_assert(kc::kCountsSum == KC_COUNTS_SUM && kc::kCountsMin == KC_COUNTS_MIN && kc::kCountsMax == KC_COUNTS_MAX &&
                  kc::kCountsA == KC_COUNTS_A && kc::kCountsB == KC_COUNTS_B, "combine_pair takes the KC_COUNTS_* values");

using namespace kc;

struct kc_run {
    int W = 1;
    uint64_t n = 0;          // records
    uint64_t skip = 0;       // leading records hidden (strict mode drops an empty key-0 record)
    uint64_t *d_keys = nullptr;
    uint32_t *d_counts = nullptr;
    // partition structure (KC_COUNT_HASH runs only): record offsets of n_sub equal key ranges
    uint32_t *d_sub_off = nullptr;
    uint32_t n_sub = 0, prefix_bits = 0;
    bool placed = false;     // arrays belong to the caller (kc_place_next_run): never freed here
};

namespace {

// A run this scope owns: kc_run_free'd when the scope ends unless released to the caller. make_run
// fills one; a run reaches a caller of the ABI only through release() on success.
struct RunFree {
    kc_ctx *c = nullptr;
    void operator()(kc_run *r) const { kc_run_free(c, r); }
};
using RunPtr = std::unique_ptr<kc_run, RunFree>;

thread_local std::string g_create_error;

enum { SC_INVALID = 0, SC_UNIQUE = 1, SC_MERGE = 2, SC_HASHNUM = 3, SC_SIDE = 4 /* 4..7 */, SC_COUNT = 16 };

struct Pending {                 // a chunk whose kernels are queued but whose run is not built yet
    bool active = false;
    uint32_t method = 0;
    uint64_t n_reads = 0, n_slots = 0;
    uint64_t *keys_a = nullptr, *keys_b = nullptr, *sorted = nullptr, *uniq = nullptr;
    uint32_t *starts = nullptr;
    void *ws_sort = nullptr, *ws_rle = nullptr;
    HashTable table{nullptr, 0, nullptr};
    unsigned long long *d_scal = nullptr;   // SC_COUNT device scalars
    unsigned long long *h_scal = nullptr;   // pinned mirror
    cudaEvent_t ev[8] = {};                  // stage k runs from ev[k] to ev[k+1]
    int n_ev = 0;                            // events recorded by count_enqueue (the emit stage adds one)
    int n_passes = 0;
    uint32_t *counts = nullptr;              // partition path: counts next to the unique keys
    void *ws_part = nullptr;
    SuperPlan splan{};                       // super-window path: plan + workspace (arena)
    void *ws_super = nullptr;
    // Chunk scratch arena: one grow-only device block per Pending, carved by a bump pointer.
    // Chunk after chunk reuses it, so the big buffers never go through the allocator again.
    uint8_t *arena = nullptr;
    uint64_t arena_cap = 0, arena_used = 0;
};

struct Slot {
    void *h_in = nullptr;        // pinned
    void *d_in = nullptr;
    uint64_t cap = 0;
    cudaStream_t stream = nullptr;
    Pending pend;
    uint64_t n_bytes = 0;
    void *d_text = nullptr;      // raw FASTQ staging (kc_submit_fastq), grown on demand
    uint64_t text_cap = 0;
};

}  // namespace

struct kc_ctx {
    kc_config cfg{};
    int W = 1, S = 12;
    bool strict = false;         // KC_COMPAT_STRICT, also set by KC_CANONICAL
    uint32_t key_flags = 0;      // kPlanStrict | kPlanCanonical: the key semantics every plan is made for
    int n_sms = 148;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    cudaStream_t copy_stream = nullptr;   // records D2H (kc_run_copy_records): its own stream, so that reading
                                          // one run back overlaps the kernels of the next on `stream`
    struct { uint64_t *keys = nullptr; uint32_t *counts = nullptr, *offs = nullptr; uint64_t cap = 0; uint32_t cap_ranges = 0; bool set = false; } place;
    std::mutex copy_mu;                   // one read-back at a time (the link is the limit anyway)
    void *copy_buf = nullptr;             // packed records staged for D2H: grow-only, not from the pool
    uint64_t copy_cap = 0;
    std::vector<Slot> slots;
    Pending direct;              // kc_count_device / kc_process_chunk without slots use this
    // Accumulating mode (kc_accum_*): chunks are only packed into super-window records; one count at the end
    struct Accum {
        bool on = false;
        SuperPlan pl{};
        void *ws = nullptr;                  // plain cudaMalloc, owned
        uint64_t ws_bytes = 0;
        unsigned long long *d_sc = nullptr, *h_sc = nullptr;
        uint64_t windows = 0, reads = 0;     // accumulated since the last reset
        uint64_t max_windows = 0;            // what the plan was made for
        uint64_t ovf_reserved = 0;           // overflow records that chunks queued so far may still produce
        std::vector<RunPtr> parts;           // runs of earlier automatic flushes
        cudaEvent_t ev[8] = {};
        bool fresh = true;                   // bins are empty
        // multi-GPU exchange (kc_xchg_*): this context is rank `rank` of `n_ranks`
        bool xchg = false;
        uint32_t rank = 0, n_ranks = 1;
        void *peer_ws[8] = {};               // the ranks' workspaces as mapped into this device
        bool peer_ipc[8] = {};               // opened with cudaIpcOpenMemHandle (to be closed)
        uint32_t *d_all_hist = nullptr;      // n_ranks x 1024, filled by the caller's all-gather
        SuperXInfo x_info{};                 // the last exchange's plan (kc_xchg_info)
        bool keep_ranges = false;            // kc_xchg_fix_ranges
        float ms_scatter = 0;
        uint64_t n_scatter = 0;
        std::vector<cudaEvent_t> sc_ev;      // begin/end event pairs of the S1 launches since the last flush
    } acc;
    std::recursive_mutex direct_mu;   // calls that take no slot (they share `direct`, its arena and `stream`) are serialised
    std::mutex mu;
    kc_stats stats{};
    unsigned long long last_scal[SC_COUNT] = {0};   // device scalars of the most recent chunk (kc_debug_scalars)
    int last_code = 0;
    char err[512] = {0};
    uint64_t fail_alloc_at = 0;           // KC_TEST_FAIL_ALLOC
    std::atomic<uint64_t> n_alloc_calls{0};

    int set_error(int code, const char *fmt, ...) {
        va_list ap;
        va_start(ap, fmt);
        vsnprintf(err, sizeof err, fmt, ap);
        va_end(ap);
        last_code = code;
        return code;
    }
};

namespace {

#define KC_TRY(expr)                         \
    do {                                     \
        int _rc = (expr);                    \
        if (_rc != KC_OK) return _rc;        \
    } while (0)

// Device memory of runs and short-lived scratch: the stream-ordered pool. If the pool cannot grow
// (the device is nearly full of plain allocations) its cached blocks are released and the request
// is retried, then made with plain cudaMalloc; dev_free knows those by address.
std::mutex g_plain_mu;
std::vector<void *> g_plain;

int dev_alloc(kc_ctx *c, cudaStream_t s, uint64_t bytes, void **out) {
    *out = nullptr;
    // KC_TEST_FAIL_ALLOC=n (test knob, read in kc_create): the context's n-th call fails once, before allocating anything
    if (c->fail_alloc_at && ++c->n_alloc_calls == c->fail_alloc_at)
        return c->set_error(KC_ERR_NOMEM, "device allocation of %llu bytes failed (KC_TEST_FAIL_ALLOC)", (unsigned long long)bytes);
    if (bytes == 0) bytes = 16;
    const bool dbg = getenv("KC_DEBUG_PLAN") != nullptr;
    if (dbg && bytes > (1ull << 30)) {
        size_t fr = 0, tot = 0;
        cudaMemGetInfo(&fr, &tot);
        fprintf(stderr, "kc dev_alloc %llu bytes (%llu of %llu free)\n", (unsigned long long)bytes, (unsigned long long)fr, (unsigned long long)tot);
    }
    cudaError_t e = cudaMallocAsync(out, bytes, s);
    if (e != cudaSuccess) {
        cudaGetLastError();
        cudaStreamSynchronize(s);
        cudaMemPool_t pool = nullptr;
        int dev = 0;
        cudaGetDevice(&dev);
        if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) cudaMemPoolTrimTo(pool, 0);
        e = cudaMallocAsync(out, bytes, s);
    }
    if (e != cudaSuccess) {
        cudaGetLastError();
        e = cudaMalloc(out, bytes);
        if (e == cudaSuccess) {
            std::lock_guard<std::mutex> g(g_plain_mu);
            g_plain.push_back(*out);
        }
    }
    if (e != cudaSuccess) {
        cudaGetLastError();
        size_t fr = 0, tot = 0;
        cudaMemGetInfo(&fr, &tot);
        *out = nullptr;
        return c->set_error(KC_ERR_NOMEM, "device allocation of %llu bytes failed: %s (%llu of %llu bytes free on the device, "
                            "accumulator workspace %llu bytes)", (unsigned long long)bytes, cudaGetErrorString(e),
                            (unsigned long long)fr, (unsigned long long)tot, (unsigned long long)c->acc.ws_bytes);
    }
    return KC_OK;
}
void dev_free(cudaStream_t s, void *p) {
    if (!p) return;
    {
        std::lock_guard<std::mutex> g(g_plain_mu);
        auto it = std::find(g_plain.begin(), g_plain.end(), p);
        if (it != g_plain.end()) {
            g_plain.erase(it);
            cudaStreamSynchronize(s);
            cudaFree(p);
            return;
        }
    }
    cudaFreeAsync(p, s);
}

// Short-lived device scratch from dev_alloc, given back on its stream when the scope ends unless released.
class DevBuf {
  public:
    explicit DevBuf(cudaStream_t s) : s_(s) {}
    DevBuf(DevBuf &&o) noexcept : s_(o.s_), p_(o.release()) {}
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
    ~DevBuf() { reset(); }
    int alloc(kc_ctx *c, uint64_t bytes) { return dev_alloc(c, s_, bytes, &p_); }
    template <class T = void> T *get() const { return static_cast<T *>(p_); }
    template <class T = void> T *release() {
        T *p = get<T>();
        p_ = nullptr;
        return p;
    }
    void reset() { dev_free(s_, release()); }

  private:
    cudaStream_t s_;
    void *p_ = nullptr;
};

int pending_init(kc_ctx *c, Pending &p) {
    if (p.d_scal) return KC_OK;
    KC_CUDA_TRY(c, cudaMalloc((void **)&p.d_scal, SC_COUNT * 8));
    KC_CUDA_TRY(c, cudaMallocHost((void **)&p.h_scal, SC_COUNT * 8));
    for (auto &e : p.ev) KC_CUDA_TRY(c, cudaEventCreate(&e));
    return KC_OK;
}
void pending_destroy(Pending &p) {
    if (p.arena) cudaFree(p.arena);
    if (p.d_scal) cudaFree(p.d_scal);
    if (p.h_scal) cudaFreeHost(p.h_scal);
    for (auto &e : p.ev)
        if (e) cudaEventDestroy(e);
    p = Pending();
}

// Reserve the scratch a chunk needs (call once per chunk, before arena_take). The stream
// is drained before a grown arena replaces the old one.
int arena_reserve(kc_ctx *c, Pending &p, uint64_t bytes, cudaStream_t s) {
    p.arena_used = 0;
    if (bytes <= p.arena_cap) return KC_OK;
    KC_CUDA_TRY(c, cudaStreamSynchronize(s));
    if (p.arena) cudaFree(p.arena);
    p.arena = nullptr;
    p.arena_cap = 0;
    bytes += bytes / 16;                           // a little headroom so that slightly larger chunks fit too
    if (cudaMalloc((void **)&p.arena, bytes) != cudaSuccess) {
        cudaGetLastError();
        return c->set_error(KC_ERR_NOMEM, "device allocation of %llu bytes of chunk scratch failed", (unsigned long long)bytes);
    }
    p.arena_cap = bytes;
    return KC_OK;
}
inline uint64_t arena_round(uint64_t b) { return (b + 511) & ~511ull; }
void *arena_take(Pending &p, uint64_t bytes) {
    void *r = p.arena + p.arena_used;
    p.arena_used += arena_round(bytes);
    return r;
}

void pending_release(cudaStream_t, Pending &p) {
    p.arena_used = 0;
    p.keys_a = p.keys_b = p.sorted = p.uniq = nullptr;
    p.starts = nullptr;
    p.counts = nullptr;
    p.ws_sort = p.ws_rle = p.ws_part = p.ws_super = nullptr;
    p.table = HashTable{nullptr, 0, nullptr};
    p.active = false;
}

// KC_TRACE=1: wall-clock milestones of the accumulating flush on stderr (development aid)
struct Trace {
    bool on;
    struct timespec t0;
    Trace() : on(getenv("KC_TRACE") != nullptr) { if (on) clock_gettime(CLOCK_MONOTONIC, &t0); }
    void mark(const char *what) {
        if (!on) return;
        struct timespec t1;
        clock_gettime(CLOCK_MONOTONIC, &t1);
        fprintf(stderr, "kc trace: %-28s %9.3f ms\n", what, (t1.tv_sec - t0.tv_sec) * 1e3 + (t1.tv_nsec - t0.tv_nsec) * 1e-6);
        t0 = t1;
    }
};

// KC_SW_FORCE_DUP=1 (test knob, read at every count): the super-window path always takes its folding variant
bool env_force_dup() {
    const char *v = getenv("KC_SW_FORCE_DUP");
    return v && v[0] == '1';
}

uint64_t pow2_ceil(uint64_t x) {
    uint64_t p = 1;
    while (p < x) p <<= 1;
    return p;
}

// low bits of the last key word that are zero for every key (masked tail): the
// radix sort skips the passes that would only see zeros
int static_zero_bits(const kc_ctx *c) {
    uint32_t m = c->cfg.k % 32;
    bool masked = c->strict ? (m != 0) : (m >= 1 && m <= 28);
    return masked ? (int)(64 - 2 * m) : 0;
}

constexpr uint64_t kMaxSortKeys = (1ull << 30) - 1;

// the super-window path takes 64/128-bit keys whose windows span at least 22 bases, from reads
// short enough for S1's shared memory (every plan super_plan makes for the shape fits it then)
bool super_ok(const kc_ctx *c) {
    SuperPlan pl;
    return c->W <= 2 && super_plan(c->cfg.k, c->cfg.read_len, c->key_flags, 1, 0, &pl);
}

// the partitioned hash takes 64/128-bit keys from reads short enough for PA's shared-memory tile
bool hash_ok(const kc_ctx *c) {
    ExtractParams ep;
    return c->W <= 2 && extract_plan(nullptr, 16, c->cfg.read_len, c->cfg.k, c->key_flags, nullptr, &ep, kPaTileBytes) &&
           partition_fits(ep, c->W);
}

uint32_t pick_method(const kc_ctx *c) {
    uint32_t m = c->cfg.method;
    if (m == KC_COUNT_SUPER) return super_ok(c) ? KC_COUNT_SUPER : (hash_ok(c) ? KC_COUNT_HASH : KC_COUNT_SORT);
    if (m == KC_COUNT_AUTO && super_ok(c)) return KC_COUNT_SUPER;
    if (m == KC_COUNT_PLACE) return KC_COUNT_PLACE;
    if (c->W > 2) return m == KC_COUNT_AUTO ? KC_COUNT_PLACE : KC_COUNT_SORT;   // 192/256-bit keys: MSD placement + fold (auto), or sort + run-length
    if ((m == KC_COUNT_AUTO || m == KC_COUNT_HASH) && !hash_ok(c)) return KC_COUNT_SORT;    // reads too long for PA
    if (c->W == 2) return (m == KC_COUNT_AUTO || m == KC_COUNT_HASH) ? KC_COUNT_HASH : KC_COUNT_SORT;
    // 64-bit keys: partitioned shared-memory hashing unless the key has too few significant
    // bits to partition on (tiny k); see DESIGN.md "method selection"
    if (m == KC_COUNT_AUTO) return (64 - static_zero_bits(c)) >= 24 ? KC_COUNT_HASH : KC_COUNT_SORT;
    return m;
}

int count_enqueue_impl(kc_ctx *c, Pending &p, const void *d_reads, uint64_t n_bytes, cudaStream_t s, uint32_t method);

// Queue extraction + counting of one chunk on stream s. Nothing is synchronised. A chunk that
// could not be queued leaves the slot idle (not "in flight"): the next submit works, a wait says
// KC_ERR_STATE.
int count_enqueue(kc_ctx *c, Pending &p, const void *d_reads, uint64_t n_bytes, cudaStream_t s, uint32_t method) {
    const int rc = count_enqueue_impl(c, p, d_reads, n_bytes, s, method);
    if (rc != KC_OK) pending_release(s, p);
    return rc;
}

int count_enqueue_impl(kc_ctx *c, Pending &p, const void *d_reads, uint64_t n_bytes, cudaStream_t s, uint32_t method) {
    KC_TRY(pending_init(c, p));
    memset(p.h_scal, 0, SC_COUNT * 8);            // an empty chunk copies nothing back: no stale counters
    const uint32_t L = c->cfg.read_len, k = c->cfg.k;
    const int W = c->W;
    p.n_reads = n_bytes / L;
    p.n_slots = p.n_reads * (uint64_t)(L - k + 1);
    p.method = method;
    p.active = true;
    p.n_passes = 0;
    int launches = 0;
    KC_CUDA_TRY(c, cudaMemsetAsync(p.d_scal, 0, SC_COUNT * 8, s));
    KC_CUDA_TRY(c, cudaEventRecord(p.ev[0], s));
    p.n_ev = 1;
    if (p.n_slots == 0) return KC_OK;
    if (p.n_slots > kMaxSortKeys) return c->set_error(KC_ERR_ARG, "chunk too large: %llu k-mer slots (max %llu)",
                                                      (unsigned long long)p.n_slots, (unsigned long long)kMaxSortKeys);
    ExtractParams ep;
    if (!extract_plan(d_reads, p.n_reads, L, k, c->key_flags, &p.d_scal[SC_INVALID], &ep))
        return c->set_error(KC_ERR_ARG, "unsupported shape k=%u read_len=%u", k, L);

    if (method == KC_COUNT_SUPER) {
        // super-window records binned by minimizer, counted in shared memory (kc_super.cu)
        if (!super_plan(k, L, c->key_flags, p.n_slots, (uint32_t)c->cfg.table_slots, &p.splan))
            return c->set_error(KC_ERR_ARG, "unsupported shape k=%u read_len=%u", k, L);
        KC_TRY(arena_reserve(c, p, arena_round(p.splan.ws_bytes), s));
        p.ws_super = arena_take(p, p.splan.ws_bytes);
        KC_CUDA_TRY(c, super_reset(p.splan, p.ws_super, p.d_scal, s));
        KC_CUDA_TRY(c, super_scatter(p.splan, d_reads, p.n_reads, p.ws_super, p.d_scal, c->n_sms, s));
        KC_CUDA_TRY(c, cudaEventRecord(p.ev[1], s));
        KC_CUDA_TRY(c, super_count(p.splan, !c->strict, p.ws_super, p.d_scal, c->n_sms, s, &p.ev[2]));
        p.n_ev = 6;
        p.n_passes = 1;
        launches += 8;
    } else if (method == KC_COUNT_PLACE) {
        // key-placement path (kc_super.cuh): keys straight into D, then S3a..S3b; S3c folds in count_finish
        if (!place_plan(k, c->strict, p.n_slots, &p.splan))
            return c->set_error(KC_ERR_ARG, "unsupported shape k=%u read_len=%u", k, L);
        KC_TRY(arena_reserve(c, p, arena_round(p.splan.ws_bytes), s));
        p.ws_super = arena_take(p, p.splan.ws_bytes);
        KC_CUDA_TRY(c, launch_extract_store(ep, W, place_keys(p.splan, p.ws_super), c->n_sms, s));
        KC_CUDA_TRY(c, cudaEventRecord(p.ev[1], s));
        KC_CUDA_TRY(c, place_init(p.splan, p.ws_super, p.d_scal, p.n_slots, c->n_sms, s));
        KC_CUDA_TRY(c, cudaEventRecord(p.ev[2], s));
        KC_CUDA_TRY(c, super_place(p.splan, p.ws_super, p.d_scal, c->n_sms, s, &p.ev[3]));
        p.n_ev = 6;
        p.n_passes = 1;
        launches += 8;
    } else if (method == KC_COUNT_HASH) {
        // partitioned shared-memory hash counting (kc_partition.cu)
        ExtractParams ep64;                     // PA's tile
        if (!extract_plan(d_reads, p.n_reads, L, k, c->key_flags, &p.d_scal[SC_INVALID], &ep64, kPaTileBytes))
            return c->set_error(KC_ERR_ARG, "unsupported shape k=%u read_len=%u", k, L);
        const uint64_t kb = p.n_slots * 8 * W + 64, cb = (p.n_slots + 2) * 4, wb = partition_workspace_bytes(p.n_slots);
        KC_TRY(arena_reserve(c, p, 2 * arena_round(kb) + arena_round(cb) + arena_round(wb), s));
        p.keys_a = static_cast<uint64_t *>(arena_take(p, kb));
        p.keys_b = static_cast<uint64_t *>(arena_take(p, kb));
        p.counts = static_cast<uint32_t *>(arena_take(p, cb));
        p.ws_part = arena_take(p, wb);
        const int sig = W == 1 ? 64 - static_zero_bits(c) : 64;        // significant bits of key word 0
        const int target = c->cfg.table_slots ? (int)c->cfg.table_slots : 0;   // keys per sub-bucket (0 = default)
        p.uniq = partition_two_levels(p.n_slots, sig, target) ? p.keys_a : p.keys_b;
        KC_CUDA_TRY(c, partition_count(W, ep64, p.n_slots, sig, !c->strict, p.keys_a, p.keys_b, p.uniq, p.counts,
                                       &p.d_scal[SC_UNIQUE], &p.d_scal[SC_SIDE + 1], &p.d_scal[SC_COUNT - 2],
                                       p.ws_part, c->n_sms, target, s, &launches, &p.ev[1]));
        p.n_ev = 6;
        p.n_passes = 1;
    } else if (method == KC_COUNT_HASH_GLOBAL) {
        uint64_t cap = c->cfg.table_slots ? pow2_ceil(c->cfg.table_slots) : pow2_ceil(p.n_slots / 2 + 1);
        if (cap < (1u << 16)) cap = 1u << 16;
        KC_TRY(arena_reserve(c, p, arena_round(hash_table_bytes(cap)), s));
        p.table.slots = static_cast<uint64_t *>(arena_take(p, hash_table_bytes(cap)));
        p.table.capacity = cap;
        p.table.side = &p.d_scal[SC_SIDE];
        KC_CUDA_TRY(c, hash_clear(p.table, s));
        KC_CUDA_TRY(c, cudaEventRecord(p.ev[1], s));
        KC_CUDA_TRY(c, launch_extract_hash(ep, p.table, c->n_sms, s));
        KC_CUDA_TRY(c, hash_touch_zero(p.table, c->strict ? &p.d_scal[SC_COUNT - 1] : &p.d_scal[SC_INVALID], s));
        KC_CUDA_TRY(c, cudaEventRecord(p.ev[2], s));
        p.n_ev = 3;
        launches += 3;
        p.n_passes = 1;
    } else {
        const uint64_t ws_bytes = sort_workspace_bytes(p.n_slots, W);
        const uint64_t kb = p.n_slots * W * 8, sb = (p.n_slots + 1) * 4, rb = rle_workspace_bytes(p.n_slots);
        KC_TRY(arena_reserve(c, p, 2 * arena_round(kb) + arena_round(sb) + arena_round(ws_bytes) + arena_round(rb), s));
        p.keys_a = static_cast<uint64_t *>(arena_take(p, kb));
        p.keys_b = static_cast<uint64_t *>(arena_take(p, kb));
        p.starts = static_cast<uint32_t *>(arena_take(p, sb));
        p.ws_sort = arena_take(p, ws_bytes);
        p.ws_rle = arena_take(p, rb);
        KC_CUDA_TRY(c, launch_extract_store(ep, W, p.keys_a, c->n_sms, s));
        KC_CUDA_TRY(c, cudaEventRecord(p.ev[1], s));
        const int lo_bit = static_zero_bits(c);
        p.n_passes = (64 * W - (lo_bit & ~7)) / 8;
        int sort_launches = 0;
        KC_CUDA_TRY(c, radix_sort(p.keys_a, p.keys_b, nullptr, nullptr, p.n_slots, W, lo_bit,
                                  SortWorkspace{p.ws_sort, ws_bytes}, s, &p.sorted, nullptr, &sort_launches,
                                  p.ev[2], p.ev[3]));
        p.uniq = (p.sorted == p.keys_a) ? p.keys_b : p.keys_a;
        KC_CUDA_TRY(c, rle_unique(p.sorted, p.n_slots, W, p.uniq, p.starts, &p.d_scal[SC_UNIQUE], p.ws_rle, s,
                                  &sort_launches));
        KC_CUDA_TRY(c, cudaEventRecord(p.ev[4], s));
        p.n_ev = 5;
        launches += 1 + sort_launches;
    }
    KC_CUDA_TRY(c, cudaMemcpyAsync(p.h_scal, p.d_scal, SC_COUNT * 8, cudaMemcpyDeviceToHost, s));
    {
        std::lock_guard<std::mutex> g(c->mu);
        c->stats.launches += launches;
    }
    return KC_OK;
}

int make_run(kc_ctx *c, cudaStream_t s, uint64_t n, RunPtr *out) {
    DevBuf keys(s), counts(s);
    KC_TRY(keys.alloc(c, n * c->W * 8));
    KC_TRY(counts.alloc(c, n * 4));
    RunPtr r(new kc_run(), RunFree{c});
    r->W = c->W;
    r->n = n;
    r->d_keys = keys.release<uint64_t>();
    r->d_counts = counts.release<uint32_t>();
    *out = std::move(r);
    return KC_OK;
}
// kc_merge_runs of runs the caller owns (they are freed with the vector)
int merge_owned(kc_ctx *c, const std::vector<RunPtr> &parts, kc_run **out) {
    std::vector<kc_run *> in;
    for (const RunPtr &p : parts) in.push_back(p.get());
    return kc_merge_runs(c, in.data(), (uint32_t)in.size(), out);
}

// Super-window path: sub-buckets S3c left out because they exceed its shared memory (skewed input:
// many distinct keys share a long prefix). Their records are gathered in sub-bucket order, sorted by
// the radix sorter and put in place (folded first if records may repeat). n_big_records comes from
// the scalars the caller has just read back; the scratch is stream-ordered.
int super_finish_big(kc_ctx *c, const SuperPlan &pl, void *ws, unsigned long long *d_sc, bool dup, uint64_t n_big_records,
                     uint64_t *out_keys, uint32_t *out_counts, cudaStream_t s) {
    if (n_big_records == 0) return KC_OK;
    if (n_big_records > kMaxSortKeys) return c->set_error(KC_ERR_CAPACITY, "%llu records in oversized key ranges", (unsigned long long)n_big_records);
    const int W = c->W;
    const uint64_t kb = n_big_records * W * 8, cb = n_big_records * 4, wsb = sort_workspace_bytes(n_big_records, W);
    DevBuf ka(s), kb2(s), ca(s), cb2(s), sw(s);
    KC_TRY(ka.alloc(c, kb));
    KC_TRY(kb2.alloc(c, kb));
    KC_TRY(ca.alloc(c, cb));
    KC_TRY(cb2.alloc(c, cb));
    KC_TRY(sw.alloc(c, wsb));
    int launches = 0;
    uint64_t *sk = nullptr;
    uint32_t *sv = nullptr;
    KC_CUDA_TRY(c, super_big_gather(pl, ws, ka.get<uint64_t>(), ca.get<uint32_t>(), c->n_sms, s));
    KC_CUDA_TRY(c, radix_sort(ka.get<uint64_t>(), kb2.get<uint64_t>(), ca.get<uint32_t>(), cb2.get<uint32_t>(), n_big_records, W,
                              static_zero_bits(c), SortWorkspace{sw.get(), wsb}, s, &sk, &sv, &launches, nullptr, nullptr));
    KC_CUDA_TRY(c, super_big_place(pl, dup, ws, d_sc, sk, sv, out_keys, out_counts, c->n_sms, s));
    std::lock_guard<std::mutex> g(c->mu);
    c->stats.launches += launches + 3;
    return KC_OK;
}

// S3c, the last stage of the super-window and key-placement paths, once S3a/S3b are queued: every
// sub-bucket is sorted in shared memory, straight into the run of n_d records, or -- if records may
// repeat (dup) -- folded into a temporary that a gather compacts into a run of the survivors.
// fpl is the plan whose S3c variant runs, h_sc the host mirror of the scalars d_sc. *run may come
// allocated (!dup: its arrays were the second record buffer E of S3a/S3b). ext_e (dup only): E is
// the caller's own allocation {keys, counts}, and the temporary: the survivors are gathered into D,
// E is given back and only then the run is allocated, so that both are never held next to the
// workspace. h_sc[SW_FAIL] set on return: the records did not fit, *run is no count.
int super_emit(kc_ctx *c, const SuperPlan &pl, const SuperPlan &fpl, void *ws, unsigned long long *d_sc,
               unsigned long long *h_sc, bool dup, uint64_t n_d, cudaStream_t s, RunPtr *run, DevBuf *ext_e = nullptr) {
    auto read_back = [&]() {
        cudaError_t e = cudaMemcpyAsync(h_sc, d_sc, SC_COUNT * 8, cudaMemcpyDeviceToHost, s);
        return e == cudaSuccess ? cudaStreamSynchronize(s) : e;
    };
    if (!dup) {
        if (!*run) KC_TRY(make_run(c, s, n_d, run));
        if (n_d) {                                  // (nothing ran otherwise: the scalars are the ones the caller holds)
            KC_CUDA_TRY(c, super_finish(fpl, false, ws, d_sc, (*run)->d_keys, (*run)->d_counts, c->n_sms, s));
            KC_CUDA_TRY(c, read_back());
        }
        if (!h_sc[SW_FAIL] && h_sc[SW_BIG])
            KC_TRY(super_finish_big(c, pl, ws, d_sc, false, h_sc[SW_BIG_RECORDS], (*run)->d_keys, (*run)->d_counts, s));
        return KC_OK;
    }
    uint64_t *tk = nullptr;
    uint32_t *tc = nullptr;
    super_tmp_buffers(pl, ws, &tk, &tc);
    KC_CUDA_TRY(c, super_finish(fpl, true, ws, d_sc, tk, tc, c->n_sms, s));
    KC_CUDA_TRY(c, read_back());
    if (!h_sc[SW_FAIL] && h_sc[SW_BIG]) KC_TRY(super_finish_big(c, pl, ws, d_sc, true, h_sc[SW_BIG_RECORDS], tk, tc, s));
    KC_CUDA_TRY(c, super_fold_offsets(pl, ws, d_sc, s));
    KC_CUDA_TRY(c, read_back());
    if (h_sc[SW_FAIL]) return KC_OK;
    const uint64_t n_out = h_sc[SW_OUT];
    if (!ext_e) {
        KC_TRY(make_run(c, s, n_out, run));
        if (n_out) KC_CUDA_TRY(c, super_gather(pl, ws, tk, tc, (*run)->d_keys, (*run)->d_counts, c->n_sms, s));
        return KC_OK;
    }
    uint64_t *dk = reinterpret_cast<uint64_t *>(static_cast<uint8_t *>(ws) + pl.off_dk);
    uint32_t *dc = reinterpret_cast<uint32_t *>(static_cast<uint8_t *>(ws) + pl.off_dc);
    if (n_out) KC_CUDA_TRY(c, super_gather(pl, ws, tk, tc, dk, dc, c->n_sms, s));
    ext_e[0].reset();
    ext_e[1].reset();
    KC_TRY(make_run(c, s, n_out, run));
    if (n_out) {
        KC_CUDA_TRY(c, cudaMemcpyAsync((*run)->d_keys, dk, n_out * c->W * 8, cudaMemcpyDeviceToDevice, s));
        KC_CUDA_TRY(c, cudaMemcpyAsync((*run)->d_counts, dc, n_out * 4, cudaMemcpyDeviceToDevice, s));
    }
    return KC_OK;
}

// kc_stats' per-stage fields of a count whose stage i took ms[i], moving bytes[i] in launches[i]
// kernels; the dominant stage is the slowest of stages 0 .. n_dom - 1. st.ms_total is set already.
void stage_stats(kc_stats &st, int n_stages, const float *ms, const uint64_t *bytes, const uint32_t *launches, int n_dom) {
    st.n_stages = (uint32_t)n_stages;
    for (int i = 0; i < 8; i++) { st.ms_stage[i] = ms[i]; st.stage_bytes[i] = bytes[i]; st.stage_launches[i] = launches[i]; }
    int dom = 0;
    for (int i = 1; i < n_dom; i++)
        if (st.ms_stage[i] > st.ms_stage[dom]) dom = i;
    st.dominant_stage = (uint32_t)dom;
    st.ms_dominant = st.ms_stage[dom];
    st.dominant_bytes = st.stage_bytes[dom];
    st.dominant_launches = st.stage_launches[dom] ? st.stage_launches[dom] : 1;
    st.ms_extract = st.ms_stage[0];
    st.ms_emit = n_stages ? st.ms_stage[n_stages - 1] : 0;
    st.ms_count = st.ms_total - st.ms_extract - st.ms_emit;
}

// What a chunk is re-counted with when method m could not take it (input far from the plan's
// assumptions): the super-window path's lists or sub-buckets overflowed -> the partitioned path,
// which sizes everything from exact histograms; a sub-bucket arrangement the placement path cannot
// take, or a full hash table -> sort + run-length.
uint32_t fallback(const kc_ctx *c, uint32_t m) {
    return m == KC_COUNT_SUPER && hash_ok(c) ? KC_COUNT_HASH : KC_COUNT_SORT;
}

int count_finish_method(kc_ctx *c, Pending &p, cudaStream_t s, RunPtr *out);

// Wait for the queued kernels, build the run, record stage timings.
int count_finish_impl(kc_ctx *c, Pending &p, const void *d_reads, uint64_t n_bytes, cudaStream_t s, RunPtr *out) {
    KC_CUDA_TRY(c, cudaStreamSynchronize(s));
    memcpy(c->last_scal, p.h_scal, sizeof c->last_scal);
    while (true) {                                // until the path the chunk was counted by gives a run
        KC_TRY(count_finish_method(c, p, s, out));
        if (*out) break;
        pending_release(s, p);
        KC_TRY(count_enqueue(c, p, d_reads, n_bytes, s, fallback(c, p.method)));
        KC_CUDA_TRY(c, cudaStreamSynchronize(s));
    }
    const uint32_t used = p.method;
    if (used != KC_COUNT_HASH) {                  // kc_place_next_run is one-shot: a chunk that took another path disarms it too
        std::lock_guard<std::mutex> g(c->mu);
        c->place.set = false;
    }
    const int n_stages = p.n_ev;                  // the last stage (emit) ends at the event recorded now
    KC_CUDA_TRY(c, cudaEventRecord(p.ev[p.n_ev], s));
    KC_CUDA_TRY(c, cudaEventSynchronize(p.ev[p.n_ev]));
    std::lock_guard<std::mutex> g(c->mu);
    kc_stats &st = c->stats;
    st.chunks++;
    st.reads += p.n_reads;
    st.kmer_slots += p.n_slots;
    const uint64_t invalid = p.h_scal[SC_INVALID];
    const uint64_t nv = p.n_slots - invalid, U = (*out)->n;
    const uint64_t in_bytes = p.n_reads * c->cfg.read_len, Kb = 8ull * c->W;
    st.kmers_valid += nv;
    st.distinct_last = (*out)->n - (*out)->skip;
    st.method_used = used;
    float ms[8] = {0};
    uint64_t b[8] = {0};
    uint32_t l[8] = {0};
    for (int i = 0; i < n_stages; i++) cudaEventElapsedTime(&ms[i], p.ev[i], p.ev[i + 1]);
    cudaEventElapsedTime(&st.ms_total, p.ev[0], p.ev[n_stages]);
    // algorithmic bytes per stage: what the stage must read and write once
    if (used == KC_COUNT_SORT && p.n_slots) {
        const uint64_t N = p.n_slots;
        b[0] = in_bytes + Kb * N;                         l[0] = 1;
        b[1] = Kb * N;                                    l[1] = 2;
        b[2] = (uint64_t)p.n_passes * 2 * Kb * N;         l[2] = (uint32_t)p.n_passes;
        b[3] = Kb * N + U * (Kb + 4);                     l[3] = 1;
        b[4] = U * (2 * Kb + 8);                          l[4] = 1;
    } else if (used == KC_COUNT_HASH && p.n_slots) {
        b[0] = in_bytes;                                  l[0] = 1;   // + a one-block scan
        b[1] = in_bytes + Kb * nv;                        l[1] = 1;
        b[2] = Kb * nv;                                   l[2] = 1;   // + a one-block scan
        b[3] = 2 * Kb * nv;                               l[3] = 1;
        b[4] = Kb * nv + (Kb + 4) * U;                    l[4] = 1;   // + a one-block scan
        b[5] = 2 * (Kb + 4) * U;                          l[5] = 1;
    } else if (used == KC_COUNT_SUPER && p.n_slots) {
        const uint64_t rec = c->last_scal[SW_RECORDS] * 16ull * c->W, ub = U * (Kb + 4);
        b[0] = in_bytes + rec;                            l[0] = 1;   // S1 scatter
        b[1] = rec + ub;                                  l[1] = 1;   // S2 count
        b[2] = 2 * ub;                                    l[2] = 1;   // S3a (+ plan)
        b[3] = U * Kb;                                    l[3] = 1;   // level-2 histogram (+ scan)
        b[4] = 2 * ub;                                    l[4] = 1;   // S3b
        b[5] = 2 * ub;                                    l[5] = 1;   // S3c
    } else if (used == KC_COUNT_PLACE && p.n_slots) {
        const uint64_t N = p.n_slots, nb = N * (Kb + 4), ub = U * (Kb + 4);
        b[0] = in_bytes + Kb * N;                         l[0] = 1;   // extract: a key per slot
        b[1] = 8 * N + 4 * N;                             l[1] = 1;   // leading word in, count out
        b[2] = 2 * nb;                                    l[2] = 1;   // S3a (+ plan)
        b[3] = 8 * N;                                     l[3] = 1;   // level-2 histogram (+ scan)
        b[4] = 2 * nb;                                    l[4] = 1;   // S3b
        b[5] = nb + 3 * ub;                               l[5] = 3;   // S3c fold, offsets, gather
    } else if (used == KC_COUNT_HASH_GLOBAL && p.n_slots) {
        b[0] = p.table.capacity * 16;                     l[0] = 1;
        b[1] = in_bytes + nv * 16;                        l[1] = 1;   // SURVEY 8(d) terms
        b[2] = p.table.capacity * 16 + U * 12 * 17;       l[2] = 10;
    }
    // every stage of the super-window and placement paths is a kernel of the path; elsewhere the emit stage is not
    const bool all_kernels = used == KC_COUNT_SUPER || used == KC_COUNT_PLACE;
    stage_stats(st, n_stages, ms, b, l, all_kernels ? n_stages : n_stages - 1);
    return KC_OK;
}

int count_finish(kc_ctx *c, Pending &p, const void *d_reads, uint64_t n_bytes, cudaStream_t s, kc_run **out) {
    *out = nullptr;
    if (!p.active) return c->set_error(KC_ERR_STATE, "no chunk queued");
    RunPtr r;
    const int rc = count_finish_impl(c, p, d_reads, n_bytes, s, &r);
    pending_release(s, p);
    if (rc == KC_OK) *out = r.release();
    return rc;
}

// Super-window path, after S1..S3b have drained: the host knows |D| now, and S3c writes the run.
// h_scal[SW_FAIL] set on return: a list or a sub-bucket overflowed, no run.
int count_finish_super(kc_ctx *c, Pending &p, cudaStream_t s, RunPtr *out) {
    if (p.h_scal[SW_FAIL]) return KC_OK;
    const bool dup = p.h_scal[SW_OVF] != 0 || env_force_dup();
    RunPtr r;
    KC_TRY(super_emit(c, p.splan, p.splan, p.ws_super, p.d_scal, p.h_scal, dup, p.h_scal[SW_D], s, &r));
    memcpy(c->last_scal, p.h_scal, sizeof c->last_scal);
    {
        std::lock_guard<std::mutex> g(c->mu);
        c->stats.launches += dup ? 3 : 1;
    }
    if (!p.h_scal[SW_FAIL]) *out = std::move(r);
    return KC_OK;
}

// strict mode: empty slots were counted as key 0; if nothing real is left there, hide that record
int strict_hide_zero(kc_ctx *c, Pending &p, kc_run *r, cudaStream_t s) {
    if (!(c->strict && r->n && p.h_scal[SC_INVALID])) return KC_OK;
    uint64_t k0[kMaxWords] = {0};
    uint32_t c0 = 0;
    KC_CUDA_TRY(c, cudaMemcpyAsync(k0, r->d_keys, c->W * 8, cudaMemcpyDeviceToHost, s));
    KC_CUDA_TRY(c, cudaMemcpyAsync(&c0, r->d_counts, 4, cudaMemcpyDeviceToHost, s));
    KC_CUDA_TRY(c, cudaStreamSynchronize(s));
    bool zero = true;
    for (int w = 0; w < c->W; w++) zero = zero && k0[w] == 0;
    if (zero && c0 == 0) r->skip = 1;
    return KC_OK;
}

// Key-placement path, after the extraction and S3a..S3b have drained: S3c sorts and folds every
// sub-bucket into the level-1 buffer (dead by now), a scan gives the survivors' offsets, a gather
// writes the run. Empty slots were placed as key 0 and are taken off that record's count.
// h_scal[SW_FAIL] set on return: a sub-bucket arrangement the path cannot take, no run.
int count_finish_place(kc_ctx *c, Pending &p, cudaStream_t s, RunPtr *out) {
    if (p.h_scal[SW_FAIL]) return KC_OK;
    RunPtr r;
    KC_TRY(super_emit(c, p.splan, p.splan, p.ws_super, p.d_scal, p.h_scal, true, 0, s, &r));
    memcpy(c->last_scal, p.h_scal, sizeof c->last_scal);
    if (p.h_scal[SW_FAIL]) return KC_OK;
    if (r->n && p.h_scal[SC_INVALID]) KC_CUDA_TRY(c, place_fix_zero(c->W, r->d_keys, r->d_counts, &p.d_scal[SC_INVALID], s));
    {
        std::lock_guard<std::mutex> g(c->mu);
        c->stats.launches += 4;
    }
    KC_TRY(strict_hide_zero(c, p, r.get(), s));
    *out = std::move(r);
    return KC_OK;
}

int count_finish_partition(kc_ctx *c, Pending &p, cudaStream_t s, RunPtr *out) {
    const uint64_t U = p.h_scal[SC_UNIQUE];
    const int sig = c->W == 1 ? 64 - static_zero_bits(c) : 64;
    const int target = c->cfg.table_slots ? (int)c->cfg.table_slots : 0;
    uint32_t n_sub = 0, prefix_bits = 0;
    const uint32_t *d_off = nullptr;
    if (U) partition_plan_info(p.n_slots, sig, target, p.ws_part, &n_sub, &prefix_bits, &d_off);
    RunPtr r;
    {
        std::lock_guard<std::mutex> g(c->mu);
        if (c->place.set && U > 0 && U <= c->place.cap && n_sub + 1 <= c->place.cap_ranges) {
            r = RunPtr(new kc_run(), RunFree{c});
            r->W = c->W;
            r->n = U;
            r->d_keys = c->place.keys;
            r->d_counts = c->place.counts;
            r->d_sub_off = c->place.offs;
            r->placed = true;
        }
        c->place.set = false;                    // one-shot, whether it fits or not
    }
    if (!r) KC_TRY(make_run(c, s, U, &r));
    if (U) {
        KC_CUDA_TRY(c, partition_gather(c->W, p.n_slots, sig, target, p.uniq, p.counts, p.ws_part, r->d_keys, r->d_counts, s));
        r->n_sub = n_sub;
        r->prefix_bits = prefix_bits;
        if (!r->placed) {
            void *mem = nullptr;
            KC_TRY(dev_alloc(c, s, (uint64_t)(n_sub + 1) * 4, &mem));
            r->d_sub_off = static_cast<uint32_t *>(mem);
        }
        KC_CUDA_TRY(c, cudaMemcpyAsync(r->d_sub_off, d_off, (uint64_t)(n_sub + 1) * 4, cudaMemcpyDeviceToDevice, s));
        std::lock_guard<std::mutex> g(c->mu);
        c->stats.launches += 1;
    }
    *out = std::move(r);
    return KC_OK;
}

int count_finish_sort(kc_ctx *c, Pending &p, cudaStream_t s, RunPtr *out) {
    const uint64_t U = p.h_scal[SC_UNIQUE];
    RunPtr r;
    KC_TRY(make_run(c, s, U, &r));
    if (U) {
        KC_CUDA_TRY(c, cudaMemcpyAsync(r->d_keys, p.uniq, U * c->W * 8, cudaMemcpyDeviceToDevice, s));
        KC_CUDA_TRY(c, starts_to_counts(p.starts, r->d_keys, c->W, U, &p.d_scal[SC_INVALID], r->d_counts, s));
        std::lock_guard<std::mutex> g(c->mu);
        c->stats.launches += 1;
    }
    // strict mode: empty slots were sorted in as key 0; if nothing real is left there, hide that record
    KC_TRY(strict_hide_zero(c, p, r.get(), s));
    *out = std::move(r);
    return KC_OK;
}

int count_finish_hash_global(kc_ctx *c, Pending &p, cudaStream_t s, RunPtr *out) {
    const uint64_t U = p.h_scal[SC_SIDE + 3] + (p.h_scal[SC_SIDE + 0] ? 1 : 0);
    RunPtr ra, rb;
    KC_TRY(make_run(c, s, U, &ra));
    KC_TRY(make_run(c, s, U, &rb));
    int launches = 0;
    KC_CUDA_TRY(c, hash_compact(p.table, ra->d_keys, ra->d_counts, &p.d_scal[SC_HASHNUM], s, &launches));
    const uint64_t ws_bytes = sort_workspace_bytes(U, 1);
    DevBuf ws(s);
    KC_TRY(ws.alloc(c, ws_bytes));
    uint64_t *sk = nullptr;
    uint32_t *sv = nullptr;
    KC_CUDA_TRY(c, radix_sort(ra->d_keys, rb->d_keys, ra->d_counts, rb->d_counts, U, 1, static_zero_bits(c),
                              SortWorkspace{ws.get(), ws_bytes}, s, &sk, &sv, &launches, nullptr, nullptr));
    {
        std::lock_guard<std::mutex> g(c->mu);
        c->stats.launches += launches;
    }
    *out = std::move(sk == ra->d_keys ? ra : rb);   // (the workspace, then the other run, go at the return)
    return KC_OK;
}

// The run of a drained chunk, built by the path it was counted by; none (and KC_OK) if that path
// could not take the chunk.
int count_finish_method(kc_ctx *c, Pending &p, cudaStream_t s, RunPtr *out) {
    if (p.n_slots == 0) return make_run(c, s, 0, out);
    const bool table_full = p.h_scal[SC_SIDE + 1] != 0;
    switch (p.method) {
    case KC_COUNT_SUPER: return count_finish_super(c, p, s, out);
    case KC_COUNT_PLACE: return count_finish_place(c, p, s, out);
    case KC_COUNT_HASH: return table_full ? KC_OK : count_finish_partition(c, p, s, out);
    case KC_COUNT_HASH_GLOBAL: return table_full ? KC_OK : count_finish_hash_global(c, p, s, out);
    default: return count_finish_sort(c, p, s, out);
    }
}

int check_ctx(const kc_ctx *c) { return c ? KC_OK : KC_ERR_ARG; }

void accum_free(kc_ctx *c);

}  // namespace

static int slot_upload_parse(kc_ctx *c, Slot &sl, const void *host_text, uint64_t n_bytes, uint64_t *n_reads,
                             uint64_t *used, uint32_t *fl);

// ---------------------------------------------------------------------- library
extern "C" {

const char *kc_version(void) { return "kc_b200 0.1 (sm_100a)"; }
uint32_t kc_key_words(uint32_t k) { return (k + 31) / 32; }
uint32_t kc_record_size(uint32_t k) { return 8 * kc_key_words(k) + 4; }
uint64_t kc_output_size(uint64_t n_bytes, uint32_t read_len, uint32_t k) {
    if (read_len == 0 || k == 0 || k > read_len) return 0;
    return (n_bytes / read_len) * (uint64_t)(read_len - k + 1) * kc_record_size(k);
}

int kc_create(const kc_config *cfg, kc_ctx **out) {
    if (out) *out = nullptr;
    if (!cfg || !out) { g_create_error = "kc_create: null argument"; return KC_ERR_ARG; }
    kc_config c0{};
    memcpy(&c0, cfg, cfg->struct_size && cfg->struct_size < sizeof(kc_config) ? cfg->struct_size : sizeof(kc_config));
    if (c0.k < 1 || c0.k > 128) { g_create_error = "kc_create: k must be in 1..128 (KMerSizes.h holds 4 words)"; return KC_ERR_ARG; }
    if (c0.read_len < c0.k || c0.read_len > 4096) { g_create_error = "kc_create: read_len must be in k..4096"; return KC_ERR_ARG; }
    if (c0.method > KC_COUNT_PLACE) { g_create_error = "kc_create: unknown method"; return KC_ERR_ARG; }
    if (c0.method == KC_COUNT_HASH && c0.k > 64) { g_create_error = "kc_create: hash counting needs k <= 64"; return KC_ERR_ARG; }
    if (c0.method == KC_COUNT_HASH_GLOBAL && c0.k > 32) { g_create_error = "kc_create: the HBM-resident table needs k <= 32"; return KC_ERR_ARG; }
    cudaError_t e = cudaSetDevice(c0.device);
    if (e != cudaSuccess) { g_create_error = std::string("kc_create: cudaSetDevice failed: ") + cudaGetErrorString(e); return KC_ERR_CUDA; }
    kc_ctx *c = new kc_ctx();
    c->cfg = c0;
    c->W = (int)kc_key_words(c0.k);
    c->S = (int)kc_record_size(c0.k);
    // a canonical key is exactly k bases: KC_CANONICAL implies KC_COMPAT_STRICT
    if (c0.flags & KC_CANONICAL) c->cfg.flags |= KC_COMPAT_STRICT;
    c->strict = (c->cfg.flags & KC_COMPAT_STRICT) != 0;
    c->key_flags = c->cfg.flags & (KC_COMPAT_STRICT | KC_CANONICAL);
    if (const char *v = getenv("KC_TEST_FAIL_ALLOC")) c->fail_alloc_at = strtoull(v, nullptr, 10);
    cudaDeviceGetAttribute(&c->n_sms, cudaDevAttrMultiProcessorCount, c0.device);
    if (c->n_sms <= 0) c->n_sms = 148;
    // keep freed blocks in the stream-ordered pool: chunk after chunk reuses the same arena
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, c0.device) == cudaSuccess) {
        uint64_t thr = UINT64_MAX;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
    }
    // merges, combines and read-backs run while later chunks' kernels fill the SMs from the slot
    // streams (default = least priority): give them the greatest priority so they are not queued behind
    int prio_lo = 0, prio_hi = 0;
    cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
    if (c0.stream) {
        c->stream = static_cast<cudaStream_t>(c0.stream);
    } else {
        e = cudaStreamCreateWithPriority(&c->stream, cudaStreamNonBlocking, prio_hi);
        if (e != cudaSuccess) { g_create_error = std::string("kc_create: stream: ") + cudaGetErrorString(e); delete c; return KC_ERR_CUDA; }
        c->own_stream = true;
    }
    if (cudaStreamCreateWithPriority(&c->copy_stream, cudaStreamNonBlocking, prio_hi) != cudaSuccess) {
        g_create_error = "kc_create: copy stream"; kc_destroy(c); return KC_ERR_CUDA;
    }
    uint32_t ns = c0.n_slots ? c0.n_slots : 2;
    if (ns > 64) ns = 64;
    c->slots.resize(ns);
    if (c0.max_chunk_bytes) {
        for (auto &sl : c->slots) {
            sl.cap = (c0.max_chunk_bytes + 255) & ~255ull;
            if (cudaMallocHost(&sl.h_in, sl.cap) != cudaSuccess || cudaMalloc(&sl.d_in, sl.cap + 256) != cudaSuccess ||
                cudaStreamCreateWithFlags(&sl.stream, cudaStreamNonBlocking) != cudaSuccess) {
                g_create_error = "kc_create: slot buffers: out of memory";
                kc_destroy(c);
                return KC_ERR_NOMEM;
            }
        }
    }
    *out = c;
    return KC_OK;
}

void kc_destroy(kc_ctx *c) {
    if (!c) return;
    cudaSetDevice(c->cfg.device);
    cudaDeviceSynchronize();
    for (auto &sl : c->slots) {
        pending_release(sl.stream ? sl.stream : c->stream, sl.pend);
        pending_destroy(sl.pend);
        if (sl.h_in) cudaFreeHost(sl.h_in);
        if (sl.d_in) cudaFree(sl.d_in);
        if (sl.d_text) cudaFree(sl.d_text);
        if (sl.stream) cudaStreamDestroy(sl.stream);
    }
    pending_release(c->stream, c->direct);
    pending_destroy(c->direct);
    accum_free(c);
    if (c->own_stream) cudaStreamDestroy(c->stream);
    if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
    if (c->copy_buf) cudaFree(c->copy_buf);
    delete c;
}

const char *kc_last_error(const kc_ctx *c) { return c ? c->err : g_create_error.c_str(); }

int kc_sync(kc_ctx *c) {
    KC_TRY(check_ctx(c));
    KC_CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    for (auto &sl : c->slots)
        if (sl.stream) KC_CUDA_TRY(c, cudaStreamSynchronize(sl.stream));
    return KC_OK;
}

int kc_stats_get(kc_ctx *c, kc_stats *out) {
    KC_TRY(check_ctx(c));
    if (!out) return c->set_error(KC_ERR_ARG, "null stats");
    std::lock_guard<std::mutex> g(c->mu);
    *out = c->stats;
    return KC_OK;
}

int kc_debug_scalars(kc_ctx *c, uint64_t *out16) {
    KC_TRY(check_ctx(c));
    if (!out16) return c->set_error(KC_ERR_ARG, "null out");
    std::lock_guard<std::mutex> g(c->mu);
    for (int i = 0; i < SC_COUNT; i++) out16[i] = c->last_scal[i];
    return KC_OK;
}

int kc_host_alloc(kc_ctx *c, uint64_t bytes, void **out) {
    KC_TRY(check_ctx(c));
    if (!out) return c->set_error(KC_ERR_ARG, "null out");
    if (cudaMallocHost(out, bytes ? bytes : 16) != cudaSuccess) {
        cudaGetLastError();
        return c->set_error(KC_ERR_NOMEM, "pinned allocation of %llu bytes failed", (unsigned long long)bytes);
    }
    return KC_OK;
}
int kc_host_free(kc_ctx *c, void *p) {
    KC_TRY(check_ctx(c));
    if (p) KC_CUDA_TRY(c, cudaFreeHost(p));
    return KC_OK;
}

}  // extern "C"

// -------------------------------------------------------------------- accumulate
namespace {

void accum_free(kc_ctx *c) {
    kc_ctx::Accum &a = c->acc;
    for (int i = 0; i < 8; i++)
        if (a.peer_ipc[i] && a.peer_ws[i]) cudaIpcCloseMemHandle(a.peer_ws[i]);
    if (a.d_all_hist) cudaFree(a.d_all_hist);
    if (a.ws) cudaFree(a.ws);
    if (a.h_sc) cudaFreeHost(a.h_sc);
    for (auto &e : a.ev) if (e) cudaEventDestroy(e);
    for (auto &e : a.sc_ev) if (e) cudaEventDestroy(e);
    a = kc_ctx::Accum();                     // (frees the parts)
}

// Counts what the bins hold into one run (S2 .. S3c) and empties them. All slot streams are
// drained first. An empty accumulator gives an empty run. *run: the run already allocated, if
// any (its arrays were the second record buffer); dup_known: force_dup is the decision; ext_e:
// see super_emit.
int accum_finish(kc_ctx *c, bool force_dup, RunPtr *run, bool dup_known = false, DevBuf *ext_e = nullptr);

int accum_count(kc_ctx *c, RunPtr *out) {
    kc_ctx::Accum &a = c->acc;
    cudaStream_t s = c->stream;
    for (auto &sl : c->slots)
        if (sl.stream) KC_CUDA_TRY(c, cudaStreamSynchronize(sl.stream));
    if (a.fresh) return make_run(c, s, 0, out);
    Trace tr;
    KC_CUDA_TRY(c, cudaEventRecord(a.ev[0], s));
    if (tr.on) { cudaStreamSynchronize(s); tr.mark("flush: S1 drained"); }
    if (!a.pl.ext_e) {
        KC_CUDA_TRY(c, super_count(a.pl, !c->strict, a.ws, a.d_sc, c->n_sms, s, &a.ev[1]));
        return accum_finish(c, false, out);
    }
    // S2 first: once the number of distinct records is known the run is allocated with exactly that
    // size and serves as the second record buffer (E) of S3a/S3b before S3c sorts the records into it
    KC_CUDA_TRY(c, super_count_bins(a.pl, !c->strict, a.ws, a.d_sc, c->n_sms, s));
    KC_CUDA_TRY(c, cudaEventRecord(a.ev[1], s));
    KC_CUDA_TRY(c, cudaMemcpyAsync(a.h_sc, a.d_sc, SC_COUNT * 8, cudaMemcpyDeviceToHost, s));
    KC_CUDA_TRY(c, cudaStreamSynchronize(s));
    tr.mark("flush: S2 count");
    if (a.h_sc[SW_FAIL])
        return c->set_error(KC_ERR_CAPACITY, "accumulated input does not fit the plan (fail bits %llu): flush more often or "
                            "raise the expected read count", (unsigned long long)a.h_sc[SW_FAIL]);
    const uint64_t n_d = a.h_sc[SW_D];
    const bool env_dup = env_force_dup();
    const bool dup = env_dup || a.h_sc[SW_OVF] != 0;
    DevBuf e[2] = {DevBuf(s), DevBuf(s)};          // if records may repeat, E is this flush's own allocation
    if (!dup) {
        KC_TRY(make_run(c, s, n_d, out));
        a.pl.ext_ek = (*out)->d_keys;
        a.pl.ext_ec = (*out)->d_counts;
    } else {
        KC_TRY(e[0].alloc(c, n_d * c->W * 8 + 64));
        KC_TRY(e[1].alloc(c, n_d * 4 + 64));
        a.pl.ext_ek = e[0].get<uint64_t>();
        a.pl.ext_ec = e[1].get<uint32_t>();
    }
    const cudaError_t err = super_place(a.pl, a.ws, a.d_sc, c->n_sms, s, &a.ev[2]);
    int rc = err == cudaSuccess ? KC_OK : c->set_error(KC_ERR_CUDA, "super_place: %s", cudaGetErrorString(err));
    if (rc == KC_OK) {
        if (tr.on) { cudaStreamSynchronize(s); tr.mark("flush: alloc + S3a/H2/S3b"); }
        rc = accum_finish(c, dup, out, true, dup ? e : nullptr);
        tr.mark("flush: S3c + emit + reset");
        if (tr.on) fprintf(stderr, "kc trace: records D %llu, overflow %llu, big ranges %llu (%llu records), aborts %llu, dup %d\n",
                           (unsigned long long)c->last_scal[SW_D], (unsigned long long)c->last_scal[SW_OVF], (unsigned long long)c->last_scal[SW_BIG],
                           (unsigned long long)c->last_scal[SW_BIG_RECORDS], (unsigned long long)c->last_scal[SW_ABORTS], (int)dup);
    }
    a.pl.ext_ek = nullptr;                         // E is attached for this flush only
    a.pl.ext_ec = nullptr;
    return rc;
}

int accum_finish(kc_ctx *c, bool force_dup, RunPtr *run, bool dup_known, DevBuf *ext_e) {
    kc_ctx::Accum &a = c->acc;
    cudaStream_t s = c->stream;
    KC_CUDA_TRY(c, cudaMemcpyAsync(a.h_sc, a.d_sc, SC_COUNT * 8, cudaMemcpyDeviceToHost, s));
    KC_CUDA_TRY(c, cudaStreamSynchronize(s));
    if (a.h_sc[SW_FAIL])
        return c->set_error(KC_ERR_CAPACITY, "accumulated input does not fit the plan (fail bits %llu): flush more often or "
                            "raise the expected read count", (unsigned long long)a.h_sc[SW_FAIL]);
    // exchange: this rank's records are the sub-buckets it pulled (n_recv), and they can only repeat if
    // some rank used its overflow list (those records are counted where they are, not by the bin's owner)
    const uint64_t n_d = a.xchg ? a.x_info.n_recv : a.h_sc[SW_D];
    const bool env_dup = env_force_dup();
    const bool dup = dup_known ? force_dup
                               : (env_dup || (a.xchg ? (force_dup && a.x_info.any_ovf != 0) : (force_dup || a.h_sc[SW_OVF] != 0)));
    SuperPlan fpl = a.pl;                                   // exchange: the S3c variant is the device plan's choice
    if (a.xchg && a.x_info.fin_large) super_use_large_finish(&fpl);
    KC_TRY(super_emit(c, a.pl, fpl, a.ws, a.d_sc, a.h_sc, dup, n_d, s, run, ext_e));
    KC_CUDA_TRY(c, cudaEventRecord(a.ev[5], s));
    KC_CUDA_TRY(c, cudaStreamSynchronize(s));
    if (a.h_sc[SW_FAIL])
        return c->set_error(KC_ERR_CAPACITY, "a key range of the accumulated input does not fit shared memory (fail bits %llu)",
                            (unsigned long long)a.h_sc[SW_FAIL]);
    const uint64_t U = (*run)->n;
    {
        std::lock_guard<std::mutex> g(c->mu);
        kc_stats &st = c->stats;
        memcpy(c->last_scal, a.h_sc, sizeof c->last_scal);
        const uint64_t Kb = 8ull * c->W, ub = U * (Kb + 4), rec = a.h_sc[SW_RECORDS] * 16ull * c->W;
        st.chunks++;
        st.kmer_slots += a.windows;
        st.kmers_valid += a.windows - a.h_sc[SW_INVALID];
        st.reads += a.reads;
        st.distinct_last = U;
        st.method_used = KC_COUNT_SUPER;
        st.launches += dup ? 11 : 9;
        float ms[8] = {0};
        a.ms_scatter = 0;                                    // summed over the chunks' S1 launches (all complete by now)
        for (uint64_t i = 0; i < a.n_scatter; i++) {
            float t = 0;
            if (cudaEventElapsedTime(&t, a.sc_ev[2 * i], a.sc_ev[2 * i + 1]) == cudaSuccess) a.ms_scatter += t;
        }
        cudaGetLastError();
        ms[0] = a.ms_scatter;
        for (int i = 1; i < 6; i++) cudaEventElapsedTime(&ms[i], a.ev[i - 1], a.ev[i]);
        st.ms_total = 0;
        for (int i = 0; i < 6; i++) st.ms_total += ms[i];
        const uint64_t b[8] = {a.reads * c->cfg.read_len + rec, rec + ub, 2 * ub, U * Kb, 2 * ub, 2 * ub};
        const uint32_t l[8] = {(uint32_t)a.n_scatter, 1, 1, 1, 1, 1};
        stage_stats(st, 6, ms, b, l, 6);
    }
    // Bins sized for the wrong redundancy cost S2 a second and third pass over most bins (too many
    // distinct keys for the table) or many nearly empty units. Now that the bins are empty and the
    // ratio is known, later flushes of this accumulator get bins of the right size (same workspace
    // if it fits, a larger one otherwise). Not with an explicit table_slots, not in exchange mode
    // (the ranks must plan alike).
    if (!a.xchg && c->cfg.table_slots == 0 && a.windows > (1u << 20) && U) {
        const double per_key = (double)a.windows / (double)U;
        double occ = 2200.0 * per_key;
        occ = occ > 8192.0 ? 8192.0 : (occ < 1024.0 ? 1024.0 : occ);
        const uint32_t want = ((uint32_t)occ + 255u) & ~255u;
        const uint32_t have = (uint32_t)((a.max_windows + a.pl.n_bins - 1) / a.pl.n_bins);
        if (want < have * 0.75 || want > have * 1.5) {
            SuperPlan np;
            if (super_plan(c->cfg.k, c->cfg.read_len, c->key_flags, a.max_windows, want, &np, 0.0, c->cfg.distinct_hint, true)) {
                bool ok = true;
                if (np.ws_bytes > a.ws_bytes) {
                    KC_CUDA_TRY(c, cudaStreamSynchronize(s));
                    void *nw = nullptr;
                    cudaFree(a.ws);
                    a.ws = nullptr;
                    a.ws_bytes = 0;
                    if (cudaMalloc(&nw, np.ws_bytes) != cudaSuccess) {
                        cudaGetLastError();
                        ok = cudaMalloc(&nw, a.pl.ws_bytes) == cudaSuccess;      // back to the old plan
                        if (!ok) return c->set_error(KC_ERR_NOMEM, "accumulator workspace of %llu bytes", (unsigned long long)a.pl.ws_bytes);
                        a.ws = nw;
                        a.ws_bytes = a.pl.ws_bytes;
                        ok = false;
                    } else {
                        a.ws = nw;
                        a.ws_bytes = np.ws_bytes;
                    }
                }
                if (ok) a.pl = np;
                a.d_sc = reinterpret_cast<unsigned long long *>(static_cast<uint8_t *>(a.ws) + a.pl.off_sc);
            }
        }
    }
    // empty bins for whatever comes next
    KC_CUDA_TRY(c, super_reset(a.pl, a.ws, a.d_sc, s));
    KC_CUDA_TRY(c, cudaStreamSynchronize(s));
    a.fresh = true;
    a.windows = a.reads = 0;
    a.ovf_reserved = 0;
    a.ms_scatter = 0;
    a.n_scatter = 0;
    return KC_OK;
}

// Room check before a chunk of n_reads joins the bins: the chunk may need up to one record per
// window in the overflow list (no read is ever dropped); if that or the plan's window budget is
// not there, what has been accumulated is counted into a part first.
int accum_make_room(kc_ctx *c, uint64_t n_reads) {
    kc_ctx::Accum &a = c->acc;
    const uint64_t nk = c->cfg.read_len - c->cfg.k + 1, w = n_reads * nk;
    if (w > a.max_windows)
        return c->set_error(KC_ERR_CAPACITY, "chunk of %llu reads exceeds what the accumulator was planned for", (unsigned long long)n_reads);
    if (a.windows + w > a.max_windows) {
        if (a.xchg) return c->set_error(KC_ERR_CAPACITY, "more reads than kc_xchg_begin planned for (%llu k-mer slots)", (unsigned long long)a.max_windows);
        RunPtr part;
        KC_TRY(accum_count(c, &part));
        a.parts.push_back(std::move(part));
    }
    return KC_OK;
}

// S1 of one chunk on stream s, timed
int accum_scatter(kc_ctx *c, const void *d_reads, uint64_t n_reads, cudaStream_t s) {
    kc_ctx::Accum &a = c->acc;
    if (n_reads == 0) return KC_OK;
    while (a.sc_ev.size() < 2 * (a.n_scatter + 1)) {
        cudaEvent_t e = nullptr;
        KC_CUDA_TRY(c, cudaEventCreate(&e));
        a.sc_ev.push_back(e);
    }
    KC_CUDA_TRY(c, cudaEventRecord(a.sc_ev[2 * a.n_scatter], s));
    KC_CUDA_TRY(c, super_scatter(a.pl, d_reads, n_reads, a.ws, a.d_sc, c->n_sms, s));
    KC_CUDA_TRY(c, cudaEventRecord(a.sc_ev[2 * a.n_scatter + 1], s));
    const uint64_t nk = c->cfg.read_len - c->cfg.k + 1;
    a.fresh = false;
    a.windows += n_reads * nk;
    a.reads += n_reads;
    a.n_scatter++;
    return KC_OK;
}

}  // namespace

extern "C" {

static int accum_begin_impl(kc_ctx *c, uint64_t expected_reads, bool exchange, uint32_t n_ranks = 1);

int kc_accum_begin(kc_ctx *c, uint64_t expected_reads) {
    KC_TRY(check_ctx(c));
    return accum_begin_impl(c, expected_reads, false);
}

// exchange: the record buffers also take what the peers send, which is this rank's share of the
// key space only on average (ranges are cut at 1/1024 of the key space): a quarter more room
static int accum_begin_impl(kc_ctx *c, uint64_t expected_reads, bool exchange, uint32_t n_ranks) {
    std::lock_guard<std::recursive_mutex> dg(c->direct_mu);
    cudaSetDevice(c->cfg.device);
    if (!super_ok(c)) {
        SuperPlan pl;
        if (c->W <= 2 && super_plan(c->cfg.k, c->cfg.k, c->key_flags, 1, 0, &pl))      // k is fine: the reads are too long
            return c->set_error(KC_ERR_ARG, "accumulating mode: reads of %u bases are too long for the super-window path at k=%u",
                                c->cfg.read_len, c->cfg.k);
        return c->set_error(KC_ERR_ARG, "accumulating mode needs k <= 64 with windows of >= 22 bases (k=%u)", c->cfg.k);
    }
    const uint64_t nk = c->cfg.read_len - c->cfg.k + 1;
    uint64_t chunk_reads = c->cfg.max_chunk_bytes / c->cfg.read_len;
    if (expected_reads < chunk_reads) expected_reads = chunk_reads;
    if (expected_reads == 0) return c->set_error(KC_ERR_ARG, "kc_accum_begin: expected_reads and max_chunk_bytes are both 0");
    const uint64_t windows = expected_reads * nk;     // (record offsets are 32-bit: at most 2^32 - 2 DISTINCT keys per flush)
    kc_ctx::Accum &a = c->acc;
    if (a.on && !a.fresh) return c->set_error(KC_ERR_STATE, "kc_accum_begin: reads are accumulated; flush first");
    SuperPlan pl;
    // exchange: a bin collects what ALL ranks put into it, so each rank plans bins 1/n_ranks the size
    uint32_t occ = (uint32_t)c->cfg.table_slots;
    if (exchange && n_ranks > 1) occ = (occ ? occ : 8192u) / n_ranks;
    if (!super_plan(c->cfg.k, c->cfg.read_len, c->key_flags, windows, occ, &pl, exchange ? 0.25 : 0.0, c->cfg.distinct_hint, !exchange))
        return c->set_error(KC_ERR_ARG, "unsupported shape k=%u read_len=%u", c->cfg.k, c->cfg.read_len);
    if (!a.h_sc) {
        KC_CUDA_TRY(c, cudaMallocHost((void **)&a.h_sc, SC_COUNT * 8));
        for (auto &e : a.ev) KC_CUDA_TRY(c, cudaEventCreate(&e));
    }
    if (getenv("KC_DEBUG_PLAN")) {
        size_t fr = 0, tot = 0;
        cudaMemGetInfo(&fr, &tot);
        fprintf(stderr, "kc accumulator: before the workspace %llu of %llu bytes free\n", (unsigned long long)fr, (unsigned long long)tot);
    }
    if (pl.ws_bytes > a.ws_bytes) {
        KC_CUDA_TRY(c, cudaDeviceSynchronize());
        if (a.ws) cudaFree(a.ws);
        a.ws = nullptr;
        a.ws_bytes = 0;
        if (cudaMalloc(&a.ws, pl.ws_bytes) != cudaSuccess) {
            cudaGetLastError();
            return c->set_error(KC_ERR_NOMEM, "accumulator workspace of %llu bytes", (unsigned long long)pl.ws_bytes);
        }
        a.ws_bytes = pl.ws_bytes;
    }
    if (getenv("KC_DEBUG_PLAN"))
        fprintf(stderr, "kc accumulator plan: windows %llu, bins %u x %u records, overflow %llu, D %llu records, ext_e %d, workspace %llu bytes\n",
                (unsigned long long)windows, pl.n_bins, pl.bin_cap, (unsigned long long)pl.ovf_cap, (unsigned long long)pl.d_cap,
                (int)pl.ext_e, (unsigned long long)pl.ws_bytes);
    a.pl = pl;
    a.d_sc = reinterpret_cast<unsigned long long *>(static_cast<uint8_t *>(a.ws) + pl.off_sc);   // (peers read the scalars too)
    a.max_windows = windows;
    a.on = true;
    a.fresh = true;
    a.windows = a.reads = 0;
    a.ovf_reserved = 0;
    KC_CUDA_TRY(c, super_reset(a.pl, a.ws, a.d_sc, c->stream));
    KC_CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    return KC_OK;
}

int kc_accum_add_device(kc_ctx *c, const void *d_reads, uint64_t n_bytes) {
    KC_TRY(check_ctx(c));
    std::lock_guard<std::recursive_mutex> dg(c->direct_mu);
    if (!c->acc.on) return c->set_error(KC_ERR_STATE, "kc_accum_begin first");
    if (n_bytes && (!d_reads || (reinterpret_cast<uintptr_t>(d_reads) & 15)))
        return c->set_error(KC_ERR_ARG, "d_reads must be a 16-byte aligned device pointer");
    cudaSetDevice(c->cfg.device);
    const uint32_t L = c->cfg.read_len;
    const uint64_t n_reads = n_bytes / L;
    // pieces the plan can take in one go (and whose worst-case overflow fits the list)
    const uint64_t nk = L - c->cfg.k + 1;
    uint64_t piece = std::min<uint64_t>(1ull << 30, c->acc.max_windows) / nk;
    piece -= piece % 16;
    if (piece == 0) return c->set_error(KC_ERR_CAPACITY, "accumulator too small for any read");
    for (uint64_t r0 = 0; r0 < n_reads; r0 += piece) {
        const uint64_t nr = std::min(piece, n_reads - r0);
        KC_TRY(accum_make_room(c, nr));
        KC_TRY(accum_scatter(c, static_cast<const uint8_t *>(d_reads) + r0 * L, nr, c->stream));
    }
    return KC_OK;
}

int kc_accum_submit(kc_ctx *c, uint32_t slot, uint64_t n_bytes) {
    KC_TRY(check_ctx(c));
    if (slot >= c->slots.size() || !c->slots[slot].h_in) return c->set_error(KC_ERR_ARG, "slot %u not available", slot);
    if (n_bytes > c->cfg.max_chunk_bytes) return c->set_error(KC_ERR_CAPACITY, "chunk of %llu bytes exceeds max_chunk_bytes", (unsigned long long)n_bytes);
    std::lock_guard<std::recursive_mutex> dg(c->direct_mu);
    if (!c->acc.on) return c->set_error(KC_ERR_STATE, "kc_accum_begin first");
    cudaSetDevice(c->cfg.device);
    Slot &sl = c->slots[slot];
    const uint64_t n_reads = n_bytes / c->cfg.read_len;
    KC_TRY(accum_make_room(c, n_reads));
    sl.n_bytes = n_bytes;
    if (n_bytes) KC_CUDA_TRY(c, cudaMemcpyAsync(sl.d_in, sl.h_in, n_bytes, cudaMemcpyHostToDevice, sl.stream));
    {
        std::lock_guard<std::mutex> g(c->mu);
        c->stats.h2d_bytes += n_bytes;
    }
    return accum_scatter(c, sl.d_in, n_reads, sl.stream);
}

int kc_accum_submit_fastq(kc_ctx *c, uint32_t slot, const void *host_text, uint64_t n_bytes, uint64_t *consumed,
                          uint32_t *flags) {
    KC_TRY(check_ctx(c));
    if (consumed) *consumed = 0;
    if (flags) *flags = 0;
    if (slot >= c->slots.size() || !c->slots[slot].d_in) return c->set_error(KC_ERR_ARG, "slot %u not available", slot);
    if (n_bytes && !host_text) return c->set_error(KC_ERR_ARG, "null text");
    std::lock_guard<std::recursive_mutex> dg(c->direct_mu);
    if (!c->acc.on) return c->set_error(KC_ERR_STATE, "kc_accum_begin first");
    cudaSetDevice(c->cfg.device);
    Slot &sl = c->slots[slot];
    uint64_t n_reads = 0, used = 0;
    uint32_t fl = 0;
    KC_TRY(slot_upload_parse(c, sl, host_text, n_bytes, &n_reads, &used, &fl));
    if (flags) *flags = fl;
    if (fl) return KC_OK;
    if (consumed) *consumed = used;
    KC_TRY(accum_make_room(c, n_reads));
    sl.n_bytes = n_reads * c->cfg.read_len;
    return accum_scatter(c, sl.d_in, n_reads, sl.stream);
}

int kc_accum_wait(kc_ctx *c, uint32_t slot) {
    KC_TRY(check_ctx(c));
    if (slot >= c->slots.size() || !c->slots[slot].stream) return c->set_error(KC_ERR_ARG, "slot %u not available", slot);
    cudaSetDevice(c->cfg.device);
    KC_CUDA_TRY(c, cudaStreamSynchronize(c->slots[slot].stream));
    return KC_OK;
}

int kc_accum_flush(kc_ctx *c, kc_run **run) {
    KC_TRY(check_ctx(c));
    if (!run) return c->set_error(KC_ERR_ARG, "null run");
    std::lock_guard<std::recursive_mutex> dg(c->direct_mu);
    if (!c->acc.on) return c->set_error(KC_ERR_STATE, "kc_accum_begin first");
    *run = nullptr;
    cudaSetDevice(c->cfg.device);
    kc_ctx::Accum &a = c->acc;
    RunPtr last;
    KC_TRY(accum_count(c, &last));
    if (a.parts.empty()) { *run = last.release(); return KC_OK; }
    std::vector<RunPtr> parts;
    parts.swap(a.parts);
    parts.push_back(std::move(last));
    return merge_owned(c, parts, run);
}

// ------------------------------------------------------------------- multi-GPU
// One context per GPU ("rank"). Every rank accumulates its own reads (kc_accum_add_device /
// kc_accum_submit), counts them locally, and the ranks then exchange DISTINCT (key, count)
// records by key range: rank r ends with the sorted unique records of the r-th key range, the
// artefact is the concatenation in rank order. The exchange is fused into the level-2 scatter
// kernel, whose loads read the peers' HBM over NVLink / NVSwitch.
int kc_xchg_begin(kc_ctx *c, uint32_t rank, uint32_t n_ranks, uint64_t expected_reads) {
    KC_TRY(check_ctx(c));
    if (n_ranks == 0 || n_ranks > 8 || rank >= n_ranks) return c->set_error(KC_ERR_ARG, "kc_xchg_begin: rank %u of %u", rank, n_ranks);
    std::lock_guard<std::recursive_mutex> dg(c->direct_mu);
    KC_TRY(accum_begin_impl(c, expected_reads, true, n_ranks));
    kc_ctx::Accum &a = c->acc;
    if (a.pl.b1 != 10) return c->set_error(KC_ERR_ARG, "kc_xchg_begin: keys of k=%u have too few bits to exchange by range", c->cfg.k);
    a.xchg = true;
    a.rank = rank;
    a.n_ranks = n_ranks;
    a.peer_ws[rank] = a.ws;
    if (!a.d_all_hist) KC_CUDA_TRY(c, cudaMalloc((void **)&a.d_all_hist, 8 * 1024 * 4));
    return KC_OK;
}

int kc_xchg_export(kc_ctx *c, void *handle64) {
    KC_TRY(check_ctx(c));
    if (!handle64 || !c->acc.xchg) return c->set_error(KC_ERR_STATE, "kc_xchg_begin first");
    cudaSetDevice(c->cfg.device);
    cudaIpcMemHandle_t h;
    KC_CUDA_TRY(c, cudaIpcGetMemHandle(&h, c->acc.ws));
    memcpy(handle64, &h, 64);
    return KC_OK;
}

int kc_xchg_import(kc_ctx *c, uint32_t peer, const void *handle64) {
    KC_TRY(check_ctx(c));
    kc_ctx::Accum &a = c->acc;
    if (!handle64 || !a.xchg || peer >= a.n_ranks || peer == a.rank) return c->set_error(KC_ERR_ARG, "kc_xchg_import: bad peer");
    cudaSetDevice(c->cfg.device);
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, 64);
    if (a.peer_ipc[peer] && a.peer_ws[peer]) cudaIpcCloseMemHandle(a.peer_ws[peer]);
    a.peer_ws[peer] = nullptr;
    KC_CUDA_TRY(c, cudaIpcOpenMemHandle(&a.peer_ws[peer], h, cudaIpcMemLazyEnablePeerAccess));
    a.peer_ipc[peer] = true;
    return KC_OK;
}

int kc_xchg_set_peer(kc_ctx *c, uint32_t peer, kc_ctx *peer_ctx) {
    KC_TRY(check_ctx(c));
    kc_ctx::Accum &a = c->acc;
    if (!peer_ctx || !a.xchg || !peer_ctx->acc.xchg || peer >= a.n_ranks)
        return c->set_error(KC_ERR_ARG, "kc_xchg_set_peer: bad peer");
    if (peer_ctx->acc.pl.ws_bytes != a.pl.ws_bytes) return c->set_error(KC_ERR_ARG, "kc_xchg_set_peer: the ranks were planned differently");
    if (peer_ctx->key_flags != c->key_flags)
        return c->set_error(KC_ERR_ARG, "kc_xchg_set_peer: the ranks count different keys (KC_COMPAT_STRICT / KC_CANONICAL)");
    cudaSetDevice(c->cfg.device);
    if (peer_ctx->cfg.device != c->cfg.device) {
        cudaError_t e = cudaDeviceEnablePeerAccess(peer_ctx->cfg.device, 0);
        if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
        else if (e != cudaSuccess) return c->set_error(KC_ERR_CUDA, "cudaDeviceEnablePeerAccess(%d): %s", peer_ctx->cfg.device, cudaGetErrorString(e));
    }
    a.peer_ws[peer] = peer_ctx->acc.ws;
    a.peer_ipc[peer] = false;
    return KC_OK;
}

int kc_xchg_count_local(kc_ctx *c) {
    KC_TRY(check_ctx(c));
    std::lock_guard<std::recursive_mutex> dg(c->direct_mu);
    kc_ctx::Accum &a = c->acc;
    if (!a.xchg) return c->set_error(KC_ERR_STATE, "kc_xchg_begin first");
    cudaSetDevice(c->cfg.device);
    cudaStream_t s = c->stream;
    for (auto &sl : c->slots)
        if (sl.stream) KC_CUDA_TRY(c, cudaStreamSynchronize(sl.stream));
    for (uint32_t i = 0; i < a.n_ranks; i++)
        if (!a.peer_ws[i]) return c->set_error(KC_ERR_STATE, "kc_xchg_count_local: rank %u's workspace is not mapped (kc_xchg_import / kc_xchg_set_peer)", i);
    KC_CUDA_TRY(c, cudaEventRecord(a.ev[0], s));
    KC_CUDA_TRY(c, super_count_bins(a.pl, !c->strict, a.ws, a.d_sc, c->n_sms, s, a.peer_ws, a.rank, a.n_ranks));
    KC_CUDA_TRY(c, cudaEventRecord(a.ev[1], s));
    a.fresh = false;                          // (a rank without reads still takes part in the exchange)
    return KC_OK;
}

int kc_xchg_hist(kc_ctx *c, void **d_hist, void **d_all_hist) {
    KC_TRY(check_ctx(c));
    if (!c->acc.xchg) return c->set_error(KC_ERR_STATE, "kc_xchg_begin first");
    if (d_hist) *d_hist = super_hist1(c->acc.pl, c->acc.ws);
    if (d_all_hist) *d_all_hist = c->acc.d_all_hist;
    return KC_OK;
}

int kc_xchg_group_local(kc_ctx *c) {
    KC_TRY(check_ctx(c));
    std::lock_guard<std::recursive_mutex> dg(c->direct_mu);
    kc_ctx::Accum &a = c->acc;
    if (!a.xchg) return c->set_error(KC_ERR_STATE, "kc_xchg_begin first");
    cudaSetDevice(c->cfg.device);
    KC_CUDA_TRY(c, super_x_local(a.pl, a.ws, a.d_sc, a.d_all_hist, a.rank, a.n_ranks, a.keep_ranges, a.peer_ws, c->n_sms, c->stream));
    KC_CUDA_TRY(c, cudaEventRecord(a.ev[2], c->stream));
    KC_CUDA_TRY(c, cudaEventRecord(a.ev[3], c->stream));
    return KC_OK;
}

int kc_xchg_pull(kc_ctx *c) {
    KC_TRY(check_ctx(c));
    std::lock_guard<std::recursive_mutex> dg(c->direct_mu);
    kc_ctx::Accum &a = c->acc;
    if (!a.xchg) return c->set_error(KC_ERR_STATE, "kc_xchg_begin first");
    for (uint32_t i = 0; i < a.n_ranks; i++)
        if (!a.peer_ws[i]) return c->set_error(KC_ERR_STATE, "kc_xchg_pull: rank %u's workspace is not mapped (kc_xchg_import / kc_xchg_set_peer)", i);
    cudaSetDevice(c->cfg.device);
    KC_CUDA_TRY(c, super_x_pull(a.pl, a.ws, a.d_sc, a.peer_ws, a.rank, a.n_ranks, c->n_sms, c->stream));
    KC_CUDA_TRY(c, cudaEventRecord(a.ev[4], c->stream));
    return KC_OK;
}

int kc_xchg_finish(kc_ctx *c, kc_run **run) {
    KC_TRY(check_ctx(c));
    if (!run) return c->set_error(KC_ERR_ARG, "null run");
    std::lock_guard<std::recursive_mutex> dg(c->direct_mu);
    if (!c->acc.xchg) return c->set_error(KC_ERR_STATE, "kc_xchg_begin first");
    cudaSetDevice(c->cfg.device);
    *run = nullptr;
    KC_CUDA_TRY(c, cudaMemcpyAsync(&c->acc.x_info, super_x_info(c->acc.pl, c->acc.ws), sizeof(SuperXInfo),
                                   cudaMemcpyDeviceToHost, c->stream));
    RunPtr r;
    KC_TRY(accum_finish(c, true, &r));        // (synchronises the stream)
    *run = r.release();
    return KC_OK;
}

int kc_xchg_fix_ranges(kc_ctx *c, int on) {
    KC_TRY(check_ctx(c));
    if (!c->acc.xchg) return c->set_error(KC_ERR_STATE, "kc_xchg_begin first");
    c->acc.keep_ranges = on != 0;
    return KC_OK;
}

int kc_xchg_info(kc_ctx *c, uint32_t *lo, uint64_t *recv_records, uint64_t *remote_records) {
    KC_TRY(check_ctx(c));
    const kc_ctx::Accum &a = c->acc;
    if (!a.xchg) return c->set_error(KC_ERR_STATE, "kc_xchg_begin first");
    if (lo) for (uint32_t i = 0; i <= a.n_ranks; i++) lo[i] = a.x_info.lo[i];
    uint64_t all = 0, remote = 0;
    for (uint32_t s2 = 0; s2 < a.n_ranks; s2++) {
        const uint64_t n = a.x_info.src_range[s2][1] - a.x_info.src_range[s2][0];
        all += n;
        if (s2 != a.rank) remote += n;
    }
    if (recv_records) *recv_records = all;
    if (remote_records) *remote_records = remote;
    return KC_OK;
}

// All ranks in one process: counts what the n contexts have accumulated and leaves rank r's key
// range in runs[r]. Cross-device ordering is by events; nothing waits inside a kernel, so the
// contexts may also share a device (tests).
int kc_xchg_run_all(kc_ctx *const *ctxs, uint32_t n, kc_run **runs) {
    if (!ctxs || !runs || n == 0 || n > 8) return KC_ERR_ARG;
    for (uint32_t r = 0; r < n; r++) {
        if (!ctxs[r] || !ctxs[r]->acc.xchg || ctxs[r]->acc.n_ranks != n || ctxs[r]->acc.rank != r) return KC_ERR_ARG;
        runs[r] = nullptr;
    }
    int rc = KC_OK;
    std::vector<cudaEvent_t> ev(n);
    for (uint32_t r = 0; r < n; r++) {
        cudaSetDevice(ctxs[r]->cfg.device);
        cudaEventCreateWithFlags(&ev[r], cudaEventDisableTiming);
    }
    // every stream waits for the events the other ranks recorded at their current position
    auto barrier = [&]() {
        for (uint32_t r = 0; r < n; r++) { cudaSetDevice(ctxs[r]->cfg.device); cudaEventRecord(ev[r], ctxs[r]->stream); }
        for (uint32_t r = 0; r < n; r++) {
            cudaSetDevice(ctxs[r]->cfg.device);
            for (uint32_t q = 0; q < n; q++)
                if (q != r) cudaStreamWaitEvent(ctxs[r]->stream, ev[q], 0);
        }
    };
    for (uint32_t r = 0; r < n && rc == KC_OK; r++)
        for (uint32_t q = 0; q < n && rc == KC_OK; q++)
            if (q != r) rc = kc_xchg_set_peer(ctxs[r], q, ctxs[q]);
    if (rc == KC_OK) barrier();                     // every rank's bins are complete
    for (uint32_t r = 0; r < n && rc == KC_OK; r++) rc = kc_xchg_count_local(ctxs[r]);
    if (rc == KC_OK) {
        barrier();                                  // the histograms are complete
        for (uint32_t r = 0; r < n; r++) {          // all-gather: rank r copies every rank's histogram
            cudaSetDevice(ctxs[r]->cfg.device);
            for (uint32_t q = 0; q < n; q++)
                cudaMemcpyPeerAsync(ctxs[r]->acc.d_all_hist + q * 1024, ctxs[r]->cfg.device,
                                    super_hist1(ctxs[q]->acc.pl, ctxs[q]->acc.ws), ctxs[q]->cfg.device, 1024 * 4,
                                    ctxs[r]->stream);
        }
    }
    for (uint32_t r = 0; r < n && rc == KC_OK; r++) rc = kc_xchg_group_local(ctxs[r]);
    if (rc == KC_OK) barrier();                     // every rank's grouped array and sub-bucket counts are final
    for (uint32_t r = 0; r < n && rc == KC_OK; r++) rc = kc_xchg_pull(ctxs[r]);
    if (rc == KC_OK) barrier();                     // nobody reads a peer's grouped array any more
    std::vector<RunPtr> got;
    for (uint32_t r = 0; r < n && rc == KC_OK; r++) {
        kc_run *run = nullptr;
        rc = kc_xchg_finish(ctxs[r], &run);
        got.emplace_back(run, RunFree{ctxs[r]});
    }
    for (uint32_t r = 0; r < n; r++) { cudaSetDevice(ctxs[r]->cfg.device); cudaEventDestroy(ev[r]); }
    if (rc == KC_OK)
        for (uint32_t r = 0; r < n; r++) runs[r] = got[r].release();
    return rc;
}

}  // extern "C"

extern "C" {

// ------------------------------------------------------------------------ chunks
int kc_count_device(kc_ctx *c, const void *d_reads, uint64_t n_bytes, kc_run **run) {
    KC_TRY(check_ctx(c));
    std::lock_guard<std::recursive_mutex> dg(c->direct_mu);
    if (!run) return c->set_error(KC_ERR_ARG, "null run");
    *run = nullptr;
    if (n_bytes && (!d_reads || (reinterpret_cast<uintptr_t>(d_reads) & 15)))
        return c->set_error(KC_ERR_ARG, "d_reads must be a 16-byte aligned device pointer");
    cudaSetDevice(c->cfg.device);
    // chunks beyond the sorter's per-call limit are cut into pieces whose runs are merged
    const uint32_t L = c->cfg.read_len;
    const uint64_t nk = L - c->cfg.k + 1;
    uint64_t n_reads = n_bytes / L;
    uint64_t max_reads = kMaxSortKeys / nk;
    max_reads -= max_reads % 16;                      // keep every piece 16-byte aligned
    std::vector<RunPtr> parts;
    for (uint64_t r0 = 0; r0 == 0 || r0 < n_reads; r0 += max_reads) {   // (an empty chunk is one piece too)
        const uint64_t nr = std::min(max_reads, n_reads - r0);
        const uint8_t *ptr = static_cast<const uint8_t *>(d_reads) + r0 * L;
        kc_run *part = nullptr;
        KC_TRY(count_enqueue(c, c->direct, ptr, nr * L, c->stream, pick_method(c)));
        KC_TRY(count_finish(c, c->direct, ptr, nr * L, c->stream, &part));
        parts.emplace_back(part, RunFree{c});
    }
    if (parts.size() == 1) { *run = parts[0].release(); return KC_OK; }
    return merge_owned(c, parts, run);
}

static int parse_fastq_impl(kc_ctx *c, Pending &ar, const void *d_text, uint64_t n_bytes, void *d_reads,
                            uint64_t reads_cap_bytes, cudaStream_t s, uint64_t *n_reads, uint64_t *consumed,
                            uint32_t *flags) {
    if (n_bytes >= (1ull << 32)) return c->set_error(KC_ERR_CAPACITY, "FASTQ chunks must be smaller than 4 GiB");
    if (n_bytes && (reinterpret_cast<uintptr_t>(d_text) & 15)) return c->set_error(KC_ERR_ARG, "d_text must be 16-byte aligned");
    KC_TRY(pending_init(c, ar));
    const uint64_t wsb = fastq_workspace_bytes(n_bytes);
    KC_TRY(arena_reserve(c, ar, arena_round(wsb) + 512, s));
    void *ws = arena_take(ar, wsb);
    unsigned long long *d_out = static_cast<unsigned long long *>(arena_take(ar, 32));
    int launches = 0;
    KC_CUDA_TRY(c, fastq_parse(d_text, n_bytes, c->cfg.read_len, d_reads, reads_cap_bytes / c->cfg.read_len, d_out, ws,
                               s, &launches));
    unsigned long long h[3] = {0, 0, 0};
    KC_CUDA_TRY(c, cudaMemcpyAsync(h, d_out, 24, cudaMemcpyDeviceToHost, s));
    KC_CUDA_TRY(c, cudaStreamSynchronize(s));
    ar.arena_used = 0;
    if (n_reads) *n_reads = h[0];
    if (consumed) *consumed = h[1];
    if (flags) *flags = (uint32_t)h[2];
    std::lock_guard<std::mutex> g(c->mu);
    c->stats.launches += launches;
    return KC_OK;
}

}  // extern "C"

// host text -> the slot's device staging -> parsed into the slot's read buffer (sl.d_in)
static int slot_upload_parse(kc_ctx *c, Slot &sl, const void *host_text, uint64_t n_bytes, uint64_t *n_reads,
                             uint64_t *used, uint32_t *fl) {
    if (n_bytes + 64 > sl.text_cap) {                    // device staging for the raw text, grown on demand
        KC_CUDA_TRY(c, cudaStreamSynchronize(sl.stream));
        if (sl.d_text) cudaFree(sl.d_text);
        sl.d_text = nullptr;
        sl.text_cap = 0;
        const uint64_t want = n_bytes + n_bytes / 8 + 4096;
        if (cudaMalloc(&sl.d_text, want) != cudaSuccess) {
            cudaGetLastError();
            return c->set_error(KC_ERR_NOMEM, "device allocation of %llu bytes for FASTQ text failed", (unsigned long long)want);
        }
        sl.text_cap = want;
    }
    if (n_bytes) KC_CUDA_TRY(c, cudaMemcpyAsync(sl.d_text, host_text, n_bytes, cudaMemcpyHostToDevice, sl.stream));
    KC_TRY(parse_fastq_impl(c, sl.pend, sl.d_text, n_bytes, sl.d_in, c->cfg.max_chunk_bytes, sl.stream, n_reads, used, fl));
    std::lock_guard<std::mutex> g(c->mu);
    c->stats.h2d_bytes += n_bytes;
    return KC_OK;
}

extern "C" {

int kc_parse_fastq_device(kc_ctx *c, const void *d_text, uint64_t n_bytes, void *d_reads, uint64_t reads_cap_bytes,
                          uint64_t *n_reads, uint64_t *consumed, uint32_t *flags) {
    KC_TRY(check_ctx(c));
    std::lock_guard<std::recursive_mutex> dg(c->direct_mu);
    if ((n_bytes && (!d_text || !d_reads))) return c->set_error(KC_ERR_ARG, "null argument");
    if (c->direct.active) return c->set_error(KC_ERR_STATE, "a chunk is in flight on this context");
    cudaSetDevice(c->cfg.device);
    return parse_fastq_impl(c, c->direct, d_text, n_bytes, d_reads, reads_cap_bytes, c->stream, n_reads, consumed, flags);
}

int kc_submit_fastq(kc_ctx *c, uint32_t slot, const void *host_text, uint64_t n_bytes, uint64_t *consumed,
                    uint32_t *flags) {
    KC_TRY(check_ctx(c));
    if (consumed) *consumed = 0;
    if (flags) *flags = 0;
    if (slot >= c->slots.size() || !c->slots[slot].d_in) return c->set_error(KC_ERR_ARG, "slot %u not available", slot);
    if (n_bytes && !host_text) return c->set_error(KC_ERR_ARG, "null text");
    Slot &sl = c->slots[slot];
    if (sl.pend.active) return c->set_error(KC_ERR_STATE, "slot %u already has a chunk in flight", slot);
    cudaSetDevice(c->cfg.device);
    uint64_t n_reads = 0, used = 0;
    uint32_t fl = 0;
    KC_TRY(slot_upload_parse(c, sl, host_text, n_bytes, &n_reads, &used, &fl));
    if (flags) *flags = fl;
    if (fl) return KC_OK;                                // not the shape the device parser handles: nothing submitted
    if (consumed) *consumed = used;
    const uint64_t nk = c->cfg.read_len - c->cfg.k + 1;
    if (n_reads * nk > kMaxSortKeys)
        return c->set_error(KC_ERR_CAPACITY, "chunk holds more than %llu k-mer slots; use a smaller max_chunk_bytes", (unsigned long long)kMaxSortKeys);
    sl.n_bytes = n_reads * c->cfg.read_len;
    return count_enqueue(c, sl.pend, sl.d_in, sl.n_bytes, sl.stream, pick_method(c));
}

int kc_slot_buffer(kc_ctx *c, uint32_t slot, void **ptr, uint64_t *cap) {
    KC_TRY(check_ctx(c));
    if (slot >= c->slots.size() || !c->slots[slot].h_in)
        return c->set_error(KC_ERR_ARG, "slot %u not available (n_slots=%zu, max_chunk_bytes=%llu)", slot,
                            c->slots.size(), (unsigned long long)c->cfg.max_chunk_bytes);
    if (ptr) *ptr = c->slots[slot].h_in;
    if (cap) *cap = c->cfg.max_chunk_bytes;
    return KC_OK;
}

static int submit_from(kc_ctx *c, uint32_t slot, const void *host_src, uint64_t n_bytes) {
    Slot &sl = c->slots[slot];
    if (sl.pend.active) return c->set_error(KC_ERR_STATE, "slot %u already has a chunk in flight", slot);
    if (n_bytes > c->cfg.max_chunk_bytes) return c->set_error(KC_ERR_CAPACITY, "chunk of %llu bytes exceeds max_chunk_bytes=%llu",
                                                              (unsigned long long)n_bytes, (unsigned long long)c->cfg.max_chunk_bytes);
    const uint64_t nk = c->cfg.read_len - c->cfg.k + 1;
    if ((n_bytes / c->cfg.read_len) * nk > kMaxSortKeys)
        return c->set_error(KC_ERR_CAPACITY, "chunk holds more than %llu k-mer slots; submit smaller chunks", (unsigned long long)kMaxSortKeys);
    cudaSetDevice(c->cfg.device);
    sl.n_bytes = n_bytes;
    if (n_bytes) KC_CUDA_TRY(c, cudaMemcpyAsync(sl.d_in, host_src, n_bytes, cudaMemcpyHostToDevice, sl.stream));
    {
        std::lock_guard<std::mutex> g(c->mu);
        c->stats.h2d_bytes += n_bytes;
    }
    return count_enqueue(c, sl.pend, sl.d_in, n_bytes, sl.stream, pick_method(c));
}

int kc_submit(kc_ctx *c, uint32_t slot, uint64_t n_bytes) {
    KC_TRY(check_ctx(c));
    if (slot >= c->slots.size() || !c->slots[slot].h_in) return c->set_error(KC_ERR_ARG, "slot %u not available", slot);
    return submit_from(c, slot, c->slots[slot].h_in, n_bytes);
}

int kc_wait(kc_ctx *c, uint32_t slot, kc_run **run) {
    KC_TRY(check_ctx(c));
    if (slot >= c->slots.size() || !run) return c->set_error(KC_ERR_ARG, "bad slot or null run");
    Slot &sl = c->slots[slot];
    cudaSetDevice(c->cfg.device);
    return count_finish(c, sl.pend, sl.d_in, sl.n_bytes, sl.stream, run);
}

int kc_process_chunk(kc_ctx *c, uint32_t slot, const char *reads, uint64_t n_bytes, void *records,
                     uint64_t records_cap, uint64_t *out_bytes) {
    KC_TRY(check_ctx(c));
    if (out_bytes) *out_bytes = 0;
    if (slot >= c->slots.size() || !c->slots[slot].d_in) return c->set_error(KC_ERR_ARG, "slot %u not available", slot);
    if (n_bytes && !reads) return c->set_error(KC_ERR_ARG, "null reads");
    KC_TRY(submit_from(c, slot, reads, n_bytes));
    kc_run *h = nullptr;
    KC_TRY(kc_wait(c, slot, &h));
    const RunPtr run(h, RunFree{c});
    uint64_t nb = (run->n - run->skip) * (uint64_t)c->S;
    if (out_bytes) *out_bytes = nb;
    if (!records) return KC_OK;
    if (nb > records_cap) return c->set_error(KC_ERR_CAPACITY, "run needs %llu bytes, buffer holds %llu", (unsigned long long)nb, (unsigned long long)records_cap);
    return kc_run_copy_records(c, run.get(), records, records_cap, out_bytes);
}

// -------------------------------------------------------------------------- runs
uint64_t kc_run_records(const kc_run *r) { return r ? r->n - r->skip : 0; }

int kc_run_free(kc_ctx *c, kc_run *r) {
    KC_TRY(check_ctx(c));
    if (!r) return KC_OK;
    cudaSetDevice(c->cfg.device);              // (may be called from a consumer thread that never touched the device)
    if (!r->placed) {
        dev_free(c->stream, r->d_keys);
        dev_free(c->stream, r->d_counts);
        dev_free(c->stream, r->d_sub_off);
    }
    delete r;
    return KC_OK;
}

int kc_place_next_run(kc_ctx *c, void *d_keys, void *d_counts, void *d_offsets, uint64_t cap_records, uint32_t cap_ranges) {
    KC_TRY(check_ctx(c));
    std::lock_guard<std::mutex> g(c->mu);
    c->place.keys = static_cast<uint64_t *>(d_keys);
    c->place.counts = static_cast<uint32_t *>(d_counts);
    c->place.offs = static_cast<uint32_t *>(d_offsets);
    c->place.cap = cap_records;
    c->place.cap_ranges = cap_ranges;
    c->place.set = d_keys && d_counts && d_offsets && cap_records;
    return KC_OK;
}

// Staging memory a peer process can map: plain cudaMalloc (CUDA IPC does not export pool or
// VMM allocations), handle = the 64-byte cudaIpcMemHandle_t.
int kc_peer_alloc(kc_ctx *c, uint64_t n_bytes, void **d_ptr, void *handle64) {
    KC_TRY(check_ctx(c));
    if (!d_ptr || !handle64 || n_bytes == 0) return c->set_error(KC_ERR_ARG, "kc_peer_alloc: null argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "handle size is part of the ABI");
    cudaSetDevice(c->cfg.device);
    void *p = nullptr;
    if (cudaMalloc(&p, n_bytes) != cudaSuccess) { cudaGetLastError(); return c->set_error(KC_ERR_NOMEM, "kc_peer_alloc: %llu bytes", (unsigned long long)n_bytes); }
    cudaIpcMemHandle_t h;
    cudaError_t e = cudaIpcGetMemHandle(&h, p);
    if (e != cudaSuccess) { cudaFree(p); return c->set_error(KC_ERR_CUDA, "cudaIpcGetMemHandle: %s", cudaGetErrorString(e)); }
    memcpy(handle64, &h, 64);
    *d_ptr = p;
    return KC_OK;
}

// Map a peer's staging memory into this context's device: opened with this device current, so
// the mapping is one its kernels can load from (peer access is enabled on the way).
int kc_peer_open(kc_ctx *c, const void *handle64, void **d_ptr) {
    KC_TRY(check_ctx(c));
    if (!d_ptr || !handle64) return c->set_error(KC_ERR_ARG, "kc_peer_open: null argument");
    cudaSetDevice(c->cfg.device);
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, 64);
    cudaError_t e = cudaIpcOpenMemHandle(d_ptr, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) { cudaGetLastError(); return c->set_error(KC_ERR_CUDA, "cudaIpcOpenMemHandle: %s", cudaGetErrorString(e)); }
    return KC_OK;
}

int kc_peer_close(kc_ctx *c, void *d_ptr) {
    KC_TRY(check_ctx(c));
    cudaSetDevice(c->cfg.device);
    KC_CUDA_TRY(c, cudaIpcCloseMemHandle(d_ptr));
    return KC_OK;
}

int kc_peer_free(kc_ctx *c, void *d_ptr) {
    KC_TRY(check_ctx(c));
    cudaSetDevice(c->cfg.device);
    KC_CUDA_TRY(c, cudaFree(d_ptr));
    return KC_OK;
}

int kc_run_parts(const kc_run *r, void **d_offsets, uint32_t *n_sub, uint32_t *prefix_bits) {
    if (!r) return KC_ERR_ARG;
    const bool has = r->d_sub_off && r->skip == 0;
    if (d_offsets) *d_offsets = has ? r->d_sub_off : nullptr;
    if (n_sub) *n_sub = has ? r->n_sub : 0;
    if (prefix_bits) *prefix_bits = has ? r->prefix_bits : 0;
    return KC_OK;
}

int kc_merge_parts(kc_ctx *c, uint32_t n_src, const void *const *d_keys, const void *const *d_counts,
                   const void *const *d_offsets, const uint64_t *n_records, uint32_t n_sub, uint32_t prefix_bits,
                   kc_run **out) {
    KC_TRY(check_ctx(c));
    std::lock_guard<std::recursive_mutex> dg(c->direct_mu);
    if (!out || n_src == 0 || n_src > 8 || !d_keys || !d_counts || !d_offsets || !n_records || n_sub == 0)
        return c->set_error(KC_ERR_ARG, "kc_merge_parts: bad argument");
    *out = nullptr;
    if (c->W != 1) return c->set_error(KC_ERR_ARG, "kc_merge_parts: 64-bit keys only");
    cudaSetDevice(c->cfg.device);
    cudaStream_t s = c->stream;
    uint64_t total = 0;
    for (uint32_t i = 0; i < n_src; i++) total += n_records[i];
    if (total >= (1ull << 32) - 2) return c->set_error(KC_ERR_CAPACITY, "kc_merge_parts: too many records");
    // temporaries come from the chunk scratch arena (idle between chunks), not from the allocator
    Pending &ar = c->direct;
    if (ar.active) return c->set_error(KC_ERR_STATE, "kc_merge_parts: a chunk is in flight on this context");
    KC_TRY(arena_reserve(c, ar, arena_round((total + 2) * 8) + arena_round((total + 2) * 4) +
                                    arena_round(merge_parts_workspace_bytes(n_sub)) + 512, s));
    void *tk = arena_take(ar, (total + 2) * 8), *tc = arena_take(ar, (total + 2) * 4);
    void *ws = arena_take(ar, merge_parts_workspace_bytes(n_sub));
    unsigned long long *d_sc = static_cast<unsigned long long *>(arena_take(ar, 16));
    int launches = 0;
    KC_CUDA_TRY(c, merge_parts_count(n_src, reinterpret_cast<const uint64_t *const *>(d_keys),
                                     reinterpret_cast<const uint32_t *const *>(d_counts),
                                     reinterpret_cast<const uint32_t *const *>(d_offsets), n_sub, (int)prefix_bits,
                                     static_cast<uint64_t *>(tk), static_cast<uint32_t *>(tc), &d_sc[0], &d_sc[1], ws,
                                     c->n_sms, s, &launches));
    unsigned long long h[2] = {0, 0};
    KC_CUDA_TRY(c, cudaMemcpyAsync(h, d_sc, 16, cudaMemcpyDeviceToHost, s));
    KC_CUDA_TRY(c, cudaStreamSynchronize(s));
    if (h[1]) return c->set_error(KC_ERR_CAPACITY, "kc_merge_parts: a key range could not be combined in shared memory");
    RunPtr r;
    KC_TRY(make_run(c, s, h[0], &r));
    void *mem = nullptr;
    KC_TRY(dev_alloc(c, s, (uint64_t)(n_sub + 1) * 4, &mem));
    r->d_sub_off = static_cast<uint32_t *>(mem);
    r->n_sub = n_sub;
    r->prefix_bits = prefix_bits;
    KC_CUDA_TRY(c, merge_parts_gather(n_sub, static_cast<uint64_t *>(tk), static_cast<uint32_t *>(tc), ws, r->d_keys,
                                      r->d_counts, r->d_sub_off, s));
    KC_CUDA_TRY(c, cudaStreamSynchronize(s));
    ar.arena_used = 0;
    {
        std::lock_guard<std::mutex> g(c->mu);
        c->stats.launches += launches + 1;
    }
    *out = r.release();
    return KC_OK;
}

int kc_run_device(const kc_run *r, void **d_keys, void **d_counts, uint64_t *n) {
    if (!r) return KC_ERR_ARG;
    if (d_keys) *d_keys = r->d_keys + r->skip * r->W;
    if (d_counts) *d_counts = r->d_counts + r->skip;
    if (n) *n = r->n - r->skip;
    return KC_OK;
}

int kc_run_copy_records(kc_ctx *c, const kc_run *r, void *dst, uint64_t cap, uint64_t *out_bytes) {
    KC_TRY(check_ctx(c));
    if (!r) return c->set_error(KC_ERR_ARG, "null run");
    const uint64_t n = r->n - r->skip, nb = n * (uint64_t)c->S;
    if (out_bytes) *out_bytes = nb;
    if (nb > cap || (nb && !dst)) return c->set_error(KC_ERR_CAPACITY, "run needs %llu bytes, buffer holds %llu", (unsigned long long)nb, (unsigned long long)cap);
    if (n == 0) return KC_OK;
    cudaSetDevice(c->cfg.device);
    std::lock_guard<std::mutex> cg(c->copy_mu);
    cudaStream_t cs = c->copy_stream;
    if (nb > c->copy_cap) {
        cudaStreamSynchronize(cs);
        if (c->copy_buf) cudaFree(c->copy_buf);
        c->copy_buf = nullptr; c->copy_cap = 0;
        const uint64_t want = nb + nb / 8 + (1u << 20);
        if (cudaMalloc(&c->copy_buf, want) != cudaSuccess) { cudaGetLastError(); return c->set_error(KC_ERR_NOMEM, "record staging buffer: %llu bytes", (unsigned long long)want); }
        c->copy_cap = want;
    }
    // everything queued on `stream` so far (the run's producer) is ordered before the copy; what
    // is queued later is not waited for
    cudaEvent_t ready;
    KC_CUDA_TRY(c, cudaEventCreateWithFlags(&ready, cudaEventDisableTiming));
    cudaEventRecord(ready, c->stream);
    cudaStreamWaitEvent(cs, ready, 0);
    cudaEventDestroy(ready);
    KC_CUDA_TRY(c, pack_records(r->d_keys + r->skip * r->W, r->d_counts + r->skip, n, r->W, c->copy_buf, cs));
    KC_CUDA_TRY(c, cudaMemcpyAsync(dst, c->copy_buf, nb, cudaMemcpyDeviceToHost, cs));
    KC_CUDA_TRY(c, cudaStreamSynchronize(cs));
    std::lock_guard<std::mutex> g(c->mu);
    c->stats.d2h_bytes += nb;
    c->stats.launches += 1;
    return KC_OK;
}

int kc_run_print(kc_ctx *c, const kc_run *r, char *dst, uint64_t cap, uint64_t *out_bytes) {
    KC_TRY(check_ctx(c));
    if (!r) return c->set_error(KC_ERR_ARG, "null run");
    std::lock_guard<std::recursive_mutex> dg(c->direct_mu);
    cudaSetDevice(c->cfg.device);
    cudaStream_t s = c->stream;
    const uint64_t n = r->n - r->skip;
    if (out_bytes) *out_bytes = 0;
    if (n == 0) return KC_OK;
    DevBuf text(s), ws(s), d_bytes(s);
    KC_TRY(text.alloc(c, print_max_bytes(n, r->W)));
    KC_TRY(ws.alloc(c, print_workspace_bytes(n)));
    KC_TRY(d_bytes.alloc(c, 8));
    unsigned long long total = 0;
    KC_CUDA_TRY(c, print_records_text(r->d_keys + r->skip * r->W, r->d_counts + r->skip, n, r->W, text.get<char>(),
                                      d_bytes.get<unsigned long long>(), ws.get(), s));
    KC_CUDA_TRY(c, cudaMemcpyAsync(&total, d_bytes.get(), 8, cudaMemcpyDeviceToHost, s));
    KC_CUDA_TRY(c, cudaStreamSynchronize(s));
    if (out_bytes) *out_bytes = total;
    if (total > cap || !dst) return c->set_error(KC_ERR_CAPACITY, "the text needs %llu bytes, buffer holds %llu", total, (unsigned long long)cap);
    KC_CUDA_TRY(c, cudaMemcpyAsync(dst, text.get(), total, cudaMemcpyDeviceToHost, s));
    KC_CUDA_TRY(c, cudaStreamSynchronize(s));
    std::lock_guard<std::mutex> g(c->mu);
    c->stats.launches += 1;
    c->stats.d2h_bytes += total;
    return KC_OK;
}

int kc_run_from_device(kc_ctx *c, const void *d_keys, const void *d_counts, uint64_t n, kc_run **out) {
    KC_TRY(check_ctx(c));
    std::lock_guard<std::recursive_mutex> dg(c->direct_mu);
    if (!out || (n && (!d_keys || !d_counts))) return c->set_error(KC_ERR_ARG, "null argument");
    *out = nullptr;
    cudaSetDevice(c->cfg.device);
    RunPtr r;
    KC_TRY(make_run(c, c->stream, n, &r));
    if (n) {
        KC_CUDA_TRY(c, cudaMemcpyAsync(r->d_keys, d_keys, n * c->W * 8, cudaMemcpyDeviceToDevice, c->stream));
        KC_CUDA_TRY(c, cudaMemcpyAsync(r->d_counts, d_counts, n * 4, cudaMemcpyDeviceToDevice, c->stream));
    }
    *out = r.release();
    return KC_OK;
}

int kc_run_upload(kc_ctx *c, const void *records, uint64_t n_bytes, kc_run **out) {
    KC_TRY(check_ctx(c));
    std::lock_guard<std::recursive_mutex> dg(c->direct_mu);
    if (!out || (n_bytes && !records)) return c->set_error(KC_ERR_ARG, "null argument");
    *out = nullptr;
    const uint64_t n = n_bytes / c->S;
    if (n >= (1ull << 32)) return c->set_error(KC_ERR_CAPACITY, "run too long for one upload");
    cudaSetDevice(c->cfg.device);
    cudaStream_t s = c->stream;
    if (n == 0) return kc_run_from_device(c, nullptr, nullptr, 0, out);
    DevBuf d_rec(s), ws(s), d_num(s);
    RunPtr raw, folded;
    KC_TRY(d_rec.alloc(c, n * c->S));
    KC_CUDA_TRY(c, cudaMemcpyAsync(d_rec.get(), records, n * c->S, cudaMemcpyHostToDevice, s));
    KC_TRY(make_run(c, s, n, &raw));
    KC_TRY(make_run(c, s, n, &folded));
    int launches = 1;
    KC_CUDA_TRY(c, unpack_records(d_rec.get(), n, c->W, raw->d_keys, raw->d_counts, s));
    KC_TRY(ws.alloc(c, ((rle_workspace_bytes(n) + 255) & ~255ull) + (n + 1) * 4 + 256));
    KC_TRY(d_num.alloc(c, 8));
    KC_CUDA_TRY(c, fold_sorted_pairs(raw->d_keys, raw->d_counts, n, c->W, folded->d_keys, folded->d_counts,
                                     d_num.get<unsigned long long>(), ws.get(), s, &launches));
    unsigned long long U = 0;
    KC_CUDA_TRY(c, cudaMemcpyAsync(&U, d_num.get(), 8, cudaMemcpyDeviceToHost, s));
    KC_CUDA_TRY(c, cudaStreamSynchronize(s));
    folded->n = U;
    {
        std::lock_guard<std::mutex> g(c->mu);
        c->stats.h2d_bytes += n * c->S;
        c->stats.launches += launches;
    }
    *out = folded.release();
    return KC_OK;
}

int kc_run_write(kc_ctx *c, const kc_run *r, const char *path, int append) {
    KC_TRY(check_ctx(c));
    if (!r || !path) return c->set_error(KC_ERR_ARG, "null argument");
    FILE *f = fopen(path, append ? "ab" : "wb");
    if (!f) return c->set_error(KC_ERR_IO, "cannot open %s", path);
    const uint64_t n = r->n - r->skip;
    const uint64_t piece = (64ull << 20) / c->S;      // 64 MiB staging
    void *h = nullptr;
    int rc = KC_OK;
    if (n) rc = kc_host_alloc(c, (n < piece ? n : piece) * c->S, &h);
    for (uint64_t i = 0; i < n && rc == KC_OK; i += piece) {
        kc_run view = *r;
        view.skip = r->skip + i;
        view.n = r->skip + (i + piece < n ? i + piece : n);
        uint64_t nb = 0;
        rc = kc_run_copy_records(c, &view, h, piece * c->S, &nb);
        if (rc == KC_OK && fwrite(h, 1, nb, f) != nb) rc = c->set_error(KC_ERR_IO, "short write to %s", path);
    }
    if (h) kc_host_free(c, h);
    if (fclose(f) != 0 && rc == KC_OK) rc = c->set_error(KC_ERR_IO, "close failed on %s", path);
    return rc;
}

int kc_run_split(kc_ctx *c, const kc_run *r, const uint64_t *splitters, uint32_t n_splitters, uint64_t *offsets) {
    KC_TRY(check_ctx(c));
    std::lock_guard<std::recursive_mutex> dg(c->direct_mu);
    if (!r || !offsets || (n_splitters && !splitters)) return c->set_error(KC_ERR_ARG, "null argument");
    const uint64_t n = r->n - r->skip;
    offsets[0] = 0;
    offsets[n_splitters + 1] = n;
    if (n_splitters == 0) return KC_OK;
    cudaSetDevice(c->cfg.device);
    cudaStream_t s = c->stream;
    DevBuf dq(s), dout(s);
    KC_TRY(dq.alloc(c, (uint64_t)n_splitters * c->W * 8));
    KC_TRY(dout.alloc(c, (uint64_t)n_splitters * 8));
    KC_CUDA_TRY(c, cudaMemcpyAsync(dq.get(), splitters, (uint64_t)n_splitters * c->W * 8, cudaMemcpyHostToDevice, s));
    KC_CUDA_TRY(c, lower_bounds(r->d_keys + r->skip * r->W, n, r->W, dq.get<uint64_t>(), n_splitters,
                                dout.get<unsigned long long>(), s));
    KC_CUDA_TRY(c, cudaMemcpyAsync(offsets + 1, dout.get(), (uint64_t)n_splitters * 8, cudaMemcpyDeviceToHost, s));
    KC_CUDA_TRY(c, cudaStreamSynchronize(s));
    std::lock_guard<std::mutex> g(c->mu);
    c->stats.launches += 1;
    return KC_OK;
}

// ------------------------------------------------------- count spectrum and filtering
int kc_run_histogram(kc_ctx *c, const kc_run *r, uint64_t *hist, uint32_t n_bins) {
    KC_TRY(check_ctx(c));
    if (!r || !hist) return c->set_error(KC_ERR_ARG, "null argument");
    if (n_bins < 2 || n_bins > (1u << 24)) return c->set_error(KC_ERR_ARG, "kc_run_histogram: n_bins %u is not in 2..2^24", n_bins);
    std::lock_guard<std::recursive_mutex> dg(c->direct_mu);
    const uint64_t n = r->n - r->skip;
    memset(hist, 0, (uint64_t)n_bins * 8);
    if (n == 0) return KC_OK;
    cudaSetDevice(c->cfg.device);
    cudaStream_t s = c->stream;
    DevBuf d_hist(s);
    KC_TRY(d_hist.alloc(c, (uint64_t)n_bins * 8));
    int launches = 0;
    KC_CUDA_TRY(c, run_histogram(r->d_counts + r->skip, n, n_bins, d_hist.get<unsigned long long>(), c->n_sms, s, &launches));
    KC_CUDA_TRY(c, cudaMemcpyAsync(hist, d_hist.get(), (uint64_t)n_bins * 8, cudaMemcpyDeviceToHost, s));
    KC_CUDA_TRY(c, cudaStreamSynchronize(s));
    std::lock_guard<std::mutex> g(c->mu);
    c->stats.launches += launches;
    c->stats.d2h_bytes += (uint64_t)n_bins * 8;
    return KC_OK;
}

int kc_run_filter(kc_ctx *c, const kc_run *r, uint32_t min_count, uint32_t max_count, kc_run **out) {
    KC_TRY(check_ctx(c));
    if (!r || !out) return c->set_error(KC_ERR_ARG, "null argument");
    *out = nullptr;
    if (min_count > max_count) return c->set_error(KC_ERR_ARG, "kc_run_filter: min_count %u > max_count %u", min_count, max_count);
    std::lock_guard<std::recursive_mutex> dg(c->direct_mu);
    cudaSetDevice(c->cfg.device);
    cudaStream_t s = c->stream;
    const uint64_t n = r->n - r->skip;
    if (n == 0) return kc_run_from_device(c, nullptr, nullptr, 0, out);
    const uint64_t *keys = r->d_keys + r->skip * r->W;
    const uint32_t *counts = r->d_counts + r->skip;
    DevBuf ws(s), d_total(s);
    KC_TRY(ws.alloc(c, filter_workspace_bytes(n)));
    KC_TRY(d_total.alloc(c, 8));
    int launches = 0;
    unsigned long long total = 0;
    KC_CUDA_TRY(c, filter_count(counts, n, min_count, max_count, ws.get(), d_total.get<unsigned long long>(), s, &launches));
    KC_CUDA_TRY(c, cudaMemcpyAsync(&total, d_total.get(), 8, cudaMemcpyDeviceToHost, s));
    KC_CUDA_TRY(c, cudaStreamSynchronize(s));
    RunPtr f;
    KC_TRY(make_run(c, s, total, &f));
    KC_CUDA_TRY(c, filter_write(keys, counts, n, r->W, min_count, max_count, ws.get(), f->d_keys, f->d_counts, s, &launches));
    KC_CUDA_TRY(c, cudaStreamSynchronize(s));
    {
        std::lock_guard<std::mutex> g(c->mu);
        c->stats.launches += launches;
        c->stats.d2h_bytes += 8;
    }
    *out = f.release();
    return KC_OK;
}

// ------------------------------------------------------------------------- merge
namespace {
// a run of one level of a merge: one of the caller's (borrowed) or one this merge made (owned)
struct LevelRun {
    const kc_run *run;
    RunPtr own;
};
LevelRun owned(RunPtr r) {
    const kc_run *p = r.get();
    return {p, std::move(r)};
}

// kc_merge_runs of runs of the partitioned path with one plan: kc_merge_parts over groups of up to 8,
// level by level
int merge_same_plan(kc_ctx *c, std::vector<LevelRun> level, kc_run **out) {
    while (level.size() > 1) {
        std::vector<LevelRun> next;
        for (size_t i = 0; i < level.size(); i += 8) {
            const uint32_t g = (uint32_t)std::min<size_t>(8, level.size() - i);
            if (g == 1) { next.push_back(std::move(level[i])); continue; }
            const void *kp[8], *cp[8], *op[8];
            uint64_t sz[8];
            for (uint32_t j = 0; j < g; j++) {
                const kc_run *r = level[i + j].run;
                kp[j] = r->d_keys; cp[j] = r->d_counts; op[j] = r->d_sub_off;
                sz[j] = r->n;
            }
            kc_run *m = nullptr;
            KC_TRY(kc_merge_parts(c, g, kp, cp, op, sz, level[0].run->n_sub, level[0].run->prefix_bits, &m));
            next.push_back(owned(RunPtr(m, RunFree{c})));
        }
        level.swap(next);                            // (the level before goes with next)
    }
    *out = level[0].own.release();
    return KC_OK;
}

// The pairwise tree of kc_merge_runs, level by level until level[0] is the one run left. The pairs of a
// level are queued back to back (each with its own output, sized for the no-overlap case, and its own
// record counter); the host reads the counters once per group of pairs instead of once per pair. A
// group closes early when its outputs would take more than a third of the free device memory.
int merge_tree(kc_ctx *c, cudaStream_t s, std::vector<LevelRun> &level, int *launches) {
    const uint32_t max_pairs = (uint32_t)(level.size() / 2 + 1);
    DevBuf d_num(s);
    KC_TRY(d_num.alloc(c, 8ull * max_pairs));
    std::vector<unsigned long long> h_num(max_pairs, 0);
    const bool trace = getenv("KC_TRACE") != nullptr;
    while (level.size() > 1) {
        std::vector<LevelRun> next;
        struct timespec t0;
        clock_gettime(CLOCK_MONOTONIC, &t0);
        uint64_t level_records = 0;
        for (size_t i = 0; i + 1 < level.size();) {
            size_t fr = 0, tot = 0;
            cudaMemGetInfo(&fr, &tot);
            const uint64_t budget = fr / 3;
            uint64_t group_bytes = 0;
            std::vector<DevBuf> group_ws;
            const size_t g0 = i, n0 = next.size();
            for (; i + 1 < level.size(); i += 2) {
                const kc_run *a = level[i].run, *b = level[i + 1].run;
                const uint64_t na = a->n - a->skip, nb = b->n - b->skip;
                const uint64_t bytes = (na + nb) * (8ull * c->W + 4);
                if (i > g0 && group_bytes + bytes > budget) break;
                RunPtr m;
                KC_TRY(make_run(c, s, na + nb, &m));
                group_ws.emplace_back(s);
                KC_TRY(group_ws.back().alloc(c, merge_workspace_bytes(na, nb)));
                const cudaError_t e = merge_pair(a->d_keys + a->skip * a->W, a->d_counts + a->skip, na,
                                                 b->d_keys + b->skip * b->W, b->d_counts + b->skip, nb, c->W, m->d_keys,
                                                 m->d_counts, d_num.get<unsigned long long>() + (next.size() - n0),
                                                 group_ws.back().get(), s, launches);
                if (e != cudaSuccess) return c->set_error(KC_ERR_CUDA, "merge failed: %s", cudaGetErrorString(e));
                next.push_back(owned(std::move(m)));
                group_bytes += bytes;
                level_records += na + nb;
            }
            const size_t n_pairs = next.size() - n0;
            KC_CUDA_TRY(c, cudaMemcpyAsync(h_num.data(), d_num.get(), 8 * n_pairs, cudaMemcpyDeviceToHost, s));
            KC_CUDA_TRY(c, cudaStreamSynchronize(s));
            for (size_t q = 0; q < n_pairs; q++) {
                next[n0 + q].own->n = h_num[q];
                level[g0 + 2 * q].own.reset();       // the pair's inputs, if this merge made them
                level[g0 + 2 * q + 1].own.reset();
            }
        }
        if (level.size() & 1) next.push_back(std::move(level.back()));
        if (trace) {
            struct timespec t1;
            clock_gettime(CLOCK_MONOTONIC, &t1);
            fprintf(stderr, "kc_merge_runs: level of %zu runs, %llu records in: %.2f ms\n", level.size(), (unsigned long long)level_records,
                    (t1.tv_sec - t0.tv_sec) * 1e3 + (t1.tv_nsec - t0.tv_nsec) * 1e-6);
        }
        level.swap(next);
    }
    return KC_OK;
}
}  // namespace


int kc_merge_runs(kc_ctx *c, kc_run *const *runs, uint32_t n, kc_run **out) {
    KC_TRY(check_ctx(c));
    std::lock_guard<std::recursive_mutex> dg(c->direct_mu);
    if (!out || (n && !runs)) return c->set_error(KC_ERR_ARG, "null argument");
    *out = nullptr;
    cudaSetDevice(c->cfg.device);
    cudaStream_t s = c->stream;
    // other streams (slots) may have produced the inputs
    for (auto &sl : c->slots)
        if (sl.stream) KC_CUDA_TRY(c, cudaStreamSynchronize(sl.stream));
    if (n == 0) return kc_run_from_device(c, nullptr, nullptr, 0, out);   // an empty run
    for (uint32_t i = 0; i < n; i++)
        if (!runs[i]) return c->set_error(KC_ERR_ARG, "null run in merge list");
    if (n == 1) {
        const kc_run *r = runs[0];
        return kc_run_from_device(c, r->d_keys + r->skip * r->W, r->d_counts + r->skip, r->n - r->skip, out);
    }
    auto borrow_all = [&]() {
        std::vector<LevelRun> v;
        for (uint32_t i = 0; i < n; i++) v.push_back({runs[i], RunPtr()});
        return v;
    };
    // Three or more runs of the partitioned path with the same plan (chunks of equal size): combine
    // them range by range in shared-memory tables, up to 8 at a time (kc_merge_parts: one pass over
    // the records instead of log2(n) merge-path passes; 4 runs of C2: 11.9 ms against 16.8 ms).
    // Two runs, or runs without a common plan, take the merge-path tree below.
    if (c->W == 1 && n >= 3 && !c->direct.active) {
        bool same = true;
        for (uint32_t i = 0; i < n && same; i++)
            same = runs[i]->d_sub_off && runs[i]->skip == 0 && runs[i]->n_sub == runs[0]->n_sub &&
                   runs[i]->prefix_bits == runs[0]->prefix_bits;
        // (a range too large for a shared-memory table, or too many records: the tree handles anything)
        if (same && merge_same_plan(c, borrow_all(), out) == KC_OK) return KC_OK;
    }
    std::vector<LevelRun> level = borrow_all();
    int launches = 0;
    const int rc = merge_tree(c, s, level, &launches);
    {
        std::lock_guard<std::mutex> g(c->mu);
        c->stats.launches += launches;
    }
    if (rc != KC_OK) return rc;
    *out = level[0].own.release();
    return KC_OK;
}

// ------------------------------------------------------------ set operations of two runs
// One merge-path pass (combine_pair: the merge's kernels with the op deciding what survives); the
// output is allocated for the most records the op can give and trimmed to what it gave.
int kc_run_combine(kc_ctx *c, const kc_run *a, const kc_run *b, uint32_t op, uint32_t counts, kc_run **out) {
    KC_TRY(check_ctx(c));
    if (!a || !b || !out) return c->set_error(KC_ERR_ARG, "null argument");
    *out = nullptr;
    if (op > KC_SET_SUBTRACT_COUNTS) return c->set_error(KC_ERR_ARG, "kc_run_combine: unknown op %u", op);
    if (counts > KC_COUNTS_B) return c->set_error(KC_ERR_ARG, "kc_run_combine: unknown count mode %u", counts);
    if (counts != KC_COUNTS_SUM && (op == KC_SET_SUBTRACT || op == KC_SET_SUBTRACT_COUNTS))
        return c->set_error(KC_ERR_ARG, "kc_run_combine: a subtract takes no count mode (got %u)", counts);
    if (a->W != c->W || b->W != c->W)
        return c->set_error(KC_ERR_ARG, "kc_run_combine: runs of %d and %d key words, the context's keys have %d", a->W, b->W, c->W);
    std::lock_guard<std::recursive_mutex> dg(c->direct_mu);
    cudaSetDevice(c->cfg.device);
    cudaStream_t s = c->stream;
    // other streams (slots) may have produced the inputs
    for (auto &sl : c->slots)
        if (sl.stream) KC_CUDA_TRY(c, cudaStreamSynchronize(sl.stream));
    const uint64_t na = a->n - a->skip, nb = b->n - b->skip;
    const uint64_t cap = op == KC_SET_UNION ? na + nb : op == KC_SET_INTERSECT ? std::min(na, nb) : na;
    RunPtr r;
    DevBuf ws(s), d_num(s);
    KC_TRY(make_run(c, s, cap, &r));
    KC_TRY(ws.alloc(c, merge_workspace_bytes(na, nb)));
    KC_TRY(d_num.alloc(c, 8));
    int launches = 0;
    const cudaError_t e = combine_pair(a->d_keys + a->skip * a->W, a->d_counts + a->skip, na, b->d_keys + b->skip * b->W,
                                       b->d_counts + b->skip, nb, c->W, op, counts, r->d_keys, r->d_counts,
                                       d_num.get<unsigned long long>(), ws.get(), s, &launches);
    if (e != cudaSuccess) return c->set_error(KC_ERR_CUDA, "combine failed: %s", cudaGetErrorString(e));
    unsigned long long n_out = 0;
    KC_CUDA_TRY(c, cudaMemcpyAsync(&n_out, d_num.get(), 8, cudaMemcpyDeviceToHost, s));
    KC_CUDA_TRY(c, cudaStreamSynchronize(s));
    r->n = n_out;
    {
        std::lock_guard<std::mutex> g(c->mu);
        c->stats.launches += launches;
        c->stats.d2h_bytes += 8;
    }
    *out = r.release();
    return KC_OK;
}

}  // extern "C"
