// RunMerger.h -- merge scheduling over sorted runs, with spill to host memory.
//
// Replaces KMerFileMergeHandler (KMerFileMergeHandler.cpp:23-123), whose polling thread
// hangs when InputComplete() arrives late or when there is a single run (SURVEY.md 5.3).
// Same shape -- AddRun / InputComplete / result -- and, like the reference's, the merges run
// on their own thread while the producer keeps counting chunks (noOfMergeThreads >= 1; the GPU
// serialises the merge kernels on the context's stream, the chunk kernels run on the slot
// streams). It terminates for 0, 1 or N runs.
//
// Schedule: runs are kept in levels, level i holding runs that are the merge of about
// fanIn^i chunk runs. Whenever a level holds noOfMergersAtOnce runs they are merged on the GPU
// (kc_merge_runs, the merge-path kernel) into one run of the next level, so every record takes
// part in O(log_fanIn(chunks)) merges instead of one per chunk.
//
// Spill (the reference spills every chunk's run to tempFileLocation and merges files,
// FileDump.cpp:51-58 + KMerFileMerger.cpp:49-135): with a run budget, a merged run that
// outgrows it is copied to pinned host memory as packed records and leaves the device.
// Finish() then merges out of core: the key space is cut at sampled splitters into ranges
// whose records fit the budget, and range by range the matching slice of every spilled run
// is uploaded (kc_run_upload), merged (kc_merge_runs) and appended to the output file --
// ranges are key-disjoint and ascending, so the file is the sorted unique artefact.
//
// An optional hook sees every final run just before it is written (or handed out by InputComplete):
// the one merged run, or each range's merged run of the out-of-core merge. Its counts are final
// there, so it may replace the run (a count filter) or read it (the count spectrum). Chunk runs and
// intermediate merges never reach it.
#pragma once

#include <stdint.h>
#include <string.h>

#include <algorithm>
#include <condition_variable>
#include <deque>
#include <functional>
#include <mutex>
#include <thread>
#include <vector>

#include "../../include/kc_api.h"

class RunMerger {
public:
    // runBudgetBytes = packed-record bytes a merged run may hold on the device (0 = no limit, never spill);
    // mergeThreads = 0: merges run inside AddRun; >= 1: on a background thread
    RunMerger(kc_ctx *ctx, uint32_t noOfMergersAtOnce, uint32_t k = 0, uint64_t runBudgetBytes = 0, uint32_t mergeThreads = 1)
        : _ctx(ctx), _fanIn(noOfMergersAtOnce < 2 ? 2 : noOfMergersAtOnce), _budget(runBudgetBytes),
          _W(k ? kc_key_words(k) : 1), _S(k ? kc_record_size(k) : 12) {
        if (mergeThreads >= 1) _worker = std::thread([this]() { workerLoop(); });
    }
    ~RunMerger() {
        stopWorker();
        for (kc_run *r : _queue) kc_run_free(_ctx, r);
        for (auto &lv : _levels)
            for (kc_run *r : lv) kc_run_free(_ctx, r);
        for (HostRun &h : _spilled) kc_host_free(_ctx, h.data);
    }
    int AddRun(kc_run *run) {                       // takes ownership
        if (!_worker.joinable()) return place(run);
        std::lock_guard<std::mutex> g(_mu);
        if (_rc != KC_OK) { kc_run_free(_ctx, run); return _rc; }
        _queue.push_back(run);
        _cv.notify_all();
        return KC_OK;
    }
    // Merges everything that is left; *out is the final run (an empty run for no input).
    // Only valid when nothing was spilled (spills() == 0); use Finish() otherwise.
    int InputComplete(kc_run **out) {
        int rc = drain();
        if (rc != KC_OK) return rc;
        if ((rc = mergeAll()) != KC_OK) return rc;
        if (!_spilled.empty()) return KC_ERR_STATE;
        kc_run *last = takeOnly();
        if (!last && (rc = kc_merge_runs(_ctx, nullptr, 0, &last)) != KC_OK) return rc;
        if ((rc = finalRun(&last)) != KC_OK) return rc;
        *out = last;
        return KC_OK;
    }
    // Merges everything that is left and writes the artefact to `path` (truncating; the reference
    // appends to whatever is there, KMerFileMerger.cpp:129). *n_records = records written.
    int Finish(const char *path, uint64_t *n_records) {
        int rc = drain();
        if (rc != KC_OK) return rc;
        if ((rc = mergeAll()) != KC_OK) return rc;
        if (_spilled.empty()) {
            kc_run *out = nullptr;
            if ((rc = InputComplete(&out)) != KC_OK) return rc;
            if (n_records) *n_records = kc_run_records(out);
            rc = kc_run_write(_ctx, out, path, 0);
            kc_run_free(_ctx, out);
            return rc;
        }
        kc_run *last = takeOnly();
        if (last && (rc = spill(last)) != KC_OK) return rc;
        return mergeOutOfCore(path, n_records);
    }
    // hook(&run): may replace *run (freeing the old one) or leave it; a non-KC_OK result aborts the merge
    void SetFinalHook(std::function<int(kc_run **)> hook) { _final = std::move(hook); }
    uint64_t merges() const { return _merges; }
    uint64_t spills() const { return _spills; }
    uint64_t ranges() const { return _ranges; }

private:
    struct HostRun {
        void *data;
        uint64_t n;                                 // records
    };
    struct KeyRef {                                 // W words, most significant first
        uint64_t w[4];
    };

    int finalRun(kc_run **run) {
        if (!_final) return KC_OK;
        const int rc = _final(run);
        if (rc != KC_OK && *run) { kc_run_free(_ctx, *run); *run = nullptr; }
        return rc;
    }
    // ---- background merging
    void workerLoop() {
        for (;;) {
            kc_run *run = nullptr;
            {
                std::unique_lock<std::mutex> g(_mu);
                _cv.wait(g, [this]() { return _stop || !_queue.empty(); });
                if (_queue.empty()) return;          // _stop and nothing left
                run = _queue.front();
                _queue.pop_front();
                _busy = true;
            }
            const int rc = place(run);
            {
                std::lock_guard<std::mutex> g(_mu);
                _busy = false;
                if (rc != KC_OK && _rc == KC_OK) _rc = rc;
                _cv.notify_all();
            }
        }
    }
    int drain() {                                   // everything queued has been placed
        if (!_worker.joinable()) return _rc;
        std::unique_lock<std::mutex> g(_mu);
        _cv.wait(g, [this]() { return _queue.empty() && !_busy; });
        return _rc;
    }
    void stopWorker() {
        if (!_worker.joinable()) return;
        {
            std::lock_guard<std::mutex> g(_mu);
            _stop = true;
            _cv.notify_all();
        }
        _worker.join();
    }
    // ---- the level schedule (one thread at a time: the worker, or the caller after drain())
    int place(kc_run *run) {
        size_t lv = 0;
        for (;;) {
            if (_levels.size() <= lv) _levels.resize(lv + 1);
            _levels[lv].push_back(run);
            if (_levels[lv].size() < _fanIn) return KC_OK;
            kc_run *merged = nullptr;
            int rc = mergeList(_levels[lv], &merged);
            if (rc != KC_OK) return rc;
            if (_budget && kc_run_records(merged) * _S > _budget) return spill(merged);
            run = merged;
            lv++;
        }
    }
    int mergeList(std::vector<kc_run *> &runs, kc_run **out) {      // frees the inputs
        int rc = kc_merge_runs(_ctx, runs.data(), (uint32_t)runs.size(), out);
        if (rc != KC_OK) return rc;
        for (kc_run *r : runs) kc_run_free(_ctx, r);
        runs.clear();
        _merges++;
        return KC_OK;
    }
    int mergeAll() {                                // what is left in the levels -> at most one run (smallest first)
        std::vector<kc_run *> rest;
        for (auto &lv : _levels) {
            for (kc_run *r : lv) rest.push_back(r);
            lv.clear();
        }
        if (rest.size() < 2) { if (!rest.empty()) { _levels.resize(1); _levels[0].push_back(rest[0]); } return KC_OK; }
        kc_run *merged = nullptr;
        int rc = kc_merge_runs(_ctx, rest.data(), (uint32_t)rest.size(), &merged);
        if (rc != KC_OK) { _levels.resize(1); _levels[0] = rest; return rc; }
        for (kc_run *r : rest) kc_run_free(_ctx, r);
        _merges++;
        _levels.resize(1);
        _levels[0].push_back(merged);
        return KC_OK;
    }
    kc_run *takeOnly() {
        for (auto &lv : _levels)
            if (!lv.empty()) { kc_run *r = lv[0]; lv.clear(); return r; }
        return nullptr;
    }
    // a run goes to pinned host memory as packed records
    int spill(kc_run *r) {
        const uint64_t n = kc_run_records(r), nb = n * _S;
        void *buf = nullptr;
        int rc = kc_host_alloc(_ctx, nb ? nb : 1, &buf);
        if (rc != KC_OK) { kc_run_free(_ctx, r); return rc; }
        uint64_t got = 0;
        rc = kc_run_copy_records(_ctx, r, buf, nb, &got);
        kc_run_free(_ctx, r);
        if (rc != KC_OK) { kc_host_free(_ctx, buf); return rc; }
        _spilled.push_back(HostRun{buf, n});
        _spills++;
        return KC_OK;
    }
    KeyRef keyAt(const HostRun &h, uint64_t i) const {
        KeyRef k = {{0, 0, 0, 0}};
        memcpy(k.w, static_cast<const uint8_t *>(h.data) + i * _S, 8 * _W);
        return k;
    }
    bool less(const KeyRef &a, const KeyRef &b) const {
        for (uint32_t i = 0; i < _W; i++)
            if (a.w[i] != b.w[i]) return a.w[i] < b.w[i];
        return false;
    }
    uint64_t lowerBound(const HostRun &h, const KeyRef &k) const {  // first record whose key is >= k
        uint64_t lo = 0, hi = h.n;
        while (lo < hi) {
            const uint64_t mid = lo + (hi - lo) / 2;
            if (less(keyAt(h, mid), k)) lo = mid + 1;
            else hi = mid;
        }
        return lo;
    }
    int mergeOutOfCore(const char *path, uint64_t *n_records) {
        uint64_t total = 0;
        for (const HostRun &h : _spilled) total += h.n * _S;
        const uint64_t per_range = _budget > 2 * _S ? _budget / 2 : _S;
        const uint64_t G = std::max<uint64_t>(1, (total + per_range - 1) / per_range);
        // splitters: 16 evenly spaced keys per range from every run, sorted, then every n_runs*16-th
        std::vector<KeyRef> samples;
        const uint64_t per_run = 16 * G;
        for (const HostRun &h : _spilled)
            for (uint64_t i = 1; i <= per_run && h.n; i++) samples.push_back(keyAt(h, (h.n - 1) * i / per_run));
        std::sort(samples.begin(), samples.end(), [this](const KeyRef &a, const KeyRef &b) { return less(a, b); });
        std::vector<uint64_t> lo(_spilled.size(), 0);
        uint64_t written = 0;
        bool first = true;
        int rc = KC_OK;
        for (uint64_t g = 0; g < G && rc == KC_OK; g++) {
            std::vector<kc_run *> parts;
            for (size_t r = 0; r < _spilled.size() && rc == KC_OK; r++) {
                const HostRun &h = _spilled[r];
                const uint64_t hi = (g + 1 == G || samples.empty()) ? h.n
                                                                   : lowerBound(h, samples[(g + 1) * samples.size() / G - 1]);
                if (hi > lo[r]) {
                    kc_run *part = nullptr;
                    rc = kc_run_upload(_ctx, static_cast<const uint8_t *>(h.data) + lo[r] * _S, (hi - lo[r]) * _S, &part);
                    if (rc == KC_OK) parts.push_back(part);
                    lo[r] = hi;
                }
            }
            if (rc == KC_OK && !parts.empty()) {
                kc_run *out = nullptr;
                rc = kc_merge_runs(_ctx, parts.data(), (uint32_t)parts.size(), &out);
                if (rc == KC_OK) rc = finalRun(&out);
                if (rc == KC_OK) {
                    rc = kc_run_write(_ctx, out, path, first ? 0 : 1);
                    written += kc_run_records(out);
                    first = false;
                    _merges++;
                    _ranges++;
                    kc_run_free(_ctx, out);
                }
            }
            for (kc_run *p : parts) kc_run_free(_ctx, p);
        }
        if (rc == KC_OK && first) {                 // nothing at all: still leave an (empty) artefact behind
            kc_run *empty = nullptr;
            if ((rc = kc_merge_runs(_ctx, nullptr, 0, &empty)) == KC_OK) {
                rc = kc_run_write(_ctx, empty, path, 0);
                kc_run_free(_ctx, empty);
            }
        }
        if (n_records) *n_records = written;
        return rc;
    }

    kc_ctx *_ctx;
    size_t _fanIn;
    uint64_t _budget;
    uint32_t _W, _S;
    std::vector<std::vector<kc_run *>> _levels;
    std::vector<HostRun> _spilled;
    uint64_t _merges = 0, _spills = 0, _ranges = 0;
    // background worker
    std::thread _worker;
    std::mutex _mu;
    std::condition_variable _cv;
    std::deque<kc_run *> _queue;
    bool _stop = false, _busy = false;
    int _rc = KC_OK;
    std::function<int(kc_run **)> _final;
};
