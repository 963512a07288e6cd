"""Object wrappers over the C ABI. No compute happens in Python."""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import KcConfig, KcStats, METHODS, METHOD_NAMES, KC_COMPAT_REF, KC_COMPAT_STRICT, KC_CANONICAL


STAGE_NAMES = {
    "sort": ["extract", "digit_histogram", "radix_scatter_passes", "run_length", "emit"],
    "hash": ["level1_histogram", "extract_scatter1", "level2_histogram", "scatter2", "smem_count_sort_write", "emit"],
    "hash_global": ["table_clear", "extract_insert", "compact_sort", "emit"],
    "super": ["encode_minimizer_scatter", "smem_count_per_bin", "record_scatter1", "record_hist2", "record_scatter2",
              "smem_sort_write"],
    "place": ["extract_keys", "count_init_hist1", "record_scatter1", "record_hist2", "record_scatter2",
              "smem_sort_fold_write"],
}

SW_SCALARS = ["invalid", "overflow_records", "d_records", "fail", "ticket", "windows", "occurrences", "aborts", "folded",
              "out_records", "records", "ticket2", "big_ranges", "big_records", "dedup_records", "multi_round_units"]


def xchg_run_all(counters):
    """All ranks in this process (kc_xchg_run_all): what the counters accumulated -> [run of rank r's key range]."""
    lib = counters[0]._lib
    n = len(counters)
    ctxs = (C.c_void_p * n)(*[c._ctx for c in counters])
    runs = (C.c_void_p * n)()
    rc = lib.kc_xchg_run_all(ctxs, n, runs)
    if rc != 0:
        msgs = [(lib.kc_last_error(c._ctx) or b"").decode() for c in counters]
        raise KcError(rc, "; ".join(m for m in msgs if m))
    return [Run(c, C.c_void_p(runs[i])) for i, c in enumerate(counters)]


class KcError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("kc error %d: %s" % (code, msg))
        self.code = code


def key_words(k):
    return _lib.load().kc_key_words(k)


def record_size(k):
    return _lib.load().kc_record_size(k)


class Run:
    """A sorted key-unique run resident on the device (the reference's run file, in HBM)."""

    def __init__(self, counter, handle):
        self._c = counter
        self._h = handle

    def __len__(self):
        return int(self._c._lib.kc_run_records(self._h)) if self._h else 0

    @property
    def nbytes(self):
        return len(self) * self._c.record_size

    def to_bytes(self) -> bytes:
        """Packed records (the SortedKMerFile format)."""
        buf = np.empty(max(self.nbytes, 1), dtype=np.uint8)
        n = C.c_uint64()
        self._c._check(self._c._lib.kc_run_copy_records(self._c._ctx, self._h, buf.ctypes.data, buf.size, C.byref(n)))
        return buf[: n.value].tobytes()

    def print_text(self) -> bytes:
        """The run in KMerPrinter's text format (KMerPrinter.cpp:35-91), formatted on the device."""
        n = len(self)
        if n == 0:
            return b""
        cap = n * (32 * self._c.words + 12)
        buf = np.empty(cap, dtype=np.uint8)
        nb = C.c_uint64()
        self._c._check(self._c._lib.kc_run_print(self._c._ctx, self._h, buf.ctypes.data, cap, C.byref(nb)))
        return buf[: nb.value].tobytes()

    def copy_into(self, host_ptr, cap) -> int:
        n = C.c_uint64()
        self._c._check(self._c._lib.kc_run_copy_records(self._c._ctx, self._h, host_ptr, cap, C.byref(n)))
        return n.value

    def write(self, path, append=False):
        self._c._check(self._c._lib.kc_run_write(self._c._ctx, self._h, path.encode(), 1 if append else 0))

    def device_arrays(self):
        """(keys_ptr, counts_ptr, n): device pointers to n*W uint64 and n uint32."""
        k, c, n = C.c_void_p(), C.c_void_p(), C.c_uint64()
        self._c._check(self._c._lib.kc_run_device(self._h, C.byref(k), C.byref(c), C.byref(n)))
        return k.value or 0, c.value or 0, n.value

    def parts(self):
        """(offsets_ptr, n_sub, prefix_bits): the run's partition structure, n_sub == 0 if it has none."""
        o, n, b = C.c_void_p(), C.c_uint32(), C.c_uint32()
        self._c._check(self._c._lib.kc_run_parts(self._h, C.byref(o), C.byref(n), C.byref(b)))
        return o.value or 0, n.value, b.value

    def split(self, splitters):
        """Lower-bound offsets of the splitter keys ([n_split, W] uint64) -> n_split+2 offsets."""
        sp = np.ascontiguousarray(splitters, dtype=np.uint64).reshape(-1, self._c.words)
        off = np.zeros(sp.shape[0] + 2, dtype=np.uint64)
        self._c._check(self._c._lib.kc_run_split(
            self._c._ctx, self._h, sp.ctypes.data_as(C.POINTER(C.c_uint64)), sp.shape[0],
            off.ctypes.data_as(C.POINTER(C.c_uint64))))
        return off

    def histogram(self, n_bins=10001) -> np.ndarray:
        """Count spectrum, computed on the device (kc_run_histogram): uint64[n_bins], where h[c] = records
        with count c and h[n_bins - 1] = records with count >= n_bins - 1. The default matches
        Jellyfish's histo: counts up to 10,000 get their own bins."""
        h = np.zeros(max(int(n_bins), 1), dtype=np.uint64)
        self._c._check(self._c._lib.kc_run_histogram(self._c._ctx, self._h, h.ctypes.data_as(C.POINTER(C.c_uint64)),
                                                     int(n_bins)))
        return h

    def filter(self, min_count=0, max_count=2**32 - 1) -> "Run":
        """A new run with the records whose count is in [min_count, max_count], in order (kc_run_filter).
        Filter only final counts: a chunk's run filtered before a merge loses k-mers."""
        h = C.c_void_p()
        self._c._check(self._c._lib.kc_run_filter(self._c._ctx, self._h, int(min_count), int(max_count), C.byref(h)))
        return Run(self._c, h)

    # KMC's count mode when none is given: union sums, intersect takes the smaller count
    _DEFAULT_COUNTS = {"union": "sum", "intersect": "min", "subtract": "sum", "subtract_counts": "sum"}

    def combine(self, other, op, counts=None) -> "Run":
        """A new run from this run (A) and `other` (B), computed on the device (kc_run_combine).
        op: "union", "intersect", "subtract" (keys of A not in B) or "subtract_counts" (also keys in
        both with a > b, counted a - b). counts: how a key in both runs is counted by union and
        intersect -- "sum", "min", "max", "a" or "b"; None = KMC's default (sum for union, min for
        intersect). The subtracts take no mode. Both runs must come from counters with the same k."""
        if op not in _lib.SET_OPS:
            raise KcError(-1, "unknown set operation %r (one of %s)" % (op, ", ".join(_lib.SET_OPS)))
        if counts is None:
            counts = self._DEFAULT_COUNTS[op]
        if counts not in _lib.COUNT_MODES:
            raise KcError(-1, "unknown count mode %r (one of %s)" % (counts, ", ".join(_lib.COUNT_MODES)))
        h = C.c_void_p()
        self._c._check(self._c._lib.kc_run_combine(self._c._ctx, self._h, other._h, _lib.SET_OPS[op],
                                                   _lib.COUNT_MODES[counts], C.byref(h)))
        return Run(self._c, h)

    def free(self):
        if self._h and self._c._ctx:
            self._c._lib.kc_run_free(self._c._ctx, self._h)
        self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Counter:
    """One kc_ctx: the replacement for PrepareGPU's GPUStream array (GPUHandler.cu:479-509)."""

    def __init__(self, k, read_len, device=0, method="auto", compat="ref", n_slots=2, max_chunk_bytes=0,
                 table_slots=0, stream=None, distinct_hint=0, canonical=False):
        """canonical=True counts every k-mer with its reverse complement under min(x, rc(x))
        (KC_CANONICAL; implies compat="strict"). Its runs must not be merged with forward runs."""
        self._lib = _lib.load()
        cfg = KcConfig()
        cfg.struct_size = C.sizeof(KcConfig)
        cfg.k, cfg.read_len, cfg.device = k, read_len, device
        cfg.flags = KC_COMPAT_STRICT if compat == "strict" else KC_COMPAT_REF
        if canonical:
            cfg.flags |= KC_CANONICAL | KC_COMPAT_STRICT
        cfg.method = METHODS[method] if isinstance(method, str) else int(method)
        cfg.n_slots, cfg.max_chunk_bytes, cfg.table_slots = n_slots, max_chunk_bytes, table_slots
        cfg.stream = stream
        cfg.distinct_hint = distinct_hint
        ctx = C.c_void_p()
        rc = self._lib.kc_create(C.byref(cfg), C.byref(ctx))
        if rc != 0:
            raise KcError(rc, (self._lib.kc_last_error(None) or b"").decode())
        self._ctx = ctx
        self.k, self.read_len, self.device = k, read_len, device
        self.canonical = bool(canonical)
        self.words = self._lib.kc_key_words(k)
        self.record_size = self._lib.kc_record_size(k)
        self.max_chunk_bytes = max_chunk_bytes

    # -- plumbing
    def _check(self, rc):
        if rc != 0:
            raise KcError(rc, (self._lib.kc_last_error(self._ctx) or b"").decode())

    def close(self):
        if getattr(self, "_ctx", None):
            self._lib.kc_destroy(self._ctx)
            self._ctx = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def sync(self):
        self._check(self._lib.kc_sync(self._ctx))

    def stats(self) -> dict:
        st = KcStats()
        self._check(self._lib.kc_stats_get(self._ctx, C.byref(st)))
        d = {name: getattr(st, name) for name, _ in KcStats._fields_}
        d["method_used"] = METHOD_NAMES.get(d["method_used"], "none")
        n = d["n_stages"]
        names = STAGE_NAMES.get(d["method_used"], [])
        d["ms_stage"] = [float(x) for x in st.ms_stage][:n]
        d["stage_bytes"] = [int(x) for x in st.stage_bytes][:n]
        d["stage_launches"] = [int(x) for x in st.stage_launches][:n]
        d["stage_names"] = (names + ["stage%d" % i for i in range(len(names), n)])[:n]
        return d

    # -- accumulating mode: many chunks, one count (kc_accum_*)
    def accum_begin(self, expected_reads=0):
        self._check(self._lib.kc_accum_begin(self._ctx, expected_reads))

    def accum_add_device(self, d_ptr, n_bytes):
        self._check(self._lib.kc_accum_add_device(self._ctx, d_ptr, n_bytes))

    def accum_submit(self, slot, n_bytes):
        self._check(self._lib.kc_accum_submit(self._ctx, slot, n_bytes))

    def accum_wait(self, slot):
        self._check(self._lib.kc_accum_wait(self._ctx, slot))

    def accum_flush(self) -> "Run":
        h = C.c_void_p()
        self._check(self._lib.kc_accum_flush(self._ctx, C.byref(h)))
        return Run(self, h)

    # -- multi-GPU exchange (kc_xchg_*): this counter is one rank
    def xchg_begin(self, rank, n_ranks, expected_reads=0):
        self._check(self._lib.kc_xchg_begin(self._ctx, rank, n_ranks, expected_reads))

    def xchg_export(self) -> bytes:
        buf = C.create_string_buffer(64)
        self._check(self._lib.kc_xchg_export(self._ctx, buf))
        return buf.raw

    def xchg_import(self, peer, handle: bytes):
        self._check(self._lib.kc_xchg_import(self._ctx, peer, C.create_string_buffer(handle, 64)))

    def xchg_set_peer(self, peer, other: "Counter"):
        self._check(self._lib.kc_xchg_set_peer(self._ctx, peer, other._ctx))

    def xchg_count_local(self):
        self._check(self._lib.kc_xchg_count_local(self._ctx))

    def xchg_hist(self):
        """(device pointer of this rank's 1024-bin histogram, of the n_ranks x 1024 gather buffer)"""
        a, b = C.c_void_p(), C.c_void_p()
        self._check(self._lib.kc_xchg_hist(self._ctx, C.byref(a), C.byref(b)))
        return a.value, b.value

    def xchg_group_local(self):
        self._check(self._lib.kc_xchg_group_local(self._ctx))

    def xchg_pull(self):
        self._check(self._lib.kc_xchg_pull(self._ctx))

    def xchg_finish(self) -> "Run":
        h = C.c_void_p()
        self._check(self._lib.kc_xchg_finish(self._ctx, C.byref(h)))
        return Run(self, h)

    def xchg_fix_ranges(self, on=True):
        self._check(self._lib.kc_xchg_fix_ranges(self._ctx, 1 if on else 0))

    def xchg_info(self, n_ranks):
        """(bucket boundaries lo[0..n_ranks], records pulled, records pulled from peers) of the last exchange"""
        lo = (C.c_uint32 * 17)()
        a, b = C.c_uint64(), C.c_uint64()
        self._check(self._lib.kc_xchg_info(self._ctx, lo, C.byref(a), C.byref(b)))
        return [int(lo[i]) for i in range(n_ranks + 1)], a.value, b.value

    def debug_scalars(self) -> dict:
        """Device scalars of the most recent chunk (super-window path: SW_* of kc_super.cuh)."""
        out = (C.c_uint64 * 16)()
        self._check(self._lib.kc_debug_scalars(self._ctx, out))
        return {name: int(out[i]) for i, name in enumerate(SW_SCALARS)}

    def host_alloc(self, nbytes) -> np.ndarray:
        """Pinned host buffer as a uint8 array (freed with host_free)."""
        p = C.c_void_p()
        self._check(self._lib.kc_host_alloc(self._ctx, nbytes, C.byref(p)))
        return np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_ubyte)), shape=(max(nbytes, 1),))

    def host_free(self, arr):
        self._check(self._lib.kc_host_free(self._ctx, arr.ctypes.data))

    # -- one chunk
    def process_chunk(self, reads, slot=0) -> bytes:
        """processKMers (GPUHandler.cu:397-477) with the sort step on: host reads in, the
        chunk's sorted unique records out."""
        a = np.frombuffer(reads, dtype=np.uint8) if isinstance(reads, (bytes, bytearray)) else \
            np.ascontiguousarray(reads, dtype=np.uint8)
        n = C.c_uint64()
        cap = self._lib.kc_output_size(a.size, self.read_len, self.k) + self.record_size
        out = np.empty(max(cap, 1), dtype=np.uint8)
        self._check(self._lib.kc_process_chunk(self._ctx, slot, a.ctypes.data, a.size, out.ctypes.data, out.size,
                                               C.byref(n)))
        return out[: n.value].tobytes()

    def slot_buffer(self, slot) -> np.ndarray:
        p, cap = C.c_void_p(), C.c_uint64()
        self._check(self._lib.kc_slot_buffer(self._ctx, slot, C.byref(p), C.byref(cap)))
        return np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_ubyte)), shape=(cap.value,))

    def submit(self, slot, n_bytes):
        self._check(self._lib.kc_submit(self._ctx, slot, n_bytes))

    def wait(self, slot) -> Run:
        h = C.c_void_p()
        self._check(self._lib.kc_wait(self._ctx, slot, C.byref(h)))
        return Run(self, h)

    def submit_fastq(self, slot, text) -> tuple:
        """Raw FASTQ text (host bytes / uint8 array, starting at a record boundary) -> H2D ->
        device parse -> count on `slot`.  Returns (consumed_bytes, flags); flags != 0 means the
        text is not plain 4-line fixed-length FASTQ and nothing was submitted."""
        a = np.frombuffer(text, dtype=np.uint8) if isinstance(text, (bytes, bytearray)) else \
            np.ascontiguousarray(text, dtype=np.uint8)
        used, fl = C.c_uint64(), C.c_uint32()
        self._check(self._lib.kc_submit_fastq(self._ctx, slot, a.ctypes.data, a.size, C.byref(used), C.byref(fl)))
        return used.value, fl.value

    def parse_fastq_device(self, d_text, n_bytes, d_reads, reads_cap) -> tuple:
        """(n_reads, consumed_bytes, flags) of a device-resident FASTQ chunk parsed into d_reads."""
        n, used, fl = C.c_uint64(), C.c_uint64(), C.c_uint32()
        self._check(self._lib.kc_parse_fastq_device(self._ctx, d_text, n_bytes, d_reads, reads_cap, C.byref(n),
                                                    C.byref(used), C.byref(fl)))
        return n.value, used.value, fl.value

    def count_fastq(self, text, block_bytes=0) -> Run:
        """A whole FASTQ file image through the device parser in blocks with carry-over, counted
        and merged. Raises KcError(-1) if the text is not of the shape the device parser handles."""
        a = np.frombuffer(text, dtype=np.uint8) if isinstance(text, (bytes, bytearray)) else \
            np.ascontiguousarray(text, dtype=np.uint8)
        if a.size and a[-1] != 10:
            a = np.concatenate([a, np.array([10], dtype=np.uint8)])
        if block_bytes <= 0:
            block_bytes = 2 * self.max_chunk_bytes + 4096
        runs, pos = [], 0
        while pos < a.size:
            used, fl = self.submit_fastq(0, a[pos:pos + block_bytes])
            if fl:
                for r in runs:
                    r.free()
                raise KcError(-1, "FASTQ text is not plain 4-line fixed-length (flags=%d)" % fl)
            if used == 0:
                raise KcError(-4, "no whole record fits a block of %d bytes" % block_bytes)
            runs.append(self.wait(0))
            pos += used
        out = self.merge(runs)
        for r in runs:
            r.free()
        return out

    def count_device(self, d_ptr, n_bytes) -> Run:
        h = C.c_void_p()
        self._check(self._lib.kc_count_device(self._ctx, d_ptr, n_bytes, C.byref(h)))
        return Run(self, h)

    # -- runs
    def upload_run(self, records) -> Run:
        a = np.frombuffer(records, dtype=np.uint8) if isinstance(records, (bytes, bytearray)) else \
            np.ascontiguousarray(records, dtype=np.uint8)
        h = C.c_void_p()
        self._check(self._lib.kc_run_upload(self._ctx, a.ctypes.data, a.size, C.byref(h)))
        return Run(self, h)

    def run_from_device(self, keys_ptr, counts_ptr, n) -> Run:
        h = C.c_void_p()
        self._check(self._lib.kc_run_from_device(self._ctx, keys_ptr, counts_ptr, n, C.byref(h)))
        return Run(self, h)

    def place_next_run(self, d_keys, d_counts, d_offsets, cap_records, cap_ranges):
        """The next partitioned-path run is written into these device arrays if it fits (kc_place_next_run)."""
        self._check(self._lib.kc_place_next_run(self._ctx, C.c_void_p(d_keys), C.c_void_p(d_counts), C.c_void_p(d_offsets),
                                                int(cap_records), int(cap_ranges)))

    def peer_alloc(self, n_bytes):
        """Staging memory peers can map (kc_peer_alloc): returns (device pointer, 64-byte handle)."""
        p, h = C.c_void_p(), C.create_string_buffer(64)
        self._check(self._lib.kc_peer_alloc(self._ctx, int(n_bytes), C.byref(p), h))
        return p.value, h.raw

    def peer_open(self, handle):
        p = C.c_void_p()
        self._check(self._lib.kc_peer_open(self._ctx, C.create_string_buffer(bytes(handle), 64), C.byref(p)))
        return p.value

    def peer_close(self, ptr):
        self._check(self._lib.kc_peer_close(self._ctx, C.c_void_p(ptr)))

    def peer_free(self, ptr):
        self._check(self._lib.kc_peer_free(self._ctx, C.c_void_p(ptr)))

    def merge_parts(self, key_ptrs, count_ptrs, offset_ptrs, n_records, n_sub, prefix_bits) -> Run:
        """Combine pre-counted parts covering the same n_sub key ranges (kc_merge_parts)."""
        n = len(key_ptrs)
        ka = (C.c_void_p * n)(*key_ptrs)
        ca = (C.c_void_p * n)(*count_ptrs)
        oa = (C.c_void_p * n)(*offset_ptrs)
        na = (C.c_uint64 * n)(*n_records)
        h = C.c_void_p()
        self._check(self._lib.kc_merge_parts(self._ctx, n, ka, ca, oa, na, n_sub, prefix_bits, C.byref(h)))
        return Run(self, h)

    # -- lookups in a run (kc_run_lookup, kc_query_reads): key semantics, L and k are this counter's; the
    # run may come from another counter with the same k
    def lookup(self, run, keys) -> np.ndarray:
        """uint32 count in `run` of every key ([n, W] uint64 host array, the record key layout), 0 if absent.
        A canonical counter looks up min(x, rc(x)), so either strand can be asked."""
        k = np.ascontiguousarray(keys, dtype=np.uint64).reshape(-1, self.words)
        out = np.zeros(k.shape[0], dtype=np.uint32)
        self._check(self._lib.kc_run_lookup(self._ctx, run._h, k.ctypes.data, k.shape[0], out.ctypes.data))
        return out

    def lookup_device(self, run, d_keys, n, d_counts):
        """kc_run_lookup with device pointers: n x W uint64 keys in, n uint32 counts out."""
        self._check(self._lib.kc_run_lookup(self._ctx, run._h, d_keys, int(n), d_counts))

    def query_reads(self, run, reads, lo=1, hi=2**32 - 1, slot_counts=True) -> tuple:
        """Host reads (packed lines of read_len) against `run`: (slot_counts uint32[R, L-k+1] or None,
        hits uint32[R]). slot_counts[r, p] = count of read r's k-mer at position p (0: absent, or no k-mer
        there); hits[r] = windows of read r holding a k-mer whose count is in [lo, hi] (absent = 0)."""
        a = np.frombuffer(reads, dtype=np.uint8) if isinstance(reads, (bytes, bytearray)) else \
            np.ascontiguousarray(reads, dtype=np.uint8)
        R, nk = a.size // self.read_len, self.read_len - self.k + 1
        sc = np.zeros((R, nk), dtype=np.uint32) if slot_counts else None
        hits = np.zeros(R, dtype=np.uint32)
        self._check(self._lib.kc_query_reads(self._ctx, run._h, a.ctypes.data, a.size, int(lo), int(hi),
                                             sc.ctypes.data if sc is not None else None, hits.ctypes.data))
        return sc, hits

    def query_reads_device(self, run, d_reads, n_bytes, d_slot_counts, d_hits, lo=1, hi=2**32 - 1):
        """kc_query_reads with device pointers (d_reads 16-byte aligned); 0 for an output that is not wanted."""
        self._check(self._lib.kc_query_reads(self._ctx, run._h, d_reads, int(n_bytes), int(lo), int(hi),
                                             d_slot_counts or None, d_hits or None))

    def merge(self, runs) -> Run:
        n = len(runs)
        arr = (C.c_void_p * max(n, 1))(*[r._h for r in runs])
        h = C.c_void_p()
        self._check(self._lib.kc_merge_runs(self._ctx, arr, n, C.byref(h)))
        return Run(self, h)

    # -- whole input held in host memory: chunk, count, merge (the path KMerCounter::Start drives)
    def count_reads(self, reads, chunk_reads=0) -> Run:
        a = np.frombuffer(reads, dtype=np.uint8) if isinstance(reads, (bytes, bytearray)) else \
            np.ascontiguousarray(reads, dtype=np.uint8)
        L = self.read_len
        n_reads = a.size // L
        if chunk_reads <= 0:
            chunk_reads = max(1, self.max_chunk_bytes // L) if self.max_chunk_bytes else max(n_reads, 1)
        if self.max_chunk_bytes == 0:
            raise KcError(-1, "Counter was created without slots (max_chunk_bytes=0)")
        chunk_reads = min(chunk_reads, self.max_chunk_bytes // L)
        n_slots = 2
        runs, inflight = [], []
        pos, slot = 0, 0
        while pos < n_reads or inflight:
            if pos < n_reads and len(inflight) < n_slots:
                nr = min(chunk_reads, n_reads - pos)
                buf = self.slot_buffer(slot)
                buf[: nr * L] = a[pos * L:(pos + nr) * L]
                self.submit(slot, nr * L)
                inflight.append(slot)
                pos += nr
                slot = (slot + 1) % n_slots
            else:
                runs.append(self.wait(inflight.pop(0)))
        out = self.merge(runs)
        for r in runs:
            r.free()
        return out
