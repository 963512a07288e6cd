"""Set operations of two runs on the GPU (kc_run_combine, Run.combine, `combine`): union, intersect,
subtract and subtract-counts, with the count modes sum, min, max, a and b for keys in both runs.

The model: numpy over oracle.records_to_arrays. Both runs' records are put in key order with a key's
A record just before its B record, and the table of kc_api.h decides which survive and with what
count. On the CPU the model is checked against a plain dict model and the identities between the
ops; on the GPU every op and mode of runs counted on the device is checked against it."""
import contextlib
import ctypes
import gc
import os
import subprocess

import numpy as np
import pytest

import oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
CLI = os.path.join(ROOT, "kmer-counter_b200", "host", "kmer_counter_b200")
U32 = 2**32

OPS = ["union", "intersect", "subtract", "subtract_counts"]
MODES = ["sum", "min", "max", "a", "b"]
DEFAULT = {"union": "sum", "intersect": "min", "subtract": "sum", "subtract_counts": "sum"}
# every (op, counts) the API takes; None = the default of the op
CASES = [(op, m) for op in OPS for m in ([None] + MODES if op in ("union", "intersect") else [None, "sum"])]
TILE = {1: 6144, 2: 4096, 3: 2048, 4: 2048}       # records per merge tile (kc_merge.cu MergeCfg) of each key width


# ---------------------------------------------------------------------------- model
def _dtype(W):
    return np.dtype([("w", "<u8", (W,)), ("c", "<u4")])


def _records(keys, counts, W):
    out = np.zeros(len(counts), dtype=_dtype(W))
    out["w"] = np.asarray(keys, dtype=np.uint64).reshape(-1, W)
    out["c"] = np.asarray(counts, dtype=np.uint64).astype(np.uint32)
    return out.tobytes()


class Pair:
    """the records of runs A and B in key order, a key's A record right before its B record"""

    def __init__(self, a: bytes, b: bytes, k):
        self.W = oracle.words(k)
        ka, ca = oracle.records_to_arrays(a, k)
        kb, cb = oracle.records_to_arrays(b, k)
        keys = np.concatenate([ka, kb])
        src = np.concatenate([np.zeros(len(ka), np.uint8), np.ones(len(kb), np.uint8)])
        order = np.lexsort((src,) + tuple(keys[:, w] for w in range(self.W - 1, -1, -1)))
        self.keys, self.src = keys[order], src[order]
        self.cnt = np.concatenate([ca, cb]).astype(np.uint64)[order]
        n = len(order)
        first = np.zeros(n, dtype=bool)                      # the A record of a key in both runs
        if n > 1:
            first[:-1] = np.all(self.keys[1:] == self.keys[:-1], axis=1)
        second = np.zeros(n, dtype=bool)
        second[1:] = first[:-1]
        assert not np.any(first & (self.src == 1)), "a run is not key-unique"
        self.pair = np.flatnonzero(first)
        self.only_a = (self.src == 0) & ~first
        self.only_b = (self.src == 1) & ~second

    def combine(self, op, counts=None) -> bytes:
        counts = counts or DEFAULT[op]
        a, b = self.cnt[self.pair], self.cnt[self.pair + 1]
        m = {"sum": (a + b) % np.uint64(U32), "min": np.minimum(a, b), "max": np.maximum(a, b), "a": a, "b": b}[counts]
        keep = np.zeros(len(self.cnt), dtype=bool)
        out = self.cnt.copy()
        if op in ("union", "intersect"):
            keep[self.pair] = True
            out[self.pair] = m
            if op == "union":
                keep |= self.only_a | self.only_b
        else:
            keep |= self.only_a
            if op == "subtract_counts":
                gt = a > b
                keep[self.pair[gt]] = True
                out[self.pair[gt]] = a[gt] - b[gt]
        return _records(self.keys[keep], out[keep], self.W)


def model(a, b, k, op, counts=None) -> bytes:
    return Pair(a, b, k).combine(op, counts)


def dict_model(a, b, k, op, counts=None) -> bytes:
    """the table of kc_api.h, one key at a time"""
    counts = counts or DEFAULT[op]
    da = {tuple(int(w) for w in key): int(c) for key, c in zip(*oracle.records_to_arrays(a, k))}
    db = {tuple(int(w) for w in key): int(c) for key, c in zip(*oracle.records_to_arrays(b, k))}
    f = {"sum": lambda x, y: (x + y) % U32, "min": min, "max": max, "a": lambda x, y: x, "b": lambda x, y: y}[counts]
    out = {}
    for key in da.keys() | db.keys():
        if key in da and key in db:
            if op in ("union", "intersect"):
                out[key] = f(da[key], db[key])
            elif op == "subtract_counts" and da[key] > db[key]:
                out[key] = da[key] - db[key]
        elif key in da:
            if op != "intersect":
                out[key] = da[key]
        elif op == "union":
            out[key] = db[key]
    ks = sorted(out)                                          # tuples of unsigned words: word 0 first
    return _records(np.array(ks, dtype=np.uint64).reshape(-1, oracle.words(k)), [out[x] for x in ks], oracle.words(k))


def derived(a: bytes, k, seed) -> bytes:
    """B from A: every third record dropped, counts changed (a > b, a = b, a < b) and keys A lacks added"""
    W = oracle.words(k)
    keys, cnt = oracle.records_to_arrays(a, k)
    rng = np.random.default_rng(seed)
    sel = np.arange(len(cnt)) % 3 != 0
    bk, bc = keys[sel], cnt[sel].astype(np.int64)
    step = np.arange(len(bc)) % 3                            # 0: b < a (where a > 0), 1: b = a, 2: b > a
    bc = np.where(step == 0, np.maximum(bc - 1, 0), np.where(step == 2, bc + rng.integers(1, 4, len(bc)), bc))
    have = {tuple(x) for x in keys.tolist()}
    extra = keys[::5].copy()
    extra[:, W - 1] += np.uint64(1 << 20)
    extra = np.array([x for x in extra.tolist() if tuple(x) not in have], dtype=np.uint64).reshape(-1, W)
    ak = np.concatenate([bk, extra])
    ac = np.concatenate([bc, rng.integers(1, 9, len(extra))])
    order = np.lexsort(tuple(ak[:, w] for w in range(W - 1, -1, -1)))
    return _records(ak[order], ac[order], W)


def _nrec(records, k):
    return len(records) // oracle.record_size(k)


def _keyset(records, k):
    return {tuple(x) for x in oracle.records_to_arrays(records, k)[0].tolist()}


# ------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("k", [31, 40])
def test_model_matches_dict_model(k):
    a = open(os.path.join(GOLD, "small_k%d.records" % k), "rb").read()
    b = derived(a, k, k)
    pa, pb = Pair(a, b, k), Pair(b, a, k)
    # the derived run has every kind of key: in both with a > b, a = b, a < b; only in A; only in B
    ca, cb = pa.cnt[pa.pair], pa.cnt[pa.pair + 1]
    assert np.any(ca > cb) and np.any(ca == cb) and np.any(ca < cb)
    assert pa.only_a.any() and pa.only_b.any()
    for op, m in CASES:
        assert pa.combine(op, m) == dict_model(a, b, k, op, m), (op, m)
        assert pb.combine(op, m) == dict_model(b, a, k, op, m), (op, m)
    assert model(a, b"", k, "union") == a and model(b"", a, k, "union") == a
    assert model(a, b"", k, "intersect") == b"" and model(a, a, k, "subtract") == b""


@pytest.mark.parametrize("k", [31, 40])
def test_identities(k):
    a = open(os.path.join(GOLD, "small_k%d.records" % k), "rb").read()
    b = derived(a, k, k + 1)
    p = Pair(a, b, k)
    union, inter, sub = p.combine("union"), p.combine("intersect"), p.combine("subtract")
    assert _nrec(union, k) + _nrec(inter, k) == _nrec(a, k) + _nrec(b, k)
    assert _keyset(sub, k) | _keyset(inter, k) == _keyset(a, k)
    assert not (_keyset(sub, k) & _keyset(inter, k))
    assert union == oracle.merge_runs([a, b], k)
    # a = b: min = max = a = b, subtract_counts keeps nothing
    q = Pair(a, a, k)
    for m in ("min", "max", "a", "b"):
        assert q.combine("intersect", m) == a
    assert q.combine("subtract_counts") == b""


# ------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def kc():
    import kmer_counter_b200 as kc
    return kc


def _counter(kc, k, L, mode, **kw):
    return kc.Counter(k, L, compat="ref" if mode == "ref" else "strict", canonical=mode == "canonical", **kw)


def _count(c, reads):
    import torch
    d = torch.from_numpy(np.ascontiguousarray(reads)).cuda()
    return c.count_device(d.data_ptr(), d.numel())


def _check_all(c, ra, rb, k, merge_too=True):
    """every op and mode of runs ra, rb against the model; the inputs are unchanged"""
    a, b = ra.to_bytes(), rb.to_bytes()
    p = Pair(a, b, k)
    for op, m in CASES:
        r = ra.combine(rb, op, m)
        want = p.combine(op, m)
        assert r.to_bytes() == want, (op, m)
        assert len(r) == _nrec(want, k)
        r.free()
    if merge_too:
        mg = c.merge([ra, rb])
        u = ra.combine(rb, "union", "sum")
        assert u.to_bytes() == mg.to_bytes()
        mg.free()
        u.free()
    assert ra.to_bytes() == a and rb.to_bytes() == b


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["ref", "strict", "canonical"])
@pytest.mark.parametrize("k", [31, 40, 63, 96, 128])
def test_every_op_and_mode_matches_model(kc, k, mode):
    """A and B: two read sets of one genome (large overlap), of two genomes (nearly disjoint), and the
    same reads (A = B)"""
    L, R, G = 150, 3000, 30000
    s1 = oracle.gen_reads(R, L, G, 0.001, 0.002, seed=k)
    pairs = {"one genome": (s1, oracle.gen_reads(R, L, G, 0.001, 0.002, seed=k, first_read=R)),
             "two genomes": (s1, oracle.gen_reads(R, L, G, 0.001, 0.002, seed=k + 1000)),
             "same reads": (s1, s1)}
    with _counter(kc, k, L, mode) as c:
        for name, (x, y) in pairs.items():
            ra, rb = _count(c, x), _count(c, y)
            if mode == "ref":
                assert ra.to_bytes() == oracle.count(x, L, k)
            elif mode == "strict":
                assert ra.to_bytes() == oracle.naive_count(x, L, k, strict=True)
            n_both = len(Pair(ra.to_bytes(), rb.to_bytes(), k).pair)
            if name == "one genome":
                assert n_both > len(ra) // 3, n_both
            elif name == "two genomes":
                assert n_both < len(ra) // 100, n_both
            _check_all(c, ra, rb, k)
            _check_all(c, rb, ra, k, merge_too=False)
            ra.free()
            rb.free()


@pytest.mark.gpu
@pytest.mark.parametrize("k", [31, 40, 96, 128])
def test_empty_inputs(kc, k):
    W = oracle.words(k)
    rec = _records(_sorted_keys(5000, W, k), np.arange(5000) % 7, W)
    with kc.Counter(k, k) as c:
        full, empty = c.upload_run(rec), c.upload_run(b"")
        for ra, rb, a, b in ((empty, full, b"", rec), (full, empty, rec, b""), (empty, empty, b"", b"")):
            for op, m in CASES:
                r = ra.combine(rb, op, m)
                assert r.to_bytes() == model(a, b, k, op, m), (len(ra), len(rb), op, m)
                r.free()
        for r in (full, empty):
            r.free()


@pytest.mark.gpu
def test_strict_skip_run(kc):
    """strict mode hides the empty slots' key-0 record of a run (skip = 1): combine does not see it"""
    L, k = 100, 31
    x = oracle.gen_reads(3000, L, 30000, 0.01, 0.02, seed=5)
    y = oracle.gen_reads(3000, L, 30000, 0.01, 0.0, seed=5, first_read=3000)
    with _counter(kc, k, L, "strict", method="sort") as c:
        ra, rb = _count(c, x), _count(c, y)
        assert ra.to_bytes() == oracle.naive_count(x, L, k, strict=True)
        assert oracle.records_to_arrays(ra.to_bytes(), k)[1].min() >= 1
        _check_all(c, ra, rb, k)
        _check_all(c, rb, ra, k, merge_too=False)
        ra.free()
        rb.free()


@pytest.mark.gpu
def test_ref_phantom_in_one_or_both(kc):
    """the ref-mode zero-count key-0 record is an ordinary record: in A only, B only, or both"""
    L, k = 100, 31
    with_n = oracle.gen_reads(3000, L, 30000, 0.01, 0.01, seed=6)
    without = oracle.gen_reads(3000, L, 30000, 0.01, 0.0, seed=6, first_read=3000)
    with _counter(kc, k, L, "ref") as c:
        ra, rb = _count(c, with_n), _count(c, without)
        ka, ca = oracle.records_to_arrays(ra.to_bytes(), k)
        assert ka[0, 0] == 0 and ca[0] == 0                     # the phantom
        kb, cb = oracle.records_to_arrays(rb.to_bytes(), k)
        assert not (kb[0, 0] == 0 and cb[0] == 0)
        rc = _count(c, oracle.gen_reads(3000, L, 30000, 0.01, 0.01, seed=6, first_read=6000))
        for x, y in ((ra, rb), (rb, ra), (ra, rc)):
            _check_all(c, x, y, k)
        for r in (ra, rb, rc):
            r.free()


@pytest.mark.gpu
@pytest.mark.parametrize("k", [31, 40, 96, 128])
def test_counts_near_2_32(kc, k):
    """sum wraps at 2^32, min / max of the extremes, subtract-counts with a = b"""
    W = oracle.words(k)
    keys = _sorted_keys(12, W, k)
    top = U32 - 1
    ca = [top, top, top, 0, 1, 2**31, top, 5, 0, top, 7, 9]
    cb = [1, top, 0, top, top, 2**31, top - 1, 5, 0, 2**31, 7, 9]
    a = _records(keys[:10], ca[:10], W)
    b = _records(np.concatenate([keys[:10], keys[10:]]), cb, W)
    with kc.Counter(k, k) as c:
        ra, rb = c.upload_run(a), c.upload_run(b)
        u = ra.combine(rb, "union")
        assert oracle.records_to_arrays(u.to_bytes(), k)[1][:3].tolist() == [0, top - 1, top]
        u.free()
        _check_all(c, ra, rb, k)
        _check_all(c, rb, ra, k, merge_too=False)
        sc = ra.combine(ra, "subtract_counts")
        assert len(sc) == 0
        for r in (ra, rb, sc):
            r.free()


def _sorted_keys(n, W, seed):
    """n distinct keys of W words, ascending (word 0 first)"""
    rng = np.random.default_rng(seed)
    lead = np.unique(rng.integers(0, 2**63, size=n + n // 8 + 16, dtype=np.uint64))[:n]
    keys = np.zeros((len(lead), W), dtype=np.uint64)
    keys[:, 0] = lead
    if W > 1:
        keys[:, 1:] = rng.integers(0, 2**63, size=(len(lead), W - 1), dtype=np.uint64)
    assert len(lead) == n
    return keys


def _pair_split_at(a, b, k, d):
    """does the merge-path diagonal d (ties to A) separate an equal (A, B) pair?"""
    p = Pair(a, b, k)
    na = int(np.count_nonzero(p.src[:d] == 0))
    nb = d - na
    ka, kb = oracle.records_to_arrays(a, k)[0], oracle.records_to_arrays(b, k)[0]
    return 0 < na and nb < len(kb) and np.array_equal(ka[na - 1], kb[nb])


@pytest.mark.gpu
@pytest.mark.parametrize("k", [31, 40, 96, 128])
def test_sizes_around_the_tile(kc, k):
    """na + nb at T - 1, T, T + 1 and 2T + 1 (T = records per tile), and an equal pair across a cut"""
    W = oracle.words(k)
    T = TILE[W]
    rng = np.random.default_rng(k)
    with kc.Counter(k, k) as c:
        cases = []
        for total in (T - 1, T, T + 1, 2 * T + 1, 3 * T):
            pool = _sorted_keys(total, W, total + k)
            side = rng.integers(0, 3, total)                 # 0: A only, 1: B only, 2: both (counted twice)
            in_a, in_b = side != 1, side != 0
            # trim B so that na + nb == total
            extra = int(in_a.sum() + in_b.sum() - total)
            in_b[np.flatnonzero(in_b)[:extra]] = False
            cases.append((pool[in_a], pool[in_b], False))
        for n in (T // 2, T // 2 + 1, T, 2 * T):
            # B = one key below all of A's, then A's keys: every cut at an even diagonal splits a pair
            pool = _sorted_keys(n + 1, W, n + k)
            cases.append((pool[1:], pool, True))
        for ka, kb, split in cases:
            a = _records(ka, rng.integers(0, 6, len(ka)), W)
            b = _records(kb, rng.integers(0, 6, len(kb)), W)
            if split:
                assert _pair_split_at(a, b, k, T)           # the partition kernel must nudge this cut
            ra, rb = c.upload_run(a), c.upload_run(b)
            _check_all(c, ra, rb, k)
            _check_all(c, rb, ra, k, merge_too=False)
            ra.free()
            rb.free()


@pytest.mark.gpu
@pytest.mark.parametrize("k", [31, 63])
def test_large_runs_built_on_the_device(kc, k):
    """about 12 M records per side from device arrays (kc_run_from_device): thousands of tiles"""
    import torch
    W = oracle.words(k)
    n = 12_000_000
    rng = np.random.default_rng(k)

    def keys_of(lead):
        keys = np.zeros((len(lead), W), dtype=np.uint64)
        keys[:, 0] = lead
        if W > 1:
            keys[:, 1] = lead * np.uint64(0x9E3779B97F4A7C15) >> np.uint64(1)
        return keys

    ka = keys_of(np.arange(n, dtype=np.uint64) * np.uint64(2 << 20))    # A: multiples of 2, B: of 3 (x 2^20)
    kb = keys_of(np.arange(n, dtype=np.uint64) * np.uint64(3 << 20))
    ca = rng.integers(0, 50, n).astype(np.uint32)
    cb = rng.integers(0, 50, n).astype(np.uint32)
    with kc.Counter(k, k) as c:
        da, db = torch.from_numpy(ka.view(np.int64)).cuda(), torch.from_numpy(kb.view(np.int64)).cuda()
        dca, dcb = torch.from_numpy(ca.view(np.int32)).cuda(), torch.from_numpy(cb.view(np.int32)).cuda()
        ra = c.run_from_device(da.data_ptr(), dca.data_ptr(), n)
        rb = c.run_from_device(db.data_ptr(), dcb.data_ptr(), n)
        a, b = _records(ka, ca, W), _records(kb, cb, W)
        del ka, kb
        p = Pair(a, b, k)
        assert len(p.pair) == 2 * (n - 1) // 6 + 1                      # the multiples of 6 up to A's last
        for op, m in (("union", None), ("union", "max"), ("intersect", None), ("subtract", None),
                      ("subtract_counts", None)):
            r = ra.combine(rb, op, m)
            assert r.to_bytes() == p.combine(op, m), (op, m)
            r.free()
        assert ra.to_bytes() == a and rb.to_bytes() == b
        ra.free()
        rb.free()


@pytest.mark.gpu
def test_argument_errors(kc):
    W31 = _records(_sorted_keys(100, 1, 1), np.ones(100), 1)
    W40 = _records(_sorted_keys(100, 2, 2), np.ones(100), 2)
    with kc.Counter(31, 31) as c31, kc.Counter(40, 40) as c40:
        a, b, x = c31.upload_run(W31), c31.upload_run(W31), c40.upload_run(W40)
        for fn in (lambda: a.combine(x, "union"), lambda: x.combine(a, "intersect"),
                   lambda: a.combine(b, "subtract", "min"), lambda: a.combine(b, "subtract_counts", "b"),
                   lambda: a.combine(b, "xor"), lambda: a.combine(b, "union", "mean")):
            with pytest.raises(kc.KcError) as e:
                fn()
            assert e.value.code == -1
        lib = c31._lib
        for op, cm in ((4, 0), (0, 5), (2, 1), (3, 4), (1, 0xFFFFFFFF)):
            h = ctypes.c_void_p(123)
            assert lib.kc_run_combine(c31._ctx, a._h, b._h, op, cm, ctypes.byref(h)) == -1, (op, cm)
            assert h.value is None
        h = ctypes.c_void_p()
        assert lib.kc_run_combine(c31._ctx, a._h, None, 0, 0, ctypes.byref(h)) == -1
        assert lib.kc_run_combine(c31._ctx, a._h, b._h, 0, 0, None) == -1
        # the runs are unchanged and still combine
        r = a.combine(b, "intersect", "max")
        assert r.to_bytes() == W31
        for q in (a, b, x, r):
            q.free()


# ------------------------------------------------- injected allocation failures
KC_ERR_NOMEM = -3
CU_MEMPOOL_ATTR_USED_MEM_CURRENT = 7


def _pool_used():
    """bytes in use from device 0's default memory pool (cudaMallocAsync without an explicit pool)"""
    cu = ctypes.CDLL("libcuda.so.1")
    cu.cuDeviceGetDefaultMemPool.argtypes = [ctypes.POINTER(ctypes.c_void_p), ctypes.c_int]
    cu.cuMemPoolGetAttribute.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p]
    dev, pool, used = ctypes.c_int(), ctypes.c_void_p(), ctypes.c_uint64()
    assert cu.cuDeviceGet(ctypes.byref(dev), 0) == 0
    assert cu.cuDeviceGetDefaultMemPool(ctypes.byref(pool), dev.value) == 0
    assert cu.cuMemPoolGetAttribute(pool, CU_MEMPOOL_ATTR_USED_MEM_CURRENT, ctypes.byref(used)) == 0
    return used.value


def _exercise(kc, monkeypatch, make_counter, scenario, want, repeat=True):
    """Inject the failure at the n-th allocation for n = 1, 2, ... until the scenario runs through;
    returns that n. repeat=False: after a failure the Counter's state is not reused (only the code
    and the absence of a leak are checked)."""
    import torch
    if "cudaMallocAsync" in os.environ.get("PYTORCH_CUDA_ALLOC_CONF", ""):
        pytest.skip("torch allocates from the same default pool")
    gc.collect()
    torch.cuda.synchronize()
    base = _pool_used()
    for n in range(1, 65):
        monkeypatch.setenv("KC_TEST_FAIL_ALLOC", str(n))
        c = make_counter()
        monkeypatch.delenv("KC_TEST_FAIL_ALLOC")
        failed = False
        try:
            try:
                got = scenario(c)
            except kc.KcError as e:
                assert e.code == KC_ERR_NOMEM, (n, str(e))
                failed = True
                got = scenario(c) if repeat else want
            assert got == want, n
        finally:
            c.close()
        torch.cuda.synchronize()
        used = _pool_used()
        assert used == base, "allocation %d failed: %d bytes left in the pool" % (n, used - base)
        if not failed:
            assert n > 1, "the scenario allocates nothing"
            return n
    pytest.fail("the scenario still fails after 64 injected allocation failures")


@pytest.mark.gpu
@pytest.mark.parametrize("op,counts", [("union", "sum"), ("union", "max"), ("intersect", None), ("subtract", None),
                                       ("subtract_counts", None)])
def test_allocation_failures(kc, monkeypatch, op, counts):
    L, k = 100, 31
    a = oracle.count(oracle.gen_reads(3000, L, 30000, 0.01, 0.002, seed=23), L, k)
    b = oracle.count(oracle.gen_reads(3000, L, 30000, 0.01, 0.002, seed=23, first_read=3000), L, k)
    want = model(a, b, k, op, counts)

    def run(c):
        with contextlib.ExitStack() as st:
            ra = c.upload_run(a)
            st.callback(ra.free)
            rb = c.upload_run(b)
            st.callback(rb.free)
            r = ra.combine(rb, op, counts)
            st.callback(r.free)
            return r.to_bytes()
    _exercise(kc, monkeypatch, lambda: kc.Counter(k, L), run, want)


# ------------------------------------------------------------------------- ranks
@pytest.mark.gpu
@pytest.mark.parametrize("P", [2, 3, 4])
def test_exchange_ranks_combine_per_rank(kc, P):
    """two exchanges, the second cut at the first's key ranges (kc_xchg_fix_ranges): rank r's runs of
    A and B cover one key range, so the per-rank results concatenate to the result over all reads"""
    import torch
    from kmer_counter_b200 import engine
    R, L, k = 12000, 100, 31
    xa = oracle.gen_reads(R, L, 60000, 0.01, 0.002, seed=P)
    xb = oracle.gen_reads(R, L, 60000, 0.01, 0.002, seed=P, first_read=R)
    want_a, want_b = oracle.count(xa, L, k), oracle.count(xb, L, k)
    p = Pair(want_a, want_b, k)
    per = (R + P - 1) // P
    cs = [kc.Counter(k, L, method="super") for _ in range(P)]
    try:
        bufs, runs = [], []
        for i, reads in enumerate((xa, xb)):
            for r, c in enumerate(cs):
                if i == 0:
                    c.xchg_begin(r, P, max(per, 16))
                part = reads[r * per * L:(r + 1) * per * L]
                d = torch.from_numpy(part.copy()).cuda()
                bufs.append(d)
                c.accum_add_device(d.data_ptr(), len(part))
            runs.append(engine.xchg_run_all(cs))
            if i == 0:
                for c in cs:
                    c.xchg_fix_ranges(True)
        ra, rb = runs
        assert b"".join(r.to_bytes() for r in ra) == want_a
        assert b"".join(r.to_bytes() for r in rb) == want_b
        for op, m in CASES:
            got = [x.combine(y, op, m) for x, y in zip(ra, rb)]
            assert b"".join(g.to_bytes() for g in got) == p.combine(op, m), (op, m)
            for g in got:
                g.free()
        for r in ra + rb:
            r.free()
    finally:
        for c in cs:
            c.close()


# ------------------------------------------------------------------- command line
def _stats(stderr):
    return dict(t.split("=") for t in stderr.split() if "=" in t and t.split("=")[1].isdigit())


def _cli(*args):
    r = subprocess.run([CLI, "combine"] + [str(x) for x in args], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return _stats(r.stderr)


@pytest.mark.gpu
@pytest.mark.parametrize("k", [31, 96])
def test_cli_combine(kc, tmp_path, k):
    L, R = 150, 6000
    xa = oracle.gen_reads(R, L, 200000, 0.005, 0.002, seed=k)
    xb = oracle.gen_reads(R, L, 200000, 0.005, 0.002, seed=k, first_read=R)
    xs = oracle.gen_reads(300, L, 200000, 0.005, 0.0, seed=k, first_read=3 * R)        # a small B: runs out first
    fa, fb, fs, out = tmp_path / "a.bin", tmp_path / "b.bin", tmp_path / "s.bin", tmp_path / "out.bin"
    with _counter(kc, k, L, "ref") as c:
        for reads, f in ((xa, fa), (xb, fb), (xs, fs)):
            r = _count(c, reads)
            r.write(str(f))
            r.free()
    a, b, s = fa.read_bytes(), fb.read_bytes(), fs.read_bytes()
    S = oracle.record_size(k)
    p, ps, pr = Pair(a, b, k), Pair(a, s, k), Pair(s, a, k)
    # every op with its default count mode, in one piece and in many
    for op in OPS:
        for extra in ((), ("pieceRecords=1000",)):
            st = _cli(op, fa, fb, out, k, *extra)
            want = p.combine(op)
            assert out.read_bytes() == want, (op, extra)
            assert int(st["a_records"]) == len(a) // S and int(st["b_records"]) == len(b) // S
            assert int(st["records"]) == len(want) // S
            if extra:          # every piece but the last empties a full buffer of 1000 records
                assert max(len(a), len(b)) // S // 1000 <= int(st["pieces"]) <= (len(a) + len(b)) // S // 1000 + 1
            else:
                assert int(st["pieces"]) == 1
    # counts= given
    for op, m in (("union", "max"), ("union", "a"), ("intersect", "sum"), ("intersect", "b"), ("subtract", "sum")):
        _cli(op, fa, fb, out, k, "counts=%s" % m, "pieceRecords=777")
        assert out.read_bytes() == p.combine(op, m), (op, m)
    # minCount= / maxCount= on the combined counts
    keys, cnt = oracle.records_to_arrays(p.combine("union", "sum"), k)
    for extra, lo, hi in ((("minCount=3",), 3, U32 - 1), (("maxCount=2",), 0, 2), (("minCount=2", "maxCount=4"), 2, 4)):
        st = _cli("union", fa, fb, out, k, *extra, "pieceRecords=5000")
        sel = (cnt >= lo) & (cnt <= hi)
        assert out.read_bytes() == _records(keys[sel], cnt[sel], oracle.words(k)), extra
        assert int(st["records"]) == int(sel.sum())
    # one file runs out in the first piece while the other goes on, from either side
    for op in OPS:
        _cli(op, fa, fs, out, k, "pieceRecords=700")
        assert out.read_bytes() == ps.combine(op), op
        _cli(op, fs, fa, out, k, "pieceRecords=700")
        assert out.read_bytes() == pr.combine(op), op
    # empty inputs
    fe = tmp_path / "e.bin"
    fe.write_bytes(b"")
    for x, y in ((fe, fa), (fa, fe), (fe, fe)):
        st = _cli("union", x, y, out, k, "pieceRecords=999")
        assert out.read_bytes() == (a if (x, y) != (fe, fe) else b"")
    # bad arguments
    for args in (("xor", fa, fb, out, k), ("union", fa, fb, out, k, "counts=mean"),
                 ("subtract", fa, fb, out, k, "counts=min"), ("union", fa, fb, out, k, "pieceRecords=0")):
        r = subprocess.run([CLI, "combine"] + [str(x) for x in args], capture_output=True, text=True)
        assert r.returncode != 0, args
