"""Error paths of the C ABI: a failed device allocation leaves no device memory behind and the
context usable.

KC_TEST_FAIL_ALLOC=n (read by kc_create) makes the context's n-th stream-ordered allocation fail once
with KC_ERR_NOMEM. Every scenario runs on a fresh Counter for n = 1, 2, ... until it no longer meets
the failure: the call must raise KcError(-3), the same call again on the same Counter must give the
oracle's answer, and once the runs are freed and the Counter is closed, the device's default memory
pool (where runs and scratch live) must hold exactly what it held before."""
import contextlib
import ctypes
import gc
import os

import numpy as np
import pytest

import oracle

pytestmark = pytest.mark.gpu

L, K, R = 100, 31, 3000
KC_ERR_NOMEM = -3
CU_MEMPOOL_ATTR_USED_MEM_CURRENT = 7


@pytest.fixture(scope="module")
def kc():
    import kmer_counter_b200 as kc
    return kc


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


# ----------------------------------------------------------------------------- inputs
@pytest.fixture(scope="module")
def data():
    import torch
    reads = oracle.gen_reads(R, L, 30000, 0.01, 0.002, seed=23)
    reads150 = oracle.gen_reads(1000, 150, 20000, 0.01, 0.002, seed=24)
    return {
        "reads": reads, "d": torch.from_numpy(reads.copy()).cuda(), "want": oracle.process_chunk(reads, L, K),
        "reads150": reads150, "d150": torch.from_numpy(reads150.copy()).cuda(),
        "want96": oracle.process_chunk(reads150, 150, 96),
    }


def _hold(stack, run):
    stack.callback(run.free)
    return run


def _records(c, d, r0, r1, read_len=L):
    """count_device of reads [r0, r1) of the device tensor d"""
    return c.count_device(d.data_ptr() + r0 * read_len, (r1 - r0) * read_len)


def _count_bytes(d, read_len=L):
    def run(c):
        with contextlib.ExitStack() as st:
            return _hold(st, _records(c, d, 0, d.numel() // read_len, read_len)).to_bytes()
    return run


@pytest.mark.parametrize("method,force_dup", [("sort", "0"), ("hash", "0"), ("hash_global", "0"), ("super", "0"),
                                              ("super", "1")])
def test_count_device(kc, monkeypatch, data, method, force_dup):
    monkeypatch.setenv("KC_SW_FORCE_DUP", force_dup)
    _exercise(kc, monkeypatch, lambda: kc.Counter(K, L, method=method), _count_bytes(data["d"]), data["want"])


def test_count_device_placement_k96(kc, monkeypatch, data):
    _exercise(kc, monkeypatch, lambda: kc.Counter(96, 150, method="place"), _count_bytes(data["d150"], 150),
              data["want96"])


def test_slot_submit_wait(kc, monkeypatch, data):
    reads = data["reads"]

    def run(c):
        c.slot_buffer(0)[:reads.size] = reads
        c.submit(0, reads.size)
        with contextlib.ExitStack() as st:
            return _hold(st, c.wait(0)).to_bytes()
    _exercise(kc, monkeypatch, lambda: kc.Counter(K, L, n_slots=1, max_chunk_bytes=reads.size), run, data["want"])


def test_accumulate_with_automatic_parts(kc, monkeypatch, data):
    """a plan for a third of the reads: the chunk is counted in automatic parts, the flush merges them"""
    def run(c):
        c.accum_begin(R // 3)
        c.accum_add_device(data["d"].data_ptr(), R * L)
        with contextlib.ExitStack() as st:
            return _hold(st, c.accum_flush()).to_bytes()
    _exercise(kc, monkeypatch, lambda: kc.Counter(K, L), run, data["want"], repeat=False)


# ---------------------------------------------------------------- what a run offers
def _on_run(d, op):
    def run(c):
        with contextlib.ExitStack() as st:
            return op(c, st, _hold(st, _records(c, d, 0, R)))
    return run


def _arrays(records, k):
    W = (k + 31) // 32
    rows = np.frombuffer(records, dtype=np.uint8).reshape(-1, 8 * W + 4)
    return np.ascontiguousarray(rows[:, :8 * W]).view("<u8"), np.ascontiguousarray(rows[:, 8 * W:]).view("<u4")[:, 0]


def test_run_filter(kc, monkeypatch, data):
    keys, counts = _arrays(data["want"], K)
    rows = np.frombuffer(data["want"], dtype=np.uint8).reshape(-1, 12)
    want = rows[(counts >= 2) & (counts <= 5)].tobytes()
    op = lambda c, st, run: _hold(st, run.filter(2, 5)).to_bytes()
    _exercise(kc, monkeypatch, lambda: kc.Counter(K, L), _on_run(data["d"], op), want)


def test_run_histogram(kc, monkeypatch, data):
    _, counts = _arrays(data["want"], K)
    want = np.bincount(np.minimum(counts, 63).astype(np.int64), minlength=64).tolist()
    op = lambda c, st, run: run.histogram(64).tolist()
    _exercise(kc, monkeypatch, lambda: kc.Counter(K, L), _on_run(data["d"], op), want)


def test_run_split(kc, monkeypatch, data):
    keys, _ = _arrays(data["want"], K)
    sp = np.array([[1 << 62], [2 << 62], [3 << 62]], dtype=np.uint64)
    want = [0] + [int(np.searchsorted(keys[:, 0], s[0], side="left")) for s in sp] + [len(keys)]
    op = lambda c, st, run: [int(x) for x in run.split(sp)]
    _exercise(kc, monkeypatch, lambda: kc.Counter(K, L), _on_run(data["d"], op), want)


def test_run_print(kc, monkeypatch, data):
    keys, counts = _arrays(data["want"], K)
    want = "".join("".join(oracle.print_word(int(w)) for w in ws) + " %d\n" % int(cn)
                   for ws, cn in zip(keys, counts)).encode()
    op = lambda c, st, run: run.print_text()
    _exercise(kc, monkeypatch, lambda: kc.Counter(K, L), _on_run(data["d"], op), want)


def test_run_upload(kc, monkeypatch, data):
    rows = np.frombuffer(data["want"], dtype=np.uint8).reshape(-1, 12)
    raw = np.repeat(rows, 2, axis=0).tobytes()     # each record twice in a row: the upload folds them
    want = oracle.merge_runs([raw], K)

    def run(c):
        with contextlib.ExitStack() as st:
            return _hold(st, c.upload_run(raw)).to_bytes()
    _exercise(kc, monkeypatch, lambda: kc.Counter(K, L), run, want)


# --------------------------------------------------------------------------- merges
def test_merge_two_runs(kc, monkeypatch, data):
    """two runs: the pairwise merge-path tree"""
    def run(c):
        with contextlib.ExitStack() as st:
            parts = [_hold(st, _records(c, data["d"], 0, R // 2)), _hold(st, _records(c, data["d"], R // 2, R))]
            return _hold(st, c.merge(parts)).to_bytes()
    _exercise(kc, monkeypatch, lambda: kc.Counter(K, L), run, data["want"])


def _thirds(c, st, d):
    parts = [_hold(st, _records(c, d, i * R // 3, (i + 1) * R // 3)) for i in range(3)]
    assert len({p.parts()[1:] for p in parts}) == 1 and parts[0].parts()[1] > 0      # one plan
    return parts


def test_merge_three_same_plan_runs(kc, monkeypatch, data):
    """three runs of the partitioned path with one plan: kc_merge_runs combines them with kc_merge_parts"""
    def run(c):
        with contextlib.ExitStack() as st:
            return _hold(st, c.merge(_thirds(c, st, data["d"]))).to_bytes()
    _exercise(kc, monkeypatch, lambda: kc.Counter(K, L, method="hash"), run, data["want"])


def test_merge_parts(kc, monkeypatch, data):
    """kc_merge_parts itself (inside kc_merge_runs a failed combine falls back to the tree)"""
    def run(c):
        with contextlib.ExitStack() as st:
            parts = _thirds(c, st, data["d"])
            arrays = [p.device_arrays() for p in parts]
            _, n_sub, prefix_bits = parts[0].parts()
            m = c.merge_parts([a[0] for a in arrays], [a[1] for a in arrays], [p.parts()[0] for p in parts],
                              [a[2] for a in arrays], n_sub, prefix_bits)
            return _hold(st, m).to_bytes()
    _exercise(kc, monkeypatch, lambda: kc.Counter(K, L, method="hash"), run, data["want"])
