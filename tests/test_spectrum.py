"""Count spectrum (kc_run_histogram, Run.histogram, multigpu.histogram, histoFile=, `histo`) and
count-range filtering (kc_run_filter, Run.filter, minCount= / maxCount=) of finished runs.

The model: np.bincount of the oracle's record counts, the last bin clipped to "count >= n_bins - 1",
and a count mask over the oracle's records. On the CPU the model is checked against hand-computed
spectra of the golden record files; on the GPU every counting path's run is checked against it."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

import oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
CLI = os.path.join(ROOT, "kmer-counter_b200", "host", "kmer_counter_b200")
U32_MAX = 2**32 - 1


# ---------------------------------------------------------------------------- model
def spectrum(counts, n_bins):
    """h[c] = records with count c for c < n_bins - 1, h[n_bins - 1] = records with count >= n_bins - 1"""
    c = np.minimum(np.asarray(counts, dtype=np.uint64), np.uint64(n_bins - 1)).astype(np.int64)
    return np.bincount(c, minlength=n_bins).astype(np.uint64)


def keep(records: bytes, k, lo, hi) -> bytes:
    """the records whose count is in [lo, hi], in order"""
    S = oracle.record_size(k)
    rows = np.frombuffer(records, dtype=np.uint8).reshape(-1, S)
    _, c = oracle.records_to_arrays(records, k)
    return rows[(c >= lo) & (c <= hi)].tobytes()


def counts_of(records: bytes, k):
    return oracle.records_to_arrays(records, k)[1]


def histo_text(hist) -> str:
    """histoFile= / `histo`: "c n" for c = 1..len(hist)-1 with n > 0 (the last line means >= c)"""
    return "".join("%d %d\n" % (c, int(n)) for c, n in enumerate(hist) if c >= 1 and n)


# canonical model, as in test_canonical.py: the oracle's strict count with every key folded by min(x, rc(x))
def _word_revcomp(x):
    """reverse complement of 32 bases per uint64 (numpy, vectorised): 2-bit groups reversed, code ^ 3"""
    x = x.copy()
    for sh, m in ((2, 0x3333333333333333), (4, 0x0F0F0F0F0F0F0F0F), (8, 0x00FF00FF00FF00FF),
                  (16, 0x0000FFFF0000FFFF), (32, 0x00000000FFFFFFFF)):
        m, sh = np.uint64(m), np.uint64(sh)
        x = ((x >> sh) & m) | ((x & m) << sh)
    return ~x


def canonical_count(reads, L, k) -> bytes:
    W = (k + 31) // 32
    dt = np.dtype([("w", "<u8", (W,)), ("c", "<u4")])
    fwd = np.frombuffer(oracle.naive_count(reads, L, k, strict=True), dtype=dt)
    if len(fwd) == 0:
        return b""
    x = np.ascontiguousarray(fwd["w"]).reshape(-1, W)
    r = _word_revcomp(x[:, ::-1])
    sh = 2 * (32 * W - k)                          # the zero tail of the last word
    if sh:
        nxt = np.concatenate([r[:, 1:], np.zeros((len(r), 1), dtype=np.uint64)], axis=1)
        r = (r << np.uint64(sh)) | (nxt >> np.uint64(64 - sh))
    lt = np.zeros(len(x), dtype=bool)
    decided = np.zeros(len(x), dtype=bool)
    for q in range(W):                             # lexicographic, word 0 first
        lt |= ~decided & (r[:, q] < x[:, q])
        decided |= r[:, q] != x[:, q]
    key = np.where(lt[:, None], r, x)
    cnt = fwd["c"].astype(np.uint64)
    order = np.lexsort(key.T[::-1])
    key, cnt = key[order], cnt[order]
    new = np.ones(len(key), dtype=bool)
    new[1:] = np.any(key[1:] != key[:-1], axis=1)
    starts = np.flatnonzero(new)
    out = np.zeros(len(starts), dtype=dt)
    out["w"] = key[starts]
    out["c"] = (np.add.reduceat(cnt, starts) & np.uint64(0xFFFFFFFF)).astype(np.uint32)
    return out.tobytes()


def model_run(reads, L, k, mode) -> bytes:
    if mode == "ref":
        return oracle.count(reads, L, k)
    if mode == "strict":
        return oracle.naive_count(reads, L, k, strict=True)
    return canonical_count(reads, L, k)


# ------------------------------------------------------------------------------ CPU
GOLDEN_SPECTRA = {                          # counted by hand from the golden files: {count: records}
    31: {0: 1, 1: 2574, 2: 498, 3: 205, 4: 48, 5: 1},
    40: {0: 1, 1: 1998, 2: 287, 3: 62, 4: 2},
}


@pytest.mark.parametrize("k", [31, 40])
def test_model_matches_hand_computed_spectra(k):
    rec = open(os.path.join(GOLD, "small_k%d.records" % k), "rb").read()
    c = counts_of(rec, k)
    want = GOLDEN_SPECTRA[k]
    assert sum(want.values()) == len(c)
    full = spectrum(c, 10001)
    assert {i: int(n) for i, n in enumerate(full) if n} == want
    # clipping into the high bin
    assert spectrum(c, 2).tolist() == [want[0], len(c) - want[0]]
    assert spectrum(c, 3).tolist() == [want[0], want[1], len(c) - want[0] - want[1]]
    # the count mask
    assert len(keep(rec, k, 2, U32_MAX)) // oracle.record_size(k) == len(c) - want[0] - want[1]
    assert len(keep(rec, k, 1, 1)) // oracle.record_size(k) == want[1]
    assert keep(rec, k, 0, U32_MAX) == rec and keep(rec, k, 6, 50) == b""


def test_histo_text_format():
    assert histo_text(spectrum(counts_of(open(os.path.join(GOLD, "small_k31.records"), "rb").read(), 31), 10001)) == \
        "1 2574\n2 498\n3 205\n4 48\n5 1\n"
    # histoMax=3: the "3" line counts every record seen 3 or more times; bin 0 (the phantom) is never printed
    assert histo_text(spectrum(counts_of(open(os.path.join(GOLD, "small_k40.records"), "rb").read(), 40), 4)) == \
        "1 1998\n2 287\n3 64\n"
    assert histo_text(np.array([5, 0, 0, 7], dtype=np.uint64)) == "3 7\n"


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


class _FakeRun:
    """stands in for a rank's Run: only its histogram is needed"""

    def __init__(self, hist):
        self.hist = hist

    def histogram(self, n_bins):
        assert n_bins == len(self.hist)
        return self.hist


def _fabricated(rank, n_bins):
    rng = np.random.default_rng(rank)
    h = rng.integers(0, 1 << 40, size=n_bins, dtype=np.uint64)
    h[rank % n_bins] = np.uint64(1 << 61)              # sums past 2^32 and past int32
    return h


def _gloo_worker(rank, world, port, n_bins, q):
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    from kmer_counter_b200 import multigpu
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    got = multigpu.histogram(_FakeRun(_fabricated(rank, n_bins)), n_bins)
    q.put((rank, got.dtype.str, got.tobytes()))
    dist.destroy_process_group()


def test_multigpu_histogram_sums_ranks_under_gloo():
    import torch.multiprocessing as mp
    world, n_bins = 2, 10001
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_gloo_worker, args=(r, world, port, n_bins, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=120) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    want = sum(_fabricated(r, n_bins) for r in range(world))
    for rank, dt, blob in res:
        assert dt == "<u8"
        assert np.array_equal(np.frombuffer(blob, dtype=np.uint64), want), rank


# ------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def kc():
    import kmer_counter_b200 as kc
    return kc


def _counter(kc, k, L, mode, method="auto", cap=1 << 23, **kw):
    return kc.Counter(k, L, method=method, compat="ref" if mode == "ref" else "strict", canonical=mode == "canonical",
                      n_slots=2, max_chunk_bytes=cap, **kw)


def _count(c, reads):
    c.slot_buffer(0)[:len(reads)] = reads
    c.submit(0, len(reads))
    return c.wait(0)


def _methods(k):
    return ["auto", "sort", "place"] + (["hash"] if k <= 64 else []) + (["super"] if 22 <= k <= 64 else [])


N_BINS = [2, 3, 17, 10001, 1 << 20]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["ref", "strict", "canonical"])
@pytest.mark.parametrize("k", [31, 40, 63, 96, 128])
def test_histogram_every_method_matches_model(kc, k, mode):
    """Zipf reads, plus two reads repeated 5000 times: counts from 1 into the thousands (past the
    shared-memory bins, into the device histogram's global bins and the high bin); N bases give ref
    mode its phantom"""
    L = 150
    reads = np.concatenate([oracle.gen_reads(20000, L, 400000, 0.002, 0.002, seed=k, zipf_loci=300),
                            np.tile(oracle.gen_reads(2, L, 0, 0.0, 0.0, seed=k + 1), 5000)])
    want = model_run(reads, L, k, mode)
    c_want = counts_of(want, k)
    assert c_want.max() > 4096
    for method in _methods(k):
        with _counter(kc, k, L, mode, method=method) as c:
            run = _count(c, reads)
            assert len(run) == len(c_want), method
            for n_bins in N_BINS:
                h = run.histogram(n_bins)
                assert h.dtype == np.uint64 and len(h) == n_bins
                assert np.array_equal(h, spectrum(c_want, n_bins)), (method, n_bins)
            assert np.array_equal(run.histogram(), spectrum(c_want, 10001))
            run.free()


def _records(keys, counts, W):
    dt = np.dtype([("w", "<u8", (W,)), ("c", "<u4")])
    out = np.zeros(len(counts), dtype=dt)
    out["w"] = np.asarray(keys, dtype=np.uint64).reshape(-1, W)
    out["c"] = counts
    return out.tobytes()


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


@pytest.mark.gpu
@pytest.mark.parametrize("k", [31, 40, 96, 128])
def test_histogram_of_uploaded_extreme_counts(kc, k):
    """counts 0, 1, 2^31 and 2^32 - 1, and counts spread up to 2^21 (global bins of a 2^20-bin histogram)"""
    W = (k + 31) // 32
    rng = np.random.default_rng(k)
    n = 50000
    counts = rng.integers(0, 1 << 21, size=n, dtype=np.uint64)
    counts[: n // 2] = rng.integers(1, 5, size=n // 2)
    counts[[3, 500, 7000, 40000]] = [0, 1, 2**31, U32_MAX]
    counts = counts.astype(np.uint32)
    rec = _records(_sorted_keys(n, W, k), counts, W)
    with kc.Counter(k, k) as c:
        run = c.upload_run(rec)
        for n_bins in N_BINS + [1 << 24]:
            assert np.array_equal(run.histogram(n_bins), spectrum(counts, n_bins)), n_bins
        for bad in (0, 1, (1 << 24) + 1):
            with pytest.raises(kc.KcError) as e:
                run.histogram(bad)
            assert e.value.code == -1
        f = run.filter(2**31, U32_MAX)
        assert f.to_bytes() == keep(rec, k, 2**31, U32_MAX)
        for r in (run, f):
            r.free()


@pytest.mark.gpu
def test_empty_run(kc):
    with kc.Counter(31, 100) as c:
        run = c.upload_run(b"")
        assert len(run) == 0
        h = run.histogram(17)
        assert h.tolist() == [0] * 17
        f = run.filter(2)
        assert len(f) == 0 and f.to_bytes() == b"" and f.parts()[1] == 0
        f.free()
        run.free()


@pytest.mark.gpu
def test_strict_skip_is_not_counted(kc):
    """strict mode hides the empty slots' key-0 record (a run with skip = 1): neither its histogram nor
    its filtered runs see it"""
    L, k = 100, 31
    reads = oracle.gen_reads(3000, L, 30000, 0.01, 0.02, seed=5)
    want = oracle.naive_count(reads, L, k, strict=True)
    c_want = counts_of(want, k)
    assert c_want.min() >= 1
    with _counter(kc, k, L, "strict", method="sort") as c:
        run = _count(c, reads)
        assert run.to_bytes() == want
        h = run.histogram(64)
        assert h[0] == 0 and np.array_equal(h, spectrum(c_want, 64))
        for lo, hi in ((0, U32_MAX), (0, 1), (2, U32_MAX)):
            f = run.filter(lo, hi)
            assert f.to_bytes() == keep(want, k, lo, hi), (lo, hi)
            f.free()
        run.free()


RANGES = [(0, U32_MAX), (2, U32_MAX), (1, 1), (5, 50), (U32_MAX, U32_MAX), (0, 0), (1, U32_MAX)]


@pytest.mark.gpu
@pytest.mark.parametrize("k,method", [(31, "hash"), (31, "super"), (40, "auto"), (96, "place"), (128, "sort")])
def test_filter_matches_model_and_every_consumer_takes_it(kc, tmp_path, k, method):
    L = 150
    reads = oracle.gen_reads(20000, L, 150000, 0.003, 0.002, seed=k + 1, zipf_loci=200)
    want = oracle.count(reads, L, k)
    S = oracle.record_size(k)
    with _counter(kc, k, L, "ref", method=method) as c:
        run = _count(c, reads)
        assert run.to_bytes() == want
        for lo, hi in RANGES:
            f = run.filter(lo, hi)
            exp = keep(want, k, lo, hi)
            assert f.to_bytes() == exp, (lo, hi)
            assert len(f) == len(exp) // S
            assert f.parts()[1] == 0
            f.free()
        with pytest.raises(kc.KcError) as e:
            run.filter(3, 2)
        assert e.value.code == -1
        f = run.filter(2)
        exp = keep(want, k, 2, U32_MAX)
        assert 0 < len(f) < len(run)
        # every consumer of a run
        keys, counts = oracle.records_to_arrays(exp, k)
        text = "".join("".join(oracle.print_word(int(w)) for w in kk) + " %d\n" % int(cn) for kk, cn in zip(keys, counts))
        assert f.print_text() == text.encode()
        p = tmp_path / "f.bin"
        f.write(str(p))
        assert p.read_bytes() == exp
        sp = keys[[len(keys) // 3, 2 * len(keys) // 3]]
        assert f.split(sp).tolist() == [0, len(keys) // 3, 2 * len(keys) // 3, len(keys)]
        ones = run.filter(1, 1)
        m = c.merge([f, ones])
        assert m.to_bytes() == keep(want, k, 1, U32_MAX)
        assert run.to_bytes() == want                              # the input is unchanged
        assert np.array_equal(run.histogram(100), spectrum(counts_of(want, k), 100))
        for r in (f, ones, m, run):
            r.free()


@pytest.mark.gpu
@pytest.mark.parametrize("k", [31, 63, 96, 128])
def test_filter_run_sizes_and_multi_tile(kc, k):
    """0, 1, tile - 1, tile, tile + 1 records (tile = 2048) and 12 M records: many tiles, one scan"""
    W = (k + 31) // 32
    sizes = [0, 1, 2047, 2048, 2049, 4097] + ([12_000_000] if k in (31, 128) else [])
    with kc.Counter(k, k) as c:
        for n in sizes:
            rng = np.random.default_rng(n + k)
            counts = rng.integers(1, 8, size=n).astype(np.uint32)
            rec = _records(_sorted_keys(n, W, n + 7), counts, W)
            run = c.upload_run(rec)
            for lo, hi in ((2, U32_MAX), (1, 1), (3, 5), (0, U32_MAX), (8, U32_MAX)):
                f = run.filter(lo, hi)
                assert f.to_bytes() == keep(rec, k, lo, hi), (n, lo, hi)
                f.free()
            assert np.array_equal(run.histogram(6), spectrum(counts, 6)), n
            run.free()


@pytest.mark.gpu
@pytest.mark.parametrize("P", [2, 3, 4, 5, 6, 7, 8])
def test_exchange_ranks_filter_and_histogram(kc, P):
    """after kc_xchg_run_all rank r holds key range r with final counts: the filtered per-rank runs
    concatenate to the filtered artefact, and the per-rank spectra add up to the artefact's"""
    import torch
    from kmer_counter_b200 import engine
    R, L, k = 12000, 100, 31
    reads = oracle.gen_reads(R, L, 60000, 0.01, 0.002, seed=P)
    want = oracle.count(reads, L, k)
    per = (R + P - 1) // P
    cs = [kc.Counter(k, L, method="super") for _ in range(P)]
    try:
        bufs = []
        for r, c in enumerate(cs):
            c.xchg_begin(r, P, max(per, 16))
            part = reads[r * per * L:(r + 1) * per * L]
            d = torch.from_numpy(part.copy()).cuda()
            bufs.append(d)
            c.accum_add_device(d.data_ptr(), len(part))
        runs = engine.xchg_run_all(cs)
        assert b"".join(r.to_bytes() for r in runs) == want
        hist = sum(r.histogram(10001) for r in runs)
        assert np.array_equal(hist, spectrum(counts_of(want, k), 10001))
        kept = [r.filter(2) for r in runs]
        assert b"".join(f.to_bytes() for f in kept) == keep(want, k, 2, U32_MAX)
        for r in runs + kept:
            r.free()
    finally:
        for c in cs:
            c.close()


# ------------------------------------------------------------------- command line
def _stats(stderr):
    return dict(t.split("=") for t in stderr.split() if "=" in t and t.split("=")[1].isdigit())


def _cli(tmp_path, reads_dir, extra, env=None):
    out = tmp_path / "out.bin"
    r = subprocess.run([CLI, "kmerLength=31", "inputFileLocation=%s" % reads_dir, "outputFile=%s" % out,
                        "tempFileLocation=%s" % tmp_path] + list(extra), capture_output=True, text=True, env=env)
    assert r.returncode == 0, r.stderr
    return out.read_bytes(), r.stderr


@pytest.mark.gpu
@pytest.mark.parametrize("args", [
    ("mode=accumulate", "gpuMemoryLimit=1500000"),
    ("mode=accumulate", "gpuMemoryLimit=1500000", "gpus=2"),
    ("mode=runs", "gpuMemoryLimit=1500000"),
    ("mode=runs", "gpuMemoryLimit=1200000", "noOfMergersAtOnce=2", "runBudget=400000"),
])
def test_cli_filter_and_histo_file(tmp_path, args):
    d = tmp_path / "in"
    d.mkdir()
    L, per, k = 100, 8000, 31
    for i in range(3):
        (d / ("part%d.fastq" % i)).write_bytes(oracle.gen_fastq(per, L, 300000, 0.01, 0.002, seed=31, first_read=i * per))
    want = oracle.count(oracle.gen_reads(3 * per, L, 300000, 0.01, 0.002, seed=31), L, k)
    c_want = counts_of(want, k)
    S = oracle.record_size(k)
    env = dict(os.environ, KC_CLI_SAME_DEVICE="1")
    # without the new flags: the artefact, and no new stderr
    got, err = _cli(tmp_path, d, args, env)
    assert got == want and "filtered=" not in err
    runs_mode = "mode=runs" in args
    assert err.splitlines()[-1] == "records=%d -> %s" % (len(want) // S, tmp_path / "out.bin")
    assert err.splitlines()[-2].startswith("parser=gpu reads=" if runs_mode else "mode=accumulate gpus=")
    if "runBudget=400000" in args:
        assert int(_stats(err)["spills"]) >= 2 and int(_stats(err)["ranges"]) >= 2, err
    for extra, lo, hi, hmax in [(("minCount=2",), 2, U32_MAX, 10000),
                                (("minCount=2", "maxCount=5", "histoMax=4"), 2, 5, 4),
                                (("maxCount=1",), 0, 1, 10000)]:
        hf = tmp_path / "histo.txt"
        got, err = _cli(tmp_path, d, args + extra + ("histoFile=%s" % hf,), env)
        exp = keep(want, k, lo, hi)
        assert got == exp, extra
        st = _stats(err)
        assert int(st["filtered"]) == (len(want) - len(exp)) // S
        assert int(st["records"]) == len(exp) // S
        assert hf.read_text() == histo_text(spectrum(c_want, hmax + 1)), extra
    # the spectrum alone: the artefact is unfiltered
    hf = tmp_path / "only.txt"
    got, err = _cli(tmp_path, d, args + ("histoFile=%s" % hf, "histoMax=3"), env)
    assert got == want and "filtered=" not in err
    assert hf.read_text() == histo_text(spectrum(c_want, 4))


@pytest.mark.gpu
@pytest.mark.parametrize("k", [31, 40, 96])
def test_cli_histo_subcommand(tmp_path, k):
    L = 150
    reads = oracle.gen_reads(6000, L, 50000, 0.003, 0.002, seed=k, zipf_loci=100)
    want = oracle.count(reads, L, k)
    p = tmp_path / "r.bin"
    p.write_bytes(want)
    r = subprocess.run([CLI, "histo", str(p), "-", str(k)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert r.stdout == histo_text(spectrum(counts_of(want, k), 10001))
    out = tmp_path / "h.txt"
    r = subprocess.run([CLI, "histo", str(p), str(out), str(k), "7"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert out.read_text() == histo_text(spectrum(counts_of(want, k), 8))
