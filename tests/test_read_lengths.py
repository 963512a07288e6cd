"""Read lengths up to 4096 bases: every counting path against the window model at the lengths where
the kernels' tiling changes shape, across the super-window path's read-length limit, with plans of
many small bins at long reads, over low-complexity long reads, and through the FASTQ parser and the
command line.

Expected records: the oracle's chunk model (process_chunk) where it applies (ref mode, L % 32 != 0),
the window model (naive_count) otherwise -- code 0 past the read end in ref mode, true k-mers in
strict mode, and the canonical fold of test_canonical for canonical runs. The CPU part pins the two
models to each other at long reads and restates the read-length limits of the super-window path and
the partitioned hash.
"""
import os
import subprocess

import numpy as np
import pytest

import oracle
from test_canonical import canonical_count

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "kmer-counter_b200", "host", "kmer_counter_b200")
HOSTILE = np.frombuffer(b"ACGT" * 12 + b"acgtNnRYKM-.*0" + bytes([0, 127, 128, 255]), dtype=np.uint8)


def _masked(k, strict):
    m = k % 32
    return m != 0 if strict else 1 <= m <= 28                          # SURVEY F4


def _extract_tile(L, target):
    """reads per extraction tile and the extraction's shared memory (extract_plan / extract_smem_layout)"""
    tr = 16 * max(1, target // (16 * L))
    stage = (tr * L + 127) & ~127
    flag_off = 2 * stage + tr * ((L + 31) // 32 + 1) * 8 + ((tr * ((L + 3) // 4) + 15) & ~15)
    return tr, ((flag_off + tr + 15) & ~15) + 16


def s1_smem(k, L, strict=False, m=12):
    """S1's shared memory (kc_super.cu, s1_smem): the extraction tile of 4800 bytes of reads (16 reads
    from L = 301 on), then per read of the tile a row of m-mer hashes (nk + w - 1, odd stride), the bin
    of every window (nk) and two words per segment of at most min(w - 1, 17) windows."""
    span = k if _masked(k, strict) else 32 * ((k + 31) // 32)
    nk, w = L - k + 1, span - m + 1
    stride = (nk + w - 1 + 8) | 1
    segs = -(-nk // min(w - 1, 17))
    tr, ext = _extract_tile(L, 4800)
    return ((ext + 15) & ~15) + tr * stride * 4 + tr * nk * 4 + 2 * tr * segs * 4


def super_max_len(k, strict=False):
    """Longest read the super-window path takes at k: S1 must fit its 200 KiB at m = 12."""
    span = k if _masked(k, strict) else 32 * ((k + 31) // 32)
    if k > 64 or span < 22:
        return 0
    return max(L for L in range(k, 4097) if s1_smem(k, L, strict) <= 200 * 1024)


# The limits, pinned. For k = 22 (window span 22, w = 11, segments of 10 windows) at L = 1140:
# extraction 2 x 18304 + 16 x 37 x 8 + 16 x 285 + 16 + 16 = 45936 bytes, hashes 16 x 1137 x 4 = 72768,
# bins 16 x 1119 x 4 = 71616, segments 2 x 16 x 112 x 4 = 14336: 204656 <= 204800. One base more adds
# 16 x 4 bytes of bins, 16 x 8 of hashes (the odd stride grows by 2) and 16 of the tile: 204864 > 204800.
# Strict and canonical keys have the same spans at these k, hence the same limits.
SUPER_MAX_L = {22: 1140, 31: 1176, 32: 1177, 63: 1190, 64: 1191}


def super_applies(k, L, strict=False):
    return L <= super_max_len(k, strict)


def pa_smem(k, L):
    """PA's shared memory (kc_partition.cu, partition_fits): the extraction tile of 6400 bytes of reads
    (16 reads from L = 201 on), three 1024-bin arrays and 64 bytes, and the tile's keys staged by digit"""
    tr, ext = _extract_tile(L, 6400)
    return ext + 3 * 1024 * 4 + 64 + tr * (L - k + 1) * 8 * ((k + 31) // 32)


def hash_applies(k, L):
    return k <= 64 and pa_smem(k, L) <= 227 * 1024


# Longest reads the partitioned hash takes (227 KiB of shared memory per CTA); beyond them the methods
# that would use it count with the sorter. For k = 31 at L = 1330: extraction 2 x 21376 + 16 x 43 x 8 +
# 16 x 333 + 16 + 16 = 53616 bytes, bins 12352, keys 16 x 1300 x 8 = 166400: 232368 <= 232448.
HASH_MAX_L = {22: 1323, 31: 1330, 32: 1331, 63: 796, 64: 797}


def expected_method(method, k, L, strict=False):
    """what pick_method (kc_api.cu) chooses"""
    W = (k + 31) // 32
    sup, hsh = super_applies(k, L, strict), hash_applies(k, L)
    if method == "super":
        return "super" if sup else ("hash" if hsh else "sort")
    if method == "hash":
        return "hash" if hsh else "sort"
    if method == "auto":
        if sup:
            return "super"
        if W > 2:
            return "place"
        if not hsh:
            return "sort"
        if W == 2:
            return "hash"
        sig = 2 * (k % 32) if _masked(k, strict) else 64                # significant bits of the key
        return "hash" if sig >= 24 else "sort"
    return method


def want_ref(reads, L, k):
    """ref-mode records: the chunk model where the reference's layout applies, the window model at L % 32 == 0"""
    return oracle.process_chunk(reads, L, k) if L % 32 else oracle.naive_count(reads, L, k, strict=False)


def n_reads_for(L):
    """three tiles of the largest extraction tile (P0's 12800 bytes) and a ragged one of 5 reads:
    R = 16 t + 5 with a whole number of tiles of every kernel's tile size in 16 t"""
    return 3 * _extract_tile(L, 12800)[0] + 5


# ------------------------------------------------------------------------------------- CPU
A0_LENGTHS = [251, 1141, 2047, 4095]
A0_K = [1, 22, 31, 33, 63, 64, 96, 128]


@pytest.mark.parametrize("L", A0_LENGTHS)
def test_oracle_models_agree_at_long_reads(L):
    """The chunk model (the reference's restatement) == the window model at long reads, over the
    hostile alphabet of test_oracle: mostly valid reads with scattered bad bytes, and reads of any
    byte. Where the reference's own code is built, it agrees too."""
    rng = np.random.default_rng(L)
    for k in A0_K:
        valid = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, size=7 * L)].copy()
        valid[rng.integers(0, valid.size, size=max(1, valid.size // 60))] = rng.choice(HOSTILE, size=max(1, valid.size // 60))
        anything = np.ascontiguousarray(HOSTILE[rng.integers(0, HOSTILE.size, size=3 * L)])
        for reads in (valid, anything, np.concatenate([valid, anything])):
            got = oracle.process_chunk(reads, L, k)
            assert got == oracle.naive_count(reads, L, k), (L, k)
            if oracle.ref_available():
                assert oracle.ref_process_chunk(reads, L, k) == got, (L, k)


def test_super_length_limits_restated():
    """The pinned limits are what the restated S1 footprint gives, in every key mode."""
    for k, L in SUPER_MAX_L.items():
        for strict in (False, True):
            assert super_max_len(k, strict) == L, (k, strict)
            assert s1_smem(k, L, strict) <= 200 * 1024 < s1_smem(k, L + 1, strict)
    assert s1_smem(22, 1140) == 204656
    assert super_max_len(21) == 0 and super_max_len(65) == 0 and super_max_len(28, strict=False) == 1174
    for k, L in HASH_MAX_L.items():
        assert hash_applies(k, L) and not hash_applies(k, L + 1), k
    assert pa_smem(31, 1330) == 232368
    # the benchmark shapes are far from the limit: S1 needs less than a quarter of it at any m
    assert max(s1_smem(k, 100, m=m) for k in (31, 63) for m in range(12, 17)) < 200 * 1024 // 4


# ------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def kc():
    import kmer_counter_b200 as kc
    return kc


def _counter(kc, k, L, method, cap=1 << 24, **kw):
    return kc.Counter(k, L, method=method, n_slots=2, max_chunk_bytes=cap, **kw)


def _count(kc, k, L, method, reads, **kw):
    """(records, method_used, device scalars) of one chunk"""
    with _counter(kc, k, L, method, cap=max(len(reads), 1 << 20), **kw) as c:
        got = c.process_chunk(reads)
        return got, c.stats()["method_used"], c.debug_scalars()


A_LENGTHS = [250, 251, 300, 301, 400, 401, 781, 782, 800, 801, 1000, 2047, 4095]
A_K = ([(k, ("sort", "hash", "super", "auto")) for k in (22, 31, 32, 63, 64)] +
       [(k, ("sort", "place", "auto")) for k in (96, 100, 128)] + [(1, ("sort",)), (5, ("sort",))])


@pytest.mark.gpu
@pytest.mark.parametrize("L", A_LENGTHS)
@pytest.mark.parametrize("k,methods", A_K, ids=["k%d" % k for k, _ in A_K])
def test_tiling_switch_points(kc, L, k, methods):
    """Lengths on both sides of where each kernel's extraction tile drops to 16 reads (S1 at L > 300,
    PA at 400, the default at 781, P0 at 800), odd lengths (reads not a multiple of 16 bytes: the
    plain-load path instead of the TMA), and up to 4095 bases (227 rolling segments per read). A few
    tiles and a ragged last one, and a single partial tile."""
    R = n_reads_for(L)
    reads = oracle.gen_reads(R, L, 50_000, 0.01, 0.002, seed=131 * L + k)
    for part in (reads, reads[:13 * L]):
        want = want_ref(part, L, k)
        for method in methods:
            got, used, _ = _count(kc, k, L, method, part)
            assert got == want, (L, k, method, len(part) // L)
            assert used == expected_method(method, k, L), (L, k, method, used)


B_LENGTHS = [64, 128, 256, 1024, 4096]
B_K = [5, 22, 29, 30, 31, 32, 61, 62, 63, 64, 94, 96, 127, 128]


def _methods_for(k):
    out = ["sort", "auto"]
    if k >= 5:
        out.append("place")
    if k <= 64:
        out += ["hash", "super"]
    if k <= 32:
        out.append("hash_global")
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("L", B_LENGTHS)
def test_read_length_multiple_of_32_ref_mode(kc, L):
    """L % 32 == 0 in ref mode, where the chunk model does not apply: every method against the window
    model, including k % 32 in {29, 30, 31, 0}, whose unmasked last window reaches past the read end."""
    R = n_reads_for(L)
    reads = oracle.gen_reads(R, L, 50_000, 0.01, 0.002, seed=L + 7)
    for k in (k for k in B_K if k <= L):
        want = oracle.naive_count(reads, L, k, strict=False)
        for method in _methods_for(k):
            got, used, _ = _count(kc, k, L, method, reads)
            assert got == want, (L, k, method)
            assert used == expected_method(method, k, L), (L, k, method, used)


@pytest.mark.gpu
@pytest.mark.parametrize("L", [250, 1000, 1177, 1178, 4095, 4096])
def test_strict_and_canonical_long_reads(kc, L):
    """strict and canonical keys against the window model and its canonical fold"""
    R = n_reads_for(L)
    reads = oracle.gen_reads(R, L, 50_000, 0.01, 0.002, seed=L + 11)
    for k in (22, 31, 32, 63, 64, 96, 128):
        strict_want = oracle.naive_count(reads, L, k, strict=True)
        canon_want = canonical_count(reads, L, k)
        for method in ("auto", "super", "hash", "sort") if k <= 64 else ("auto", "place", "sort"):
            got, used, _ = _count(kc, k, L, method, reads, compat="strict")
            assert got == strict_want, (L, k, method)
            assert used == expected_method(method, k, L, strict=True), (L, k, method, used)
            got, used, _ = _count(kc, k, L, method, reads, canonical=True)
            assert got == canon_want, (L, k, method, "canonical")
            assert used == expected_method(method, k, L, strict=True), (L, k, method, used)


@pytest.mark.gpu
@pytest.mark.parametrize("k", sorted(SUPER_MAX_L))
def test_super_window_length_limit(kc, k):
    """At the longest read the super-window path takes, auto and super count there and the accumulating
    mode is accepted; one base longer, they count with the partitioned hash (the sorter for 128-bit keys,
    whose reads are then too long for the hash too), with the same records, and the accumulating mode is
    refused with KC_ERR_ARG."""
    import torch
    Lmax = SUPER_MAX_L[k]
    for L, path in ((Lmax, "super"), (Lmax + 1, "hash" if k <= 32 else "sort")):
        R = n_reads_for(L)
        reads = oracle.gen_reads(R, L, 50_000, 0.01, 0.002, seed=L * 3 + k)
        want = want_ref(reads, L, k)
        for method in ("auto", "super", "hash"):
            got, used, _ = _count(kc, k, L, method, reads)
            assert got == want, (k, L, method)
            assert used == (path if method != "hash" else expected_method("hash", k, L)), (k, L, method, used)
        got, used, _ = _count(kc, k, L, "auto", reads, canonical=True)
        assert got == canonical_count(reads, L, k) and used == path, (k, L, "canonical")
        with kc.Counter(k, L, method="auto") as c:
            if path == "super":
                c.accum_begin(R)
                d = torch.from_numpy(reads.copy()).cuda()
                c.accum_add_device(d.data_ptr(), len(reads))
                run = c.accum_flush()
                assert run.to_bytes() == want, (k, L, "accumulate")
                run.free()
            else:
                with pytest.raises(kc.KcError) as e:
                    c.accum_begin(R)
                assert e.value.code == -1, str(e.value)


@pytest.mark.gpu
def test_accumulate_refusal_names_the_read_length(kc):
    """k = 31 is fine for the accumulating mode; reads of 1177 bases are not"""
    with kc.Counter(31, SUPER_MAX_L[31] + 1) as c:
        with pytest.raises(kc.KcError) as e:
            c.accum_begin(1000)
    assert e.value.code == -1 and "reads of 1177 bases are too long" in str(e.value), str(e.value)
    with kc.Counter(21, 100) as c:
        with pytest.raises(kc.KcError) as e:
            c.accum_begin(1000)
    assert e.value.code == -1 and "windows of >= 22 bases" in str(e.value), str(e.value)


# Plans with many bins at reads near the limit. super_plan lengthens the minimizer with the bin count
# (m = 13 from 87 382 bins, 14 from 349 526); a longer minimizer means shorter segments and more of S1's
# shared memory per read. Each of these plans would take m = 13 or 14 and S1 more than 200 KiB; the
# plan keeps m where S1 fits. table_slots = 64 is the occurrences per bin.
D_CHUNK = [(22, 1140, 5000, False), (22, 1140, 5000, True), (24, 1150, 5000, False), (28, 1170, 20000, False)]
_D_CACHE = {}


def _d_reads(k, L, R, canonical=False):
    key = (k, L, R, canonical)
    if key not in _D_CACHE:
        reads = oracle.gen_reads(R, L, 2_000_000, 0.01, 0.001, seed=L + R)
        _D_CACHE[key] = (reads, canonical_count(reads, L, k) if canonical else oracle.process_chunk(reads, L, k))
    return _D_CACHE[key]


@pytest.mark.gpu
@pytest.mark.parametrize("k,L,R,canonical", D_CHUNK)
def test_long_reads_many_small_bins_chunk(kc, k, L, R, canonical):
    reads, want = _d_reads(k, L, R, canonical)
    got, used, sc = _count(kc, k, L, "super", reads, table_slots=64, canonical=canonical)
    assert used == "super"
    assert got == want, sc
    assert sc["windows"] == R * (L - k + 1) - sc["invalid"]


@pytest.mark.gpu
def test_long_reads_many_small_bins_accumulate(kc):
    k, L, R = 22, 1140, 5000
    reads, want = _d_reads(k, L, R)
    per = 1000
    with kc.Counter(k, L, method="super", n_slots=2, max_chunk_bytes=per * L, table_slots=64) as c:
        c.accum_begin(R)
        sl, busy = 0, [False, False]
        for r0 in range(0, R, per):
            part = reads[r0 * L:(r0 + per) * L]
            if busy[sl]:
                c.accum_wait(sl)
            c.slot_buffer(sl)[:len(part)] = part
            c.accum_submit(sl, len(part))
            busy[sl] = True
            sl ^= 1
        run = c.accum_flush()
        assert run.to_bytes() == want
        run.free()


@pytest.mark.gpu
def test_long_reads_many_small_bins_exchange(kc):
    """two ranks on one device; each plans bins of table_slots / 2 occurrences"""
    import torch
    from kmer_counter_b200 import engine
    k, L, per = 22, 1140, 2600
    reads = oracle.gen_reads(2 * per, L, 2_000_000, 0.01, 0.001, seed=77)
    want = oracle.process_chunk(reads, L, k)
    cs = [kc.Counter(k, L, method="super", table_slots=64) for _ in range(2)]
    try:
        bufs = []
        for r, c in enumerate(cs):
            c.xchg_begin(r, 2, per)
            d = torch.from_numpy(reads[r * per * L:(r + 1) * per * L].copy()).cuda()
            bufs.append(d)
            c.accum_add_device(d.data_ptr(), d.numel())
        runs = engine.xchg_run_all(cs)
        got = b"".join(r.to_bytes() for r in runs)
        for r in runs:
            r.free()
        assert got == want
    finally:
        for c in cs:
            c.close()


@pytest.mark.gpu
def test_long_reads_default_plan_accumulate(kc):
    """the plan of an accumulator for 660 000 reads of 1140 bases (0.75 Gbase): 90 154 bins by default"""
    import torch
    k, L, R = 22, 1140, 5000
    reads, want = _d_reads(k, L, R)
    with kc.Counter(k, L, method="auto") as c:
        c.accum_begin(660_000)
        d = torch.from_numpy(reads.copy()).cuda()
        c.accum_add_device(d.data_ptr(), len(reads))
        run = c.accum_flush()
        assert run.to_bytes() == want
        run.free()


@pytest.mark.gpu
def test_long_reads_default_plan_large_chunk(kc):
    """one chunk of 660 000 reads of 1140 bases generated on the device: the super-window path (a
    default plan of 90 154 bins) and the partitioned hash give the same run; its counts add up to the
    number of k-mers, and its keys are strictly ascending"""
    import torch
    from kmer_counter_b200 import synth
    from kmer_counter_b200.multigpu import run_as_tensors
    k, L, R = 22, 1140, 660_000
    d = torch.empty(R * L, dtype=torch.uint8, device="cuda")
    synth.synth_reads_device(d.data_ptr(), R, L, 200_000_000, 1e-3, 0.0, seed=23)
    torch.cuda.synchronize()
    runs = {}
    for method in ("super", "hash"):
        with kc.Counter(k, L, method=method) as c:
            run = c.count_device(d.data_ptr(), R * L)
            assert c.stats()["method_used"] == method
            keys, counts = run_as_tensors(run, d.device)
            runs[method] = (keys.clone(), counts.clone())
            run.free()
    del d
    assert torch.equal(runs["super"][0], runs["hash"][0]) and torch.equal(runs["super"][1], runs["hash"][1])
    keys, counts = runs["super"]
    assert int(counts.to(torch.int64).sum()) == R * (L - k + 1)
    kk = keys[:, 0] ^ torch.tensor(-2**63, dtype=torch.int64, device=keys.device)      # unsigned order
    assert bool((kk[1:] > kk[:-1]).all())


@pytest.mark.gpu
@pytest.mark.parametrize("L", [1100, 4095])
@pytest.mark.parametrize("k", [31, 63])
def test_low_complexity_long_reads(kc, L, k):
    """Reads whose minimizer never changes: poly-A, poly-T, period-2 and period-3 repeats, and 500
    copies of one read, next to reads with an N every 300 bases. Records are cut every cmax windows
    and crowd one bin, so the super-window path fills its overflow list."""
    def rep(unit, n):
        return np.frombuffer((unit * (L // len(unit) + 1))[:L] * n, dtype=np.uint8)
    with_n = oracle.gen_reads(40, L, 0, 0, 0, seed=L + k).reshape(-1, L).copy()
    with_n[:, 299::300] = ord("N")
    reads = np.concatenate([rep(b"A", 150), rep(b"T", 150), rep(b"AC", 60), rep(b"ACG", 60), with_n.reshape(-1),
                            np.tile(oracle.gen_reads(1, L, 0, 0, 0, seed=L * k), 500)])
    want = want_ref(reads, L, k)
    for method in ("auto", "super", "hash", "sort"):
        got, used, sc = _count(kc, k, L, method, reads)
        assert got == want, (L, k, method, sc)
        assert used == expected_method(method, k, L), (L, k, method, used)
        if used == "super":
            assert sc["overflow_records"] > 0, sc


@pytest.mark.gpu
@pytest.mark.parametrize("L", [1000, 4095])
def test_fastq_long_reads(kc, L):
    """FASTQ text of long reads parsed on the device: blocks that cut a record in the middle of its
    sequence line, CRLF line ends, and the parser alone against the oracle's restatement."""
    import torch
    k, R = 31, (400 if L == 1000 else 150)
    fq = oracle.gen_fastq(R, L, 200_000, 0.01, 0.002, seed=L)
    reads = oracle.parse_fastq(fq)
    assert reads == oracle.gen_reads(R, L, 200_000, 0.01, 0.002, seed=L).tobytes()
    want = oracle.count(reads, L, k)
    rec = len(fq) // R                                   # bytes of one record (fixed-width headers)
    with _counter(kc, k, L, "auto", cap=1 << 22) as c:
        for text, block in ((fq, 0), (fq, 3 * rec + rec // 4), (fq, 7 * rec + rec // 3),
                            (fq.replace(b"\n", b"\r\n"), 3 * rec + rec // 4)):
            run = c.count_fastq(text, block_bytes=block)
            assert run.to_bytes() == want, (block, len(text))
            run.free()
            assert c.stats()["method_used"] == expected_method("auto", k, L)
        d_text = torch.from_numpy(np.frombuffer(fq, dtype=np.uint8).copy()).cuda()
        d_reads = torch.empty(R * L, dtype=torch.uint8, device="cuda")
        n, used, fl = c.parse_fastq_device(d_text.data_ptr(), d_text.numel(), d_reads.data_ptr(), d_reads.numel())
        assert (n, used, fl) == (R, len(fq), 0)
        assert bytes(d_reads.cpu().numpy()) == reads
        n, used, fl = c.parse_fastq_device(d_text.data_ptr(), len(fq) - rec + 20 + L // 2, d_reads.data_ptr(),
                                           d_reads.numel())
        assert (n, used, fl) == (R - 1, len(fq) - rec, 0)          # the record cut in its sequence is left over


@pytest.mark.gpu
@pytest.mark.parametrize("L,accumulates", [(1000, True), (1500, False)])
def test_cli_default_mode_long_reads(tmp_path, L, accumulates):
    """The command line's default mode accumulates where the super-window path takes the reads, and
    counts chunk by chunk into runs beyond its length limit (k = 31: 1176 bases); the file is the
    oracle's artefact either way."""
    k, per = 31, 500
    d = tmp_path / "in"
    d.mkdir()
    for i in range(2):
        (d / ("part%d.fastq" % i)).write_bytes(oracle.gen_fastq(per, L, 300_000, 0.01, 0.002, seed=L, first_read=i * per))
    out = tmp_path / "out.bin"
    r = subprocess.run([CLI, "kmerLength=%d" % k, "inputFileLocation=%s" % d, "outputFile=%s" % out,
                        "gpuMemoryLimit=3000000", "tempFileLocation=%s" % tmp_path], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert ("mode=accumulate" in r.stderr) == accumulates, r.stderr
    stats = dict(t.split("=") for t in r.stderr.split() if "=" in t and t.split("=")[1].isdigit())
    assert int(stats["chunks"]) >= 4, r.stderr
    assert out.read_bytes() == oracle.count(oracle.gen_reads(2 * per, L, 300_000, 0.01, 0.002, seed=L), L, k)
