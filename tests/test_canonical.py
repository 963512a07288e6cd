"""Canonical k-mer counting (KC_CANONICAL): a k-mer and its reverse complement are counted under
one key, min(x, rc(x)) in record order. The model (the oracle's strict count folded by
min(x, rc(x))) is checked against a string model and known answers on the CPU; every counting path
of the library is checked against the model on the GPU."""
import os
import re
import subprocess

import numpy as np
import pytest

import oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "kmer-counter_b200", "host", "kmer_counter_b200")
CODE = {"A": 0, "C": 1, "G": 2, "T": 3}
COMP = bytes.maketrans(b"ACGT", b"TGCA")


# ------------------------------------------------------------------ string model (CPU)
def _revcomp(s: bytes) -> bytes:
    return s.translate(COMP)[::-1]


def _encode(kmer: str):
    W = (len(kmer) + 31) // 32
    v = 0
    for ch in kmer.ljust(32 * W, "A"):
        v = (v << 2) | CODE[ch]
    return tuple((v >> (64 * (W - 1 - i))) & (2**64 - 1) for i in range(W))


def _model(reads: bytes, L, k) -> bytes:
    """Reverse-complement the k-mer text, encode both, take the smaller; windows with a
    byte other than A, C, G, T are dropped."""
    counts = {}
    for r in range(len(reads) // L):
        s = reads[r * L:(r + 1) * L]
        for p in range(L - k + 1):
            w = s[p:p + k]
            if any(c not in b"ACGT" for c in w):
                continue
            key = min(_encode(w.decode()), _encode(_revcomp(w).decode()))
            counts[key] = counts.get(key, 0) + 1
    W = (k + 31) // 32
    dt = np.dtype([("w", "<u8", (W,)), ("c", "<u4")])
    out = np.zeros(len(counts), dtype=dt)
    for i, key in enumerate(sorted(counts)):
        out[i]["w"] = key
        out[i]["c"] = counts[key]
    return out.tobytes()


def _records(run: bytes, k):
    W = (k + 31) // 32
    a = np.frombuffer(run, dtype=np.dtype([("w", "<u8", (W,)), ("c", "<u4")]))
    return [(tuple(int(x) for x in r["w"]), int(r["c"])) for r in a]


def _u8(b: bytes):
    return np.frombuffer(b, dtype=np.uint8)


def _revcomp_reads(reads, L):
    """every read reverse-complemented (other bytes stay where the reversal puts them)"""
    rows = np.asarray(reads, dtype=np.uint8).reshape(-1, L)[:, ::-1]
    lut = np.arange(256, dtype=np.uint8)
    for a, b in zip(b"ACGT", b"TGCA"):
        lut[a] = b
    return np.ascontiguousarray(lut[rows]).reshape(-1)


_M1 = np.uint64(0x5555555555555555)


def _word_revcomp(x):
    """reverse complement of 32 bases per uint64 (numpy, vectorised): 2-bit groups reversed, code ^ 3"""
    x = x.copy()
    for sh, m in ((2, 0x3333333333333333), (4, 0x0F0F0F0F0F0F0F0F), (8, 0x00FF00FF00FF00FF),
                  (16, 0x0000FFFF0000FFFF), (32, 0x00000000FFFFFFFF)):
        m, sh = np.uint64(m), np.uint64(sh)
        x = ((x >> sh) & m) | ((x & m) << sh)
    return ~x


def canonical_count(reads, L, k) -> bytes:
    """The canonical model: the oracle's strict (true k-mer) count, every key replaced by
    min(x, rc(x)) in record order, equal keys summed, sorted."""
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


KNOWN = [
    (b"ACGTTGCAAC", 5, [((0x06c0000000000000,), 1), ((0x4180000000000000,), 1), ((0x9040000000000000,), 2),
                        ((0xe400000000000000,), 2)]),
    (b"ACGTNACGTACG", 5, [((0x1b00000000000000,), 1), ((0x6c40000000000000,), 2)]),
    (b"GGGTTTAAACCC", 6, [((0x0150000000000000,), 2), ((0xafc0000000000000,), 2), ((0xbf00000000000000,), 2),
                          ((0xfc00000000000000,), 1)]),
]
A4_READ = b"ACGTACGTACGTACGTACGTACGTACGTACGTTTGGCCAAC"      # SURVEY A.4's 41-base read

K_LIST = [1, 2, 5, 16, 31, 32, 33, 63, 64, 65, 96, 100, 128]


@pytest.mark.parametrize("read,k,want", KNOWN)
def test_known_answers(read, k, want):
    got = _records(canonical_count(_u8(read), len(read), k), k)
    assert got == want
    assert _model(read, len(read), k) == canonical_count(_u8(read), len(read), k)


def test_known_answer_survey_a4_read():
    assert len(A4_READ) == 41
    got = _records(canonical_count(_u8(A4_READ), 41, 33), 33)
    assert got[:3] == [((0x01b1b1b1b1b1b1b1, 0x8000000000000000), 1), ((0x06c6c6c6c6c6c6c6, 0xc000000000000000), 1),
                       ((0x1b1b1b1b1b1b1bfa, 0x4000000000000000), 1)]


@pytest.mark.parametrize("k", K_LIST)
def test_oracle_matches_string_model(k):
    rng = np.random.default_rng(1000 + k)
    for trial in range(3):
        L = int(rng.integers(k, k + 40))
        R = int(rng.integers(1, 12))
        alphabet = np.frombuffer(b"ACGTACGTACGTACGTNacgt", dtype=np.uint8)
        reads = alphabet[rng.integers(0, len(alphabet), size=R * L)]
        if trial == 2 and k % 2 == 0:
            # reads built from palindromes: x == rc(x) counts once per occurrence
            half = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, size=k // 2)].tobytes()
            pal = half + _revcomp(half)
            reads = _u8((pal * (L // k + 2))[:L] * R)
        assert canonical_count(reads, L, k) == _model(bytes(reads), L, k), (k, trial)


@pytest.mark.parametrize("k", K_LIST)
def test_oracle_strand_properties(k):
    L = max(k + 30, 60)
    reads = oracle.gen_reads(40, L, 3000, 0.01, 0.01, seed=k)
    rc = _revcomp_reads(reads, L)
    canon = canonical_count(reads, L, k)
    assert canon == canonical_count(rc, L, k)
    both = canonical_count(np.concatenate([reads, rc]), L, k)
    assert [key for key, _ in _records(both, k)] == [key for key, _ in _records(canon, k)]
    assert [c for _, c in _records(both, k)] == [2 * c for _, c in _records(canon, k)]


def test_flag_value_matches_header():
    import kmer_counter_b200._lib as _lib
    hdr = open(os.path.join(ROOT, "include", "kc_api.h")).read()
    m = re.search(r"#define KC_CANONICAL\s+(0x[0-9a-fA-F]+)u", hdr)
    assert m and int(m.group(1), 16) == _lib.KC_CANONICAL == 2


# -------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def kc():
    import kmer_counter_b200 as kc
    return kc


def _counter(kc, k, L, method="auto", cap=1 << 24, **kw):
    return kc.Counter(k, L, method=method, n_slots=2, max_chunk_bytes=cap, canonical=True, **kw)


CASES = [
    # (reads, L, k, genome, sub, n_rate)
    (2000, 100, 31, 30000, 0.01, 0.002),
    (2000, 100, 31, 30000, 0.0, 0.0),
    (1500, 100, 32, 20000, 0.01, 0.001),
    (1500, 100, 28, 20000, 0.0, 0.001),
    (1500, 100, 29, 20000, 0.0, 0.001),
    (700, 70, 63, 5000, 0.001, 0.001),
    (700, 70, 64, 5000, 0.001, 0.0),
    (700, 70, 60, 5000, 0.001, 0.001),
    (500, 41, 33, 0, 0.0, 0.01),
    (300, 150, 96, 2000, 0.01, 0.01),
    (300, 150, 128, 2000, 0.01, 0.01),
    (300, 150, 100, 2000, 0.01, 0.0),
    (300, 45, 5, 0, 0.0, 0.02),
    (64, 10, 1, 0, 0.0, 0.1),
]
METHODS = ["auto", "sort", "hash", "hash_global", "super", "place"]


def _expected_method(method, k):
    if method == "auto":
        return "super" if 22 <= k <= 64 else ("place" if k > 64 else None)
    if method == "super":
        return "super" if 22 <= k <= 64 else None
    return method


@pytest.mark.gpu
@pytest.mark.parametrize("method", METHODS)
@pytest.mark.parametrize("R,L,k,G,e,n", CASES)
def test_every_method_matches_oracle(kc, method, R, L, k, G, e, n):
    if method == "hash" and k > 64:
        pytest.skip("hash counting needs k <= 64")
    reads = oracle.gen_reads(R, L, G, e, n, seed=R + k)
    want = canonical_count(reads, L, k)
    if method == "hash_global" and k > 32:
        with pytest.raises(kc.KcError):
            _counter(kc, k, L, method=method)
        return
    with _counter(kc, k, L, method=method) as c:
        assert c.process_chunk(reads) == want
        used = c.stats()["method_used"]
    exp = _expected_method(method, k)
    if exp in ("super", "place", "sort"):
        assert used == exp, (method, k, used)
    elif exp in ("hash", "hash_global"):
        assert used in (exp, "sort"), (method, k, used)      # a full table falls back to sort


@pytest.mark.gpu
def test_submit_wait_count_device_and_fastq(kc):
    """kc_submit / kc_wait, kc_count_device, kc_submit_fastq and kc_run_print of a canonical run
    (kc_accum_submit_fastq: the command line's parser=gpu, below)"""
    import torch
    L, k, R = 100, 31, 5000
    fq = oracle.gen_fastq(R, L, 60000, 0.01, 0.002, seed=41)
    reads = _u8(oracle.parse_fastq(fq))
    want = canonical_count(reads, L, k)
    with _counter(kc, k, L, cap=1 << 20) as c:
        c.slot_buffer(0)[:len(reads)] = reads
        c.submit(0, len(reads))
        run = c.wait(0)
        assert run.to_bytes() == want
        run.free()
        d = torch.from_numpy(reads.copy()).cuda()
        run = c.count_device(d.data_ptr(), len(reads))
        assert run.to_bytes() == want
        # kc_run_print of a canonical run: KMerPrinter's format over the same records
        rows = np.frombuffer(want, dtype=np.uint8).reshape(-1, 12)
        words = np.ascontiguousarray(rows[:, :8]).view("<u8")[:, 0]
        counts = np.ascontiguousarray(rows[:, 8:]).view("<u4")[:, 0]
        assert run.print_text() == "".join("%s %d\n" % (oracle.print_word(int(w)), int(cn))
                                           for w, cn in zip(words, counts)).encode()
        run.free()
        for block in (0, 77_777):
            run = c.count_fastq(fq, block_bytes=block)
            assert run.to_bytes() == want, block
            run.free()


@pytest.mark.gpu
def test_merge_of_canonical_runs(kc):
    L, k = 100, 31
    a = oracle.gen_reads(1500, L, 20000, 0.01, 0.002, seed=3)
    b = oracle.gen_reads(1500, L, 20000, 0.01, 0.002, seed=4)
    ra, rb = canonical_count(a, L, k), canonical_count(b, L, k)
    with _counter(kc, k, L) as c:
        runs = [c.count_reads(a), c.count_reads(b)]
        assert [r.to_bytes() for r in runs] == [ra, rb]
        m = c.merge(runs)
        assert m.to_bytes() == oracle.merge_runs([ra, rb], k) == canonical_count(np.concatenate([a, b]), L, k)
        for r in runs + [m]:
            r.free()


@pytest.mark.gpu
@pytest.mark.parametrize("occ", [256, 1024, 60000])
def test_super_split_passes_and_bin_sizes(kc, occ):
    for k in (31, 63):
        reads = np.concatenate([oracle.gen_reads(6000, 100, 0, 0.0, 0.001, seed=77),
                                np.tile(oracle.gen_reads(2, 100, 0, 0, 0, seed=79), 500),
                                _u8((b"T" * 100) * 7 + (b"A" * 100) * 5)])
        want = canonical_count(reads, 100, k)
        with _counter(kc, k, 100, method="super", table_slots=occ, cap=1 << 26) as c:
            assert c.process_chunk(reads) == want, k
            assert c.stats()["method_used"] == "super"


@pytest.mark.gpu
def test_super_heavy_hitters_and_oversized_ranges(kc):
    """the overflow list (tens of thousands of copies of a few reads), and Zipf reads plus reads
    that share 45 leading bases: sub-buckets too large for the shared-memory sort"""
    L = 100
    hot = oracle.gen_reads(3, L, 0, 0, 0, seed=5)
    rng = np.random.default_rng(11)
    body = rng.integers(0, 4, size=(9000, L))
    body[:, :45] = rng.integers(0, 4, size=45)
    skew = np.frombuffer(b"ACGT", dtype=np.uint8)[body].reshape(-1)
    inputs = [np.concatenate([np.tile(hot, 30000), oracle.gen_reads(2000, L, 50000, 0.01, 0.001, seed=6)]),
              np.concatenate([skew, oracle.gen_reads(3000, L, 40000, 0.01, 0.001, seed=12)]),
              oracle.gen_reads(20000, L, 50000, 0.005, 0.001, seed=13, zipf_loci=2000)]
    for i, reads in enumerate(inputs):
        for k in (31, 63):
            want = canonical_count(reads, L, k)
            for force_dup in ("0", "1"):
                os.environ["KC_SW_FORCE_DUP"] = force_dup
                try:
                    with _counter(kc, k, L, method="super", cap=1 << 26) as c:
                        assert c.process_chunk(reads) == want, (i, k, force_dup, c.debug_scalars())
                finally:
                    os.environ["KC_SW_FORCE_DUP"] = "0"


@pytest.mark.gpu
def test_accumulate_many_chunks_one_count(kc):
    import torch
    for (R, L, k, expected, chunk_reads) in [(30000, 100, 31, 30000, 7000), (30000, 100, 31, 7000, 7000),
                                             (20000, 100, 63, 20000, 4096), (5000, 70, 28, 0, 1000)]:
        reads = oracle.gen_reads(R, L, 100000, 0.01, 0.002, seed=R + k)
        want = canonical_count(reads, L, k)
        with kc.Counter(k, L, method="super", n_slots=2, max_chunk_bytes=chunk_reads * L, canonical=True) as c:
            c.accum_begin(expected)
            sl, busy = 0, [False, False]
            for r0 in range(0, R, chunk_reads):
                part = reads[r0 * L:(r0 + chunk_reads) * L]
                if busy[sl]:
                    c.accum_wait(sl)
                c.slot_buffer(sl)[:len(part)] = part
                c.accum_submit(sl, len(part))
                busy[sl] = True
                sl ^= 1
            run = c.accum_flush()
            assert run.to_bytes() == want, (R, k, expected)
            run.free()
            d = torch.from_numpy(reads.copy()).cuda()
            c.accum_add_device(d.data_ptr(), len(reads))
            run = c.accum_flush()
            assert run.to_bytes() == want, (R, k, "device")
            run.free()


@pytest.mark.gpu
@pytest.mark.parametrize("P", [2, 3, 5, 8])
@pytest.mark.parametrize("k", [31, 63])
def test_exchange_all_ranks_on_one_device(kc, P, k):
    import torch
    from kmer_counter_b200 import engine
    R, L = 12000, 100
    reads = oracle.gen_reads(R, L, 80000, 0.01, 0.002, seed=P * 100 + k)
    want = canonical_count(reads, L, k)
    per = (R + P - 1) // P
    cs = [kc.Counter(k, L, method="super", canonical=True) for _ in range(P)]
    try:
        bufs = []
        for r, c in enumerate(cs):
            c.xchg_begin(r, P, max(per, 16))
            part = reads[r * per * L:(r + 1) * per * L]
            d = torch.from_numpy(part.copy()).cuda()
            bufs.append(d)
            c.accum_add_device(d.data_ptr(), len(part))
        runs = engine.xchg_run_all(cs)
        parts = [r.to_bytes() for r in runs]
        for r in runs:
            r.free()
        assert b"".join(parts) == want
        keys = [_records(p, k) for p in parts]
        last = None
        for ks in keys:                                   # ranks hold disjoint, ascending key ranges
            if ks:
                assert last is None or ks[0][0] > last
                last = ks[-1][0]
    finally:
        for c in cs:
            c.close()


@pytest.mark.gpu
def test_exchange_refuses_a_peer_with_other_keys(kc):
    L, k = 100, 31
    a = kc.Counter(k, L, method="super", canonical=True)
    b = kc.Counter(k, L, method="super", compat="strict")
    try:
        a.xchg_begin(0, 2, 1000)
        b.xchg_begin(1, 2, 1000)
        with pytest.raises(kc.KcError):
            a.xchg_set_peer(1, b)
    finally:
        a.close()
        b.close()


@pytest.mark.gpu
def test_strand_invariance_at_scale(kc):
    """count(R) == count(revcomp(R)), and R ++ revcomp(R) doubles every count: 1 M reads, auto path
    and accumulator"""
    import torch
    L, k, R = 100, 31, 1_000_000
    reads = oracle.gen_reads(R, L, 5_000_000, 0.01, 0.001, seed=99)
    rc = _revcomp_reads(reads, L)
    with _counter(kc, k, L, cap=R * L) as c:
        a = c.process_chunk(reads)
        assert c.stats()["method_used"] == "super"
        b = c.process_chunk(rc)
    assert a == b
    with kc.Counter(k, L, method="super", canonical=True) as c:
        c.accum_begin(2 * R)
        d1, d2 = torch.from_numpy(reads.copy()).cuda(), torch.from_numpy(rc).cuda()
        c.accum_add_device(d1.data_ptr(), len(reads))
        c.accum_add_device(d2.data_ptr(), len(rc))
        run = c.accum_flush()
        both = run.to_bytes()
        run.free()
    ra = np.frombuffer(a, dtype=np.dtype([("w", "<u8"), ("c", "<u4")]))
    rb = np.frombuffer(both, dtype=np.dtype([("w", "<u8"), ("c", "<u4")]))
    assert np.array_equal(ra["w"], rb["w"]) and np.array_equal(2 * ra["c"].astype(np.uint64), rb["c"].astype(np.uint64))


@pytest.mark.gpu
@pytest.mark.parametrize("args", [("mode=runs",), ("mode=accumulate",), ("mode=accumulate", "gpus=2"),
                                  ("mode=accumulate", "parser=host")])
def test_cli_canonical(tmp_path, args):
    d = tmp_path / "in"
    d.mkdir()
    L, per, k = 100, 2500, 31
    for i in range(3):
        (d / ("part%d.fastq" % i)).write_bytes(oracle.gen_fastq(per, L, 60000, 0.01, 0.002, seed=28, first_read=i * per))
    out = tmp_path / "out.bin"
    env = dict(os.environ, KC_CLI_SAME_DEVICE="1")
    r = subprocess.run([CLI, "kmerLength=%d" % k, "inputFileLocation=%s" % d, "outputFile=%s" % out,
                        "gpuMemoryLimit=1500000", "canonical=1", "tempFileLocation=%s" % tmp_path] + list(args),
                       capture_output=True, text=True, env=env)
    assert r.returncode == 0, r.stderr
    reads = oracle.gen_reads(3 * per, L, 60000, 0.01, 0.002, seed=28)
    assert out.read_bytes() == canonical_count(reads, L, k)
