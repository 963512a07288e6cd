"""GPU parity: the CUDA path (through the C ABI) against the CPU oracle, bit-exact.

Every comparison is on packed record bytes -- the parity artefact of SURVEY.md 0.
"""
import hashlib
import os

import numpy as np
import pytest

import oracle

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def kc():
    import kmer_counter_b200 as kc
    return kc


def _counter(kc, k, L, method="sort", compat="ref", cap=1 << 24, **kw):
    return kc.Counter(k, L, method=method, compat=compat, n_slots=2, max_chunk_bytes=cap, **kw)


CASES = [
    # (reads, L, k, genome, sub, n_rate)
    (2000, 100, 31, 30000, 0.01, 0.002),     # headline k, with N (phantom record, SURVEY F7)
    (2000, 100, 31, 30000, 0.0, 0.0),        # no N: no phantom
    (1500, 100, 32, 20000, 0.01, 0.001),     # k % 32 == 0
    (1500, 100, 28, 20000, 0.0, 0.001),      # masked tail (k % 32 in 1..28)
    (1500, 100, 29, 20000, 0.0, 0.001),      # first unmasked k (SURVEY F4)
    (700, 70, 63, 5000, 0.001, 0.001),       # 128-bit keys, unmasked
    (700, 70, 60, 5000, 0.001, 0.001),       # 128-bit keys, masked
    (500, 41, 33, 0, 0.0, 0.01),             # iid reads, 1 base in the second word
    (300, 150, 96, 2000, 0.01, 0.01),        # 3 words
    (300, 150, 128, 2000, 0.01, 0.01),       # 4 words, k % 32 == 0
    (300, 150, 100, 2000, 0.01, 0.0),        # 4 words masked
    (300, 45, 5, 0, 0.0, 0.02),              # tiny k: few distinct keys, heavy duplication
    (257, 33, 33, 0, 0.0, 0.0),              # one k-mer per read
    (1000, 133, 31, 8000, 0.002, 0.0),       # L % 4 != 0
    (64, 10, 1, 0, 0.0, 0.1),                # k = 1, shortest read the reference handles
]


@pytest.mark.parametrize("R,L,k,G,e,n", CASES)
def test_chunk_matches_oracle_sort(kc, R, L, k, G, e, n):
    reads = oracle.gen_reads(R, L, G, e, n, seed=R + k)
    want = oracle.process_chunk(reads, L, k)
    with _counter(kc, k, L) as c:
        got = c.process_chunk(reads)
    assert got == want


@pytest.mark.parametrize("method", ["hash", "hash_global"])
@pytest.mark.parametrize("R,L,k,G,e,n", [c for c in CASES if c[2] <= 64])
def test_chunk_matches_oracle_hash(kc, R, L, k, G, e, n, method):
    if method == "hash_global" and k > 32:
        with pytest.raises(kc.KcError):                # the HBM-resident table is for 64-bit keys
            _counter(kc, k, L, method=method)
        return
    reads = oracle.gen_reads(R, L, G, e, n, seed=R + k)
    want = oracle.process_chunk(reads, L, k)
    with _counter(kc, k, L, method=method) as c:
        got = c.process_chunk(reads)
        assert c.stats()["method_used"] == method
    assert got == want


@pytest.mark.parametrize("R,L,k,G,e,n", [c for c in CASES if c[2] >= 5])
def test_chunk_matches_oracle_place(kc, R, L, k, G, e, n):
    """The key-placement path (what auto picks for k > 64): a key per slot, two MSD placement passes,
    shared-memory sort + fold per sub-bucket. Every key width, with and without the phantom."""
    reads = oracle.gen_reads(R, L, G, e, n, seed=R + k)
    want = oracle.process_chunk(reads, L, k)
    with _counter(kc, k, L, method="place") as c:
        got = c.process_chunk(reads)
        assert c.stats()["method_used"] == "place"
        sc = c.debug_scalars()
    assert got == want, sc


@pytest.mark.parametrize("k", [96, 128, 100, 65])
def test_place_path_heavy_hitters_deep_plans_and_strict(kc, monkeypatch, k):
    """192/256-bit keys: many copies of one read (a sub-bucket crowded by one key goes through the
    radix sorter), all-T and all-A reads (all-ones and zero keys), a forced deep level-2 plan, and
    strict masking against the window model."""
    L = 150
    reads = np.concatenate([oracle.gen_reads(1500, L, 20000, 0.005, 0.002, seed=k),
                            np.tile(oracle.gen_reads(1, L, 0, 0, 0, seed=k + 1), 4000),      # 4000 copies of every k-mer of one read
                            np.frombuffer((b"T" * L) * 9 + (b"A" * L) * 6, dtype=np.uint8)])
    want = oracle.process_chunk(reads, L, k)
    for sub_target in (None, "3"):
        if sub_target:
            monkeypatch.setenv("KC_SW_SUB_TARGET", sub_target)
        with _counter(kc, k, L, method="auto") as c:
            got = c.process_chunk(reads)
            assert c.stats()["method_used"] == "place"
            sc = c.debug_scalars()
        assert got == want, (sub_target, sc)
    monkeypatch.delenv("KC_SW_SUB_TARGET")
    want = oracle.naive_count(reads, L, k, strict=True)
    with _counter(kc, k, L, compat="strict", method="place") as c:
        assert c.process_chunk(reads) == want


@pytest.mark.parametrize("k", [31, 63, 96, 128])
def test_run_print_matches_kmerprinter_format(kc, k):
    """kc_run_print (the run as text, formatted on the device) against KMerPrinter's format applied to the
    same records on the host (KMerPrinter.cpp:35-91: 32 letters per key word, a blank, the count): a hundred
    tiles of records, counts of one to five digits and the zero-count phantom record."""
    L = 150
    reads = np.concatenate([oracle.gen_reads(900, L, 9000, 0.01, 0.003, seed=k),              # N bases: phantom (0, 0)
                            np.tile(oracle.gen_reads(1, L, 0, 0, 0, seed=k + 1), 12345)])     # counts of 12345
    with _counter(kc, k, L, method="auto", cap=1 << 26) as c:
        run = c.count_reads(reads, chunk_reads=len(reads) // L)
        rec, text = run.to_bytes(), run.print_text()
        run.free()
    assert rec == oracle.process_chunk(reads, L, k)
    W = (k + 31) // 32
    rows = np.frombuffer(rec, dtype=np.uint8).reshape(-1, 8 * W + 4)
    words = np.ascontiguousarray(rows[:, :8 * W]).view("<u8")
    counts = np.ascontiguousarray(rows[:, 8 * W:]).view("<u4")[:, 0]
    assert counts.min() == 0 and counts.max() >= 12345
    want = "".join("".join(oracle.print_word(int(w)) for w in ws) + " %d\n" % int(cn) for ws, cn in zip(words, counts))
    assert text == want.encode()


SUPER_CASES = [c for c in CASES if 22 <= c[2] <= 64]


@pytest.mark.parametrize("R,L,k,G,e,n", SUPER_CASES)
def test_chunk_matches_oracle_super(kc, R, L, k, G, e, n):
    """The super-window path (minimizer-binned 2-bit records, per-bin shared-memory count, MSD
    placement of the distinct records), also with its folding variant forced."""
    reads = oracle.gen_reads(R, L, G, e, n, seed=R + k)
    want = oracle.process_chunk(reads, L, k)
    for force_dup in ("0", "1"):
        os.environ["KC_SW_FORCE_DUP"] = force_dup
        try:
            with _counter(kc, k, L, method="super") as c:
                got = c.process_chunk(reads)
                assert c.stats()["method_used"] == "super"
                sc = c.debug_scalars()
        finally:
            os.environ["KC_SW_FORCE_DUP"] = "0"
        assert got == want, (force_dup, sc)
        assert sc["windows"] == R * (L - k + 1) - sc["invalid"]          # S1 packed every k-mer into a record


def test_auto_picks_super_where_it_applies(kc):
    reads = oracle.gen_reads(500, 100, 9000, 0.01, 0.002, seed=3)
    for k, want_method in ((31, "super"), (63, "super"), (22, "super"), (21, "hash"), (5, "sort"), (96, "place"), (100, "place")):
        with _counter(kc, k, 100, method="auto") as c:
            assert c.process_chunk(reads) == oracle.process_chunk(reads, 100, k)
            assert c.stats()["method_used"] == want_method, k


@pytest.mark.parametrize("occ", [64, 1000, 100000])
def test_super_bin_sizes_and_split_passes(kc, occ):
    """table_slots = k-mer occurrences per minimizer bin: tiny bins, and bins whose distinct keys
    exceed the shared-memory table (counted in 2, 4, ... passes). The artefact must not depend on it."""
    for k in (31, 63):
        reads = np.concatenate([oracle.gen_reads(6000, 100, 0, 0.0, 0.001, seed=77),          # iid: all distinct
                                np.tile(oracle.gen_reads(2, 100, 0, 0, 0, seed=79), 500),      # heavy hitters
                                np.frombuffer((b"T" * 100) * 7 + (b"A" * 100) * 5, dtype=np.uint8)])
        want = oracle.process_chunk(reads, 100, k)
        with _counter(kc, k, 100, method="super", table_slots=occ, cap=1 << 26) as c:
            assert c.process_chunk(reads) == want, k
            assert c.stats()["method_used"] == "super"


def test_super_heavy_hitters_overflow_list(kc):
    """Tens of thousands of copies of a few reads overflow their minimizer bins: the surplus goes to
    the shared overflow list, is counted in slices, and the duplicates are folded after the sort."""
    L = 100
    hot = oracle.gen_reads(3, L, 0, 0, 0, seed=5)
    for reps, kk in ((4000, 31), (30000, 31), (30000, 63)):
        reads = np.concatenate([np.tile(hot, reps), oracle.gen_reads(2000, L, 50000, 0.01, 0.001, seed=6)])
        want = oracle.process_chunk(reads, L, kk)
        with _counter(kc, kk, L, method="super", cap=1 << 26) as c:
            assert c.process_chunk(reads) == want, (reps, kk)
            st, sc = c.stats(), c.debug_scalars()
        if st["method_used"] == "super":
            assert sc["overflow_records"] > 0 and sc["folded"] > 0, (reps, kk, sc)


def test_super_oversized_key_ranges(kc):
    """Skew in key space: thousands of distinct k-mers share their leading bases (reads that start
    with the same 45 bases and then differ), so some sub-buckets of the placement exceed what the
    shared-memory sort takes. They go through the radix sorter instead -- in chunk mode, in the
    accumulating mode, and with the folding variant forced."""
    import torch
    L = 100
    rng = np.random.default_rng(11)
    head = rng.integers(0, 4, size=45)
    n_skew = 9000
    body = rng.integers(0, 4, size=(n_skew, L))
    body[:, :45] = head
    skew = np.frombuffer(b"ACGT", dtype=np.uint8)[body].reshape(-1)
    reads = np.concatenate([skew, oracle.gen_reads(3000, L, 40000, 0.01, 0.001, seed=12)])
    for k in (31, 63):
        want = oracle.process_chunk(reads, L, k)
        for force_dup in ("0", "1"):
            os.environ["KC_SW_FORCE_DUP"] = force_dup
            try:
                with _counter(kc, k, L, method="super", cap=1 << 26) as c:
                    got = c.process_chunk(reads)
                    st, sc = c.stats(), c.debug_scalars()
                assert got == want, (k, force_dup, sc)
                assert st["method_used"] == "super" and sc["big_ranges"] > 0, (k, force_dup, sc)
                with kc.Counter(k, L, method="super") as c:
                    c.accum_begin(len(reads) // L)
                    d = torch.from_numpy(reads.copy()).cuda()
                    c.accum_add_device(d.data_ptr(), len(reads))
                    run = c.accum_flush()
                    sc = c.debug_scalars()
                    assert run.to_bytes() == want, (k, force_dup, "accumulate", sc)
                    assert sc["big_ranges"] > 0
                    run.free()
            finally:
                os.environ["KC_SW_FORCE_DUP"] = "0"


def test_super_accumulate_many_chunks_one_count(kc):
    """kc_accum_*: chunks are only packed into super-window records; one count at the end gives the
    artefact of counting the chunks separately and merging (KMerFileMerger). Also with a plan that
    is too small, so that parts are counted early and merged by the flush."""
    import torch
    for (R, L, k, G, e, n, expected, chunk_reads) in [
            (30000, 100, 31, 200000, 0.01, 0.002, 30000, 7000),
            (30000, 100, 31, 200000, 0.01, 0.002, 7000, 7000),
            (20000, 100, 63, 100000, 0.001, 0.001, 20000, 4096),
            (5000, 70, 28, 0, 0.0, 0.01, 0, 1000)]:
        reads = oracle.gen_reads(R, L, G, e, n, seed=R + k + 1)
        want = oracle.count(reads, L, k)
        for how in ("slots", "device"):
            with kc.Counter(k, L, method="super", n_slots=2, max_chunk_bytes=chunk_reads * L) as c:
                c.accum_begin(expected)
                if how == "slots":
                    sl, busy = 0, [False, False]
                    for r0 in range(0, R, chunk_reads):
                        part = reads[r0 * L:(r0 + chunk_reads) * L]
                        if busy[sl]:
                            c.accum_wait(sl)
                        c.slot_buffer(sl)[:len(part)] = part
                        c.accum_submit(sl, len(part))
                        busy[sl] = True
                        sl ^= 1
                else:
                    d = torch.from_numpy(reads.copy()).cuda()
                    c.accum_add_device(d.data_ptr(), len(reads))
                run = c.accum_flush()
                assert run.to_bytes() == want, (how, R, k, expected)
                run.free()
                run = c.accum_flush()                              # nothing accumulated: an empty run
                assert len(run) == 0
                run.free()


@pytest.mark.parametrize("target", [16, 300, 4000])
def test_partitioned_hash_128bit_keys_bucket_sizes_and_rounds(kc, target):
    R, L, k = 4000, 100, 63
    reads = np.concatenate([oracle.gen_reads(R, L, 0, 0.0, 0.001, seed=78),             # iid: all distinct
                            np.tile(oracle.gen_reads(2, L, 0, 0, 0, seed=79), 500),      # heavy hitters
                            np.frombuffer((b"T" * L) * 7 + (b"A" * L) * 5, dtype=np.uint8)])  # all-ones / zero keys
    want = oracle.process_chunk(reads, L, k)
    with _counter(kc, k, L, method="hash", table_slots=target, cap=1 << 26) as c:
        got = c.process_chunk(reads)
        assert c.stats()["method_used"] == "hash"
    assert got == want


@pytest.mark.parametrize("target", [16, 64, 300, 4000])
def test_partitioned_hash_bucket_sizes_and_rounds(kc, target):
    """table_slots doubles as the keys-per-sub-bucket target of the partitioned hash: small
    targets give many tiny sub-buckets, large ones overflow one shared-memory table and go
    through the multi-round path.  The artefact must not depend on it."""
    R, L, k = 6000, 100, 31
    reads = oracle.gen_reads(R, L, 0, 0.0, 0.001, seed=77)          # iid reads: almost every k-mer distinct
    want = oracle.process_chunk(reads, L, k)
    with _counter(kc, k, L, method="hash", table_slots=target) as c:
        got = c.process_chunk(reads)
        assert c.stats()["method_used"] == "hash"
    assert got == want


def test_partitioned_hash_heavy_hitters(kc):
    """A few keys with huge counts (skew): they stream through one table without overflowing it."""
    L, k = 100, 31
    hot = oracle.gen_reads(3, L, 0, 0, 0, seed=5)
    for reps, kk in ((4000, 31), (30000, 31), (30000, 63)):       # 30000 copies: the warp-aggregated path of hot sub-buckets
        reads = np.concatenate([np.tile(hot, reps), oracle.gen_reads(2000, L, 50000, 0.01, 0.001, seed=6)])
        want = oracle.process_chunk(reads, L, kk)
        with _counter(kc, kk, L, method="hash", cap=1 << 26) as c:
            assert c.process_chunk(reads) == want, (reps, kk)


def test_empty_and_ragged_inputs(kc):
    L, k = 100, 31
    with _counter(kc, k, L) as c:
        assert c.process_chunk(b"") == b""
        assert c.process_chunk(b"ACGT" * 10) == b""              # shorter than one read: ignored
        reads = oracle.gen_reads(10, L, 0, 0, 0, seed=3)
        ragged = np.concatenate([reads, np.frombuffer(b"ACGTACGTAC", dtype=np.uint8)])
        assert c.process_chunk(ragged) == oracle.process_chunk(reads, L, k)   # partial tail ignored
        one = oracle.gen_reads(1, L, 0, 0, 0, seed=4)
        assert c.process_chunk(one) == oracle.process_chunk(one, L, k)


def test_all_invalid_reads_give_only_the_phantom(kc):
    L, k = 50, 31
    reads = np.frombuffer(b"N" * (L * 40), dtype=np.uint8)
    want = oracle.process_chunk(reads, L, k)
    assert want == bytes(12)                                      # key 0, count 0
    for method in ("sort", "hash", "hash_global", "super"):
        with _counter(kc, k, L, method=method) as c:
            assert c.process_chunk(reads) == want


def test_poly_a_and_poly_t(kc):
    L, k = 64 + 5, 31
    reads = np.frombuffer((b"A" * L) * 30 + (b"T" * L) * 20 + (b"A" * 40 + b"N" + b"A" * (L - 41)) * 3, dtype=np.uint8)
    want = oracle.process_chunk(reads, L, k)
    for method in ("sort", "hash", "hash_global", "super"):
        with _counter(kc, k, L, method=method) as c:
            assert c.process_chunk(reads) == want


def test_lowercase_is_invalid(kc):
    L, k = 40, 9
    reads = np.frombuffer((b"ACGTacgtACGTACGTNNACGTACGTACGTACGTACGTAC") * 7, dtype=np.uint8)
    want = oracle.process_chunk(reads, L, k)
    with _counter(kc, k, L) as c:
        assert c.process_chunk(reads) == want


def test_random_shapes_and_hostile_alphabet(kc):
    """Random (L, k, R) over an alphabet with lower case, N, IUPAC letters, digits and bytes >= 0x80:
    validity runs start and stop everywhere. Sort path for every k, partitioned hash for k <= 64."""
    rng = np.random.default_rng(20261019)
    alphabet = np.frombuffer(b"ACGT" * 12 + b"acgtNnRYKM-.*0" + bytes([0, 127, 128, 255]), dtype=np.uint8)
    done = 0
    while done < 24:
        L = int(rng.integers(10, 201))
        if L % 32 == 0 or 2 + 8 * ((L + 31) // 32) > L:            # shapes the reference corrupts (SURVEY F8)
            continue
        k = int(rng.integers(1, min(L, 128) + 1))
        R = int(rng.integers(1, 400))
        reads = np.ascontiguousarray(alphabet[rng.integers(0, alphabet.size, size=R * L)])
        if done % 2 == 0:
            reads = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, size=R * L)].copy()
            reads[rng.integers(0, R * L, size=max(1, R * L // 40))] = rng.choice(alphabet, size=max(1, R * L // 40))
        want = oracle.process_chunk(reads, L, k)
        for method in (("sort", "hash", "super") if k <= 64 else ("sort", "place")):       # super falls back where it does not apply
            with _counter(kc, k, L, method=method) as c:
                assert c.process_chunk(reads) == want, (L, k, R, method)
        done += 1


def test_strict_mode_matches_naive_model(kc):
    for (R, L, k) in [(800, 100, 31), (500, 80, 63), (500, 60, 28)]:
        reads = oracle.gen_reads(R, L, 9000, 0.005, 0.003, seed=k)
        want = oracle.naive_count(reads, L, k, strict=True)
        for method in (("sort", "hash", "hash_global", "super", "place") if k <= 32 else ("sort", "hash", "super", "place")):
            with _counter(kc, k, L, compat="strict", method=method) as c:
                assert c.process_chunk(reads) == want, (k, method)


def test_chunking_invariance_and_merge(kc):
    R, L, k = 5000, 100, 31
    reads = oracle.gen_reads(R, L, 40000, 0.01, 0.002, seed=11)
    want = oracle.count(reads, L, k, chunk_reads=777)
    assert want == oracle.process_chunk(reads, L, k)              # the artefact ignores chunking
    with _counter(kc, k, L) as c:
        for chunk in (R, 1000, 777, 64):
            run = c.count_reads(reads, chunk_reads=chunk)
            assert run.to_bytes() == want
            run.free()


def test_merge_of_same_plan_hash_runs(kc):
    """Three or more partitioned-path runs with one plan (equal chunks) are combined range by range in
    shared-memory tables, up to 8 at a time (kc_merge_runs' fast path); the result is the merge-path
    tree's. 11 equal chunks exercise two levels (8 + 3), the ragged count the mixed case (tree)."""
    L, k, per = 100, 31, 1200
    reads = oracle.gen_reads(11 * per + 500, L, 40000, 0.01, 0.002, seed=31)
    with _counter(kc, k, L, method="hash") as c:
        def chunk_run(part):
            c.slot_buffer(0)[:part.size] = part
            c.submit(0, part.size)
            return c.wait(0)
        d_runs = [chunk_run(reads[i * per * L:(i + 1) * per * L]) for i in range(11)]
        assert len({r.parts()[1:] for r in d_runs}) == 1 and d_runs[0].parts()[1] > 0        # one plan
        for n in (3, 8, 11):
            m = c.merge(d_runs[:n])
            assert m.to_bytes() == oracle.count(reads[:n * per * L], L, k), n
            assert m.parts()[1] == d_runs[0].parts()[1]                                      # structure is kept
            m.free()
        tail = chunk_run(reads[11 * per * L:])
        m = c.merge(d_runs + [tail])                                                         # another plan: the tree
        assert m.to_bytes() == oracle.count(reads, L, k)
        m.free()


def test_merge_runs_against_oracle_merger(kc):
    L, k = 100, 63
    parts = [oracle.gen_reads(400 + 37 * i, L, 6000, 0.01, 0.003, seed=100 + i) for i in range(5)]
    runs_bytes = [oracle.process_chunk(p, L, k) for p in parts]
    want = oracle.merge_runs(runs_bytes, k)
    with _counter(kc, k, L) as c:
        runs = [c.upload_run(b) for b in runs_bytes]
        for n in (0, 1, 2, 3, 5):
            m = c.merge(runs[:n])
            assert m.to_bytes() == oracle.merge_runs(runs_bytes[:n], k)
            m.free()
        m = c.merge(runs)
        assert m.to_bytes() == want


def test_upload_folds_adjacent_duplicates(kc):
    # a run file may repeat a key; SortedKMerFile::ReadKmer folds them (SortedKMerFile.cpp:57-82)
    k = 31
    rec = np.zeros(6, dtype=[("key", "<u8"), ("cnt", "<u4")])
    rec["key"] = [5, 5, 9, 9, 9, 12]
    rec["cnt"] = [1, 2, 0xFFFFFFFF, 2, 1, 7]
    raw = rec.tobytes()
    assert len(raw) == 72
    want = oracle.merge_runs([raw], k)
    with _counter(kc, k, 100) as c:
        assert c.upload_run(raw).to_bytes() == want


def test_count_wraps_at_32_bits(kc):
    # uint32 counts wrap (SURVEY F9): merge two runs whose counts overflow
    k = 31
    a = np.zeros(2, dtype=[("key", "<u8"), ("cnt", "<u4")]); a["key"] = [3, 8]; a["cnt"] = [0xFFFFFFF0, 5]
    b = np.zeros(2, dtype=[("key", "<u8"), ("cnt", "<u4")]); b["key"] = [3, 9]; b["cnt"] = [0x20, 6]
    want = oracle.merge_runs([a.tobytes(), b.tobytes()], k)
    with _counter(kc, k, 100) as c:
        m = c.merge([c.upload_run(a.tobytes()), c.upload_run(b.tobytes())])
        assert m.to_bytes() == want


def test_config1_full_size(kc):
    """BASELINE config 1: 100k reads x 100 bp, k=31, against the oracle."""
    R, L, k = 100_000, 100, 31
    reads = oracle.gen_reads(R, L, 1_000_000, 0.0, 1e-3, seed=1)
    want = oracle.count(reads, L, k, chunk_reads=89364, threads=4)
    for method in ("sort", "hash", "hash_global", "super"):
        with _counter(kc, k, L, method=method) as c:
            got = c.process_chunk(reads)
        assert hashlib.sha256(got).hexdigest() == hashlib.sha256(want).hexdigest(), method


def test_device_resident_input(kc):
    import torch
    R, L, k = 3000, 100, 31
    reads = oracle.gen_reads(R, L, 20000, 0.01, 0.001, seed=5)
    d = torch.from_numpy(reads).cuda()
    want = oracle.process_chunk(reads, L, k)
    with kc.Counter(k, L, method="sort") as c:
        run = c.count_device(d.data_ptr(), d.numel())
        assert run.to_bytes() == want
        st = c.stats()
        assert st["reads"] == R and st["kmer_slots"] == R * (L - k + 1)
        assert st["launches"] > 0 and st["method_used"] == "sort"
        assert st["stage_names"][2] == "radix_scatter_passes" and st["stage_launches"][2] == 8   # 64-bit key, 8-bit digits


def test_run_placed_in_caller_arrays_and_peer_staging(kc):
    """kc_place_next_run: the next partitioned-path run lands in caller-owned arrays (here: staging
    memory from kc_peer_alloc, as the multi-GPU combine uses it) if it fits, and is allocated as
    usual if it does not; a placed run does not own its arrays."""
    import torch
    from kmer_counter_b200 import multigpu
    R, L, k = 4000, 100, 31
    reads = oracle.gen_reads(R, L, 30000, 0.01, 0.001, seed=15)
    d = torch.from_numpy(reads).cuda()
    want = oracle.process_chunk(reads, L, k)
    n_want = len(want) // 12
    with kc.Counter(k, L, method="hash") as c:
        cap, ranges = n_want + 10, 1 << 16
        o_counts, o_offs = 8 * cap, (12 * cap + 255) // 256 * 256
        base, handle = c.peer_alloc(o_offs + 4 * ranges)
        assert len(handle) == 64
        c.place_next_run(base, base + o_counts, base + o_offs, cap, ranges)
        run = c.count_device(d.data_ptr(), d.numel())
        kptr, cptr, n = run.device_arrays()
        off_ptr, n_sub, pbits = run.parts()
        assert (kptr, cptr, off_ptr, n) == (base, base + o_counts, base + o_offs, n_want)
        assert run.to_bytes() == want
        run.free()                                           # leaves the staging memory alone:
        keys = torch.as_tensor(multigpu._CudaView(base, (n_want,), "<i8"), device=d.device).cpu().numpy()
        assert keys.view(np.uint64).tolist() == np.frombuffer(want, dtype=[("k", "<u8"), ("c", "<u4")])["k"].tolist()
        run = c.count_device(d.data_ptr(), d.numel())        # one-shot: the next run is allocated normally
        assert run.device_arrays()[0] != base and run.to_bytes() == want
        run.free()
        c.place_next_run(base, base + o_counts, base + o_offs, n_want - 1, ranges)   # one record too small
        run = c.count_device(d.data_ptr(), d.numel())
        assert run.device_arrays()[0] != base and run.to_bytes() == want
        run.free()
        c.peer_free(base)


def test_run_split_and_file_write(kc, tmp_path):
    R, L, k = 2000, 100, 31
    reads = oracle.gen_reads(R, L, 20000, 0.0, 0.0, seed=6)
    want = oracle.process_chunk(reads, L, k)
    keys, _ = oracle.records_to_arrays(want, k)
    with _counter(kc, k, L) as c:
        run = c.count_reads(reads)
        sp = np.array([[1 << 62], [2 << 62], [3 << 62]], dtype=np.uint64)
        off = run.split(sp)
        exp = [0] + [int(np.searchsorted(keys[:, 0], s[0], side="left")) for s in sp] + [len(keys)]
        assert list(map(int, off)) == exp
        p = str(tmp_path / "out.bin")
        run.write(p)
        assert open(p, "rb").read() == want
        run.write(p)                                   # truncates, unlike KMerFileMerger.cpp:129
        assert os.path.getsize(p) == len(want)


def test_device_generator_matches_host_generator(kc):
    import torch
    from kmer_counter_b200 import synth
    for kw in (dict(genome_len=50000, sub_rate=0.01, n_rate=0.002, seed=3),
               dict(genome_len=0, sub_rate=0.0, n_rate=0.0, seed=4),
               dict(genome_len=80000, sub_rate=0.001, n_rate=0.0, seed=5, zipf_loci=1000)):
        R, L = 3000, 100
        d = torch.empty(R * L, dtype=torch.uint8, device="cuda")
        synth.synth_reads_device(d.data_ptr(), R, L, first_read=17, **kw)
        torch.cuda.synchronize()
        want = oracle.gen_reads(R, L, kw["genome_len"], kw["sub_rate"], kw["n_rate"], seed=kw["seed"], first_read=17,
                                zipf_loci=kw.get("zipf_loci", 0))
        assert bytes(d.cpu().numpy()) == bytes(want)


def test_full_size_properties_config2(kc):
    """BASELINE config 2 at full size (10M reads): size-independent properties -- strictly
    ascending keys, counts sum to the number of k-mers, methods agree byte for byte, and a
    2e5-read prefix is bit-exact against the oracle."""
    import torch
    from kmer_counter_b200 import synth
    R, L, k = 10_000_000, 100, 31
    d = torch.empty(R * L + 256, dtype=torch.uint8, device="cuda")
    synth.synth_reads_device(d.data_ptr(), R, L, 100_000_000, 1e-3, 0.0, seed=2)
    torch.cuda.synchronize()
    digests = {}
    for method in ("super", "hash", "sort"):
        with kc.Counter(k, L, method=method) as c:
            run = c.count_device(d.data_ptr(), R * L)
            kptr, cptr, n = run.device_arrays()
            from kmer_counter_b200.multigpu import run_as_tensors
            keys_t, counts_t = run_as_tensors(run, torch.device("cuda", 0))
            ku = keys_t[:, 0]
            # unsigned order on int64 storage: flip the sign bit
            kk = ku ^ torch.tensor(-2**63, dtype=torch.int64, device="cuda")
            assert bool((kk[1:] > kk[:-1]).all()), "keys not strictly ascending"
            assert int(counts_t.to(torch.int64).sum()) == R * (L - k + 1)
            digests[method] = (n, int(ku.sum()), int((ku * counts_t.to(torch.int64)).sum()))
            if method in ("hash", "super"):
                pre = 200_000
                r2 = c.count_device(d.data_ptr(), pre * L)
                host = d[: pre * L].cpu().numpy()
                assert r2.to_bytes() == oracle.count(host, L, k, threads=8)
                r2.free()
            run.free()
    assert digests["hash"] == digests["sort"] == digests["super"]


def test_fastq_parse_on_device(kc):
    """N1: raw FASTQ text parsed on the GPU, in blocks with carry-over, against the oracle's
    restatement of the reference reader + counter."""
    import torch
    L, k, R = 100, 31, 5000
    fq = oracle.gen_fastq(R, L, 60000, 0.01, 0.002, seed=31)
    assert oracle.parse_fastq(fq) == oracle.gen_reads(R, L, 60000, 0.01, 0.002, seed=31).tobytes()
    want = oracle.count(oracle.parse_fastq(fq), L, k)
    with _counter(kc, k, L, method="auto", cap=1 << 20) as c:
        for block in (0, 50_000, 7_777, 1_000_003):
            run = c.count_fastq(fq, block_bytes=block)
            assert run.to_bytes() == want, block
            run.free()
        # no trailing newline, CRLF line ends
        run = c.count_fastq(fq[:-1]); assert run.to_bytes() == want; run.free()
        run = c.count_fastq(fq.replace(b"\n", b"\r\n")); assert run.to_bytes() == want; run.free()
        # parse only, device buffers
        d_text = torch.from_numpy(np.frombuffer(fq, dtype=np.uint8).copy()).cuda()
        d_reads = torch.empty(R * L, dtype=torch.uint8, device="cuda")
        n, used, fl = c.parse_fastq_device(d_text.data_ptr(), d_text.numel(), d_reads.data_ptr(), d_reads.numel())
        assert (n, used, fl) == (R, len(fq), 0)
        assert bytes(d_reads.cpu().numpy()) == oracle.parse_fastq(fq)
        n, used, fl = c.parse_fastq_device(d_text.data_ptr(), len(fq) - 150, d_reads.data_ptr(), d_reads.numel())
        assert (n, fl) == (R - 1, 0) and used == len(fq) - 220                 # the cut record is left to the caller
        # shapes the device parser refuses (the host chunker handles them)
        ragged = fq[:220] + b"@x\nACGT\n+\nIIII\n" + fq[220:]
        assert c.submit_fastq(0, ragged)[1] == 2
        multi = b"@r\nACGT\nACGT\n+\nIIIIIIII\n" * 4
        assert c.submit_fastq(0, multi)[1] & 1
        with pytest.raises(kc.KcError):
            c.count_fastq(ragged)
