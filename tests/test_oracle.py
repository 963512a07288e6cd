"""CPU tests: the oracle (oracle/kc_oracle.c) against the golden vectors produced by the
reference's own code (tests/golden, made by make_golden.py from oracle/_ref) and against
SURVEY.md Appendix A.4's known answers."""
import hashlib
import json
import os

import numpy as np
import pytest

import oracle

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

# shapes of the comparisons with the reference build (tests/golden/reference_digests.json)
REFERENCE_CASES = [(1500, 100, 31, 20000, 0.01, 0.003), (600, 70, 63, 5000, 0.0, 0.002),
                   (300, 150, 96, 2000, 0.01, 0.01), (300, 150, 128, 2000, 0.01, 0.01),
                   (400, 45, 5, 0, 0.0, 0.02), (900, 100, 28, 9000, 0.0, 0.0),
                   (400, 133, 100, 3000, 0.001, 0.001), (500, 41, 33, 0, 0.0, 0.01),
                   (300, 37, 29, 0, 0.0, 0.0), (300, 100, 64, 4000, 0.0, 0.004)]


def _hexkeys(data, k):
    keys, counts = oracle.records_to_arrays(data, k)
    return [[["%016x" % int(w) for w in row], int(c)] for row, c in zip(keys, counts)]


def _sha(data):
    return hashlib.sha256(bytes(data)).hexdigest()


def _reference_digests():
    with open(os.path.join(GOLD, "reference_digests.json")) as f:
        return json.load(f)


def case_key(R, L, k, G, e, n):
    return "R=%d L=%d k=%d G=%d e=%r n=%r" % (R, L, k, G, e, n)


def random_shapes():
    """60 random shapes (k 1..128, L up to 200, L % 32 != 0) over a hostile alphabet -- lower case,
    N, IUPAC letters, digits, bytes >= 0x80 -- so that validity runs start and stop everywhere.
    Yields (L, k, R, reads)."""
    rng = np.random.default_rng(20261018)
    alphabet = np.frombuffer(b"ACGT" * 12 + b"acgtNnRYKM-.*0" + bytes([0, 127, 128, 255]), dtype=np.uint8)
    done = 0
    while done < 60:
        L = int(rng.integers(10, 201))
        if L % 32 == 0 or 2 + 8 * ((L + 31) // 32) > L:            # shapes the reference corrupts (SURVEY F8)
            continue
        k = int(rng.integers(1, min(L, 128) + 1))
        R = int(rng.integers(1, 60))
        reads = alphabet[rng.integers(0, alphabet.size, size=R * L)]
        if done % 3 == 0:                                           # mostly valid reads with a few bad letters
            reads = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, size=R * L)].copy()
            reads[rng.integers(0, R * L, size=max(1, R * L // 50))] = ord("N")
        yield L, k, R, np.ascontiguousarray(reads)
        done += 1


def test_survey_appendix_a4_known_answers():
    """SURVEY.md Appendix A.4 (values produced by the reference's kernel code)."""
    r = b"ACGTACGTACGTACGTACGTACGTACGTACGTTTGGCCAAC"
    w, f = oracle.encode_read(r)
    assert [int(x) for x in w] == [0x1b1b1b1b1b1b1b1b, 0xfa50400000000000] and int(f[0]) == 0

    def keys(k):
        raw, n = oracle.extract_read(r, k)
        ks, _ = oracle.records_to_arrays(raw.tobytes(), k)
        return n, ks

    n, ks = keys(31)
    assert n == 11 and [int(x) for x in ks[:3, 0]] == [0x1b1b1b1b1b1b1b1b, 0x6c6c6c6c6c6c6c6f, 0xb1b1b1b1b1b1b1bf]
    assert int(ks[10, 0]) == 0xb1b1b1b1b1bfa504
    n, ks32 = keys(32)
    assert n == 10 and (ks32[:3, 0] == ks[:3, 0]).all() and int(ks32[9, 0]) == 0x6c6c6c6c6c6fe941      # F4
    n, ks = keys(28)
    assert n == 14 and [int(x) for x in ks[:3, 0]] == [0x1b1b1b1b1b1b1b00, 0x6c6c6c6c6c6c6c00, 0xb1b1b1b1b1b1b100]
    assert int(ks[13, 0]) == 0x6c6c6c6c6fe94100
    n, ks = keys(33)
    assert n == 9 and [int(x) for x in ks[0]] == [0x1b1b1b1b1b1b1b1b, 0xc000000000000000]
    assert [int(x) for x in ks[2]] == [0xb1b1b1b1b1b1b1bf, 0x8000000000000000]
    assert [int(x) for x in ks[8]] == [0x1b1b1b1b1b1bfa50, 0x4000000000000000]
    # the N read: filter word, and the zero-count phantom record (F7)
    w, f = oracle.encode_read(b"ACGTNACGTACG")
    assert int(w[0]) == 0x1bc6c60000000000 and int(f[0]) == 0x0800000000000000
    got = _hexkeys(oracle.process_chunk(b"ACGTNACGTACG", 12, 5, do_sort=False), 5)
    assert got == [[["1b00000000000000"], 1], [["6c40000000000000"], 1], [["b180000000000000"], 1],
                   [["0000000000000000"], 0]]


def test_golden_kat_from_reference_kernels():
    kat = json.load(open(os.path.join(GOLD, "kat.json")))
    assert len(kat["cases"]) >= 15
    for c in kat["cases"]:
        read, k = c["read"].encode(), c["k"]
        got = _hexkeys(oracle.process_chunk(read, len(read), k, do_sort=False), k)
        assert got == c["records_unsorted_reduced"], (c["read"], k)


def test_golden_pipeline_b_artefacts():
    fix = json.load(open(os.path.join(GOLD, "pipeline_b.json")))
    for c in fix["cases"]:
        reads = oracle.gen_reads(c["reads"], c["L"], c["genome"], c["sub"], c["n"], seed=c["seed"])
        assert hashlib.sha256(reads.tobytes()).hexdigest() == c["reads_sha256"], "generator drifted"
        art = oracle.count(reads, c["L"], c["k"], chunk_reads=c["chunk_reads"], threads=2)
        assert len(art) // oracle.record_size(c["k"]) == c["records"]
        assert hashlib.sha256(art).hexdigest() == c["artefact_sha256"], c


def test_golden_small_artefacts_bytes():
    reads = np.fromfile(os.path.join(GOLD, "small_reads_L60.bin"), dtype=np.uint8)
    for k in (31, 40):
        want = open(os.path.join(GOLD, "small_k%d.records" % k), "rb").read()
        assert oracle.count(reads, 60, k, chunk_reads=64) == want
        assert oracle.count(reads, 60, k, chunk_reads=7, threads=3) == want        # chunking / threads invariant
        assert oracle.naive_count(reads, 60, k) == want                            # independent window model
        keys, counts = oracle.records_to_arrays(want, k)
        order = [tuple(int(x) for x in row) for row in keys]
        assert order == sorted(order) and len(set(order)) == len(order)           # strictly ascending


@pytest.mark.parametrize("R,L,k,G,e,n", REFERENCE_CASES)
def test_oracle_equals_reference_build(R, L, k, G, e, n):
    """The chunk artefact (sorted and unsorted) and Pipeline B's merged file against the reference
    build's on the same reads (sha256, tests/golden/reference_digests.json)."""
    want = _reference_digests()["chunks"][case_key(R, L, k, G, e, n)]
    reads = oracle.gen_reads(R, L, G, e, n, seed=1000 + R + k)
    assert _sha(reads) == want["reads_sha256"], "generator drifted"
    assert _sha(oracle.process_chunk(reads, L, k, True)) == want["sorted_sha256"]
    assert _sha(oracle.process_chunk(reads, L, k, False)) == want["unsorted_sha256"]
    art = oracle.count(reads, L, k, chunk_reads=max(1, R // 5), threads=2)
    assert _sha(art) == want["artefact_sha256"]
    assert oracle.naive_count(reads, L, k) == art


def test_random_shapes_and_alphabets_three_way():
    """random_shapes(): restatement == reference build (sha256 of its output, sorted and unsorted)
    == independent window model."""
    want = _reference_digests()["random_shapes"]
    done = 0
    for (L, k, R, reads), w in zip(random_shapes(), want):
        assert (L, k, R, _sha(reads)) == (w["L"], w["k"], w["R"], w["reads_sha256"]), "shape generator drifted"
        assert _sha(oracle.process_chunk(reads, L, k, True)) == w["sorted_sha256"], (L, k, R)
        assert _sha(oracle.process_chunk(reads, L, k, False)) == w["unsorted_sha256"], (L, k, R)
        assert oracle.count(reads, L, k, chunk_reads=7) == oracle.naive_count(reads, L, k), (L, k, R)
        done += 1
    assert done == len(want) == 60


def test_merge_semantics():
    k = 31
    mk = lambda pairs: np.array(pairs, dtype=[("key", "<u8"), ("cnt", "<u4")]).tobytes()
    a = mk([(1, 2), (5, 1), (5, 3), (9, 0xFFFFFFFF)])          # intra-run duplicate is folded
    b = mk([(0, 0), (5, 10), (9, 2)])
    c = mk([])
    assert oracle.merge_runs([a, b, c], k) == mk([(0, 0), (1, 2), (5, 14), (9, 1)])     # uint32 wrap (F9)
    assert oracle.merge_runs([], k) == b""
    assert oracle.merge_runs([a], k) == mk([(1, 2), (5, 4), (9, 0xFFFFFFFF)])


def test_unsupported_shapes_are_rejected():
    reads = oracle.gen_reads(4, 64, 0, 0, 0, seed=1)
    with pytest.raises(ValueError):
        oracle.process_chunk(reads, 64, 31)           # L % 32 == 0: the reference corrupts its last word (F8)
    with pytest.raises(ValueError):
        oracle.process_chunk(oracle.gen_reads(4, 20, 0, 0, 0, seed=1), 20, 31)     # k > L


def test_fastq_parser_restatement():
    fq = oracle.gen_fastq(50, 100, 5000, 0.01, 0.01, seed=3)
    packed = oracle.parse_fastq(fq)
    assert packed == oracle.gen_reads(50, 100, 5000, 0.01, 0.01, seed=3).tobytes()
    # what the reference's reader (FASTQFileReader / InputFileHandler) made of the same file
    want = _reference_digests()["fastq_reader"]
    assert (want["fastq_sha256"], want["L"], want["sha256"]) == (_sha(fq), 100, _sha(packed))
    # a quality line that starts with '+' is harmless; lower-case bases survive the reader
    txt = b"@r1\nACGTACGTAC\n+\n+IIIIIIIII\n@r2\nacgtNNACGT\n+\nIIIIIIIIII\n"
    assert oracle.parse_fastq(txt) == b"ACGTACGTACacgtNNACGT"


def test_printer_restatement():
    assert oracle.print_word(0x1b1b1b1b1b1b1b1b) == "ACGT" * 8
    assert oracle.print_word(0) == "A" * 32 and oracle.print_word(2**64 - 1) == "T" * 32


def test_generator_is_deterministic_and_shardable():
    a = oracle.gen_reads(1000, 100, 50000, 0.01, 0.001, seed=9)
    b = np.concatenate([oracle.gen_reads(400, 100, 50000, 0.01, 0.001, seed=9),
                        oracle.gen_reads(600, 100, 50000, 0.01, 0.001, seed=9, first_read=400)])
    assert (a == b).all()
    z = oracle.gen_reads(2000, 100, 50000, 0.0, 0.0, seed=9, zipf_loci=100)
    assert set(np.unique(z)) <= set(b"ACGT")
