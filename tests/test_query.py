"""Lookups in a run on the GPU (kc_run_lookup, kc_query_reads, Counter.lookup / query_reads, `query`).

The model: every slot r*(L-k+1)+p of a read set gets the key counting puts its occurrence under and a
validity mark (the window holds only A, C, G, T), in numpy; its count is looked up in the run's records
(oracle.records_to_arrays). On the CPU the model is checked against oracle.extract_read (the reference's
own extraction, KC_COMPAT_REF) and a string model (strict, canonical); on the GPU both calls are checked
against it for runs of every method and mode."""
import contextlib
import ctypes
import gc
import os
import subprocess

import numpy as np
import pytest

import oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "kmer-counter_b200", "host", "kmer_counter_b200")
U32 = 2**32
CODE = {"A": 0, "C": 1, "G": 2, "T": 3}
COMP = bytes.maketrans(b"ACGT", b"TGCA")
MODES = ["ref", "strict", "canonical"]
KC_ERR_ARG, KC_ERR_NOMEM = -1, -3


# ---------------------------------------------------------------------------- model
def _word_revcomp(x):
    """reverse complement of 32 bases per uint64: 2-bit groups reversed, code ^ 3"""
    x = x.copy()
    for sh, m in ((2, 0x3333333333333333), (4, 0x0F0F0F0F0F0F0F0F), (8, 0x00FF00FF00FF00FF),
                  (16, 0x0000FFFF0000FFFF), (32, 0x00000000FFFFFFFF)):
        m, sh = np.uint64(m), np.uint64(sh)
        x = ((x >> sh) & m) | ((x & m) << sh)
    return ~x


def canonical_keys(x, k):
    """min(x, rc(x)) in record order of strict keys x[..., W]"""
    W = x.shape[-1]
    r = _word_revcomp(x[..., ::-1])
    sh = 2 * (32 * W - k)
    if sh:
        nxt = np.concatenate([r[..., 1:], np.zeros(r.shape[:-1] + (1,), dtype=np.uint64)], axis=-1)
        r = (r << np.uint64(sh)) | (nxt >> np.uint64(64 - sh))
    lt = np.zeros(x.shape[:-1], dtype=bool)
    decided = np.zeros(x.shape[:-1], dtype=bool)
    for q in range(W):
        lt |= ~decided & (r[..., q] < x[..., q])
        decided |= r[..., q] != x[..., q]
    return np.where(lt[..., None], r, x)


def last_mask(k, mode):
    m = k % 32
    masked = m != 0 if mode != "ref" else 1 <= m <= 28
    return ((2**64 - 1) << (64 - 2 * m)) & (2**64 - 1) if masked else 2**64 - 1


def slot_model(reads, L, k, mode):
    """(keys[R, nk, W] uint64, valid[R, nk] bool) of every slot: the 2-bit codes of bases p .. p + 32W
    (past the read end 0, a byte other than A, C, G, T 3), word W-1 masked to the mode's span"""
    a = np.asarray(reads, dtype=np.uint8)
    R = a.size // L
    rows = a[:R * L].reshape(R, L)
    W, nk = (k + 31) // 32, L - k + 1
    code = np.full((R, L + 32 * W), 0, dtype=np.uint64)
    lut = np.full(256, 3, dtype=np.uint64)
    for ch, v in CODE.items():
        lut[ord(ch)] = v
    code[:, :L] = lut[rows]
    bad = np.ones(256, dtype=np.int32)
    for ch in b"ACGT":
        bad[ch] = 0
    cb = np.zeros((R, L + 1), dtype=np.int32)
    cb[:, 1:] = np.cumsum(bad[rows], axis=1)
    valid = (cb[:, k:k + nk] - cb[:, :nk]) == 0
    keys = np.zeros((R, nk, W), dtype=np.uint64)
    for q in range(W):
        acc = np.zeros((R, nk), dtype=np.uint64)
        for j in range(32):
            acc |= code[:, 32 * q + j:32 * q + j + nk] << np.uint64(62 - 2 * j)
        keys[:, :, q] = acc
    keys[:, :, W - 1] &= np.uint64(last_mask(k, mode))
    if mode == "canonical":
        keys = canonical_keys(keys, k)
    return keys, valid


def find(run: bytes, k, q):
    """counts in the run's records of keys q[..., W] (0 if absent)"""
    W = (k + 31) // 32
    rk, rc = oracle.records_to_arrays(run, k)
    flat = np.ascontiguousarray(q.reshape(-1, W))
    if len(rk) == 0:
        return np.zeros(q.shape[:-1], dtype=np.uint32)
    as_bytes = lambda x: np.ascontiguousarray(x.astype(">u8")).view("S%d" % (8 * W)).reshape(-1)
    idx = np.searchsorted(as_bytes(rk), as_bytes(flat))
    idx_c = np.minimum(idx, len(rk) - 1)
    hit = (idx < len(rk)) & np.all(rk[idx_c] == flat, axis=1)
    return np.where(hit, rc[idx_c], 0).astype(np.uint32).reshape(q.shape[:-1])


def query_model(run: bytes, reads, L, k, mode, lo=1, hi=U32 - 1):
    """(slot_counts[R, nk], hits[R]) of kc_query_reads"""
    keys, valid = slot_model(reads, L, k, mode)
    c = np.where(valid, find(run, k, keys), 0).astype(np.uint32)
    hits = np.sum(valid & (c >= lo) & (c <= hi), axis=1).astype(np.uint32)
    return c, hits


def _encode(kmer: bytes):
    W = (len(kmer) + 31) // 32
    v = 0
    for ch in kmer.decode().ljust(32 * W, "A"):
        v = (v << 2) | CODE[ch]
    return [(v >> (64 * (W - 1 - i))) & (2**64 - 1) for i in range(W)]


def string_model(read: bytes, k, mode):
    """(keys, valid) of one read from the k-mer text: strict = the k letters, canonical = the smaller of
    the text and its reverse complement"""
    W, nk = (k + 31) // 32, len(read) - k + 1
    keys, valid = np.zeros((nk, W), dtype=np.uint64), np.zeros(nk, dtype=bool)
    for p in range(nk):
        w = read[p:p + k]
        if all(ch in b"ACGT" for ch in w):
            valid[p] = True
            x = _encode(w)
            if mode == "canonical":
                x = min(x, _encode(w.translate(COMP)[::-1]))
            keys[p] = x
    return keys, valid


def model_run(reads, L, k, mode) -> bytes:
    """the run counted from the reads: every valid slot's key, counted"""
    keys, valid = slot_model(reads, L, k, mode)
    W = (k + 31) // 32
    v = keys[valid].reshape(-1, W)
    if len(v) == 0:
        return b""
    u, c = np.unique(v, axis=0, return_counts=True)
    out = np.zeros(len(u), dtype=np.dtype([("w", "<u8", (W,)), ("c", "<u4")]))
    out["w"], out["c"] = u, c
    return out.tobytes()


HAND = [b"ACGTNACGTACGTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTGCA", b"A" * 70, b"T" * 70,
        b"ACGTACGTACGTACGTACGTACGTACGTACGTTTGGCCAAC" * 2 + b"NACGT",
        b"AAAACCCCGGGGTTTT" * 8 + b"A", b"ACGTNNNNACGTAGCTAGCTAGCTAGCTACGATCGATGCATGCA" * 3 + b"N",
        b"GATC" * 40 + b"G", b"CCCCCCCCCCCCCCCCCCCCCCCCCCCCCCCCCCGGGGGGGGGGGGGGGGGGGGGGGGGGGGGGG" * 2]
K_CPU = [1, 2, 5, 16, 28, 29, 30, 31, 32, 33, 60, 63, 64, 65, 96, 97, 128]


# ------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("k", K_CPU)
def test_ref_model_matches_the_reference_extraction(k):
    for read in HAND:
        if len(read) < k:
            continue
        keys, valid = slot_model(np.frombuffer(read, np.uint8), len(read), k, "ref")
        recs, n = oracle.extract_read(read, k)
        want = oracle.records_to_arrays(recs.tobytes(), k)[0][:n]
        assert n == valid.sum()
        assert np.array_equal(keys[0][valid[0]], want), read


@pytest.mark.parametrize("mode", ["strict", "canonical"])
@pytest.mark.parametrize("k", K_CPU)
def test_strict_and_canonical_model_match_the_string_model(k, mode):
    for read in HAND:
        if len(read) < k:
            continue
        keys, valid = slot_model(np.frombuffer(read, np.uint8), len(read), k, mode)
        sk, sv = string_model(read, k, mode)
        assert np.array_equal(valid[0], sv)
        assert np.array_equal(keys[0][sv], sk[sv]), read


def test_canonical_model_palindrome_and_strands():
    k = 6
    pal = b"ACGCGT"                                            # its own reverse complement
    keys, _ = slot_model(np.frombuffer(pal, np.uint8), 6, k, "canonical")
    assert keys[0, 0].tolist() == _encode(pal)
    read = b"ACGTTGCAACGGA"
    rc = read.translate(COMP)[::-1]
    a, _ = slot_model(np.frombuffer(read, np.uint8), len(read), k, "canonical")
    b, _ = slot_model(np.frombuffer(rc, np.uint8), len(rc), k, "canonical")
    assert np.array_equal(a[0], b[0][::-1])


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("k", [5, 31, 33, 96])
def test_slot_count_identity_on_the_model(k, mode):
    """for a run counted from exactly the queried reads, the valid slots with count c number c * hist[c],
    and every valid slot has a count >= 1"""
    L = 120
    reads = oracle.gen_reads(200, L, 3000, 0.01, 0.01, seed=k)
    if mode == "ref":
        run = oracle.count(reads, L, k)
    elif mode == "strict":
        run = oracle.naive_count(reads, L, k, strict=True)
    else:
        run = model_run(reads, L, k, mode)
    if mode != "canonical":
        assert run == model_run(reads, L, k, mode) or mode == "ref"
    c, hits = query_model(run, reads, L, k, mode)
    _, valid = slot_model(reads, L, k, mode)
    assert (c[valid] >= 1).all() and (c[~valid] == 0).all()
    assert np.array_equal(hits, valid.sum(axis=1))
    counts = oracle.records_to_arrays(run, k)[1].astype(np.int64)
    hist = np.bincount(counts)
    seen = np.bincount(c[valid].astype(np.int64), minlength=len(hist))
    assert np.array_equal(seen[1:], np.arange(1, len(hist)) * hist[1:])


def _cli_nodev(*args):
    return subprocess.run([CLI, "query"] + list(args), capture_output=True, text=True,
                          env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), timeout=120)


@pytest.mark.skipif(not os.path.exists(CLI), reason="command line not built")
def test_cli_rejects_bad_usage_before_touching_a_device(tmp_path):
    rec = tmp_path / "r.bin"
    rec.write_bytes(b"")
    for args in ((), (str(rec),), (str(rec), "31", "-"), (str(rec), "0", "-", "-"), (str(rec), "129", "-", "-"),
                 (str(rec), "x", "-", "-"), (str(rec), "31", "-", "-", "compat=strict", "bogus=1")):
        r = _cli_nodev(*args)
        assert r.returncode == 2 and "usage" in r.stderr, args
    for k in (29, 30, 31, 61, 95, 127):                       # a REF key spans 32 bases there
        r = _cli_nodev(str(rec), str(k), "-", "-")
        assert r.returncode == 2 and "compat=ref" in r.stderr, k
        r = _cli_nodev(str(rec), str(k), "-", "-", "canonical=1", "canonical=0")     # the last word is REF
        assert r.returncode == 2 and "compat=ref" in r.stderr, k
        # canonical keys are strict whatever compat= says (as counting has it): not refused, it goes on to
        # the device, which this process does not see
        for flags in (("canonical=1", "compat=ref"), ("compat=ref", "canonical=1"), ("compat=strict",)):
            r = _cli_nodev(str(rec), str(k), "-", "-", *flags)
            assert r.returncode == 1 and "kc_create" in r.stderr, (k, flags, r.stderr)


# ------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def kc():
    import kmer_counter_b200 as kc
    return kc


def _counter(kc, k, L, mode, **kw):
    return kc.Counter(k, L, compat="ref" if mode == "ref" else "strict", canonical=mode == "canonical", **kw)


def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _count(c, reads):
    d = _dev(reads)
    return c.count_device(d.data_ptr(), d.numel())


def _records(keys, counts, W):
    out = np.zeros(len(counts), dtype=np.dtype([("w", "<u8", (W,)), ("c", "<u4")]))
    out["w"] = np.asarray(keys, dtype=np.uint64).reshape(-1, W)
    out["c"] = np.asarray(counts, dtype=np.uint64).astype(np.uint32)
    return out.tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("k", [1, 5, 31, 32, 33, 63, 64, 96, 128])
def test_lookup_every_key_of_a_counted_run(kc, k, mode):
    L = max(150, k)
    reads = oracle.gen_reads(2000, L, 20000, 0.01, 0.005, seed=k)
    W = (k + 31) // 32
    with _counter(kc, k, L, mode) as c:
        run = _count(c, reads)
        keys, counts = oracle.records_to_arrays(run.to_bytes(), k)
        assert np.array_equal(c.lookup(run, keys), counts)
        # perturbed keys: the lowest base of the k-mer changed (where the result is not in the run)
        pert = keys.copy()
        pert[:, W - 1] ^= np.uint64(1 << (64 - 2 * (k - 32 * (W - 1))))
        want = find(run.to_bytes(), k, pert)
        if mode == "canonical":
            want = find(run.to_bytes(), k, canonical_keys(pert, k))
        assert np.array_equal(c.lookup(run, pert), want)
        if k >= 16:
            assert (want == 0).mean() > 0.9
        if mode == "canonical":
            rc = _word_revcomp(keys[:, ::-1])
            sh = 2 * (32 * W - k)
            if sh:
                nxt = np.concatenate([rc[:, 1:], np.zeros((len(rc), 1), dtype=np.uint64)], axis=1)
                rc = (rc << np.uint64(sh)) | (nxt >> np.uint64(64 - sh))
            assert np.array_equal(c.lookup(run, rc), counts)          # either strand
        if mode != "ref" and k % 32:
            stray = keys.copy()
            stray[:, W - 1] |= np.uint64(1)                            # a bit past the k bases
            assert not c.lookup(run, stray).any()
        run.free()


@pytest.mark.gpu
@pytest.mark.parametrize("k", [31, 32, 128])
def test_lookup_uploaded_edge_runs(kc, k):
    W = (k + 31) // 32
    rng = np.random.default_rng(k)
    ones = np.full((1, W), 2**64 - 1, dtype=np.uint64)
    zero = np.zeros((1, W), dtype=np.uint64)
    if k % 32:
        ones[0, W - 1] &= np.uint64(last_mask(k, "ref"))
    with kc.Counter(k, k) as c:
        empty = c.upload_run(b"")
        q = rng.integers(0, 2**63, size=(1001, W), dtype=np.uint64)
        assert not c.lookup(empty, q).any()
        assert len(c.lookup(empty, q[:0])) == 0
        one = c.upload_run(_records(q[:1], [7], W))
        assert c.lookup(one, q[:3]).tolist() == [7, 0, 0]
        for n in (2, 3, 1000, 4097, 100_003):
            body = np.unique(rng.integers(1, 2**63, size=(n, W), dtype=np.uint64), axis=0)
            keys = np.concatenate([zero, body, ones])
            counts = rng.integers(0, U32, len(keys), dtype=np.uint64)
            counts[:3] = [0, U32 - 1, 1]
            rec = _records(keys, counts, W)
            run = c.upload_run(rec)
            assert np.array_equal(c.lookup(run, keys), counts.astype(np.uint32))
            perm = rng.permutation(len(keys))
            assert np.array_equal(c.lookup(run, keys[perm]), counts.astype(np.uint32)[perm])
            miss = keys.copy()
            miss[:, W - 1] ^= np.uint64(1 << 40)
            assert np.array_equal(c.lookup(run, miss), find(rec, k, miss))
            run.free()
        empty.free()
        one.free()


@pytest.mark.gpu
@pytest.mark.parametrize("k", [31, 64, 128])
def test_lookup_device_keys_at_any_alignment(kc, k):
    """device keys and counts used in place when aligned for the kernel's loads, staged otherwise (128- and
    256-bit keys at an 8-byte offset, counts at a 2-byte offset)"""
    import torch
    W = (k + 31) // 32
    rng = np.random.default_rng(k)
    keys = np.unique(rng.integers(0, 2**63, size=(5000, W), dtype=np.uint64), axis=0)
    if k % 32:
        keys[:, W - 1] &= np.uint64(last_mask(k, "strict"))
        keys = np.unique(keys, axis=0)
    counts = rng.integers(1, 100, len(keys))
    q = np.concatenate([keys, keys ^ np.uint64(1 << 40)])
    want = find(_records(keys, counts, W), k, q)
    with kc.Counter(k, k) as c:
        run = c.upload_run(_records(keys, counts, W))
        buf = torch.zeros(q.size + W, dtype=torch.int64, device="cuda")
        out = torch.zeros(len(q) + 2, dtype=torch.int32, device="cuda")
        assert buf.data_ptr() % 16 == 0 and out.data_ptr() % 16 == 0
        for key_off in (0, 1):                              # in words: 8 and 16-byte aligned
            buf[key_off:key_off + q.size] = torch.from_numpy(q.reshape(-1).view(np.int64)).cuda()
            for count_off in (0, 2):                        # in bytes: 4- and 2-byte aligned
                out.zero_()
                torch.cuda.synchronize()                # torch's writes are on its own stream
                c.lookup_device(run, buf.data_ptr() + 8 * key_off, len(q), out.data_ptr() + count_off)
                raw = out.cpu().numpy().view(np.uint8)[count_off:count_off + 4 * len(q)]
                assert np.array_equal(np.frombuffer(raw.tobytes(), np.uint32), want), (key_off, count_off)
        # query_reads with device outputs at a 2-byte offset
        L = k + 20
        reads = oracle.gen_reads(300, L, 5000, 0.01, 0.01, seed=k)
        run2 = c.upload_run(model_run(reads, L, k, "ref"))
        with kc.Counter(k, L) as cl:
            d = _dev(reads)
            sc = torch.zeros(300 * 21 + 1, dtype=torch.int32, device="cuda")
            h = torch.zeros(301, dtype=torch.int32, device="cuda")
            torch.cuda.synchronize()                # torch's writes are on its own stream
            cl.query_reads_device(run2, d.data_ptr(), d.numel(), sc.data_ptr() + 2, h.data_ptr() + 2, 1, 1)
            want_sc, want_h = query_model(model_run(reads, L, k, "ref"), reads, L, k, "ref", 1, 1)
            got_sc = np.frombuffer(sc.cpu().numpy().view(np.uint8)[2:2 + 4 * want_sc.size].tobytes(), np.uint32)
            got_h = np.frombuffer(h.cpu().numpy().view(np.uint8)[2:2 + 4 * 300].tobytes(), np.uint32)
            assert np.array_equal(got_sc, want_sc.reshape(-1)) and np.array_equal(got_h, want_h)
        run.free()
        run2.free()


@pytest.mark.gpu
@pytest.mark.parametrize("k", [31, 63])
def test_lookup_of_host_keys_in_several_pieces(kc, k):
    """a little over 2^24 host keys: kc_run_lookup stages them in two pieces"""
    W = (k + 31) // 32
    rng = np.random.default_rng(k)
    keys = np.unique(rng.integers(0, 2**62, size=(100_000, W), dtype=np.uint64), axis=0) << np.uint64(2)
    counts = rng.integers(1, 1000, len(keys))
    rec = _records(keys, counts, W)
    n = (1 << 24) + 4099
    q = keys[rng.integers(0, len(keys), n)]
    q[1::2, W - 1] ^= np.uint64(1)                        # every other key absent (the low bits of keys are 0)
    with kc.Counter(k, k) as c:
        run = c.upload_run(rec)
        got = c.lookup(run, q)
        assert np.array_equal(got, find(rec, k, q))
        assert (got[1::2] == 0).all() and (got[0::2] > 0).all()
        run.free()


@pytest.mark.gpu
@pytest.mark.parametrize("spread", [0, 10, 40])
def test_index_of_keys_crowded_into_few_buckets(kc, spread):
    """2^20 keys whose word 0 is below 2^spread: a few buckets hold them all and the index's long empty
    stretch (up to 2^19 buckets) is filled by the bucket pass"""
    k, W = 64, 2
    rng = np.random.default_rng(spread)
    n = 1 << 20
    lead = rng.integers(0, 1 << spread, n, dtype=np.uint64) if spread else np.zeros(n, dtype=np.uint64)
    keys = np.unique(np.stack([lead, rng.integers(0, 2**63, n, dtype=np.uint64)], axis=1), axis=0)
    top = keys.copy()
    top[:, 0] |= np.uint64(0xF000000000000000)          # a second crowd at the other end of the key space
    keys = np.concatenate([keys, top])
    counts = rng.integers(1, 1000, len(keys))
    with kc.Counter(k, k) as c:
        run = c.upload_run(_records(keys, counts, W))
        assert np.array_equal(c.lookup(run, keys), counts.astype(np.uint32))
        miss = keys ^ np.array([1 << 50, 0], dtype=np.uint64)
        assert np.array_equal(c.lookup(run, miss), find(_records(keys, counts, W), k, miss))
        run.free()


@pytest.mark.gpu
def test_lookup_one_huge_bucket(kc):
    """10^5 keys share their leading 40 bits: one bucket of the index holds them all"""
    k, W = 64, 2
    rng = np.random.default_rng(3)
    lead = np.uint64(0x5A5A5A5A5A << 24)
    a = np.unique(rng.integers(0, 2**63, size=100_000, dtype=np.uint64))
    hot = np.stack([lead | (a >> np.uint64(40)), a], axis=1)
    cold = np.unique(rng.integers(0, 2**63, size=(100_000, W), dtype=np.uint64), axis=0)
    keys = np.unique(np.concatenate([hot, cold]), axis=0)
    counts = rng.integers(1, 1000, len(keys))
    with kc.Counter(k, k) as c:
        run = c.upload_run(_records(keys, counts, W))
        assert np.array_equal(c.lookup(run, keys), counts.astype(np.uint32))
        miss = hot.copy()
        miss[:, 1] ^= np.uint64(1)
        assert np.array_equal(c.lookup(run, miss), find(_records(keys, counts, W), k, miss))
        run.free()


@pytest.mark.gpu
def test_strict_hidden_key0_and_ref_phantom(kc):
    """strict mode hides the empty slots' key-0 record (skip): not found; the REF phantom (0, 0) is a record"""
    L, k = 100, 31
    reads = oracle.gen_reads(3000, L, 30000, 0.01, 0.02, seed=5)
    zero = np.zeros((1, 1), dtype=np.uint64)
    with _counter(kc, k, L, "strict", method="sort") as c:
        run = _count(c, reads)
        assert oracle.records_to_arrays(run.to_bytes(), k)[0][0, 0] != 0
        assert c.lookup(run, zero).tolist() == [0]
        sc, hits = c.query_reads(run, reads, lo=0)
        want_sc, want_hits = query_model(run.to_bytes(), reads, L, k, "strict", lo=0)
        assert np.array_equal(sc, want_sc) and np.array_equal(hits, want_hits)
        run.free()
    with _counter(kc, k, L, "ref") as c:
        run = _count(c, reads)
        kk, cc = oracle.records_to_arrays(run.to_bytes(), k)
        assert kk[0, 0] == 0 and cc[0] == 0
        assert c.lookup(run, zero).tolist() == [0]
        sc, hits = c.query_reads(run, reads, lo=0, hi=0)
        want_sc, want_hits = query_model(run.to_bytes(), reads, L, k, "ref", lo=0, hi=0)
        assert np.array_equal(sc, want_sc) and np.array_equal(hits, want_hits)
        run.free()


SHAPES = [(31, 31), (31, 100), (33, 257), (64, 1000), (96, 150), (128, 4096), (5, 4096)]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("k,L,method", [(k, L, m) for k, L in SHAPES for m in ("super", "hash", "sort", "place")
                                        if m != "hash" or k <= 64])            # (hash counting is for k <= 64)
def test_query_reads_matches_model(kc, k, L, mode, method):
    R = max(40, 60000 // L)
    reads = oracle.gen_reads(R, L, 20000, 0.01, 0.005, seed=k + L)
    tail = oracle.gen_reads(1, L, 20000, 0.01, 0.0, seed=1)[: L // 2]      # a partial trailing read
    with _counter(kc, k, L, mode, method=method) as c:
        run = _count(c, reads)
        rb = run.to_bytes()
        for lo, hi in ((1, U32 - 1), (0, 0), (0, U32 - 1), (2, 3), (1, 1)):
            sc, hits = c.query_reads(run, np.concatenate([reads, tail]), lo, hi)
            want_sc, want_hits = query_model(rb, reads, L, k, mode, lo, hi)
            assert sc.shape == (R, L - k + 1)
            assert np.array_equal(sc, want_sc), (lo, hi)
            assert np.array_equal(hits, want_hits), (lo, hi)
        _, valid = slot_model(reads, L, k, mode)
        assert (sc[valid] >= 1).all()
        run.free()


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
def test_query_against_other_reads_and_other_read_length(kc, mode):
    """contaminant removal: reads of one sample against the run of another; and a run counted with
    another read length on a context with the same k"""
    k, L = 31, 150
    sample = oracle.gen_reads(3000, L, 40000, 0.01, 0.005, seed=11)
    other = oracle.gen_reads(3000, L, 40000, 0.01, 0.005, seed=11, first_read=3000)
    with _counter(kc, k, L, mode) as c, _counter(kc, k, 90, mode) as c90:
        run = _count(c, other)
        run90 = _count(c90, oracle.gen_reads(4000, 90, 40000, 0.01, 0.005, seed=11, first_read=6000))
        for r in (run, run90):
            sc, hits = c.query_reads(r, sample, 2, 10)
            want_sc, want_hits = query_model(r.to_bytes(), sample, L, k, mode, 2, 10)
            assert np.array_equal(sc, want_sc) and np.array_equal(hits, want_hits)
            assert 0 < (sc > 0).mean() < 1
        run.free()
        run90.free()


@pytest.mark.gpu
def test_errors(kc):
    reads = oracle.gen_reads(100, 100, 0, 0.0, 0.0, seed=2)
    with kc.Counter(31, 100) as c, kc.Counter(40, 100) as c40:
        run, run40 = _count(c, reads), _count(c40, reads)
        with pytest.raises(kc.KcError) as e:
            c.query_reads(run40, reads)
        assert e.value.code == KC_ERR_ARG
        with pytest.raises(kc.KcError) as e:
            c.lookup(run40, np.zeros((3, 1), dtype=np.uint64))
        assert e.value.code == KC_ERR_ARG
        with pytest.raises(kc.KcError) as e:
            c.query_reads(run, reads, lo=5, hi=4)
        assert e.value.code == KC_ERR_ARG
        lib = c._lib
        assert lib.kc_query_reads(c._ctx, run._h, reads.ctypes.data, reads.size, 1, 10, None, None) == KC_ERR_ARG
        assert lib.kc_query_reads(c._ctx, None, reads.ctypes.data, reads.size, 1, 10, None, None) == KC_ERR_ARG
        assert lib.kc_run_lookup(c._ctx, run._h, None, 3, None) == KC_ERR_ARG
        assert lib.kc_run_lookup(None, run._h, None, 0, None) == KC_ERR_ARG
        # nothing to do: success, nothing written
        sc, hits = c.query_reads(run, reads[:99])
        assert sc.shape == (0, 70) and len(hits) == 0
        assert len(c.lookup(run, np.zeros((0, 1), dtype=np.uint64))) == 0
        d = _dev(np.concatenate([np.zeros(1, np.uint8), reads]))
        h = _dev(np.zeros(100, np.uint32))
        with pytest.raises(kc.KcError) as e:                   # device reads not 16-byte aligned
            c.query_reads_device(run, d.data_ptr() + 1, reads.size, 0, h.data_ptr())
        assert e.value.code == KC_ERR_ARG
        run.free()
        run40.free()


@pytest.mark.gpu
def test_pieces_of_a_large_query(kc):
    """400 k reads of 137 bases: three internal pieces (whole reads, a multiple of 16 of them), the
    boundaries at slots that are not aligned to anything; the whole equals the parts, and the reads
    around the boundaries match the model"""
    import torch
    k, L, R = 31, 137, 400_000
    reads = oracle.gen_reads(R, L, 1_000_000, 0.01, 0.002, seed=21)
    with _counter(kc, k, L, "strict") as c:
        d = _dev(reads)
        run = c.count_device(d.data_ptr(), d.numel())
        nk = L - k + 1
        sc = torch.zeros(R * nk, dtype=torch.int32, device="cuda")
        hits = torch.zeros(R, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()                # torch's writes are on its own stream
        c.query_reads_device(run, d.data_ptr(), d.numel(), sc.data_ptr(), hits.data_ptr(), 2, 5)
        sc_h, hits_h = sc.cpu().numpy().view(np.uint32).reshape(R, nk), hits.cpu().numpy().view(np.uint32)
        piece = ((1 << 24) // nk) & ~15
        assert piece * 2 < R < piece * 3
        rb = run.to_bytes()
        for b in (piece, 2 * piece):
            lo_r, hi_r = b - 37, b + 41
            want_sc, want_hits = query_model(rb, reads[lo_r * L:hi_r * L], L, k, "strict", 2, 5)
            assert np.array_equal(sc_h[lo_r:hi_r], want_sc) and np.array_equal(hits_h[lo_r:hi_r], want_hits)
        parts_sc, parts_hits = [], []
        for r0 in range(0, R, 65_536 + 3):
            r1 = min(R, r0 + 65_536 + 3)
            s, h = c.query_reads(run, reads[r0 * L:r1 * L], 2, 5)
            parts_sc.append(s)
            parts_hits.append(h)
        assert np.array_equal(np.concatenate(parts_sc), sc_h) and np.array_equal(np.concatenate(parts_hits), hits_h)
        run.free()


@pytest.mark.gpu
@pytest.mark.parametrize("k", [31, 64, 96])
def test_canonical_reverse_complemented_reads(kc, k):
    L = 151
    reads = oracle.gen_reads(2000, L, 20000, 0.01, 0.005, seed=k)
    rows = reads.reshape(-1, L)[:, ::-1]
    lut = np.arange(256, dtype=np.uint8)
    for a, b in zip(b"ACGT", b"TGCA"):
        lut[a] = b
    rc = np.ascontiguousarray(lut[rows]).reshape(-1)
    with _counter(kc, k, L, "canonical") as c:
        run = _count(c, reads)
        s1, h1 = c.query_reads(run, reads)
        s2, h2 = c.query_reads(run, rc)
        assert np.array_equal(s1, s2[:, ::-1]) and np.array_equal(h1, h2)
        run.free()


@pytest.mark.gpu
def test_host_and_device_pointers_agree(kc):
    import torch
    k, L = 31, 100
    reads = oracle.gen_reads(5000, L, 30000, 0.01, 0.005, seed=8)
    with _counter(kc, k, L, "canonical") as c:
        run = _count(c, reads)
        sc, hits = c.query_reads(run, reads, 1, 3)
        d = _dev(reads)
        dsc = torch.zeros(sc.size, dtype=torch.int32, device="cuda")
        dh = torch.zeros(len(hits), dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()                # torch's writes are on its own stream
        c.query_reads_device(run, d.data_ptr(), d.numel(), dsc.data_ptr(), dh.data_ptr(), 1, 3)
        assert np.array_equal(dsc.cpu().numpy().view(np.uint32).reshape(sc.shape), sc)
        assert np.array_equal(dh.cpu().numpy().view(np.uint32), hits)
        # one output only; pinned host reads
        dh.zero_()
        torch.cuda.synchronize()                # torch's writes are on its own stream
        c.query_reads_device(run, d.data_ptr(), d.numel(), 0, dh.data_ptr(), 1, 3)
        assert np.array_equal(dh.cpu().numpy().view(np.uint32), hits)
        pinned = torch.from_numpy(reads.copy()).pin_memory()
        torch.cuda.synchronize()                # torch's writes are on its own stream
        c.query_reads_device(run, pinned.data_ptr(), pinned.numel(), dsc.data_ptr(), 0, 1, 3)
        assert np.array_equal(dsc.cpu().numpy().view(np.uint32).reshape(sc.shape), sc)
        assert c.query_reads(run, reads, 1, 3, slot_counts=False)[0] is None
        # lookup: device keys and counts
        keys, counts = oracle.records_to_arrays(run.to_bytes(), k)
        dk = _dev(keys.view(np.int64))
        dc = torch.zeros(len(counts), dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()                # torch's writes are on its own stream
        c.lookup_device(run, dk.data_ptr(), len(counts), dc.data_ptr())
        assert np.array_equal(dc.cpu().numpy().view(np.uint32), counts)
        st = c.stats()
        assert st["launches"] > 0 and st["h2d_bytes"] > 0 and st["d2h_bytes"] > 0
        if torch.cuda.device_count() > 1:
            other = torch.zeros(len(hits), dtype=torch.int32, device="cuda:1")
            with pytest.raises(kc.KcError) as e:
                c.query_reads_device(run, d.data_ptr(), d.numel(), 0, other.data_ptr())
            assert e.value.code == KC_ERR_ARG
        run.free()


@pytest.mark.gpu
def test_scale_identity_on_the_device(kc):
    """3 M reads x 100 bp against their own run: the valid slots with count c number c * hist[c], and
    every valid slot has a count >= 1; checked on the device"""
    import torch
    k, L, R = 31, 100, 3_000_000
    reads = oracle.gen_reads(R, L, 50_000_000, 0.005, 0.001, seed=31)
    nk = L - k + 1
    with _counter(kc, k, L, "canonical") as c:
        d = _dev(reads)
        run = c.count_device(d.data_ptr(), d.numel())
        sc = torch.zeros(R * nk, dtype=torch.int32, device="cuda")
        hits = torch.zeros(R, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()                # torch's writes are on its own stream
        c.query_reads_device(run, d.data_ptr(), d.numel(), sc.data_ptr(), hits.data_ptr())
        rows = d.view(R, L)
        bad = ~((rows == 65) | (rows == 67) | (rows == 71) | (rows == 84))
        cb = torch.nn.functional.pad(torch.cumsum(bad.int(), dim=1), (1, 0))
        valid = (cb[:, k:k + nk] - cb[:, :nk]) == 0
        sc = sc.view(R, nk)
        assert bool((sc[valid] >= 1).all()) and bool((sc[~valid] == 0).all())
        assert torch.equal(hits, valid.sum(dim=1).int())
        nb = 4096
        hist = torch.from_numpy(run.histogram(nb).astype(np.int64)).cuda()
        seen = torch.bincount(sc[valid].long().clamp(max=nb - 1), minlength=nb)
        c_ = torch.arange(nb, device="cuda")
        assert torch.equal(seen[1:nb - 1], (c_ * hist)[1:nb - 1])
        run.free()


# ------------------------------------------------------------------ allocation failure
CU_MEMPOOL_ATTR_USED_MEM_CURRENT = 7


def _pool_used():
    cu = ctypes.CDLL("libcuda.so.1")
    cu.cuDeviceGetDefaultMemPool.argtypes = [ctypes.POINTER(ctypes.c_void_p), ctypes.c_int]
    cu.cuMemPoolGetAttribute.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p]
    dev, pool, used = ctypes.c_int(), ctypes.c_void_p(), ctypes.c_uint64()
    assert cu.cuDeviceGet(ctypes.byref(dev), 0) == 0
    assert cu.cuDeviceGetDefaultMemPool(ctypes.byref(pool), dev.value) == 0
    assert cu.cuMemPoolGetAttribute(pool, CU_MEMPOOL_ATTR_USED_MEM_CURRENT, ctypes.byref(used)) == 0
    return used.value


def _exercise_alloc_failures(kc, monkeypatch, make_counter, scenario, want):
    """the n-th allocation of a fresh counter fails for n = 1, 2, ...: KC_ERR_NOMEM, then the right answer
    from the same call again, and the pool back to its base once the counter is closed"""
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
            with contextlib.ExitStack() as st:
                try:
                    got = scenario(c, st)
                except kc.KcError as e:
                    assert e.code == KC_ERR_NOMEM, (n, str(e))
                    failed = True
                    got = scenario(c, st)
                assert got == want, n
        finally:
            c.close()
        torch.cuda.synchronize()
        assert _pool_used() == base, "allocation %d failed: memory left in the pool" % n
        if not failed:
            assert n > 1
            return n
    pytest.fail("still failing after 64 injected allocation failures")


@pytest.mark.gpu
@pytest.mark.parametrize("call", ["lookup", "query_host", "query_device"])
def test_allocation_failure(kc, monkeypatch, call):
    import torch
    k, L = 31, 100
    reads = oracle.gen_reads(3000, L, 30000, 0.01, 0.002, seed=23)
    run_bytes = oracle.count(reads, L, k)
    keys, counts = oracle.records_to_arrays(run_bytes, k)
    d = _dev(reads)
    want_sc, want_hits = query_model(run_bytes, reads, L, k, "ref", 2, 9)

    def scenario(c, st):
        run = c.upload_run(run_bytes)
        st.callback(run.free)
        if call == "lookup":
            return c.lookup(run, keys).tolist()
        if call == "query_host":
            sc, hits = c.query_reads(run, reads, 2, 9)
            return sc.tolist(), hits.tolist()
        dh = torch.zeros(len(want_hits), dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()                # torch's writes are on its own stream
        c.query_reads_device(run, d.data_ptr(), d.numel(), 0, dh.data_ptr(), 2, 9)
        return dh.cpu().numpy().view(np.uint32).tolist()

    want = {"lookup": counts.tolist(), "query_host": (want_sc.tolist(), want_hits.tolist()),
            "query_device": want_hits.tolist()}[call]
    _exercise_alloc_failures(kc, monkeypatch, lambda: kc.Counter(k, L), scenario, want)


# ------------------------------------------------------------------------ command line
@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["strict", "canonical"])
@pytest.mark.parametrize("k", [25, 31, 40])
def test_cli_query(tmp_path, mode, k):
    d = tmp_path / "in"
    d.mkdir()
    L, R = 100, 3000
    (d / "a.fastq").write_bytes(oracle.gen_fastq(R, L, 50000, 0.01, 0.002, seed=k))
    rec = tmp_path / "rec.bin"
    flag = ["compat=strict"] if mode == "strict" else ["canonical=1"]
    r = subprocess.run([CLI, "kmerLength=%d" % k, "inputFileLocation=%s" % d, "outputFile=%s" % rec,
                        "tempFileLocation=%s" % tmp_path] + flag, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    reads = oracle.gen_reads(R, L, 50000, 0.01, 0.002, seed=k)
    rows = reads.reshape(R, L)
    rng = np.random.default_rng(k)
    lines = [bytes(rows[i, p:p + k]) for i, p in zip(rng.integers(0, R, 3000), rng.integers(0, L - k + 1, 3000))]
    lines += [bytes(rng.choice(list(b"ACGT"), k).astype(np.uint8)) for _ in range(500)]
    lines += [b"N" * k, b"A" * k, b"T" * k]
    text = b"".join(x + b"\n" for x in lines)
    kf, out = tmp_path / "kmers.txt", tmp_path / "out.txt"
    kf.write_bytes(text)
    run = rec.read_bytes()
    keys, valid = slot_model(np.frombuffer(b"".join(lines), np.uint8), k, k, mode)
    want_c = np.where(valid[:, 0], find(run, k, keys[:, 0]), 0)
    want = b"".join(b"%s %d\n" % (x, int(cn)) for x, cn in zip(lines, want_c))
    assert (want_c > 0).sum() >= 2500
    r = subprocess.run([CLI, "query", str(rec), str(k), str(kf), str(out)] + flag, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert out.read_bytes() == want
    r = subprocess.run([CLI, "query", str(rec), str(k), "-", "-"] + flag, input=text, capture_output=True)
    assert r.returncode == 0, r.stderr
    assert r.stdout == want
    bad = subprocess.run([CLI, "query", str(rec), str(k), "-", "-"] + flag, input=text + b"ACGT\n", capture_output=True)
    assert bad.returncode != 0 and b"letters" in bad.stderr
