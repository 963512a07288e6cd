"""S2 of the super-window path (sw_count_kernel): the per-bin shared-memory count.

Each case is checked bit-exact against the CPU oracle, and the debug scalars show that the path
it is about really ran: units of more than one round (the record table is handed back slot by
slot between rounds), split passes after an abort, the overflow slices of heavy hitters, the
phantom key-0 record, 128-bit keys, canonical keys and the exchange with every rank on one device.
"""
import numpy as np
import pytest

import oracle
from test_canonical import canonical_count

pytestmark = pytest.mark.gpu
L = 100


@pytest.fixture(scope="module")
def kc():
    import kmer_counter_b200 as kc
    return kc


def _count(kc, reads, k, canonical=False, **kw):
    with kc.Counter(k, L, method="super", n_slots=2, max_chunk_bytes=1 << 26, canonical=canonical, **kw) as c:
        got = c.process_chunk(reads)
        st, sc = c.stats(), c.debug_scalars()
    assert st["method_used"] == "super"
    assert sc["fail"] == 0, sc
    return got, sc


def _want(reads, k, canonical=False):
    return canonical_count(reads, L, k) if canonical else oracle.process_chunk(reads, L, k)


def _deep_reads():
    """20000 reads of a 3 kbase genome: bins of ~2500 records (several rounds of 1024), most of them
    copies of each other, and few distinct keys per bin (no split passes)"""
    return oracle.gen_reads(20000, L, 3000, 0.0, 0.001, seed=41)


@pytest.mark.parametrize("canonical", [False, True])
@pytest.mark.parametrize("k", [31, 63])
def test_units_of_several_rounds(kc, k, canonical):
    reads = _deep_reads()
    got, sc = _count(kc, reads, k, canonical=canonical, table_slots=20000)
    assert got == _want(reads, k, canonical), sc
    assert sc["multi_round_units"] > 0, sc
    assert sc["aborts"] == 0, sc
    if k <= 32:                                    # the record table exists for 64-bit keys
        assert sc["dedup_records"] > 0, sc
        assert sc["occurrences"] < sc["windows"], sc
    else:
        assert sc["dedup_records"] == 0 and sc["occurrences"] == sc["windows"], sc


@pytest.mark.parametrize("canonical", [False, True])
@pytest.mark.parametrize("k", [31, 63])
def test_abort_and_split_passes(kc, k, canonical):
    """iid reads: every key distinct, so a bin of 100000 occurrences overfills the table and is
    counted again in 2, 4, ... passes"""
    reads = oracle.gen_reads(12000, L, 0, 0.0, 0.001, seed=43)
    got, sc = _count(kc, reads, k, canonical=canonical, table_slots=100000)
    assert got == _want(reads, k, canonical), sc
    assert sc["aborts"] > 0 and sc["multi_round_units"] > 0, sc


@pytest.mark.parametrize("k", [31, 63])
def test_heavy_hitters_fill_the_overflow_list(kc, k):
    """4000 copies of three reads: more records than their bins hold, so the surplus is counted in
    overflow slices (far more copies fill the overflow list too, and the chunk goes to the hash path)"""
    hot = oracle.gen_reads(3, L, 0, 0, 0, seed=45)
    reads = np.concatenate([np.tile(hot, 4000), oracle.gen_reads(2000, L, 50000, 0.01, 0.001, seed=46)])
    got, sc = _count(kc, reads, k)
    assert got == _want(reads, k), sc
    assert sc["overflow_records"] > 0 and sc["folded"] > 0, sc
    if k <= 32:
        assert sc["dedup_records"] > 0, sc


@pytest.mark.parametrize("k", [31, 63])
def test_phantom_record(kc, k):
    """N bases leave k-mer slots empty: key 0 joins with count += 0 (the phantom record of bin 0),
    next to the real key-0 occurrences of the poly-A reads"""
    reads = np.concatenate([oracle.gen_reads(3000, L, 20000, 0.01, 0.02, seed=47),
                            np.frombuffer(b"A" * L * 3, dtype=np.uint8)])
    want = _want(reads, k)
    got, sc = _count(kc, reads, k, table_slots=20000)
    assert got == want, sc
    assert sc["invalid"] > 0, sc
    W = (k + 31) // 32
    assert want[:8 * W] == bytes(8 * W)            # the run starts with key 0
    # no N and no poly-A: no key-0 record at all
    clean = oracle.gen_reads(3000, L, 20000, 0.01, 0.0, seed=48)
    got, sc = _count(kc, clean, k)
    assert got == _want(clean, k) and sc["invalid"] == 0, sc


@pytest.mark.parametrize("P", [2, 3])
@pytest.mark.parametrize("k", [31, 63])
def test_exchange_all_ranks_on_one_device(kc, P, k):
    """every rank counts its share of the bins from the records of all ranks"""
    import torch
    from kmer_counter_b200 import engine
    reads = _deep_reads()
    R = len(reads) // L
    want = _want(reads, k)
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
        got = b"".join(r.to_bytes() for r in runs)
        for r in runs:
            r.free()
        assert got == want
    finally:
        for c in cs:
            c.close()
