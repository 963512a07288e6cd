"""CPU tests of the boundary: the shared library loads, exports every symbol include/kc_api.h
declares, fails loudly without a device, and the host-side helpers behave."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "kc_api.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(kc_[a-z_0-9]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    import kmer_counter_b200 as kc
    lib = kc._lib.load()
    declared = _declared_symbols()
    assert len(declared) >= 25
    for name in declared:
        assert hasattr(lib, name), "libkc_b200.so does not export %s" % name
    assert set(kc._lib.SYMBOLS) == set(declared), "python binding and header disagree"


def test_pure_functions():
    import kmer_counter_b200 as kc
    lib = kc._lib.load()
    assert [lib.kc_key_words(k) for k in (1, 31, 32, 33, 63, 64, 65, 96, 97, 128)] == [1, 1, 1, 2, 2, 2, 3, 3, 4, 4]
    assert [lib.kc_record_size(k) for k in (31, 63, 96, 128)] == [12, 20, 28, 36]       # KMerSizes.h:10-28
    assert lib.kc_output_size(89364 * 100, 100, 31) == 89364 * 70 * 12                   # calculateOutputSize
    assert lib.kc_output_size(1000, 100, 101) == 0
    assert b"sm_100a" in lib.kc_version()


def test_config_struct_layout_matches_header():
    import kmer_counter_b200 as kc
    assert C.sizeof(kc._lib.KcConfig) == 64                      # grew by distinct_hint (struct_size keeps old callers working)
    assert kc._lib.KcConfig.max_chunk_bytes.offset == 32 and kc._lib.KcConfig.stream.offset == 48
    assert kc._lib.KcConfig.distinct_hint.offset == 56
    assert kc._lib.KcStats.ms_stage.offset % 4 == 0


def test_no_cpu_fallback():
    """Without a CUDA device the product path must fail loudly, not compute on the CPU. The check
    runs in a child process that sees no device, so it runs on GPU machines too."""
    code = ("import kmer_counter_b200 as kc\n"
            "try:\n    kc.Counter(31, 100)\nexcept kc.KcError as e:\n    print('code', e.code)\n")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    assert r.stdout.split() == ["code", "-2"], r.stdout


def test_bad_arguments_are_rejected_before_touching_the_device():
    import kmer_counter_b200 as kc
    for k, L in ((0, 100), (129, 200), (31, 30), (31, 5000)):
        with pytest.raises(kc.KcError) as ei:
            kc.Counter(k, L)
        assert ei.value.code == -1
    with pytest.raises(kc.KcError):
        kc.Counter(65, 100, method="hash")            # partitioned hash counting is for k <= 64
    with pytest.raises(kc.KcError):
        kc.Counter(63, 100, method="hash_global")     # the HBM-resident table is for k <= 32


def test_product_package_does_not_import_the_oracle():
    pkg = os.path.join(ROOT, "kmer-counter_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp", ".hpp")):
                text = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in text and "from oracle" not in text and "kc_oracle" not in text, f
                assert "/root/reference" not in text, f


def test_range_ownership_model():
    from kmer_counter_b200 import multigpu
    sp = multigpu.range_splitters(4, 2)
    assert sp.shape == (3, 2) and [int(x) for x in sp[:, 0]] == [1 << 62, 2 << 62, 3 << 62] and (sp[:, 1] == 0).all()
    keys_hi = np.array([0, (1 << 62) - 1, 1 << 62, (3 << 62) + 5, 2**64 - 1], dtype=np.uint64)
    assert list(multigpu.owner_of(keys_hi, 4)) == [0, 0, 1, 3, 3]
    keys = np.array([[1, 0], [1 << 62, 0], [1 << 62, 7], [3 << 62, 0]], dtype=np.uint64)
    assert list(multigpu.slice_offsets_host(keys, sp)) == [0, 1, 3, 3, 4]
