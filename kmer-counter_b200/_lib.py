"""ctypes binding of libkc_b200.so (include/kc_api.h).

The library is the product: if it is missing or cannot be loaded this module
raises -- there is no Python/CPU fallback for any compute call.
"""
import ctypes as C
import os
import subprocess

_PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG_DIR, "libkc_b200.so")
CSRC_DIR = os.path.join(_PKG_DIR, "csrc")

KC_OK = 0
KC_COMPAT_REF, KC_COMPAT_STRICT = 0, 1
KC_CANONICAL = 0x2          # count a k-mer and its reverse complement under min(x, rc(x)); implies strict
KC_COUNT_AUTO, KC_COUNT_SORT, KC_COUNT_HASH, KC_COUNT_HASH_GLOBAL, KC_COUNT_SUPER, KC_COUNT_PLACE = 0, 1, 2, 3, 4, 5
METHODS = {"auto": KC_COUNT_AUTO, "sort": KC_COUNT_SORT, "hash": KC_COUNT_HASH, "hash_global": KC_COUNT_HASH_GLOBAL,
           "super": KC_COUNT_SUPER, "place": KC_COUNT_PLACE}
METHOD_NAMES = {v: k for k, v in METHODS.items()}
# kc_run_combine: the set operation, and how a key in both runs is counted
KC_SET_UNION, KC_SET_INTERSECT, KC_SET_SUBTRACT, KC_SET_SUBTRACT_COUNTS = 0, 1, 2, 3
KC_COUNTS_SUM, KC_COUNTS_MIN, KC_COUNTS_MAX, KC_COUNTS_A, KC_COUNTS_B = 0, 1, 2, 3, 4
SET_OPS = {"union": KC_SET_UNION, "intersect": KC_SET_INTERSECT, "subtract": KC_SET_SUBTRACT,
           "subtract_counts": KC_SET_SUBTRACT_COUNTS}
COUNT_MODES = {"sum": KC_COUNTS_SUM, "min": KC_COUNTS_MIN, "max": KC_COUNTS_MAX, "a": KC_COUNTS_A, "b": KC_COUNTS_B}


class KcConfig(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32), ("k", C.c_uint32), ("read_len", C.c_uint32), ("device", C.c_int32),
        ("flags", C.c_uint32), ("method", C.c_uint32), ("n_slots", C.c_uint32), ("reserved0", C.c_uint32),
        ("max_chunk_bytes", C.c_uint64), ("table_slots", C.c_uint64), ("stream", C.c_void_p),
        ("distinct_hint", C.c_uint64),
    ]


class KcStats(C.Structure):
    _fields_ = [
        ("chunks", C.c_uint64), ("reads", C.c_uint64), ("kmer_slots", C.c_uint64), ("kmers_valid", C.c_uint64),
        ("distinct_last", C.c_uint64), ("launches", C.c_uint64), ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64),
        ("ms_extract", C.c_float), ("ms_count", C.c_float), ("ms_emit", C.c_float), ("ms_total", C.c_float),
        ("ms_dominant", C.c_float), ("dominant_launches", C.c_uint32), ("method_used", C.c_uint32),
        ("dominant_bytes", C.c_uint64),
        ("n_stages", C.c_uint32), ("dominant_stage", C.c_uint32),
        ("ms_stage", C.c_float * 8), ("stage_bytes", C.c_uint64 * 8), ("stage_launches", C.c_uint32 * 8),
    ]


# every symbol include/kc_api.h declares: (restype, argtypes)
_vp, _u32, _u64, _i = C.c_void_p, C.c_uint32, C.c_uint64, C.c_int
_pp = C.POINTER(C.c_void_p)
_pu64 = C.POINTER(C.c_uint64)
SYMBOLS = {
    "kc_version": (C.c_char_p, []),
    "kc_key_words": (_u32, [_u32]),
    "kc_record_size": (_u32, [_u32]),
    "kc_output_size": (_u64, [_u64, _u32, _u32]),
    "kc_create": (_i, [C.POINTER(KcConfig), _pp]),
    "kc_destroy": (None, [_vp]),
    "kc_last_error": (C.c_char_p, [_vp]),
    "kc_sync": (_i, [_vp]),
    "kc_stats_get": (_i, [_vp, C.POINTER(KcStats)]),
    "kc_debug_scalars": (_i, [_vp, _pu64]),
    "kc_accum_begin": (_i, [_vp, _u64]),
    "kc_accum_add_device": (_i, [_vp, _vp, _u64]),
    "kc_accum_submit": (_i, [_vp, _u32, _u64]),
    "kc_accum_submit_fastq": (_i, [_vp, _u32, _vp, _u64, _pu64, C.POINTER(C.c_uint32)]),
    "kc_accum_wait": (_i, [_vp, _u32]),
    "kc_accum_flush": (_i, [_vp, _pp]),
    "kc_xchg_begin": (_i, [_vp, _u32, _u32, _u64]),
    "kc_xchg_export": (_i, [_vp, _vp]),
    "kc_xchg_import": (_i, [_vp, _u32, _vp]),
    "kc_xchg_set_peer": (_i, [_vp, _u32, _vp]),
    "kc_xchg_count_local": (_i, [_vp]),
    "kc_xchg_hist": (_i, [_vp, _pp, _pp]),
    "kc_xchg_group_local": (_i, [_vp]),
    "kc_xchg_pull": (_i, [_vp]),
    "kc_xchg_finish": (_i, [_vp, _pp]),
    "kc_xchg_fix_ranges": (_i, [_vp, _i]),
    "kc_xchg_info": (_i, [_vp, C.POINTER(C.c_uint32), _pu64, _pu64]),
    "kc_xchg_run_all": (_i, [_pp, _u32, _pp]),
    "kc_host_alloc": (_i, [_vp, _u64, _pp]),
    "kc_host_free": (_i, [_vp, _vp]),
    "kc_process_chunk": (_i, [_vp, _u32, _vp, _u64, _vp, _u64, _pu64]),
    "kc_slot_buffer": (_i, [_vp, _u32, _pp, _pu64]),
    "kc_submit": (_i, [_vp, _u32, _u64]),
    "kc_wait": (_i, [_vp, _u32, _pp]),
    "kc_count_device": (_i, [_vp, _vp, _u64, _pp]),
    "kc_parse_fastq_device": (_i, [_vp, _vp, _u64, _vp, _u64, _pu64, _pu64, C.POINTER(C.c_uint32)]),
    "kc_submit_fastq": (_i, [_vp, _u32, _vp, _u64, _pu64, C.POINTER(C.c_uint32)]),
    "kc_run_records": (_u64, [_vp]),
    "kc_run_free": (_i, [_vp, _vp]),
    "kc_run_copy_records": (_i, [_vp, _vp, _vp, _u64, _pu64]),
    "kc_run_print": (_i, [_vp, _vp, _vp, _u64, _pu64]),
    "kc_run_upload": (_i, [_vp, _vp, _u64, _pp]),
    "kc_run_device": (_i, [_vp, _pp, _pp, _pu64]),
    "kc_run_from_device": (_i, [_vp, _vp, _vp, _u64, _pp]),
    "kc_run_write": (_i, [_vp, _vp, C.c_char_p, _i]),
    "kc_run_split": (_i, [_vp, _vp, _pu64, _u32, _pu64]),
    "kc_run_histogram": (_i, [_vp, _vp, _pu64, _u32]),
    "kc_run_filter": (_i, [_vp, _vp, _u32, _u32, _pp]),
    "kc_merge_runs": (_i, [_vp, _pp, _u32, _pp]),
    "kc_run_combine": (_i, [_vp, _vp, _vp, _u32, _u32, _pp]),
    "kc_run_lookup": (_i, [_vp, _vp, _vp, _u64, _vp]),
    "kc_query_reads": (_i, [_vp, _vp, _vp, _u64, _u32, _u32, _vp, _vp]),
    "kc_place_next_run": (_i, [_vp, _vp, _vp, _vp, _u64, _u32]),
    "kc_peer_alloc": (_i, [_vp, _u64, C.POINTER(_vp), _vp]),
    "kc_peer_open": (_i, [_vp, _vp, C.POINTER(_vp)]),
    "kc_peer_close": (_i, [_vp, _vp]),
    "kc_peer_free": (_i, [_vp, _vp]),
    "kc_run_parts": (_i, [_vp, _pp, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]),
    "kc_merge_parts": (_i, [_vp, _u32, _pp, _pp, _pp, _pu64, _u32, _u32, _pp]),
    "kc_synth_reads": (_i, [_vp, _u64, _u64, _u32, _u64, C.c_double, C.c_double, _u64, _u64, _vp]),
}


def build(verbose=False):
    """Compile the CUDA library in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    cmd = ["make", "-C", CSRC_DIR, "-j8"]
    if not verbose:
        cmd.insert(1, "-s")
    subprocess.check_call(cmd)
    return LIB_PATH


_lib = None


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "%s is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C kmer-counter_b200/csrc`). There is no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)      # AttributeError here = header and library disagree
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib
