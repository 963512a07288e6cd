"""Where the cycles of S2 (sw_count_kernel) go, phase by phase.

usage: s2_profile.py [--reads R] [--k K] [--iters N] [--canonical] [--json OUT]
       s2_profile.py --sass-check

The first form builds libkc_b200.so with -DKC_SW_PROFILE into a temporary directory (the tree is
not written), counts configs[1]'s reads (10M x 100 bp of a 100 Mbase genome, 1e-3 substitutions,
seed 2; generated on the device) with the super-window path, and prints each phase's share of the
warps' cycles in S2 together with the collision-queue counters and the debug scalars. The timer's
clock reads slow S2 down a little: the shares are what to read, not the stage time of this build.

--sass-check needs no GPU: it compiles kc_super.cu as it is and with every KC_SW_PROFILE hook
removed from the text, both without the switch, and checks that cuobjdump -sass prints the same
instructions for both (function names aside: they carry the file name).
"""
import argparse
import ctypes as C
import json
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "kmer-counter_b200", "csrc")
sys.path.insert(0, ROOT)

PHASES = ["unit", "dedupe", "scan", "open", "insert", "drain", "round_end", "emit"]
COUNTERS = ["queued", "drain_probes", "warps", "total_cycles"]
NVFLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-O3", "-lineinfo", "-Xcompiler", "-fPIC"]


def sass_check():
    src = open(os.path.join(CSRC, "kc_super.cu")).read()
    i = src.index("#ifdef KC_SW_PROFILE")
    stripped = src[:i] + src[src.index("#endif", i) + len("#endif"):]
    stripped = re.sub(r"\s*if \(lane == 0\) SWP_ADD\([^;]*\);", "", stripped)
    stripped = re.sub(r"\s*SWP_(MARK|ADD|ADD_ACTIVE|FLUSH)\([^;]*\);", "", stripped)
    stripped = re.sub(r"\s*SWP_DECL;", "", stripped)
    assert "SWP_MARK" not in stripped and "SWP_DECL" not in stripped
    with tempfile.TemporaryDirectory() as td:
        open(os.path.join(td, "kc_super.cu"), "w").write(stripped)
        out = {}
        for name, path in (("hooks", os.path.join(CSRC, "kc_super.cu")), ("no_hooks", os.path.join(td, "kc_super.cu"))):
            obj = os.path.join(td, name + ".o")
            subprocess.check_call(["nvcc"] + NVFLAGS + ["-I" + CSRC, "-c", path, "-o", obj])
            sass = subprocess.check_output(["cuobjdump", "-sass", obj]).decode()
            # keep the instructions; function names embed the translation unit's name and path hash
            out[name] = [re.sub(r"_GLOBAL__N__\w+?_kc_super_cu_[0-9a-f]+", "ANON", l)
                         for l in sass.splitlines() if "/*" in l or "Function :" in l]
        n_clock = sum("SR_CLOCK" in l for l in out["hooks"])
        same = out["hooks"] == out["no_hooks"]
        print("sass lines %d, identical without the hooks: %s, clock reads in the default build: %d"
              % (len(out["hooks"]), same, n_clock))
        return 0 if same and n_clock == 0 else 1


def build_profiled(td):
    lib = os.path.join(td, "libkc_b200.so")
    subprocess.check_call(["make", "-s", "-C", CSRC, "-j8", "OBJDIR=" + os.path.join(td, "build"), "TARGET=" + lib,
                           "EXTRA_NVFLAGS=-DKC_SW_PROFILE"])
    return lib


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=10_000_000)
    ap.add_argument("--k", type=int, default=31)
    ap.add_argument("--iters", type=int, default=3)
    ap.add_argument("--canonical", action="store_true")
    ap.add_argument("--json", default=None)
    ap.add_argument("--sass-check", action="store_true")
    a = ap.parse_args()
    if a.sass_check:
        return sass_check()
    import torch
    with tempfile.TemporaryDirectory() as td:
        lib_path = build_profiled(td)
        from kmer_counter_b200 import _lib
        _lib.LIB_PATH = lib_path
        import kmer_counter_b200 as kc
        from kmer_counter_b200 import synth
        lib = _lib.load()
        rd = lib.kc_sw_profile_read
        rd.restype, rd.argtypes = C.c_int, [C.POINTER(C.c_uint64), C.c_int]
        buf = (C.c_uint64 * (len(PHASES) + len(COUNTERS)))()
        L, G = 100, 100_000_000
        dev = torch.device("cuda", 0)
        d_reads = torch.empty(a.reads * L + 256, dtype=torch.uint8, device=dev)
        synth.synth_reads_device(d_reads.data_ptr(), a.reads, L, G, 1e-3, 0.0, 2)
        torch.cuda.synchronize()
        rows = []
        with kc.Counter(a.k, L, method="super", canonical=a.canonical) as c:
            for it in range(a.iters):
                assert rd(buf, 1) == 0
                run = c.count_device(d_reads.data_ptr(), a.reads * L)
                n = len(run)
                run.free()
                torch.cuda.synchronize()
                assert rd(buf, 0) == 0
                st, sc = c.stats(), c.debug_scalars()
                v = [int(x) for x in buf]
                ph = dict(zip(PHASES, v[:len(PHASES)]))
                cnt = dict(zip(COUNTERS, v[len(PHASES):]))
                tot = sum(ph.values())
                row = {"iter": it, "records": n, "ms_stage": dict(zip(st["stage_names"], [round(x, 3) for x in st["ms_stage"]])),
                       "share": {k: round(x / tot, 4) for k, x in ph.items()}, "cycles": ph, "counters": cnt,
                       "queued_per_occurrence": round(cnt["queued"] / max(sc["occurrences"], 1), 4),
                       "drain_probes_per_queued": round(cnt["drain_probes"] / max(cnt["queued"], 1), 3),
                       "scalars": sc}
                rows.append(row)
                print(json.dumps(row), flush=True)
        if a.json:
            os.makedirs(os.path.dirname(os.path.abspath(a.json)), exist_ok=True)
            with open(a.json, "w") as f:
                json.dump(rows, f, indent=1)
    return 0


if __name__ == "__main__":
    sys.exit(main())
