"""Time of the set operations of two runs (kc_run_combine) against kc_merge_runs of the same pair.

Two C2-shaped samples (10 M x 100 bp reads each, one 100 Mbase genome, different reads; about 129 M
records each) are counted on GPU 0. Then every op with its default count mode, and union with min, is
timed with kc_merge_runs of the same pair alternating, warm; each line has the median of --reps calls
of each. Algorithmic bytes: S * (nA + nB) read + S * U written, S = record bytes, U = records out. The
card's name and power limit are read in the same run. One JSON line per op on stdout (and --out)."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import kmer_counter_b200 as kc
from kmer_counter_b200 import synth

CASES = [("union", None), ("union", "min"), ("intersect", None), ("subtract", None), ("subtract_counts", None)]


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else "%s (nvidia-smi unavailable)" % torch.cuda.get_device_name(0)


def timed(fn):
    torch.cuda.synchronize()
    t = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return r, (time.perf_counter() - t) * 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=10_000_000)
    ap.add_argument("--reps", type=int, default=9)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    R, L, k = a.reads, 100, 31
    gpu = card()
    d = torch.empty(R * L + 256, dtype=torch.uint8, device="cuda")
    lines = []
    with kc.Counter(k, L) as c:
        runs = []
        for s in range(2):
            synth.synth_reads_device(d.data_ptr(), R, L, 100_000_000, 1e-3, 0.0, 2, first_read=s * R)
            torch.cuda.synchronize()
            runs.append(c.count_device(d.data_ptr(), R * L))
        ra, rb = runs
        na, nb, S = len(ra), len(rb), c.record_size
        for op, counts in CASES:                            # warm every kernel the timed calls use
            ra.combine(rb, op, counts).free()
        c.merge([ra, rb]).free()
        for op, counts in CASES:
            t_comb, t_merge, n_out = [], [], 0
            for _ in range(a.reps):
                m, t = timed(lambda: c.merge([ra, rb]))
                n_merge = len(m)
                m.free()
                t_merge.append(t)
                r, t = timed(lambda: ra.combine(rb, op, counts))
                n_out = len(r)
                r.free()
                t_comb.append(t)
            mc, mm = statistics.median(t_comb), statistics.median(t_merge)
            line = {"op": op, "counts": counts or "default", "records_a": na, "records_b": nb, "records_out": n_out,
                    "records_merge": n_merge, "ms_combine": round(mc, 3), "ms_merge": round(mm, 3),
                    "combine_over_merge": round(mc / mm, 3),
                    "combine_GB_per_s": round(S * (na + nb + n_out) / mc / 1e6, 1),
                    "merge_GB_per_s": round(S * (na + nb + n_merge) / mm / 1e6, 1),
                    "ms_combine_all": [round(x, 3) for x in t_comb], "ms_merge_all": [round(x, 3) for x in t_merge],
                    "reps": a.reps, "gpu": gpu}
            print(json.dumps(line), flush=True)
            lines.append(line)
        ra.free()
        rb.free()
    if a.out:
        with open(a.out, "w") as f:
            f.write("".join(json.dumps(x) + "\n" for x in lines))


if __name__ == "__main__":
    main()
