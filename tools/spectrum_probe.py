"""Cost of the count spectrum and of the count filter on the device, and the D2H time the filter saves.

Device-resident synthetic reads with the values of bench.py's configs[1] (C2: 10M x 100 bp, 10x of a
100 Mbase genome, substitution rate 1e-3, seed 2), counted once per k: k=31 and k=63 (super-window
path) and k=96 (key placement). Before anything is timed, the spectrum and the min_count=2 filter of
a 20,000-read prefix are checked against the oracle. Then, per k:
  - records, and the fraction a min_count=2 filter keeps;
  - histogram ms: wall time of Run.histogram(10001) (memset, kernel, 80 KB D2H, synchronise);
  - filter ms: wall time of Run.filter(2) (count pass, scan, total D2H, allocation, write pass);
  - D2H ms of kc_run_copy_records into pinned memory, for the unfiltered run and for the filtered
    one, alternating.
Every time is the median of --reps repetitions after one warm-up call. Prints one JSON line.

    python tools/spectrum_probe.py [--reps 7] [--out FILE]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

C2 = dict(reads=10_000_000, read_len=100, genome=100_000_000, sub_rate=1e-3, n_rate=0.0, seed=2)
PREFIX = 20_000


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [x.strip() for x in q.split(",")]
        return {"gpu": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:                     # the name is still known to torch
        import torch
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": "unknown (%s)" % e}


def check_prefix(kc, oracle, k):
    """spectrum and min_count=2 filter of a prefix of the same reads against the oracle"""
    L = C2["read_len"]
    reads = oracle.gen_reads(PREFIX, L, C2["genome"], C2["sub_rate"], C2["n_rate"], seed=C2["seed"])
    want = oracle.count(reads, L, k)
    S = oracle.record_size(k)
    _, counts = oracle.records_to_arrays(want, k)
    rows = np.frombuffer(want, dtype=np.uint8).reshape(-1, S)
    with kc.Counter(k, L, max_chunk_bytes=PREFIX * L) as c:
        c.slot_buffer(0)[:len(reads)] = reads
        c.submit(0, len(reads))
        run = c.wait(0)
        h = run.histogram(10001)
        f = run.filter(2)
        ok = (run.to_bytes() == want and
              np.array_equal(h, np.bincount(np.minimum(counts, 10000), minlength=10001).astype(np.uint64)) and
              f.to_bytes() == rows[counts >= 2].tobytes())
        run.free()
        f.free()
    if not ok:
        sys.exit("spectrum_probe: k=%d differs from the oracle on the %d-read prefix" % (k, PREFIX))


def timed(fn):
    t0 = time.perf_counter()
    out = fn()
    return (time.perf_counter() - t0) * 1e3, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    import kmer_counter_b200 as kc
    import oracle
    from kmer_counter_b200 import synth
    if not torch.cuda.is_available():
        sys.exit("spectrum_probe: no CUDA device")
    R, L = C2["reads"], C2["read_len"]
    d = torch.empty(R * L, dtype=torch.uint8, device="cuda:0")
    synth.synth_reads_device(d.data_ptr(), R, L, C2["genome"], C2["sub_rate"], C2["n_rate"], seed=C2["seed"])
    torch.cuda.synchronize()
    res = {"probe": "spectrum_and_filter", **C2, "reps": a.reps, "min_count": 2, "n_bins": 10001, **gpu_info(),
           "shapes": {}}
    for k in (31, 63, 96):
        check_prefix(kc, oracle, k)
        with kc.Counter(k, L, max_chunk_bytes=R * L) as c:
            run = c.count_device(d.data_ptr(), R * L)
            c.sync()
            n = len(run)
            hist = run.histogram(10001)
            t_hist, t_filt, t_full, t_kept = [], [], [], []
            buf = c.host_alloc(run.nbytes)
            kept = run.filter(2)
            for rep in range(a.reps + 1):
                ms_h, _ = timed(lambda: run.histogram(10001))
                ms_f, f = timed(lambda: run.filter(2))
                f.free()
                ms_full, nb_full = timed(lambda: run.copy_into(buf.ctypes.data, buf.size))
                ms_kept, nb_kept = timed(lambda: kept.copy_into(buf.ctypes.data, buf.size))
                if rep:
                    t_hist.append(ms_h)
                    t_filt.append(ms_f)
                    t_full.append(ms_full)
                    t_kept.append(ms_kept)
            shape = {"method_used": c.stats()["method_used"], "records": n, "records_kept": len(kept),
                     "kept_fraction": round(len(kept) / n, 4), "singletons": int(hist[1]),
                     "histogram_ms": round(statistics.median(t_hist), 3), "filter_ms": round(statistics.median(t_filt), 3),
                     "d2h_unfiltered_ms": round(statistics.median(t_full), 3), "d2h_unfiltered_bytes": nb_full,
                     "d2h_filtered_ms": round(statistics.median(t_kept), 3), "d2h_filtered_bytes": nb_kept,
                     "spectrum_head": [int(x) for x in hist[:12]]}
            shape["d2h_saved_ms"] = round(shape["d2h_unfiltered_ms"] - shape["d2h_filtered_ms"], 3)
            shape["counts_gb_per_s_histogram"] = round(n * 4 / (shape["histogram_ms"] * 1e6), 1)
            kept.free()
            run.free()
            c.host_free(buf)
        res["shapes"]["k%d" % k] = shape
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
