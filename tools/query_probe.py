"""Time of the lookups in a run (kc_query_reads, kc_run_lookup) on C2's reads against their own run.

C2's reads (10 M x 100 bp of a 100 Mbase genome, device-resident) are counted on GPU 0 at each k; then
kc_query_reads of the same reads, device pointers in and out (slot counts and read hits), is timed warm:
the wall time of the call (median of --reps), and in a separate profiled pass the device time of its
kernels by name -- the index build, the extraction of the slots' keys, the lookups. The count of the
same reads is timed too, as scale. Then kc_run_lookup of 128 M device keys, half of them keys of the run
and half absent (a key of the run with one base changed). The floor: each lookup touches about four
random 32-byte sectors (index, one or two of keys, count), so 128 B / lookup over 7.7 TB/s. The card's
name and power limit are read in the same run. One JSON line per k on stdout (and --out).

Then, with 64-bit keys (k = 32) on runs built from uniform random keys: the lookup kernel's rate for 2^27
keys against runs of 2^20, 2^23 and 2^26 records (the first fits in L2 with its index, the last is 0.8 GB),
and the index build of a run of 2^26 records whose keys all fall below 2^40 (two of its 2^25 buckets hold
every record; the rest are filled by the index's bucket pass) against a uniform run of the same size."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import kmer_counter_b200 as kc
from kmer_counter_b200 import synth

HBM_BYTES_PER_S = 7.7e12


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else "%s (nvidia-smi unavailable)" % torch.cuda.get_device_name(0)


def timed(fn, reps):
    out = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        out.append((time.perf_counter() - t) * 1e3)
    return out


def kernel_ms(fn, reps):
    """device time per call of each kernel family fn launches, from torch.profiler (median over reps)"""
    from torch.profiler import ProfilerActivity, profile
    per = {}
    for _ in range(reps):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        sums = {}
        for e in prof.events():
            if e.device_type.name != "CUDA":
                continue
            name = e.name
            fam = ("index" if "query_index" in name else "extract" if "KeyValidSink" in name else
                   "lookup" if "query_lookup_kernel" in name else None)
            if fam:
                sums[fam] = sums.get(fam, 0.0) + e.device_time / 1e3
        for f, v in sums.items():
            per.setdefault(f, []).append(v)
    return {f: round(statistics.median(v), 3) for f, v in per.items()}


def sweep(gpu, n_q):
    # keys, picks and counts are made on the host and uploaded before any library call: the library runs
    # on its own stream, which does not wait for work queued on torch's
    out = []
    rng = np.random.default_rng(5)
    with kc.Counter(32, 32) as c:
        for log_n, crowd in ((20, False), (23, False), (26, False), (26, True)):
            hi = 2**40 if crowd else 2**62
            keys_h = np.unique(rng.integers(0, hi, int(1.05 * (1 << log_n)), dtype=np.uint64))[:1 << log_n]
            q_h = keys_h[rng.integers(0, len(keys_h), n_q)]
            keys = torch.from_numpy(keys_h.view(np.int64)).cuda()
            counts = torch.ones(len(keys_h), dtype=torch.int32, device="cuda")
            q = torch.from_numpy(q_h.view(np.int64)).cuda()
            res = torch.empty(n_q, dtype=torch.int32, device="cuda")
            torch.cuda.synchronize()
            run = c.run_from_device(keys.data_ptr(), counts.data_ptr(), len(keys_h))
            c.sync()
            del keys_h, q_h
            lk = lambda: c.lookup_device(run, q.data_ptr(), n_q, res.data_ptr())
            lk()
            parts = kernel_ms(lk, 3)
            line = {"sweep": "crowded below 2^40" if crowd else "uniform", "k": 32, "records": len(run),
                    "lookup_keys": n_q, "kernel_ms": parts, "all_found": bool((res == 1).all()),
                    "lookup_kernel_per_s": round(n_q / (parts["lookup"] / 1e3)), "gpu": gpu}
            print(json.dumps(line), flush=True)
            out.append(line)
            run.free()
            del keys, counts, q, res
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=10_000_000)
    ap.add_argument("--ks", default="31,63,96")
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--lookup-keys", type=int, default=128 << 20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    R, L = a.reads, 100
    gpu = card()
    d = torch.empty(R * L + 256, dtype=torch.uint8, device="cuda")
    synth.synth_reads_device(d.data_ptr(), R, L, 100_000_000, 1e-3, 0.0, 2)
    torch.cuda.synchronize()
    lines = []
    for k in [int(x) for x in a.ks.split(",")]:
        nk = L - k + 1
        slots = R * nk
        with kc.Counter(k, L) as c:
            count_ms = timed(lambda: c.count_device(d.data_ptr(), R * L).free(), 3)
            run = c.count_device(d.data_ptr(), R * L)
            W = c.words
            sc = torch.empty(slots, dtype=torch.int32, device="cuda")
            hits = torch.empty(R, dtype=torch.int32, device="cuda")
            q = lambda: c.query_reads_device(run, d.data_ptr(), R * L, sc.data_ptr(), hits.data_ptr())
            q()                                                  # warm
            q_ms = timed(q, a.reps)
            parts = kernel_ms(q, 3)
            ok = bool((sc > 0).all()) and int(hits.sum()) == slots      # no N in C2: every slot is a k-mer of the run
            # kc_run_lookup: half keys of the run, half absent (one base changed)
            n_run, n_q = len(run), a.lookup_keys
            rows = np.frombuffer(run.to_bytes(), dtype=np.uint8).reshape(n_run, c.record_size)
            pick = np.random.default_rng(k).integers(0, n_run, n_q)
            keys = np.ascontiguousarray(rows[pick, :8 * W]).view(np.uint64).reshape(n_q, W)
            del rows
            half = n_q // 2
            keys[half:, W - 1] ^= np.uint64(1 << (64 - 2 * (k - 32 * (W - 1))))
            qk = torch.from_numpy(keys.view(np.int64)).cuda()
            del keys
            out = torch.empty(n_q, dtype=torch.int32, device="cuda")
            lk = lambda: c.lookup_device(run, qk.data_ptr(), n_q, out.data_ptr())
            lk()
            lk_ms = timed(lk, a.reps)
            found = int((out[:half] > 0).sum()), int((out[half:] > 0).sum())
            lk_parts = kernel_ms(lk, 3)
            med = statistics.median(q_ms)
            floor_ms = slots * 128 / HBM_BYTES_PER_S * 1e3
            line = {"k": k, "reads": R, "read_len": L, "slots": slots, "records": n_run,
                    "ms_query_reads": round(med, 3), "ms_query_reads_all": [round(x, 3) for x in q_ms],
                    "kernel_ms": parts, "lookups_per_s": round(slots / (med / 1e3)),
                    "lookup_kernel_per_s": round(slots / (parts.get("lookup", 0) / 1e3)) if parts.get("lookup") else None,
                    "sector_floor_ms": round(floor_ms, 2), "floor_over_lookup_kernel": round(floor_ms / parts["lookup"], 3)
                    if parts.get("lookup") else None,
                    "ms_count_same_reads": round(statistics.median(count_ms), 3), "all_slots_found": ok,
                    "run_lookup_keys": n_q, "ms_run_lookup": round(statistics.median(lk_ms), 3),
                    "run_lookup_kernel_ms": lk_parts, "run_lookup_found_present_absent": found,
                    "run_lookup_per_s": round(n_q / (statistics.median(lk_ms) / 1e3)), "gpu": gpu}
            print(json.dumps(line), flush=True)
            lines.append(line)
            del sc, hits, qk, out
            run.free()
            torch.cuda.empty_cache()
    lines += sweep(gpu, a.lookup_keys)
    if a.out:
        with open(a.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
