"""Cost of canonical counting (KC_CANONICAL) against forward strict counting, on the GPU.

Device-resident synthetic reads (kc_synth_reads, the shape of configs[1]: 10M x 100 bp of a
100 Mbase genome); k=31 and k=63 (super-window path) and k=96 (key placement). For every shape
both settings are warmed up, then timed alternately step by step (events around kc_count_device
on the counter's stream, ending in a synchronise). Prints one JSON line: the GPU and its power
limit, and per shape and setting the median ms per step, G k-mers/s and the per-stage device
times of kc_stats.

    python tools/canonical_probe.py [--steps 10] [--warmup 3] [--out FILE]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [x.strip() for x in q.split(",")]
        return {"gpu": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:                     # the name is still known to torch
        import torch
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": "unknown (%s)" % e}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=10_000_000)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    import kmer_counter_b200 as kc
    from kmer_counter_b200 import synth
    if not torch.cuda.is_available():
        sys.exit("canonical_probe: no CUDA device")
    R, L = a.reads, 100
    d = torch.empty(R * L, dtype=torch.uint8, device="cuda:0")
    synth.synth_reads_device(d.data_ptr(), R, L, 100_000_000, 1e-3, 0.0, seed=2)
    torch.cuda.synchronize()
    res = {"probe": "canonical_vs_forward_strict", "reads": R, "read_len": L, "steps": a.steps, "warmup": a.warmup,
           "input": "device-resident synthetic reads, 10x of a 100 Mbase genome, sub 1e-3", **gpu_info(), "shapes": {}}
    for k in (31, 63, 96):
        cs = {"forward_strict": kc.Counter(k, L, compat="strict", max_chunk_bytes=R * L),
              "canonical": kc.Counter(k, L, canonical=True, max_chunk_bytes=R * L)}
        slots = R * (L - k + 1)
        times = {n: [] for n in cs}
        stats, distinct = {}, {}
        for step in range(a.warmup + a.steps):
            for name, c in cs.items():
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                run = c.count_device(d.data_ptr(), R * L)
                c.sync()
                ms = (time.perf_counter() - t0) * 1e3
                distinct[name] = len(run)
                run.free()
                if step >= a.warmup:
                    times[name].append(ms)
                    stats[name] = c.stats()
        shape = {}
        for name in cs:
            st = stats[name]
            med = statistics.median(times[name])
            shape[name] = {"ms_per_step": round(med, 3), "ms_min": round(min(times[name]), 3),
                           "gkmers_per_s": round(slots / med / 1e6, 2), "method_used": st["method_used"],
                           "distinct": distinct[name],
                           "stages_ms": {n: round(v, 3) for n, v in zip(st["stage_names"], st["ms_stage"])}}
            cs[name].close()
        shape["canonical_over_forward"] = round(shape["canonical"]["ms_per_step"] / shape["forward_strict"]["ms_per_step"], 3)
        res["shapes"]["k%d" % k] = shape
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
