#!/usr/bin/env python
"""bench.py -- k-mers counted per second at k=31 (BASELINE.json's metric).

    python bench.py --gpus N --steps K --warmup W            (ours; torchrun for N > 1)
    python bench.py --impl reference --gpus N --steps K ...   (the reference's CPU path)
    python bench.py --config c3|c4|c5 ...                     (the other BASELINE configurations)
    python bench.py ... --dump-outputs DIR                    (also write the last timed step's run to DIR/*.npy)

A step is one pass of the whole counting path over one batch of synthetic reads:
reads -> super-window records -> per-bin count -> distinct records in key order
[-> exchange over NVLink for N > 1] -> sorted key-unique run.
  value : whole-job k-mers/s with the reads already resident in HBM
  e2e   : the same through the host-buffer API: pinned host reads -> H2D -> count ->
          packed records D2H into pinned host memory, every step
  parity: before anything is timed, a prefix of every rank's reads goes through the SAME path
          that is timed and is compared with the CPU oracle (bit-exact, sha256); a mismatch
          fails the run
  roofline      : dominant kernel of the step; algorithmic bytes over its device time (CUDA
                  events inside libkc_b200 on the stream the kernels run on), against
                  MEASURED_PEAKS.json's HBM copy bandwidth
  path_roofline : SURVEY.md 8(d)'s whole-path figure B_alg = B_in + N*(Kb+8) + U*S over step time
  cpu_baseline  : oracle/_ref (the reference's own sources) on bounded samples, host cores
One JSON line on stdout (rank 0).
"""
import argparse
import hashlib
import json
import os
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "k-mers counted/s at k=31"          # BASELINE.json's metric; a line run with another k says so (metric_for)
UNIT = "kmers/s"
REF_CHUNK = 89364           # reads per chunk at the reference's defaults (KMerCounter.cpp:193-212, SURVEY 3.1)
DUMP_BYTES = 48 << 20       # --dump-outputs writes at most this much; larger runs are sampled at seeded record indices
DUMP_SEED = 20261020

# BASELINE.json configs[0..4] (SURVEY.md 8(d) "Synthetic inputs"); reads are per GPU
CONFIGS = {
    "c1": dict(reads=100_000, k=31, genome=1_000_000, sub_rate=0.0, n_rate=1e-3, seed=1, zipf_loci=0, runs=1,
               name="configs[0]: synthetic 100k x 100 bp reads, k=31"),
    "c2": dict(reads=10_000_000, k=31, genome=100_000_000, sub_rate=1e-3, n_rate=0.0, seed=2, zipf_loci=0, runs=1,
               name="configs[1]: synthetic 10M x 100 bp reads (1 Gbase, 10x of a 100 Mbase genome), k=31"),
    "c3": dict(reads=200_000_000, k=63, genome=1_000_000_000, sub_rate=1e-3, n_rate=0.0, seed=3, zipf_loci=0, runs=1,
               name="configs[2]: synthetic 200M x 100 bp reads (20 Gbase, 20x of a 1 Gbase genome), k=63 (128-bit keys)"),
    "c4": dict(reads=125_000_000, k=31, genome=3_330_000_000, sub_rate=1e-3, n_rate=0.0, seed=4, zipf_loci=0, runs=1,
               name="configs[3]: 125M x 100 bp reads per GPU of a 3.33 Gbase genome (100 Gbase = 30x at 8 GPUs), k=31"),
    "c5": dict(reads=125_000_000, k=31, genome=3_330_000_000, sub_rate=1e-3, n_rate=0.0, seed=5, zipf_loci=1_000_000, runs=16,
               name="configs[4]: 125M x 100 bp reads per GPU, half of them at 1M Zipf-distributed hot loci, counted "
                    "in 16 runs per GPU that are merged on the GPU (merge path), k=31"),
}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default=None, choices=sorted(CONFIGS), help="default: c2 (per GPU, scaled out for N > 1)")
    ap.add_argument("--reads", type=int, default=None, help="reads per GPU (overrides the config)")
    ap.add_argument("--read-len", type=int, default=100)
    ap.add_argument("--k", type=int, default=None)
    ap.add_argument("--genome", type=int, default=None)
    ap.add_argument("--sub-rate", type=float, default=None)
    ap.add_argument("--n-rate", type=float, default=None)
    ap.add_argument("--seed", type=int, default=None)
    ap.add_argument("--zipf-loci", type=int, default=None)
    ap.add_argument("--runs", type=int, default=None, help="count every GPU's reads in this many runs and merge them")
    ap.add_argument("--method", default="auto", choices=["auto", "sort", "hash", "super"])
    ap.add_argument("--parity-reads", type=int, default=200_000, help="reads per rank of the in-run parity check (0 = off)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--occ", type=int, default=0, help="k-mer occurrences per minimizer bin (0 = library default)")
    ap.add_argument("--bench", default="count", choices=["count", "merge"],
                    help="merge: time kc_merge_runs (GPU KMerFileMerger) over --runs runs of --reads reads each")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the run the last step computed to DIR as float64 .npy files "
                         "(a seeded sample of its records beyond %d MB)" % (DUMP_BYTES >> 20))
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs writes what this project's GPU path computed; the reference arm computes on the host")
    cfg = dict(CONFIGS[a.config or "c2"])
    changed = []
    for key in ("reads", "k", "genome", "sub_rate", "n_rate", "seed", "zipf_loci", "runs"):
        v = getattr(a, key)
        if v is not None and v != cfg[key]:
            cfg[key] = v
            changed.append("%s=%s" % (key, v))
    if changed:                                     # not a BASELINE configuration any more: say so in the workload name
        cfg["name"] = "%s-shaped synthetic reads with %s (k=%d)" % ((a.config or "c2"), ", ".join(changed), cfg["k"])
    world = int(os.environ.get("WORLD_SIZE", "1"))
    cfg["scaled_out"] = False
    if a.config is None and world > 1 and a.genome is None:
        # weak scaling of configs[1]: the job is N x 10M reads of a genome N times as long (10x coverage of
        # the whole job, as in configs[1]); rank r counts reads [r*R, (r+1)*R) of it
        cfg["genome"] *= world
        cfg["scaled_out"] = True
        cfg["name"] = ("configs[1] scaled out: %d x 10M x 100 bp reads of a %d Mbase genome (10x), 10M reads per GPU, k=31"
                       % (world, cfg["genome"] // 1_000_000))
    a.cfg = cfg
    return a


E2E_SLOTS = 2           # pinned input slots of the end-to-end pipeline (chunks whose H2D / kernels are in flight)


def metric_for(k):
    return METRIC if k == 31 else "k-mers counted/s at k=%d" % k


def workload(a, world, mode=None):
    c = a.cfg
    L = a.read_len
    return {"workload": c["name"], "reads_per_gpu": c["reads"], "read_len": L, "k": c["k"], "genome_len": c["genome"],
            "sub_rate": c["sub_rate"], "n_rate": c["n_rate"], "seed": c["seed"], "zipf_loci": c["zipf_loci"],
            "runs_per_gpu": c["runs"], "kmers_per_step_per_gpu": c["reads"] * (L - c["k"] + 1), "mode": mode,
            "l2_policy": "inputs larger than L2 (%.1f GB of reads per GPU per step vs 126 MB L2)" % (c["reads"] * L / 1e9)}


def bind_near_gpu(index):
    """Run this process on the CPUs next to GPU `index` (NVML's ideal affinity) before anything is
    allocated. Returns the CPU count bound to, or None (KC_NO_BIND=1 skips it)."""
    if os.environ.get("KC_NO_BIND") == "1":
        return None
    try:
        import pynvml
        pynvml.nvmlInit()
        pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(index))
        return len(os.sched_getaffinity(0))
    except Exception:
        return None


# ------------------------------------------------------------------ clocks
class ClockSampler:
    """SM clock and throttle reasons sampled through NVML every 5 ms while the timed region runs."""

    def __init__(self, index):
        self.index, self.sm, self.mx, self.reasons, self.stop, self.th = index, [], 0, set(), threading.Event(), None
        self.nv = self.h = None
        try:
            import pynvml as nv
            nv.nvmlInit()
            self.nv, self.h = nv, nv.nvmlDeviceGetHandleByIndex(index)
            self.mx = nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)
            self.flags = {"hw_slowdown": nv.nvmlClocksThrottleReasonHwSlowdown,
                          "hw_thermal_slowdown": nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                          "sw_thermal_slowdown": nv.nvmlClocksThrottleReasonSwThermalSlowdown,
                          "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap}
        except Exception as e:
            self.reasons.add("nvml_unavailable: %s" % type(e).__name__)

    def _sample(self):
        if self.h is None:
            return
        self.sm.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
        r = self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
        for name, bit in self.flags.items():
            if r & bit:
                self.reasons.add(name)

    def _run(self):
        while not self.stop.is_set():
            self._sample()
            self.stop.wait(0.005)

    def __enter__(self):
        self.th = threading.Thread(target=self._run, daemon=True)
        self.th.start()
        return self

    def __exit__(self, *a):
        self._sample()
        self.stop.set()
        self.th.join(timeout=5)

    def summary(self):
        sm = sorted(self.sm)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.mx or None,
                "reasons": sorted(self.reasons), "samples": len(sm)}


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


class StdoutToStderr:
    """The reference's own code prints progress on stdout (e.g. FASTQFileReader.cpp:40); while it runs, file
    descriptor 1 points at stderr so that this program's stdout stays ONE JSON line."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)


# --------------------------------------------------------- the reference's CPU path
def _ref_row(oracle, reads, L, k, threads, fan_in, merge_threads, tmp_root):
    """One timed run of the reference's Pipeline B (oracle/_ref) -> row with per-stage seconds."""
    n_reads = len(reads) // L
    kmers = n_reads * (L - k + 1)
    t0 = time.perf_counter()
    if oracle.ref_available() and hasattr(oracle.ref(), "ref_count_packed_ex"):
        with tempfile.TemporaryDirectory(dir=tmp_root) as d:
            st = oracle.ref_count_packed_ex(reads, L, k, REF_CHUNK, threads, fan_in, merge_threads, d, os.path.join(d, "out.bin"))
        kind = "reference"
    else:
        oracle.count(reads, L, k, REF_CHUNK, threads=threads)
        st, kind = {}, "port"
    dt = time.perf_counter() - t0
    row = {"threads": threads, "merge_threads": merge_threads, "merge_fan_in": fan_in, "reads": n_reads, "kmers": kmers,
           "seconds": dt, "value": kmers / dt, "unit": UNIT, "kind": kind}
    row.update({"stage_seconds": {kx: round(v, 4) for kx, v in st.items() if kx.endswith("_s")},
                "runs": st.get("runs"), "threads_busy": st.get("threads_busy")})
    return row


def _read_stage_seconds(oracle, n_reads, L, c, tmp_root):
    """The reference's reader (FASTQFileReader / InputFileHandler) on the same sample written as a FASTQ file."""
    if not oracle.ref_available():
        return None
    try:
        fq = oracle.gen_fastq(n_reads, L, c["genome"], c["sub_rate"], c["n_rate"], seed=c["seed"])
        with tempfile.TemporaryDirectory(dir=tmp_root) as d:
            with open(os.path.join(d, "sample.fastq"), "wb") as f:
                f.write(fq)
            t0 = time.perf_counter()
            oracle.ref_read_fastq_dir(d)
            return time.perf_counter() - t0
    except Exception:
        return None


def cpu_rows(a, budget_reads=None):
    """SURVEY 8(d): (i) 1 thread, (ii) 8 chunk workers (the reference's 8 GPUStream threads,
    KMerCounter.cpp:117) + noOfMergeThreads=2 mergers with fan-in 2, on bounded samples of the workload."""
    import oracle
    c, L = a.cfg, a.read_len
    cores = os.cpu_count() or 1
    tmp_root = "/dev/shm" if os.path.isdir("/dev/shm") else None
    n8 = min(c["reads"], budget_reads or 8 * REF_CHUNK)
    n1 = min(c["reads"], 2 * REF_CHUNK)
    gen = lambda n: oracle.gen_reads(n, L, c["genome"], c["sub_rate"], c["n_rate"], seed=c["seed"], zipf_loci=c["zipf_loci"])
    rows = []
    reads8 = gen(n8)
    rows.append(_ref_row(oracle, reads8[: n1 * L], L, c["k"], 1, 2, 1, tmp_root))
    rows.append(_ref_row(oracle, reads8, L, c["k"], min(8, cores), 2, 2, tmp_root))
    rd = _read_stage_seconds(oracle, n1, L, c, tmp_root)
    if rd is not None:
        rows[0]["stage_seconds"]["read_fastq_s"] = round(rd, 4)
    return rows, cores


def reference_gpu_seam(a):
    """SURVEY F10 / 8(d) "reference-on-B200": the reference's own GPUHandler.cu, compiled unmodified for
    sm_100a (oracle/_ref/ref_gpu, built by oracle/build_ref.sh), driven like KMerCounter::dispatchWork drives
    it: PrepareGPU once, processKMers per default-sized chunk. The host hash accumulate that follows
    at HEAD (KMerCounter.cpp:61-82) is not in it. None when the binary is not there."""
    import subprocess
    import oracle
    exe = os.path.join(ROOT, "oracle", "_ref", "ref_gpu")
    if not os.path.isfile(exe):
        return None
    c, L = a.cfg, a.read_len
    n = min(c["reads"], 16 * REF_CHUNK)
    tmp_root = "/dev/shm" if os.path.isdir("/dev/shm") else None
    try:
        reads = oracle.gen_reads(n, L, c["genome"], c["sub_rate"], c["n_rate"], seed=c["seed"], zipf_loci=c["zipf_loci"])
        with tempfile.TemporaryDirectory(dir=tmp_root) as d:
            path = os.path.join(d, "reads.bin")
            with open(path, "wb") as f:
                f.write(bytes(reads))
            r = subprocess.run([exe, path, str(L), str(c["k"]), str(REF_CHUNK)], capture_output=True, timeout=300)
        row = json.loads(r.stderr.decode().strip().splitlines()[-1])
    except Exception as e:
        return {"unavailable": "%s: %s" % (type(e).__name__, e)}
    return {"value": row["kmers_per_s"], "unit": UNIT, "kind": "reference GPUHandler.cu (unmodified) built for sm_100a",
            "seconds": row["seconds"], "reads": row["reads"], "chunks": row["chunks"], "chunk_reads": REF_CHUNK,
            "what": "PrepareGPU + processKMers per chunk (GPUHandler.cu:397-508): H2D, bitEncode, extractKMers, D2H of the "
                    "record block, host reduceKMers; one GPUStream; the TBB accumulate of KMerCounter.cpp:61-82 is not included"}


def cpu_baseline(a):
    with StdoutToStderr():
        rows, cores = cpu_rows(a)
        gpu_seam = reference_gpu_seam(a)
    best = max(rows, key=lambda r: r["value"])
    return {"value": best["value"], "unit": UNIT, "cores": best["threads"], "host_cores": cores, "kind": best["kind"],
            "reference_gpu_seam": gpu_seam,
            "sample": "first %d reads (%d k-mers) of the workload in chunks of %d reads (the reference's default), %d chunk-worker "
                      "threads busy, KMerFileMerger with fan-in %d on %d merger threads; rows: 1 thread and 8+2 threads"
                      % (best["reads"], best["kmers"], REF_CHUNK, best.get("threads_busy") or best["threads"],
                         best["merge_fan_in"], best["merge_threads"]),
            "rows": rows}


def run_reference(a, rank):
    """The reference's own CPU implementation of the path (oracle/_ref: its sources compiled in
    place) on the host cores; each step a bounded sample of this arm's workload."""
    if rank != 0:
        return
    import oracle
    c, L = a.cfg, a.read_len
    cores = os.cpu_count() or 1
    tmp_root = "/dev/shm" if os.path.isdir("/dev/shm") else None
    # ~40k reads/s on 8 threads: size the per-step sample so that K + 1 steps stay within ~150 s
    per_step = int(150.0 / (max(a.steps, 1) + 1) * 40_000)
    sample = max(2 * REF_CHUNK, min(8 * REF_CHUNK, per_step, c["reads"]))
    sample = min(sample, c["reads"])
    reads = oracle.gen_reads(sample, L, c["genome"], c["sub_rate"], c["n_rate"], seed=c["seed"], zipf_loci=c["zipf_loci"])
    threads = min(8, cores)
    rows = []
    with StdoutToStderr():
        for _ in range(min(a.warmup, 1)):
            _ref_row(oracle, reads, L, c["k"], threads, 2, 2, tmp_root)
        for _ in range(max(a.steps, 1)):
            rows.append(_ref_row(oracle, reads, L, c["k"], threads, 2, 2, tmp_root))
    dt = sum(r["seconds"] for r in rows) / len(rows)
    kmers = sample * (L - c["k"] + 1)
    val = kmers / dt
    line = {"metric": metric_for(c["k"]), "value": val, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps, "warmup": min(a.warmup, 1),
            "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u64" if c["k"] <= 32 else "u128", "data": "synthetic", "impl": "reference",
            "config": workload(a, max(a.gpus, 1), "reference CPU path"),
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "host_cores": cores, "kind": rows[-1]["kind"],
                             "sample": "%d reads (%d k-mers) of the workload per step, chunks of %d reads through FileDump run files in %s, "
                                       "%d chunk-worker threads (%s busy), KMerFileMerger fan-in 2 on 2 merger threads"
                                       % (sample, kmers, REF_CHUNK, tmp_root or "tmp", threads, rows[-1].get("threads_busy")),
                             "stage_seconds_last_step": rows[-1]["stage_seconds"]},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------- our arm
def dump_run(run, out_dir, device, budget, suffix=""):
    """--dump-outputs: the records of a device-resident run as float64 .npy files in out_dir --
    keys[m, 2W] (every key word as its high and low 32 bits, exact in float64), counts[m], record_index[m]
    (the records' positions in the run) and run_summary = [records, sum of counts]. A run whose m = n
    records do not fit `budget` bytes is sampled at seeded, sorted record indices."""
    import numpy as np
    import torch
    from kmer_counter_b200.multigpu import run_as_tensors
    keys, counts = run_as_tensors(run, device)
    n, W = keys.shape
    cap = budget // (8 * (2 * W + 2))
    idx = np.arange(n) if n <= cap else np.unique(np.random.default_rng(DUMP_SEED).integers(0, n, size=cap))
    sel = torch.from_numpy(idx).to(device)
    k = keys.index_select(0, sel).cpu().numpy().view(np.uint64)
    c = counts.index_select(0, sel).cpu().numpy().view(np.uint32)
    halves = np.empty((len(idx), 2 * W), dtype=np.float64)
    halves[:, 0::2] = k >> np.uint64(32)
    halves[:, 1::2] = k & np.uint64(0xFFFFFFFF)
    total = int((counts.to(torch.int64) & 0xFFFFFFFF).sum().item())
    os.makedirs(out_dir, exist_ok=True)
    for name, arr in (("keys", halves), ("counts", c), ("record_index", idx), ("run_summary", [n, total])):
        np.save(os.path.join(out_dir, name + suffix + ".npy"), np.asarray(arr, dtype=np.float64))


class Job:
    """One rank's share of the workload and the path it is counted through."""

    def __init__(self, a, rank, world, local_rank):
        import torch
        import torch.distributed as dist
        import kmer_counter_b200 as kc
        from kmer_counter_b200 import multigpu
        self.torch, self.dist, self.kc, self.multigpu = torch, dist, kc, multigpu
        self.a, self.c, self.rank, self.world = a, a.cfg, rank, world
        c = a.cfg
        self.L, self.k, self.R = a.read_len, c["k"], c["reads"]
        self.nk = self.L - self.k + 1
        self.n_bytes = self.R * self.L
        self.dev = torch.device("cuda", local_rank)
        self.stream = torch.cuda.Stream(device=self.dev, priority=-1)
        torch.cuda.set_stream(self.stream)
        windows = self.R * self.nk
        self.runs = max(1, c["runs"])
        if world > 1:
            self.mode = "exchange"
        elif self.runs > 1 or windows > (1 << 30) - 1:
            self.mode = "accumulate"
        else:
            self.mode = "chunk"
        self.e2e = not a.no_e2e and self.runs == 1 and windows <= (1 << 30) - 1
        per_run = (self.R + self.runs - 1) // self.runs
        # distinct keys a flush may see: the genome's k-mers + ~k per sequencing error (bounded by the windows)
        # (with several GPUs a rank counts 1/N of the bins of the whole job: its share of the job's distinct keys)
        est_u = 0
        if c["genome"]:
            est_u = (c["genome"] + int(per_run * world * self.L * c["sub_rate"] * self.k * 1.2)) // world + (1 << 20)
            est_u = min(per_run * self.nk, est_u)
        self.counter = kc.Counter(self.k, self.L, device=local_rank, method=a.method, n_slots=E2E_SLOTS,
                                  max_chunk_bytes=self.n_bytes if self.e2e else 0, table_slots=a.occ,
                                  stream=self.stream.cuda_stream,
                                  distinct_hint=est_u if self.mode != "chunk" and per_run * self.nk > (1 << 31) else 0)
        self.exchange = None
        if self.mode == "exchange":
            self.exchange = multigpu.Exchange(self.counter, self.dev, per_run + 4096)
        elif self.mode == "accumulate":
            self.counter.accum_begin(per_run + 4096)          # (pieces are whole multiples of 16 reads: the last one is a little longer)
        self.per_run = per_run
        self.d_reads = None
        self.last_run = None
        self.acc = self.new_acc()

    @staticmethod
    def new_acc():
        return {"dom_ms": 0.0, "dom_bytes": 0, "dom_launch": 0, "tot_ms": 0.0, "counts": 0}

    def note_count(self):
        """Stage timers of the count / flush that just finished (libkc_b200 keeps the last one's)."""
        s, acc = self.counter.stats(), self.acc
        acc["dom_ms"] += s["ms_dominant"]; acc["dom_bytes"] += s["dominant_bytes"]; acc["dom_launch"] += s["dominant_launches"]
        acc["tot_ms"] += s["ms_total"]
        acc["counts"] += 1

    def make_reads(self):
        from kmer_counter_b200 import synth
        c = self.c
        self.d_reads = self.torch.empty(self.n_bytes + 256, dtype=self.torch.uint8, device=self.dev)
        synth.synth_reads_device(self.d_reads.data_ptr(), self.R, self.L, c["genome"], c["sub_rate"], c["n_rate"], c["seed"],
                                 first_read=self.rank * self.R, zipf_loci=c["zipf_loci"], stream=self.stream.cuda_stream)
        self.stream.synchronize()

    def count(self, ptr, n_reads):
        """n_reads device-resident reads at ptr through the timed path -> Run of this rank's records."""
        c, L = self.counter, self.L
        if self.mode == "chunk":
            run = c.count_device(ptr, n_reads * L)
            self.note_count()
            return run
        # `runs` pieces of about equal size (whole multiples of 16 reads: device pieces stay 16-byte aligned),
        # each counted into its own run; the runs are then merged on the GPU (merge path = KMerFileMerger)
        # Merge schedule = the tiered one of host/RunMerger.h (KMerFileMergeHandler's fan-in 2): two runs of the
        # same level are merged as soon as both exist, so at most log2(runs) runs wait at any time.
        runs = self.runs if n_reads >= 16 * self.runs else 1
        per = (n_reads // runs) // 16 * 16 if runs > 1 else n_reads
        stack = []                                   # (level, run)
        for i in range(runs):
            r0 = i * per
            nr = per if i + 1 < runs else n_reads - r0
            c.accum_add_device(ptr + r0 * L, nr * L)
            stack.append((0, self.exchange.finish() if self.exchange is not None else c.accum_flush()))
            self.note_count()
            if self.exchange is not None and runs > 1 and i == 0:
                c.xchg_fix_ranges(True)              # every run of this count is cut at the first run's key ranges
            while len(stack) >= 2 and stack[-1][0] == stack[-2][0]:
                (lv, b), (_, a2) = stack.pop(), stack.pop()
                m = c.merge([a2, b])
                a2.free()
                b.free()
                stack.append((lv + 1, m))
        if self.exchange is not None and runs > 1:
            c.xchg_fix_ranges(False)
        while len(stack) >= 2:                       # a run count that is not a power of two
            (lv, b), (_, a2) = stack.pop(), stack.pop()
            m = c.merge([a2, b])
            a2.free()
            b.free()
            stack.append((lv + 1, m))
        return stack[0][1]

    def step(self, keep=False):
        """One pass over this rank's reads -> records in its run; keep=True holds the run in last_run."""
        run = self.count(self.d_reads.data_ptr(), self.R)
        n = len(run)
        if keep:
            self.last_run = run
        else:
            run.free()
        return n


def parity_check(job, a):
    """A prefix of every rank's reads through the path that is timed, against the CPU oracle."""
    import numpy as np
    import oracle
    torch, dist = job.torch, job.dist
    pre = min(job.R, a.parity_reads)
    if pre <= 0:
        return {"checked": False}
    c, L, k = job.c, job.L, job.k
    run = job.count(job.d_reads.data_ptr(), pre)
    got = run.to_bytes()
    run.free()
    S = job.counter.record_size
    mine = {"n": len(got) // S, "sha": hashlib.sha256(got).hexdigest()}
    if job.world > 1:
        lo, _, _ = job.counter.xchg_info(job.world)
        mine["lo"] = lo
        everyone = [None] * job.world
        dist.all_gather_object(everyone, mine)
    else:
        everyone = [mine]
    ok, detail = True, None
    if job.rank == 0:
        host = job.d_reads[: pre * L].cpu().numpy()
        gen = oracle.gen_reads(pre, L, c["genome"], c["sub_rate"], c["n_rate"], seed=c["seed"], zipf_loci=c["zipf_loci"])
        assert bytes(host) == bytes(gen), "device generator != host generator"
        shards = [gen] + [oracle.gen_reads(pre, L, c["genome"], c["sub_rate"], c["n_rate"], seed=c["seed"], zipf_loci=c["zipf_loci"],
                                           first_read=r * job.R) for r in range(1, job.world)]
        want = oracle.count(np.concatenate(shards), L, k, chunk_reads=REF_CHUNK, threads=os.cpu_count() or 1)
        if job.world == 1:
            ok = hashlib.sha256(want).hexdigest() == mine["sha"]
        else:
            # rank r holds the keys whose leading 10 bits lie in [lo[r], lo[r+1]): cut the oracle's artefact there
            keys, _ = oracle.records_to_arrays(want, k)
            b = (keys[:, 0] >> np.uint64(54)).astype(np.int64)
            lo = everyone[0]["lo"]
            cuts = [int(np.searchsorted(b, x, side="left")) for x in lo]
            for r, e in enumerate(everyone):
                piece = want[cuts[r] * S: cuts[r + 1] * S]
                if e["lo"] != lo or e["n"] != cuts[r + 1] - cuts[r] or hashlib.sha256(piece).hexdigest() != e["sha"]:
                    ok, detail = False, "rank %d: %d records, oracle has %d in its key range" % (r, e["n"], cuts[r + 1] - cuts[r])
                    break
        res = {"checked": True, "ok": ok, "reads_per_rank": pre, "ranks": job.world, "records": sum(e["n"] for e in everyone),
               "sha256": hashlib.sha256(want).hexdigest(), "oracle": "oracle.count (C restatement pinned to oracle/_ref)",
               "path": job.mode}
        if detail:
            res["detail"] = detail
    else:
        res = None
    if job.world > 1:
        box = [res]
        dist.broadcast_object_list(box, src=0)
        res = box[0]
    if not res["ok"]:
        if job.rank == 0:
            sys.stderr.write("bench.py: PARITY FAILED: %s\n" % json.dumps(res))
        sys.exit(3)
    return res


def run_ours(a, rank, world, local_rank):
    import torch
    import torch.distributed as dist

    numa = bind_near_gpu(local_rank)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    job = Job(a, rank, world, local_rank)
    counter, stream = job.counter, job.stream
    L, k, R, nk, n_bytes = job.L, job.k, job.R, job.nk, job.n_bytes
    job.make_reads()

    parity = parity_check(job, a)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(a.warmup):
        job.step()
    barrier()
    st0 = counter.stats()
    acc = job.acc = job.new_acc()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clk:
        ev0.record(stream)
        t0 = time.perf_counter()
        distinct = 0
        for i in range(a.steps):
            distinct = job.step(keep=a.dump_outputs is not None and i == a.steps - 1)
        ev1.record(stream)
        barrier()
        wall = time.perf_counter() - t0
    dev_ms = ev0.elapsed_time(ev1)
    st1 = counter.stats()
    t = torch.tensor([dev_ms, float(distinct)], dtype=torch.float64, device=dev)
    tsum = t.clone()
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
    ms_per_step = float(t[0].item()) / a.steps
    distinct_total = int(tsum[1].item()) if world > 1 else distinct
    kmers_step = R * nk * world
    value = kmers_step / (ms_per_step * 1e-3)
    method_used = st1["method_used"]
    launches = st1["launches"] - st0["launches"]
    nvlink = None
    if world > 1:
        _, recv, remote = counter.xchg_info(world)
        # bytes this rank pulled from its peers in the last step: super-window records of its bins + its key range's records
        rec_bytes = 16 * counter.words
        sc = counter.debug_scalars()
        pulled_rec = sc["records"] * (world - 1) // world * rec_bytes      # this rank's bins hold 1/P of every rank's records
        pulled_d = remote * (8 * counter.words + 4)
        x = torch.tensor([float(pulled_rec + pulled_d)], dtype=torch.float64, device=dev)
        dist.all_reduce(x, op=dist.ReduceOp.MAX)
        # per-stage device times of the last step over the ranks (a stage ends when its kernels end on that
        # rank: a rank that waits for a slower peer shows the wait in the stage that follows the barrier)
        stg = torch.tensor(list(st1["ms_stage"])[:6] + [float(sc["overflow_records"] != 0), float(sc["big_ranges"])],
                           dtype=torch.float64, device=dev)
        smax, smin = stg.clone(), stg.clone()
        dist.all_reduce(smax, op=dist.ReduceOp.MAX)
        dist.all_reduce(smin, op=dist.ReduceOp.MIN)
        nvlink = {"bytes_in_per_step_per_gpu": int(x.item()),
                  "stage_ms_max_over_ranks": [round(v, 3) for v in smax.tolist()[:6]],
                  "stage_ms_min_over_ranks": [round(v, 3) for v in smin.tolist()[:6]],
                  "ranks_with_overflow_records": bool(smax.tolist()[6]), "max_oversized_ranges": int(smax.tolist()[7]), "super_window_records_bytes": int(pulled_rec),
                  "distinct_records_bytes": int(pulled_d),
                  "achieved_gbs_over_step": x.item() / (ms_per_step * 1e-3) / 1e9, "peak": 900, "measured_peer_copy": 770,
                  "note": "both exchanges are the load side of the consuming kernels (peer loads over NVLink/NVSwitch), "
                          "spread over the step: the rate is bytes over the whole step time, not a link saturation figure"}

    if job.last_run is not None:
        dump_run(job.last_run, a.dump_outputs, dev, DUMP_BYTES // world, "_rank%d" % rank if world > 1 else "")
        job.last_run.free()
        job.last_run = None

    # ---- end to end through the host-buffer API (pinned in, pinned out)
    e2e = None
    if job.e2e:
        e2e = run_e2e(job, a, distinct, kmers_step, barrier, numa)

    clocks = clk.summary()
    peak, peak_src = measured_peak_gbs()
    if rank == 0:
        dom_ms, dom_bytes, dom_launch, tot_ms = acc["dom_ms"], acc["dom_bytes"], acc["dom_launch"], acc["tot_ms"]
        names = st1["stage_names"]
        dom_name = names[st1["dominant_stage"]] if names else "none"
        Kb, S = 8 * counter.words, counter.record_size
        U = distinct_total // world if world > 1 else distinct
        N = R * nk
        # SURVEY 8(d): per occurrence one key-sized read + a 4-byte count read and write of its table slot.
        # The kernel that does those N table updates is the per-bin count (it keeps the table in shared
        # memory); its share of B_alg is N*(Kb+8). Its own HBM input/output is reported beside it.
        survey_bytes = N * (Kb + 8) * a.steps if dom_name == "smem_count_per_bin" else dom_bytes
        achieved = survey_bytes / (dom_ms * 1e-3) / 1e9 if dom_ms > 0 else 0.0
        io_achieved = dom_bytes / (dom_ms * 1e-3) / 1e9 if dom_ms > 0 else 0.0
        traffic, traffic_src = None, None
        try:
            with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
                tj = json.load(f)
            ent = tj.get("%s/%s/k%d/R%d/G%d/z%d" % (method_used, dom_name, k, R, a.cfg["genome"], a.cfg["zipf_loci"]))
            if ent:
                traffic, traffic_src = ent["dram_bytes_per_launch"], ent["source"]
        except Exception:
            pass
        b_alg = R * L + N * (Kb + 8) + U * S
        # (several runs per GPU: the step also merges them -- the whole step counts)
        path_ms = ms_per_step if world > 1 or job.runs > 1 else (tot_ms / a.steps if tot_ms > 0 else ms_per_step)
        path_ach = b_alg / (path_ms * 1e-3) / 1e9
        line = {
            "metric": metric_for(k), "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u%d" % (64 * counter.words), "data": "synthetic",
            "config": dict(workload(a, world, job.mode), method=method_used,
                           exchange=None if world == 1 else
                           "fused into the consuming kernels: the per-bin count loads every rank's super-window records of its bins, "
                           "the level-2 placement loads its key range of every rank's distinct records (peer memory over NVLink, CUDA IPC)"),
            "parity": parity,
            "bases_per_s": R * L * world / (ms_per_step * 1e-3),
            "distinct_per_gpu": U,
            "roofline": {"bound": "hbm", "kernel": dom_name,
                         "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak if peak else None,
                         "definition": "SURVEY 8(d) algorithmic bytes of the kernel's work: N*(Kb+8) for the per-bin count "
                                       "(one key read + count read/write per k-mer occurrence; the table lives in shared memory), "
                                       "the stage's HBM input+output for any other kernel",
                         "hbm_io_achieved": io_achieved, "hbm_io_frac": io_achieved / peak if peak else None,
                         "hbm_io_bytes_per_launch": dom_bytes / max(dom_launch, 1),
                         "peak_source": peak_src + " HBM copy bandwidth (MEASURED_PEAKS.json)",
                         "bytes_per_launch": survey_bytes / max(dom_launch, 1), "launches_per_step": dom_launch / a.steps,
                         "ms_per_launch": dom_ms / max(dom_launch, 1),
                         "share_of_step": dom_ms / (path_ms * a.steps) if path_ms else None, "traffic": traffic,
                         "traffic_source": traffic_src},
            "path_roofline": {"bound": "hbm", "b_alg_bytes": b_alg, "achieved": path_ach, "peak": peak, "unit": "GB/s",
                              "frac": path_ach / peak if peak else None, "ms": path_ms,
                              "definition": "SURVEY 8(d): B_in + N*(Kb+8) + U*S per GPU over the step time (device time of the "
                                            "counting path on one GPU; the whole step, exchange included, for N > 1)"},
            "counts_per_step": acc["counts"] / a.steps,
            "merge_ms_per_step": (ms_per_step - tot_ms / a.steps) if job.runs > 1 and world == 1 else None,
            "stages_last_step": {n: round(m, 4) for n, m in zip(names, st1["ms_stage"])},
            "stage_hbm_io_bytes_last_step": {n: int(b) for n, b in zip(names, st1["stage_bytes"])},
            "nvlink": nvlink,
            "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
            "wall_ms_per_step": wall / a.steps * 1e3,
        }
        if not a.no_cpu_baseline and world == 1:
            line["cpu_baseline"] = cpu_baseline(a)
        print(json.dumps(line), flush=True)
    counter.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_e2e(job, a, distinct, kmers_step, barrier, numa):
    """K steps through the host-buffer API: pinned reads -> H2D -> count -> records D2H into pinned memory."""
    import queue
    torch, dist = job.torch, job.dist
    counter, world, rank, dev = job.counter, job.world, job.rank, job.dev
    n_bytes, R, nk = job.n_bytes, job.R, job.nk
    host_reads = job.d_reads[:n_bytes].cpu().numpy()
    for sl in range(E2E_SLOTS):                         # every pinned input slot holds the step's reads
        counter.slot_buffer(sl)[:n_bytes] = host_reads
    out_cap = (distinct + distinct // 4 + 4096) * counter.record_size
    pinned_out = counter.host_alloc(out_cap)
    parts = {"h2d_count": 0.0, "records_d2h": 0.0}

    if world == 1:
        def one(sl):
            t_a = time.perf_counter()
            counter.submit(sl, n_bytes)
            run = counter.wait(sl)
            t_b = time.perf_counter()
            nb = run.copy_into(pinned_out.ctypes.data, out_cap)
            run.free()
            parts["h2d_count"] += t_b - t_a
            parts["records_d2h"] += time.perf_counter() - t_b
            return nb
    else:
        def one(sl):
            t_a = time.perf_counter()
            counter.accum_submit(sl, n_bytes)
            run = job.exchange.finish()
            t_b = time.perf_counter()
            nb = run.copy_into(pinned_out.ctypes.data, out_cap)
            run.free()
            parts["h2d_count"] += t_b - t_a
            parts["records_d2h"] += time.perf_counter() - t_b
            return nb

    # (1) one step at a time: the latency of a single chunk, with its parts
    for _ in range(2):
        one(0)
    for kx in parts:
        parts[kx] = 0.0
    barrier()
    t0 = time.perf_counter()
    d2h = 0
    for _ in range(a.steps):
        d2h = one(0)
    barrier()
    single_ms = (time.perf_counter() - t0) / a.steps * 1e3
    parts_ms = {kx: v / a.steps * 1e3 for kx, v in parts.items()}
    # (2) the reported number: the same K steps pipelined, which is how the API is meant to be driven: the
    # records are read back by a consumer thread (kc_run_copy_records on its own stream) while the producer
    # is already submitting the next step.
    todo, res = queue.Queue(maxsize=1), {"nb": 0, "err": None}

    def reader():
        while True:
            run = todo.get()
            if run is None:
                return
            try:
                res["nb"] = run.copy_into(pinned_out.ctypes.data, out_cap)
                run.free()
            except Exception as e:
                res["err"] = e

    if world == 1:
        # kc_submit / kc_wait over the pinned slots: H2D of step i, the kernels of step i-1 and the records
        # D2H of step i-2 overlap
        def pipelined(n_steps):
            th = threading.Thread(target=reader, daemon=True)
            th.start()
            for i in range(n_steps + 1):
                if i < n_steps:
                    counter.submit(i % E2E_SLOTS, n_bytes)
                if i >= 1:
                    todo.put(counter.wait((i - 1) % E2E_SLOTS))
            todo.put(None)
            th.join()
            if res["err"] is not None:
                raise res["err"]

        timing = ("wall clock around K steps pipelined over %d pinned slots (kc_submit/kc_wait, records read back by a consumer "
                  "thread), sync on both sides; every step copies its reads H2D and its records D2H" % E2E_SLOTS)
    else:
        # exchange: the bins are shared by the ranks, so step i+1's reads are submitted once step i's exchange
        # has returned (every peer has read this rank's bins by then); the records D2H of step i overlaps the
        # H2D and the kernels of step i+1
        def pipelined(n_steps):
            th = threading.Thread(target=reader, daemon=True)
            th.start()
            for i in range(n_steps):
                counter.accum_submit(i % E2E_SLOTS, n_bytes)
                todo.put(job.exchange.finish())
            todo.put(None)
            th.join()
            if res["err"] is not None:
                raise res["err"]

        timing = ("wall clock around K steps (kc_accum_submit -> exchange over NVLink -> kc_run_copy_records by a consumer thread: "
                  "the records D2H of step i overlaps step i+1), sync on both sides, max over ranks; every step copies its reads "
                  "H2D and its records D2H")
    pipelined(max(a.warmup, 2 * E2E_SLOTS))
    barrier()
    t0 = time.perf_counter()
    pipelined(a.steps)
    d2h = res["nb"]
    barrier()
    e2e_dt = (time.perf_counter() - t0) / a.steps
    t = torch.tensor([e2e_dt, single_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_dt, single_ms = float(t[0].item()), float(t[1].item())
    out = {"value": kmers_step / e2e_dt, "unit": UNIT, "h2d_bytes_per_step": n_bytes, "d2h_bytes_per_step": int(d2h),
           "ms_per_step": e2e_dt * 1e3, "timing": timing,
           "pcie_gbs": {"h2d": n_bytes / e2e_dt / 1e9, "d2h": d2h / e2e_dt / 1e9},
           "single_step_ms": single_ms, "single_step_value": kmers_step / (single_ms * 1e-3),
           "single_step_parts_ms_rank0": parts_ms, "cpus_bound_near_gpu": numa}
    counter.host_free(pinned_out)
    return out


def run_merge_bench(a):
    """kc_merge_runs (merge path, KMerFileMerger.cpp:49-135) over `runs` sorted unique runs, each the count of
    `reads` reads of the workload (consecutive read ranges, so the runs overlap like chunks of one input do).
    Algorithmic bytes per pairwise merge: S*(nA + nB) in, S*U out; a tree of log2(runs) levels."""
    import torch
    import kmer_counter_b200 as kc
    from kmer_counter_b200 import synth
    import oracle
    c, L = a.cfg, a.read_len
    k, R, runs = c["k"], c["reads"], max(2, c["runs"])
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    stream = torch.cuda.Stream(device=dev, priority=-1)
    torch.cuda.set_stream(stream)
    counter = kc.Counter(k, L, device=0, method=a.method, stream=stream.cuda_stream)
    S = counter.record_size
    parts = []
    d = torch.empty(R * L + 256, dtype=torch.uint8, device=dev)
    for i in range(runs):
        synth.synth_reads_device(d.data_ptr(), R, L, c["genome"], c["sub_rate"], c["n_rate"], c["seed"], first_read=i * R,
                                 zipf_loci=c["zipf_loci"], stream=stream.cuda_stream)
        parts.append(counter.count_device(d.data_ptr(), R * L))
    del d
    n_in = sum(len(p) for p in parts)
    # parity on a small instance of the same shape: merge of the runs of 4 x 20k reads against the oracle's merger
    small = [oracle.gen_reads(20000, L, c["genome"], c["sub_rate"], c["n_rate"], seed=c["seed"], first_read=i * 20000) for i in range(4)]
    sruns = [counter.upload_run(oracle.process_chunk(x, L, k)) for x in small]
    mg = counter.merge(sruns)
    import numpy as np
    want = oracle.count(np.concatenate(small), L, k, chunk_reads=20000)
    ok = mg.to_bytes() == want
    mg.free()
    for r in sruns:
        r.free()
    if not ok:
        sys.stderr.write("bench.py: merge PARITY FAILED\n")
        sys.exit(3)
    for _ in range(a.warmup):
        counter.merge(parts).free()
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(0) as clk:
        ev0.record(stream)
        for i in range(a.steps):
            m = counter.merge(parts)
            U = len(m)
            if a.dump_outputs is None or i + 1 < a.steps:
                m.free()
        ev1.record(stream)
        torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1) / a.steps
    if a.dump_outputs is not None:
        dump_run(m, a.dump_outputs, dev, DUMP_BYTES)
        m.free()
    peak, peak_src = measured_peak_gbs()
    # bytes of the tree: every level reads its inputs and writes its outputs once
    sizes, tree_bytes = [len(p) for p in parts], 0
    # (upper bound on the intermediate sizes: what the final level reads is at least U; use measured sizes of the first level
    #  and U for the last when runs == 2)
    if runs == 2:
        tree_bytes = S * (n_in + U)
    line = {"bench": "merge", "metric": "records merged/s (kc_merge_runs: merge path summing counts)", "unit": "records/s",
            "value": n_in / (ms * 1e-3), "ms_per_merge": ms, "runs": runs, "records_in": n_in, "records_out": U,
            "record_bytes": S, "steps": a.steps, "warmup": a.warmup, "parity": {"checked": True, "ok": True,
            "what": "4 runs of 20k reads merged on the GPU == oracle.count of the 80k reads"},
            "config": workload(a, 1, "merge"), "clocks": clk.summary()}
    if runs == 2:
        ach = tree_bytes / (ms * 1e-3) / 1e9
        line["roofline"] = {"bound": "hbm", "kernel": "merge_tile_kernel", "achieved": ach, "peak": peak, "unit": "GB/s",
                            "frac": ach / peak, "bytes_per_launch": tree_bytes, "definition": "S*(nA+nB) read + S*U written over the "
                            "device time of kc_merge_runs (partition + tile kernels, allocation and the count read-back included)",
                            "peak_source": peak_src + " HBM copy bandwidth (MEASURED_PEAKS.json)"}
    print(json.dumps(line), flush=True)
    for p in parts:
        p.free()
    counter.close()


def main():
    a = parse_args()
    if a.bench == "merge" and a.impl == "ours":
        run_merge_bench(a)
        return
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if a.impl == "reference":
        run_reference(a, rank)
        return
    if world != a.gpus and world == 1 and a.gpus > 1:
        sys.stderr.write("bench.py: --gpus %d needs torchrun (WORLD_SIZE=%d)\n" % (a.gpus, world))
        sys.exit(2)
    run_ours(a, rank, world, local_rank)


if __name__ == "__main__":
    main()
