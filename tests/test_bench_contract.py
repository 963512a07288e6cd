"""bench.py's contract: on a box without a GPU, the reference arm prints exactly one JSON line with
the keys the driver reads, and workloads that are not a BASELINE configuration say so; on the GPU,
--dump-outputs writes the run the last timed step computed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [x for x in r.stdout.splitlines() if x.strip()]
    assert len(lines) == 1, lines                      # the reference's own chatter goes to stderr
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "k-mers counted/s at k=31" and d["unit"] == "kmers/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["n_gpus"] == 1 and d["steps"] == 1
    assert d["config"]["workload"].startswith("configs[1]")
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == d["value"]
    assert set(cb["stage_seconds_last_step"]) >= {"sort_thread_s", "merge_wall_s"} or cb["kind"] == "port"
    assert d["e2e"] == {"value": d["value"], "unit": "kmers/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1"],
                       capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_overridden_workloads_are_labelled():
    sys.path.insert(0, ROOT)
    import bench
    argv = sys.argv
    try:
        sys.argv = ["bench.py", "--k", "96"]
        a = bench.parse_args()
        assert a.cfg["k"] == 96 and "k=96" in a.cfg["name"] and "configs[" not in a.cfg["name"]
        assert bench.metric_for(96) == "k-mers counted/s at k=96" and bench.metric_for(31) == bench.METRIC
        sys.argv = ["bench.py", "--config", "c3"]
        a = bench.parse_args()
        assert a.cfg["name"].startswith("configs[2]") and a.cfg["k"] == 63 and a.cfg["reads"] == 200_000_000
    finally:
        sys.argv = argv


def test_steps_and_dump_outputs_arguments_are_checked():
    sys.path.insert(0, ROOT)
    import bench
    argv = sys.argv
    try:
        for args in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]):
            sys.argv = ["bench.py"] + args
            with pytest.raises(SystemExit):
                bench.parse_args()
        sys.argv = ["bench.py", "--steps", "7", "--dump-outputs", "out"]
        a = bench.parse_args()
        assert a.steps == 7 and a.dump_outputs == "out"
    finally:
        sys.argv = argv


def _dumped_records(d, suffix=""):
    """The .npy files of --dump-outputs -> (keys[m, W] uint64, counts[m], record_index[m], run_summary)."""
    load = lambda name: np.load(os.path.join(d, name + suffix + ".npy"))
    halves, counts, idx, summary = load("keys"), load("counts"), load("record_index"), load("run_summary")
    assert all(x.dtype == np.float64 for x in (halves, counts, idx, summary))
    keys = (halves[:, 0::2].astype(np.uint64) << np.uint64(32)) | halves[:, 1::2].astype(np.uint64)
    return keys, counts.astype(np.uint32), idx.astype(np.int64), summary


@pytest.mark.gpu
def test_dump_outputs_writes_the_last_steps_run(tmp_path):
    """A small c2-shaped workload: the files hold every record of the run, equal to the oracle's artefact,
    and --steps sets the number of timed steps."""
    import oracle
    R = 10000
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--reads", str(R), "--steps", "3", "--warmup", "1",
                        "--no-cpu-baseline", "--no-e2e", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == 3 and line["parity"]["ok"]
    want = oracle.count(oracle.gen_reads(R, 100, 100_000_000, 1e-3, 0.0, seed=2), 100, 31)
    wk, wc = oracle.records_to_arrays(want, 31)
    keys, counts, idx, summary = _dumped_records(str(tmp_path))
    assert list(summary) == [len(wk), R * (100 - 31 + 1)]
    assert (idx == np.arange(len(wk))).all() and (keys == wk).all() and (counts == wc).all()


@pytest.mark.gpu
@pytest.mark.parametrize("k", [31, 96])
def test_dump_run_samples_large_runs(tmp_path, k):
    """A run over the byte budget is sampled at seeded record indices: the same sample every time, and
    every sampled row is the run's record at that index."""
    import torch
    import bench
    import kmer_counter_b200 as kc
    import oracle
    L = 100
    reads = oracle.gen_reads(3000, L, 50000, 0.01, 0.002, seed=4)
    wk, wc = oracle.records_to_arrays(oracle.process_chunk(reads, L, k), k)
    W = wk.shape[1]
    budget = 8 * (2 * W + 2) * 1000
    dev = torch.device("cuda", 0)
    d_reads = torch.from_numpy(reads).to(dev)
    with kc.Counter(k, L) as c:
        run = c.count_device(d_reads.data_ptr(), reads.size)
        for d in ("a", "b"):
            bench.dump_run(run, str(tmp_path / d), dev, budget)
        run.free()
    keys, counts, idx, summary = _dumped_records(str(tmp_path / "a"))
    assert len(wk) > 1000 >= len(idx) > 900 and (np.diff(idx) > 0).all()
    assert (keys == wk[idx]).all() and (counts == wc[idx]).all()
    assert list(summary) == [len(wk), int(wc.astype(np.int64).sum())]
    for name in ("keys", "counts", "record_index", "run_summary"):
        assert (tmp_path / "a" / (name + ".npy")).read_bytes() == (tmp_path / "b" / (name + ".npy")).read_bytes()
