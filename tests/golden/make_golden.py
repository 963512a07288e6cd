"""Generates tests/golden/*.json|bin from the REFERENCE'S OWN code (oracle/_ref, built from
/root/reference by oracle/build_ref.sh).  Run in the build container only; the outputs are
committed so that the GPU box (which has no /root/reference) can check against them.

    python tests/golden/make_golden.py
"""
import hashlib
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import numpy as np  # noqa: E402
import oracle  # noqa: E402

assert oracle.ref_available(), "build oracle/_ref first (bash oracle/build_ref.sh)"


def hexkeys(data, k):
    keys, counts = oracle.records_to_arrays(data, k)
    return [[["%016x" % int(w) for w in row], int(c)] for row, c in zip(keys, counts)]


# known-answer reads of SURVEY.md Appendix A.4, answered by the reference's kernels
kat = {"source": "reference kernels via oracle/_ref (bitEncode + extractKMers + reduceKMers, no sort)", "cases": []}
for read, ks in [("ACGTACGTACGTACGTACGTACGTACGTACGTTTGGCCAAC", [31, 32, 28, 33, 5, 29, 30]),
                 ("ACGTNACGTACG", [5, 3, 1]),
                 ("ACGT" * 18, [63, 61, 60, 64, 33]),
                 ("TTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTT", [31, 32]),
                 ("AAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAANAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAA", [31])]:
    for k in ks:
        raw = oracle.ref_process_chunk(read.encode(), len(read), k, do_sort=False)
        kat["cases"].append({"read": read, "k": k, "records_unsorted_reduced": hexkeys(raw, k)})
json.dump(kat, open(os.path.join(HERE, "kat.json"), "w"), indent=1)

# seeded chunks: sha256 of the reference's Pipeline-B artefact (sorted, reduced, merged)
fix = {"source": "reference Pipeline B via oracle/_ref (ref_count_packed: kernels, std::sort with the reference "
                 "comparators, reduceKMers, FileDump, KMerFileMerger)", "cases": []}
import tempfile
for (R, L, k, G, e, n, seed, chunk) in [(3000, 100, 31, 40000, 0.01, 0.002, 11, 700),
                                        (1500, 100, 63, 20000, 0.005, 0.001, 12, 400),
                                        (800, 150, 96, 6000, 0.01, 0.01, 13, 300),
                                        (800, 150, 128, 6000, 0.01, 0.0, 14, 800),
                                        (2000, 41, 28, 0, 0.0, 0.01, 15, 333),
                                        (2000, 100, 32, 30000, 0.0, 0.0, 16, 2000),
                                        (20000, 100, 31, 200000, 0.001, 0.001, 17, 4096)]:
    reads = oracle.gen_reads(R, L, G, e, n, seed=seed)
    with tempfile.TemporaryDirectory() as d:
        out = os.path.join(d, "out.bin")
        oracle.ref_count_packed(reads, L, k, chunk, 2, d, out)
        data = open(out, "rb").read()
    fix["cases"].append({"reads": R, "L": L, "k": k, "genome": G, "sub": e, "n": n, "seed": seed, "chunk_reads": chunk,
                         "reads_sha256": hashlib.sha256(reads.tobytes()).hexdigest(),
                         "records": len(data) // oracle.record_size(k),
                         "artefact_sha256": hashlib.sha256(data).hexdigest()})
json.dump(fix, open(os.path.join(HERE, "pipeline_b.json"), "w"), indent=1)

# a small artefact kept in full (bytes), for format-level tests
reads = oracle.gen_reads(200, 60, 3000, 0.01, 0.01, seed=21)
open(os.path.join(HERE, "small_reads_L60.bin"), "wb").write(reads.tobytes())
with tempfile.TemporaryDirectory() as d:
    out = os.path.join(d, "out.bin")
    oracle.ref_count_packed(reads, 60, 31, 64, 1, d, out)
    open(os.path.join(HERE, "small_k31.records"), "wb").write(open(out, "rb").read())
    oracle.ref_count_packed(reads, 60, 40, 64, 1, d, out)
    open(os.path.join(HERE, "small_k40.records"), "wb").write(open(out, "rb").read())

# sha256 of the reference's outputs on the inputs of test_oracle.py's reference comparisons
sys.path.insert(0, os.path.dirname(HERE))
import test_oracle  # noqa: E402

sha = lambda b: hashlib.sha256(bytes(b)).hexdigest()
dig = {"source": "reference build via oracle/_ref (ref_process_chunk, ref_count_packed, ref_read_fastq_dir)",
       "chunks": {}, "random_shapes": []}
for (R, L, k, G, e, n) in test_oracle.REFERENCE_CASES:
    reads = oracle.gen_reads(R, L, G, e, n, seed=1000 + R + k)
    with tempfile.TemporaryDirectory() as d:
        out = os.path.join(d, "out.bin")
        oracle.ref_count_packed(reads, L, k, max(1, R // 5), 2, d, out)
        art = open(out, "rb").read()
    dig["chunks"][test_oracle.case_key(R, L, k, G, e, n)] = {
        "reads_sha256": sha(reads), "sorted_sha256": sha(oracle.ref_process_chunk(reads, L, k, True)),
        "unsorted_sha256": sha(oracle.ref_process_chunk(reads, L, k, False)), "artefact_sha256": sha(art)}
for L, k, R, reads in test_oracle.random_shapes():
    dig["random_shapes"].append({"L": L, "k": k, "R": R, "reads_sha256": sha(reads),
                                 "sorted_sha256": sha(oracle.ref_process_chunk(reads, L, k, True)),
                                 "unsorted_sha256": sha(oracle.ref_process_chunk(reads, L, k, False))})
fq = oracle.gen_fastq(50, 100, 5000, 0.01, 0.01, seed=3)
with tempfile.TemporaryDirectory() as d:
    open(os.path.join(d, "a.fastq"), "wb").write(fq)
    data, L = oracle.ref_read_fastq_dir(d)
dig["fastq_reader"] = {"fastq_sha256": sha(fq), "L": L, "sha256": sha(data)}
json.dump(dig, open(os.path.join(HERE, "reference_digests.json"), "w"), indent=1)
print("golden vectors written to", HERE)
