// Options.h -- the reference's key=value flags (main.cpp:25-70, Options.h:26-43).
#pragma once

#include <stdint.h>

#include <string>

struct Options {
    std::string inputFileDirectory;           // inputFileLocation=
    std::string tempFileLocation = "/tmp";    // tempFileLocation=   (run spill directory)
    std::string outputFile = "output.bin";    // outputFile=
    int64_t gpuMemoryLimit = 100000000;       // gpuMemoryLimit=     (main.cpp:28)
    int64_t kmerLength = 32;                  // kmerLength=         (Options.cpp default)
    uint32_t noOfMergersAtOnce = 2;           // noOfMergersAtOnce=
    uint32_t noOfMergeThreads = 2;            // noOfMergeThreads=   (0: merge inside the producer loop; >= 1: merges run on a
                                              // background thread while chunks are counted -- the GPU serialises them)
    // additions
    std::string method = "auto";              // method=auto|sort|hash
    std::string compat = "ref";               // compat=ref|strict
    bool canonical = false;                   // canonical=1: count each k-mer with its reverse complement under
                                              // min(x, rc(x)) (KC_CANONICAL, implies compat=strict)
    int device = 0;                           // device=
    bool keepRuns = false;                    // keepRuns=1: also write every chunk's run to tempFileLocation/<id>
    int64_t runBudget = 0;                    // runBudget=BYTES: a merged run larger than this is spilled to pinned host
                                              // memory and the final merge runs out of core, range by range (0 = never)
    int gpus = 1;                             // gpus=N: N contexts on devices device .. device+N-1; reads are dealt to them
                                              // chunk by chunk, super-window records and distinct records are exchanged
                                              // over NVLink inside the counting kernels (kc_xchg_*)
    std::string mode = "auto";                // mode=auto|accumulate|runs: accumulate = chunks are only packed into
                                              // super-window records, one count at the end (k <= 64); runs = one sorted run
                                              // per chunk, merged on the GPU (the reference's shape; keepRuns, runBudget)
    int64_t expectedReads = 0;                // expectedReads=: plan the accumulator for this many reads (0 = from file sizes)
    std::string parser = "gpu";               // parser=gpu|host: where FASTQ text is parsed (gpu falls back to host
                                              // for input that is not plain 4-line fixed-length FASTQ)
    int64_t minCount = -1;                    // minCount=N / maxCount=N: the artefact keeps only k-mers whose final
    int64_t maxCount = -1;                    // count is in [minCount, maxCount] (KMC -ci/-cx, Jellyfish -L/-U); -1 = no bound
    std::string histoFile;                    // histoFile=PATH: the count spectrum of the final (unfiltered) counts as
                                              // "c n" lines, c = 1..histoMax with n > 0; the histoMax line means >= histoMax
    int64_t histoMax = 10000;                 // histoMax=N (Jellyfish's default high)

    // Same prefix matching as the reference. Unknown tokens are ignored, as there.
    static Options parse(int argc, char **argv);
    bool filtering() const { return minCount >= 0 || maxCount >= 0; }
    // KMerCounter::GetChunkSize (KMerCounter.cpp:193-212): bytes of reads per chunk
    int64_t chunkSize(int64_t lineLength) const;
};
