#include "Options.h"

#include <stdlib.h>
#include <string.h>

static bool take(const char *arg, const char *key, const char **value) {
    size_t n = strlen(key);
    if (strncmp(arg, key, n) != 0) return false;
    *value = arg + n;
    return true;
}

Options Options::parse(int argc, char **argv) {
    Options o;
    for (int i = 1; i < argc; i++) {
        const char *v = nullptr;
        if (take(argv[i], "kmerLength=", &v)) o.kmerLength = strtoll(v, nullptr, 10);
        else if (take(argv[i], "gpuMemoryLimit=", &v)) o.gpuMemoryLimit = strtoll(v, nullptr, 10);
        else if (take(argv[i], "inputFileLocation=", &v)) o.inputFileDirectory = v;
        else if (take(argv[i], "tempFileLocation=", &v)) o.tempFileLocation = v;
        else if (take(argv[i], "outputFile=", &v)) o.outputFile = v;
        else if (take(argv[i], "noOfMergersAtOnce=", &v)) o.noOfMergersAtOnce = (uint32_t)atoi(v);
        else if (take(argv[i], "noOfMergeThreads=", &v)) o.noOfMergeThreads = (uint32_t)atoi(v);
        else if (take(argv[i], "method=", &v)) o.method = v;
        else if (take(argv[i], "compat=", &v)) o.compat = v;
        else if (take(argv[i], "canonical=", &v)) o.canonical = atoi(v) != 0;
        else if (take(argv[i], "device=", &v)) o.device = atoi(v);
        else if (take(argv[i], "keepRuns=", &v)) o.keepRuns = atoi(v) != 0;
        else if (take(argv[i], "parser=", &v)) o.parser = v;
        else if (take(argv[i], "gpus=", &v)) o.gpus = atoi(v);
        else if (take(argv[i], "mode=", &v)) o.mode = v;
        else if (take(argv[i], "expectedReads=", &v)) o.expectedReads = strtoll(v, nullptr, 10);
        else if (take(argv[i], "runBudget=", &v)) o.runBudget = strtoll(v, nullptr, 10);
        else if (take(argv[i], "minCount=", &v)) o.minCount = strtoll(v, nullptr, 10);
        else if (take(argv[i], "maxCount=", &v)) o.maxCount = strtoll(v, nullptr, 10);
        else if (take(argv[i], "histoFile=", &v)) o.histoFile = v;
        else if (take(argv[i], "histoMax=", &v)) o.histoMax = strtoll(v, nullptr, 10);
    }
    if (o.noOfMergersAtOnce < 2) o.noOfMergersAtOnce = 2;
    if (o.gpus < 1) o.gpus = 1;
    if (o.gpus > 8) o.gpus = 8;
    if (o.histoMax < 1) o.histoMax = 1;
    if (o.histoMax > (1 << 24) - 1) o.histoMax = (1 << 24) - 1;
    return o;
}

// The reference sizes a chunk so that its raw per-occurrence records fit the "GPU memory
// limit": 8 bytes per started 32 bases plus 8 for the count, per k-mer slot.
int64_t Options::chunkSize(int64_t lineLength) const {
    int64_t keyBytes = (kmerLength + 3) / 4;
    int64_t words = (keyBytes + 7) / 8 + 1;
    int64_t perRead = words * 8 * (lineLength - kmerLength + 1);
    if (perRead <= 1) return lineLength;
    int64_t reads = (gpuMemoryLimit - lineLength) / (perRead - 1);
    if (reads < 1) reads = 1;
    return lineLength * reads;
}
