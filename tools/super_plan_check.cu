// super_plan_check.cu -- host only, no GPU needed: the super-window plans of long reads, and S1's shared
// memory recomputed from each plan as super_scatter lays it out. Every plan super_plan accepts must fit
// S1's 200 KiB; prints the shapes of profiles/read-lengths/INDEX.md and the longest read per k.
//   nvcc -gencode arch=compute_100a,code=sm_100a -std=c++17 -I../kmer-counter_b200/csrc super_plan_check.cu \
//        -L../kmer-counter_b200 -lkc_b200 -Xlinker -rpath=$PWD/../kmer-counter_b200 -o super_plan_check
#include <cstdio>

#include "kc_internal.h"
#include "kc_super.cuh"

using namespace kc;

static unsigned s1_smem(const SuperPlan &pl) {
    ExtractParams ep;
    if (!extract_plan((void *)16, 16, pl.L, pl.k, pl.flags, nullptr, &ep, 4800)) return ~0u;
    const unsigned h = (ep.smem_total + 15u) & ~15u;
    return h + ep.tile_reads * pl.nh_stride * 4 + ep.tile_reads * pl.nk * 4 + 2 * ep.tile_reads * pl.segs_per_read * 4;
}

int main() {
    struct C { const char *what; unsigned k, L, flags; unsigned long long reads; unsigned occ; double head; bool ext; } cs[] = {
        {"one window", 22, 1140, 0, 1, 0, 0, false},
        {"chunk, occ 64", 22, 1140, 0, 5000, 64, 0, false}, {"chunk, occ 64, canon", 22, 1140, 2, 5000, 64, 0, false},
        {"chunk, occ 64", 24, 1150, 0, 5000, 64, 0, false}, {"chunk, occ 64", 28, 1170, 0, 20000, 64, 0, false},
        {"chunk, default", 22, 1140, 0, 660000, 0, 0, false}, {"accumulate, default", 22, 1140, 0, 660000, 0, 0, true},
        {"exchange 2 ranks", 22, 1140, 0, 330000, 4096, 0.25, false}, {"chunk, occ 64", 22, 1139, 0, 5000, 64, 0, false},
        {"C2", 31, 100, 0, 10000000, 0, 0, false}, {"C3", 63, 100, 0, 200000000, 0, 0, true},
        {"C4 accumulate", 31, 100, 0, 1000000000, 0, 0, true}};
    for (const C &c : cs) {
        SuperPlan p;
        const bool ok = super_plan(c.k, c.L, c.flags, c.reads * (c.L - c.k + 1), c.occ, &p, c.head, 0, c.ext);
        printf("%-22s k=%u L=%u flags=%u reads=%llu occ=%u: %s bins=%u m=%u S1 smem=%u\n", c.what, c.k, c.L, c.flags,
               c.reads, c.occ, ok ? "planned" : "refused", ok ? p.n_bins : 0, ok ? p.m : 0, ok ? s1_smem(p) : 0);
    }
    unsigned over = 0;
    for (unsigned flags = 0; flags < 3; flags++)
        for (unsigned k = 22; k <= 64; k++) {
            unsigned longest = 0;
            for (unsigned L = k; L <= 4096; L++) {
                for (unsigned long long windows : {1ull, 1ull << 22, 1ull << 26, 1ull << 30, 1ull << 34})
                    for (unsigned occ : {0u, 16u, 64u}) {
                        SuperPlan p;
                        if (!super_plan(k, L, flags, windows, occ, &p)) continue;
                        if (windows == 1 && occ == 0) longest = L;
                        if (s1_smem(p) > 200 * 1024) over++;
                    }
            }
            if (flags == 0) printf("k=%u: reads of up to %u bases\n", k, longest);
        }
    printf("accepted plans whose S1 exceeds 200 KiB: %u\n", over);
    return over != 0;
}
