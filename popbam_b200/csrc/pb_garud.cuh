// pb_garud.cuh -- Garud's H statistics per (window, population) (PB_AN_GARUD; include/popbam_b200.h, pb_region_garud).
// No reference counterpart; restated in plain C by tests/garud_oracle.c.
//
// Samples i and j carry the same haplotype in a window iff bit i equals bit j in every segregating-site type of the
// window.  eq[i] = the samples that agree with sample i at every site, so the identity classes of population p are the
// distinct eq[i] & pop_mask[p] over its members i; the class of i is represented by its lowest sample.
//
// One CTA of PB_GARUD_WARPS warps per window.
//   Phase 1: lane l keeps eq[l] and eq[l + 32], starting from the all-samples mask.  The warps stride over the window's
//            sites in coalesced chunks of 32 words; each word is broadcast by shuffle and every lane applies
//            eq[i] &= (t >> i & 1) ? t : ~t.
//   Phase 2: the warps' eq arrays are AND-reduced in shared memory (exact and order-free).
//   Phase 3: one warp per population: class sizes popc(r), r = eq[i] & pop_mask[p], counted at the representatives
//            i == ctz(r); warp sums give n_hap and hh = sum c^2, three rounds of warp max on (size, sample) keys give
//            c1 >= c2 >= c3.  Lane 0 writes the integers and the four ratios.
// The window's site count and offset are read from device memory, so the kernel runs unchanged when the host does not
// know the number of segregating sites (asynchronous regions).  No atomics.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define PB_GARUD_WARPS 8

struct PbGarudArgs {
    int n, P;
    uint64_t pop_mask[64];
    int32_t pop_nsmpl[64];
    const int32_t *segsites;
    const int64_t *seg_off;
    const uint64_t *seg_type;
    int32_t *n_hap, *c1, *c2, *c3, *hh;           // [NW*P], index w*P + p
    double *h1, *h12, *h123, *h2h1;
};

__global__ void __launch_bounds__(PB_GARUD_WARPS * 32) k_garud(const PbGarudArgs a) {
    __shared__ uint64_t s_eq[PB_GARUD_WARPS][64];
    const int w = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint64_t all = a.n >= 64 ? ~0ull : (1ull << a.n) - 1;
    const uint64_t *__restrict__ T = a.seg_type + a.seg_off[w];
    const int S = a.segsites[w];
    uint64_t e0 = all, e1 = all;                  // eq[lane], eq[lane + 32]
    for (int base = warp * 32; base < S; base += PB_GARUD_WARPS * 32) {
        const uint64_t mine = base + lane < S ? T[base + lane] : 0;
        const int cnt = min(32, S - base);
        for (int k = 0; k < cnt; ++k) {
            const uint64_t t = __shfl_sync(0xffffffffu, mine, k);
            e0 &= (t >> lane & 1) ? t : ~t;
            e1 &= (t >> (lane + 32) & 1) ? t : ~t;
        }
    }
    s_eq[warp][lane] = e0;
    s_eq[warp][lane + 32] = e1;
    __syncthreads();
    if (threadIdx.x < 64) {
        uint64_t e = s_eq[0][threadIdx.x];
        for (int k = 1; k < PB_GARUD_WARPS; ++k) e &= s_eq[k][threadIdx.x];
        s_eq[0][threadIdx.x] = e;
    }
    __syncthreads();
    for (int p = warp; p < a.P; p += PB_GARUD_WARPS) {
        const uint64_t mask = a.pop_mask[p];
        // key = size * 64 + sample of every class representative held by this lane (0: none); unique per class
        unsigned k0 = 0, k1 = 0;
        int reps = 0, sq = 0;
        if (mask >> lane & 1) {
            const uint64_t r = s_eq[0][lane] & mask;
            if (__ffsll((long long)r) - 1 == lane) { const int c = __popcll(r); k0 = (unsigned)(c * 64 + lane); reps += 1; sq += c * c; }
        }
        if (mask >> (lane + 32) & 1) {
            const uint64_t r = s_eq[0][lane + 32] & mask;
            if (__ffsll((long long)r) - 1 == lane + 32) { const int c = __popcll(r); k1 = (unsigned)(c * 64 + lane + 32); reps += 1; sq += c * c; }
        }
        const int nh = (int)__reduce_add_sync(0xffffffffu, (unsigned)reps);
        const int h = (int)__reduce_add_sync(0xffffffffu, (unsigned)sq);
        int top[3];
        for (int q = 0; q < 3; ++q) {
            const unsigned m = __reduce_max_sync(0xffffffffu, max(k0, k1));
            top[q] = (int)(m >> 6);
            if (k0 == m) k0 = 0;
            if (k1 == m) k1 = 0;
        }
        if (lane == 0) {
            const size_t x = (size_t)w * a.P + p;
            const int n = a.pop_nsmpl[p], c1 = top[0], c2 = top[1], c3 = top[2];
            a.n_hap[x] = nh; a.c1[x] = c1; a.c2[x] = c2; a.c3[x] = c3; a.hh[x] = h;
            if (n < 2) {
                a.h1[x] = a.h12[x] = a.h123[x] = a.h2h1[x] = nan("");
            } else {
                const double nn = (double)(n * n);
                a.h1[x] = (double)h / nn;
                a.h12[x] = (double)(h + 2 * c1 * c2) / nn;
                a.h123[x] = (double)(h + 2 * (c1 * c2 + c1 * c3 + c2 * c3)) / nn;
                a.h2h1[x] = (double)(h - c1 * c1) / (double)h;
            }
        }
    }
}
