// pb_spectrum.cuh -- unfolded site frequency spectra of 1-3 populations per window (PB_AN_SPECTRUM;
// include/popbam_b200.h, pb_region_spectrum).  No reference counterpart; restated in plain C by tests/spectrum_oracle.c.
//
// Per segregating site and set: a_k = popc(t & mask_k), all flipped to n_k - a_k when the outgroup sample carries the
// derived allele (PB_FLAG_OUTGROUP, as the sfs pass of k_window_stats), bin = a1 * st1 + a2 * st2 + a3 (row-major, the
// last population fastest).  Unused slots of a one- or two-population set have mask 0 and n 0, so they add nothing.
//
// Grid (window, group).  The host packs the sets, in order, into groups of at most PB_SPECTRUM_GROUP_BINS bins, so one
// group's histogram fits the 48 KB of static shared memory.  The threads stride over the window's segregating sites, read
// each seg_type word once and add 1 to the bin of every set of the group with warp-aggregated shared atomics: lanes
// that hit the same bin (rare variants put most sites into a few low-frequency bins) are merged by __match_any_sync and
// their leader adds the count.  One thread adds num_sites - segsites to each set's all-zero bin, and the group's bins
// go to `counts` with coalesced stores.  Every count is an exact integer written once; there are no global atomics.
// The window's site counts and offset are read from device memory, so the kernel runs unchanged on asynchronous
// regions and relaunches.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define PB_SPECTRUM_THREADS 256
#define PB_SPECTRUM_GROUP_BINS 12288      // int32 bins of one group: 48 KB of static shared memory

struct PbSpecSet {
    uint64_t mask[3];                     // population masks (0 in unused slots)
    int32_t n[3];                         // population sizes (0 in unused slots)
    int32_t stride[3];                    // bin strides: (n2+1)(n3+1), n3+1, 1 for a three-population set
    int32_t off;                          // first bin of the set within its group
};
struct PbSpecGroup {
    int32_t s0, s1;                       // sets [s0, s1)
    int32_t b0, nb;                       // their bins: [b0, b0 + nb) of a window's B
};

struct PbSpectrumArgs {
    const PbSpecSet *sets;
    const PbSpecGroup *groups;
    int B;                                // bins per window over all sets
    int outg, outidx;                     // polarise by sample outidx
    const int32_t *num_sites, *segsites;
    const int64_t *seg_off;
    const uint64_t *seg_type;
    int32_t *counts;                      // [NW*B]
};

__global__ void __launch_bounds__(PB_SPECTRUM_THREADS) k_spectrum(const PbSpectrumArgs a) {
    __shared__ int32_t hist[PB_SPECTRUM_GROUP_BINS];
    const int w = blockIdx.x, tid = threadIdx.x, lane = tid & 31;
    const PbSpecGroup g = a.groups[blockIdx.y];
    for (int i = tid; i < g.nb; i += PB_SPECTRUM_THREADS) hist[i] = 0;
    __syncthreads();
    const int S = a.segsites[w];
    const uint64_t *__restrict__ T = a.seg_type + a.seg_off[w];
    // whole warps run every round, so __match_any_sync sees every lane that has a site
    for (int base = tid - lane; base < S; base += PB_SPECTRUM_THREADS) {
        const bool have = base + lane < S;
        const unsigned act = __ballot_sync(0xffffffffu, have);
        if (!have) continue;
        const uint64_t t = T[base + lane];
        const bool flip = a.outg && (t >> a.outidx & 1);
        for (int s = g.s0; s < g.s1; ++s) {
            const PbSpecSet &q = a.sets[s];
            int bin = q.off;
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                const int c = __popcll(t & q.mask[k]);
                bin += (flip ? q.n[k] - c : c) * q.stride[k];
            }
            const unsigned peers = __match_any_sync(act, bin);
            if (lane == __ffs(peers) - 1) atomicAdd(&hist[bin], __popc(peers));
        }
    }
    __syncthreads();
    if (tid == 0) {
        const int rest = a.num_sites[w] - S;
        for (int s = g.s0; s < g.s1; ++s) hist[a.sets[s].off] += rest;
    }
    __syncthreads();
    int32_t *out = a.counts + (size_t)w * a.B + g.b0;
    for (int i = tid; i < g.nb; i += PB_SPECTRUM_THREADS) out[i] = hist[i];
}
