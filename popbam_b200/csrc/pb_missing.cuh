// pb_missing.cuh -- pi and dxy over sites with missing calls, as sums of pairwise differences and comparisons among the
// samples called at each position (PB_AN_NUCDIV_MISSING; include/popbam_b200.h, pb_region_nucdiv_missing; the estimator of
// Korunes & Samuk 2021, pixy).  No reference counterpart; restated in plain C by tests/missing_oracle.c.
//
// Per position of a window: cov = the samples whose cell passes qfilter (acc_cov), der = the derived-allele bits
// (site_type), cleared where segbase's value pb_site_fq(acc_cnt4) < 0 (two different derived bases).  Per population p,
// k_p = popc(cov & m_p), c_p = popc(der & m_p); per population and per pair i < j:
//   pi:  the position counts when k_p >= 2;        diffs += c_p (k_p - c_p),               comps += C(k_p, 2)
//   dxy: the position counts when k_i, k_j >= 1;   diffs += c_i (k_j - c_j) + c_j (k_i - c_i), comps += k_i k_j
// Neither term needs the condition (both are 0 where it fails), only the site count does.  missing = sites * C(n_p, 2)
// - comps (pi) and sites * n_i n_j - comps (dxy).
//
// Grid (window, slice of PB_MISSING_SLICE positions), so one long window (-w 0) spreads over the whole GPU.  A CTA walks its
// slice in chunks of 256 positions.  Phase 1: one thread per position reads its acc_cov, site_type and acc_cnt4 words once
// (20 bytes, coalesced; the loads of the next PB_MISSING_AHEAD chunks are in flight) and writes (k_p | c_p << 8) of every population into shared memory.  Phase 2: the threads are
// mapped to (item, stripe), an item being a population or a pair, and add the chunk's positions of their stripe into
// registers.  Within a slice every sum fits uint32 (per-position terms <= 2016, 8192 * 2016 < 2^32).  After the slice the
// stripes of an item are summed by shuffles and one thread issues one int64 atomic per (item, counter) into arrays the host
// zeroed on the stream: integer addition is order-free, so the sums are exact and do not depend on the grid.
// k_nucdiv_missing_ratio then divides.  The kernels read window bounds and per-position arrays only from device memory,
// so asynchronous regions and relaunches work unchanged.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "pb_cell.cuh"

#define PB_MISSING_THREADS 256
#define PB_MISSING_SLICE 2048              // positions per CTA and pass (every per-item sum of a slice fits uint32 up to 8192)
#define PB_MISSING_PITCH 258               // uint16 per population row: 129 words, odd, so the rows start in different banks
#define PB_MISSING_MAXR 9                  // items per thread: ceil((64 + 2016) / 256)
#define PB_MISSING_AHEAD 4                 // chunks of 256 positions whose loads are in flight per thread

struct PbMissingArgs {
    int P;                                 // populations
    int stripes;                           // threads per item (a power of two <= 32; 1 when there are more than 256 items)
    uint64_t pop_mask[64];
    int32_t pop_nsmpl[64];
    int span_beg;
    const int32_t *win_beg, *win_end;
    const uint64_t *acc_cov;               // [span]
    const uint32_t *acc_cnt4;              // [span]
    const uint64_t *site_type;             // [span]
    int32_t *pi_sites; int64_t *pi_diffs, *pi_comps, *pi_missing; double *pi;             // [NW*P]
    int32_t *dxy_sites; int64_t *dxy_diffs, *dxy_comps, *dxy_missing; double *dxy;        // [NW*P*P], i*P + (j-(i+1))
};

// threads per item: every item gets the same power of two, as many as 256 threads allow, at most a warp
static inline int pb_missing_stripes(int P) {
    const int items = P + P * (P - 1) / 2;
    int s = 32;
    while (s > 1 && s * items > PB_MISSING_THREADS) s >>= 1;
    return s;
}

__global__ void __launch_bounds__(PB_MISSING_THREADS, 4) k_nucdiv_missing(const PbMissingArgs a) {
    __shared__ uint16_t kc[64 * PB_MISSING_PITCH];     // (k | c << 8) per population and position of the chunk
    __shared__ uint64_t mask_s[64];
    __shared__ uint8_t pair_s[2 * 2016];               // (i, j) of every pair in dxy order
    const int w = blockIdx.x, tid = threadIdx.x;
    const int P = a.P, I = P + P * (P - 1) / 2;
    const int S = a.stripes, R = PB_MISSING_THREADS / S, slot = tid / S, stripe = tid % S;
    if (tid < P) {
        mask_s[tid] = a.pop_mask[tid];
        int q = tid * P - tid * (tid + 1) / 2;
        for (int j = tid + 1; j < P; ++j, ++q) { pair_s[2 * q] = (uint8_t)tid; pair_s[2 * q + 1] = (uint8_t)j; }
    }
    const int beg = a.win_beg[w], len = a.win_end[w] - beg;
    const int64_t off = (int64_t)beg - a.span_beg;
    for (int s0 = (int)blockIdx.y * PB_MISSING_SLICE; s0 < len; s0 += (int)gridDim.y * PB_MISSING_SLICE) {
        const int s1 = min(len, s0 + PB_MISSING_SLICE);
        uint32_t sites[PB_MISSING_MAXR], diffs[PB_MISSING_MAXR], comps[PB_MISSING_MAXR];
#pragma unroll
        for (int r = 0; r < PB_MISSING_MAXR; ++r) sites[r] = diffs[r] = comps[r] = 0;
        // the words of PB_MISSING_AHEAD chunks are in flight: chunk u of a group of AHEAD comes from register slot u, which is
        // refilled with the chunk AHEAD further on as soon as it is used (one chunk at a time leaves the loop waiting on DRAM)
        uint64_t cov_r[PB_MISSING_AHEAD], der_r[PB_MISSING_AHEAD];
        uint32_t cnt_r[PB_MISSING_AHEAD];
        auto fetch = [&](int u, int pos) {
            if (pos < s1) { const int64_t o = off + pos; cov_r[u] = a.acc_cov[o]; der_r[u] = a.site_type[o]; cnt_r[u] = a.acc_cnt4[o]; }
        };
#pragma unroll
        for (int u = 0; u < PB_MISSING_AHEAD; ++u) fetch(u, s0 + u * PB_MISSING_THREADS + tid);
        for (int g0 = s0; g0 < s1; g0 += PB_MISSING_AHEAD * PB_MISSING_THREADS)
#pragma unroll
        for (int u = 0; u < PB_MISSING_AHEAD; ++u) {
            const int c0 = g0 + u * PB_MISSING_THREADS;
            if (c0 >= s1) break;
            const int m = min(PB_MISSING_THREADS, s1 - c0);
            __syncthreads();                           // the chunk before is read (and mask_s / pair_s are written)
            if (tid < m) {
                const uint64_t cov = cov_r[u], der = pb_site_fq(cnt_r[u]) < 0 ? 0 : der_r[u];
                for (int p = 0; p < P; ++p)
                    kc[p * PB_MISSING_PITCH + tid] = (uint16_t)(__popcll(cov & mask_s[p]) | __popcll(der & mask_s[p]) << 8);
            }
            fetch(u, c0 + PB_MISSING_AHEAD * PB_MISSING_THREADS + tid);
            __syncthreads();
#pragma unroll
            for (int r = 0; r < PB_MISSING_MAXR; ++r) {
                const int it = slot + r * R;
                if (it >= I) break;
                if (it < P) {
                    const uint16_t *x = kc + it * PB_MISSING_PITCH;
                    for (int j = stripe; j < m; j += S) {
                        const uint32_t v = x[j], k = v & 255u, c = v >> 8;
                        sites[r] += k >= 2u;
                        diffs[r] += c * (k - c);
                        comps[r] += k * (k - 1u) / 2u;
                    }
                } else {
                    const int q = it - P;
                    const uint16_t *xi = kc + pair_s[2 * q] * PB_MISSING_PITCH, *xj = kc + pair_s[2 * q + 1] * PB_MISSING_PITCH;
                    for (int j = stripe; j < m; j += S) {
                        const uint32_t u = xi[j], v = xj[j];
                        const uint32_t ki = u & 255u, ci = u >> 8, kj = v & 255u, cj = v >> 8;
                        sites[r] += (ki != 0u) & (kj != 0u);
                        diffs[r] += ci * (kj - cj) + cj * (ki - ci);
                        comps[r] += ki * kj;
                    }
                }
            }
        }
        // more than one stripe only when every thread has one item (r = 0); the stripes of an item are adjacent lanes
        for (int d = S >> 1; d > 0; d >>= 1) {
            sites[0] += __shfl_xor_sync(0xffffffffu, sites[0], d);
            diffs[0] += __shfl_xor_sync(0xffffffffu, diffs[0], d);
            comps[0] += __shfl_xor_sync(0xffffffffu, comps[0], d);
        }
        if (stripe == 0) {
#pragma unroll
            for (int r = 0; r < PB_MISSING_MAXR; ++r) {
                const int it = slot + r * R;
                if (it >= I) break;
                if (sites[r] == 0) continue;           // then diffs and comps are 0 too
                if (it < P) {
                    const int64_t np = a.pop_nsmpl[it];
                    const size_t x = (size_t)w * P + it;
                    atomicAdd(a.pi_sites + x, (int)sites[r]);
                    atomicAdd(reinterpret_cast<unsigned long long *>(a.pi_diffs + x), (unsigned long long)diffs[r]);
                    atomicAdd(reinterpret_cast<unsigned long long *>(a.pi_comps + x), (unsigned long long)comps[r]);
                    atomicAdd(reinterpret_cast<unsigned long long *>(a.pi_missing + x),
                              (unsigned long long)((int64_t)sites[r] * (np * (np - 1) / 2) - (int64_t)comps[r]));
                } else {
                    const int q = it - P, i = pair_s[2 * q], j = pair_s[2 * q + 1];
                    const size_t x = (size_t)w * P * P + i * P + (j - (i + 1));
                    const int64_t nn = (int64_t)a.pop_nsmpl[i] * a.pop_nsmpl[j];
                    atomicAdd(a.dxy_sites + x, (int)sites[r]);
                    atomicAdd(reinterpret_cast<unsigned long long *>(a.dxy_diffs + x), (unsigned long long)diffs[r]);
                    atomicAdd(reinterpret_cast<unsigned long long *>(a.dxy_comps + x), (unsigned long long)comps[r]);
                    atomicAdd(reinterpret_cast<unsigned long long *>(a.dxy_missing + x),
                              (unsigned long long)((int64_t)sites[r] * nn - (int64_t)comps[r]));
                }
            }
        }
    }
}

// the ratios, once every sum is complete: (double) diffs / (double) comps, NaN where comps is 0.  The slots of a window's
// P*P dxy block that name no pair (j <= i) stay 0 in every array.
__global__ void __launch_bounds__(256) k_nucdiv_missing_ratio(const PbMissingArgs a, int NW) {
    const int P = a.P;
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i < (int64_t)NW * P) {
        const int64_t den = a.pi_comps[i];
        a.pi[i] = den ? (double)a.pi_diffs[i] / (double)den : __longlong_as_double(0x7ff8000000000000LL);
    }
    if (i < (int64_t)NW * P * P) {
        const int r = (int)(i % ((int64_t)P * P)), pi = r / P, pj = pi + 1 + r % P;
        if (pj < P) {
            const int64_t den = a.dxy_comps[i];
            a.dxy[i] = den ? (double)a.dxy_diffs[i] / (double)den : __longlong_as_double(0x7ff8000000000000LL);
        }
    }
}
