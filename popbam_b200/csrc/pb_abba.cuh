// pb_abba.cuh -- ABBA-BABA statistics per (window, triple) (PB_AN_ABBA; include/popbam_b200.h, pb_region_abba).
// No reference counterpart; restated in plain C by tests/abba_oracle.c.
//
// Triple (P1, P2, P3) against the outgroup population O; per segregating site a_k = popc(T & mask_k), k = 1..4 (O = 4),
// polarised so that O carries the derived allele at frequency <= 1/2 (all a_k <-> m_k = n_k - a_k if 2 a_4 > n_4).
// On the scale K = n1^2 n2^2 n3^2 n4 every site term is an exact integer of magnitude <= K < 2^29 (n1+n2+n3+n4 <= 64):
//   abba    = m1 a2 a3 m4 * n1 n2 n3,   baba = a1 m2 a3 m4 * n1 n2 n3
//   fd_den  = (m1 a2^2 - a1 m2 a2) m4 * n1 n3^2        if a2 n3 >= a3 n2   (pD = p2)
//             (m1 a3^2 - a1 m3 a3) m4 * n1 n2^2        otherwise           (pD = p3)
//   fdm_den = fd_den's term                             if a2 n1 >= a1 n2   (p2 >= p1)
//             (a1^2 m2 - m1 a2 a1) m4 * n2 n3^2        else if a1 n3 >= a3 n1 (pD = p1)
//             (a3^2 m2 - m3 a2 a3) m4 * n1^2 n2        otherwise           (pD = p3)
// so the int64 window sums (< 2^31 sites) are exact and independent of the summation order.
//
// Grid (window, block of PB_ABBA_WARPS triples), one warp per triple: lanes stride over the window's segregating sites
// (the CTA's warps read the same seg_type words, which stay in L1), a shuffle reduction gives the sums, lane 0 writes
// them and the three ratios.  No atomics.  The window's site count and offset are read from device memory, so the
// kernel runs unchanged when the host does not know the number of segregating sites (asynchronous regions).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define PB_ABBA_WARPS 4

// one triple's masks, sizes and scale factors (built on the host by pb_region_begin)
struct PbAbbaTriple {
    uint64_t m1, m2, m3, m4;
    int32_t n1, n2, n3, n4;
    long long s_ab;        // n1 n2 n3     (abba, baba)
    long long s_d2;        // n1 n3^2      (fd_den, pD = p2)
    long long s_d3;        // n1 n2^2      (fd_den, pD = p3)
    long long s_m1;        // n2 n3^2      (fdm_den, pD = p1)
    long long s_m3;        // n1^2 n2      (fdm_den, pD = p3)
};

struct PbAbbaArgs {
    const PbAbbaTriple *tri;
    int nt;
    const int32_t *segsites;
    const int64_t *seg_off;
    const uint64_t *seg_type;
    int32_t *sites;                               // [NW*nt], index w*nt + t
    int64_t *abba, *baba, *fd_den, *fdm_den;
    double *d, *fd, *fdm;
};

__global__ void __launch_bounds__(PB_ABBA_WARPS * 32) k_abba(const PbAbbaArgs a) {
    const int w = blockIdx.x, lane = threadIdx.x & 31;
    const int t = blockIdx.y * PB_ABBA_WARPS + (threadIdx.x >> 5);
    if (t >= a.nt) return;
    const PbAbbaTriple q = a.tri[t];
    const uint64_t *__restrict__ T = a.seg_type + a.seg_off[w];
    const int S = a.segsites[w];
    long long ab = 0, ba = 0, fdd = 0, fmd = 0;
    int ns = 0;
    for (int s = lane; s < S; s += 32) {
        const uint64_t x = T[s];
        int a1 = __popcll(x & q.m1), a2 = __popcll(x & q.m2), a3 = __popcll(x & q.m3), a4 = __popcll(x & q.m4);
        if (2 * a4 > q.n4) { a1 = q.n1 - a1; a2 = q.n2 - a2; a3 = q.n3 - a3; a4 = q.n4 - a4; }
        const int m1 = q.n1 - a1, m2 = q.n2 - a2, m3 = q.n3 - a3, m4 = q.n4 - a4;
        // every int product below is at most 64^4
        const long long tab = (long long)(m1 * a2 * a3 * m4) * q.s_ab, tba = (long long)(a1 * m2 * a3 * m4) * q.s_ab;
        const long long tfd = a2 * q.n3 >= a3 * q.n2 ? (long long)((m1 * a2 * a2 - a1 * m2 * a2) * m4) * q.s_d2
                                                     : (long long)((m1 * a3 * a3 - a1 * m3 * a3) * m4) * q.s_d3;
        const long long tfm = a2 * q.n1 >= a1 * q.n2 ? tfd
                            : a1 * q.n3 >= a3 * q.n1 ? (long long)((a1 * a1 * m2 - m1 * a2 * a1) * m4) * q.s_m1
                                                     : (long long)((a3 * a3 * m2 - m3 * a2 * a3) * m4) * q.s_m3;
        ab += tab; ba += tba; fdd += tfd; fmd += tfm;
        ns += tab + tba > 0;
    }
    for (int o = 16; o > 0; o >>= 1) {
        ab += __shfl_xor_sync(0xffffffffu, ab, o);
        ba += __shfl_xor_sync(0xffffffffu, ba, o);
        fdd += __shfl_xor_sync(0xffffffffu, fdd, o);
        fmd += __shfl_xor_sync(0xffffffffu, fmd, o);
        ns += __shfl_xor_sync(0xffffffffu, ns, o);
    }
    if (lane == 0) {
        const size_t i = (size_t)w * a.nt + t;
        const long long num = ab - ba;
        a.sites[i] = ns;
        a.abba[i] = ab; a.baba[i] = ba; a.fd_den[i] = fdd; a.fdm_den[i] = fmd;
        a.d[i] = ab + ba != 0 ? (double)num / (double)(ab + ba) : nan("");
        a.fd[i] = fdd != 0 ? (double)num / (double)fdd : nan("");
        a.fdm[i] = fmd != 0 ? (double)num / (double)fmd : nan("");
    }
}
