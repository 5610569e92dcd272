// pb_stats.cuh -- per-window statistics on the segregating-site type words: one CTA per window.
//
//   haplotype bit-packing          hap.seq[i][s/64] |= 1<<(s%64)          (pop_nucdiv.cpp:190-193)
//   calc_diff_matrix               pop_nucdiv.cpp:242-256, hamming_distance pop_utils.cpp:51-64
//   calc_nucdiv / calc_minDxy      pop_nucdiv.cpp:206-239, pop_haplo.cpp:325-363
//   calc_sfs                       pop_sfs.cpp:227-291 (+ calc_a1/a2/e1/e2, :511-571)
//   (calc_zns / calc_omegamax: pb_ld.cuh)
//   calc_wall                      pop_ld.cpp:375-458
//   calc_diverge                   pop_diverge.cpp:220-257
//   calc_nhaps / calc_ehhs         pop_haplo.cpp:208-254, :256-323
//   extensions (no reference counterpart): Watterson's theta and Fu & Li's D / D* on calc_sfs's spectrum,
//   the closed forms of tests/ext_oracle.c in the same operation order; F_ST and Snn between population pairs
//   (PB_AN_FST, pb_fst_pairs and k_snn_perm below, restated by tests/fst_oracle.c)
//
// Integer results are exact.  Floating-point statistics use the reference's formulas term by term
// (the library is compiled with -fmad=false so products and sums round separately, as on x86-64);
// only the ORDER of the O(S^2) r^2 summations differs (parallel partial sums), which is inside the
// 1e-9 relative tolerance of the parity contract.  The small sequential routines with order-dependent
// quirks (Wall's B/Q, haplotype counting; SURVEY.md Q11-Q12) are literal single-thread restatements.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define PB_ST_THREADS 256

struct PbStatArgs {
    int n, P;
    uint64_t pop_mask[64];
    uint8_t pop_nsmpl[64];
    uint32_t analyses, flags;
    int outidx, min_freq;
    const int32_t *num_sites, *segsites;
    const int64_t *seg_off;
    const uint64_t *seg_type;
    // scratch
    uint64_t *hap;        // n * (S_total/64 + NW + 1) words
    uint64_t *kt;         // [S_total + NW] kept / list entries of the current population
    uint8_t *km;          // [S_total + NW] marginal counts
    uint64_t *wall_u;     // [P * S_total] unique partitions (ld -o 2) or null
    int64_t s_total;
    // outputs (see pb_region_result)
    double *piw, *pib; uint16_t *min_dxy;
    int32_t *sfs_num_snps; double *td, *fwh;
    int32_t *wall_num_snps; double *wallb, *wallq;
    uint16_t *ind_div, *pop_div; int32_t *div_num_snps;
    int32_t *nhaps; double *hdiv, *ehhs;
    uint16_t *tree_diff;  // [NW][(n+1)*(n+1)]
    int32_t *pop_segsites; double *theta_w, *fuli_d, *fuli_ds; int32_t *fuli_eta_e, *fuli_eta_s;
    // PB_AN_FST, [NW][P*P] indexed like pib; snn_nn [NW][P*P][n]: nearest-neighbour masks for k_snn_perm (null without permutations)
    int64_t *hud_num, *hud_den, *wc_num, *wc_den; double *fst_hudson, *fst_wc, *snn;
    uint64_t *snn_nn;
};

// analysis bits (include/popbam_b200.h)
#define PBA_NUCDIV 0x001u
#define PBA_SFS 0x002u
#define PBA_LD_ZNS 0x004u
#define PBA_LD_OMEGA 0x008u
#define PBA_LD_WALL 0x010u
#define PBA_DIVERGE_IND 0x020u
#define PBA_DIVERGE_POP 0x040u
#define PBA_TREE 0x800u
#define PBA_HAPLO_K 0x080u
#define PBA_HAPLO_EHHS 0x100u
#define PBA_HAPLO_DXY 0x200u
#define PBA_THETA_W 0x1000u
#define PBA_FULI 0x2000u
#define PBA_FST 0x8000u
#define PBA_FLAG_OUTGROUP 0x40u

__device__ __forceinline__ int pb_block_sum_int(int v, int *sh /* [32] */) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
    __syncthreads();
    int t = 0;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) t += sh[i];
    return t;
}

// ordered compaction of the sites of one population that satisfy `pred`; returns the count (all threads)
template <class Pred>
__device__ int pb_compact_sites(const uint64_t *__restrict__ T, int S, uint64_t mask, Pred pred, uint64_t *__restrict__ out_t,
                                uint8_t *__restrict__ out_m, int limit_excl /* count only sites < limit in *n_before */,
                                int *n_before, uint32_t *sh /* [33] */) {
    int carry = 0, before = 0;
    for (int b0 = 0; b0 < S; b0 += PB_ST_THREADS) {
        const int s = b0 + (int)threadIdx.x;
        uint64_t t = 0; int m = 0; bool keep = false;
        if (s < S) { t = T[s] & mask; m = __popcll(t); keep = pred(t, m); }
        // block exclusive scan of keep
        const uint32_t bal = __ballot_sync(0xffffffffu, keep);
        const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
        __syncthreads();
        if (lane == 0) sh[wid] = __popc(bal);
        __syncthreads();
        int base = 0, tot = 0;
        for (int i = 0; i < (int)(blockDim.x >> 5); ++i) { if (i < wid) base += sh[i]; tot += sh[i]; }
        const int idx = carry + base + __popc(bal & ((1u << lane) - 1u));
        if (keep) { out_t[idx] = t; out_m[idx] = (uint8_t)m; }
        // number kept among sites < limit_excl
        int nb = 0;
        if (b0 + PB_ST_THREADS <= limit_excl) nb = tot;
        else if (b0 < limit_excl) {
            int c = (keep && s < limit_excl) ? 1 : 0;
            for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
            __syncthreads();
            if (lane == 0) sh[wid] = c;
            __syncthreads();
            for (int i = 0; i < (int)(blockDim.x >> 5); ++i) nb += sh[i];
        }
        before += nb;
        carry += tot;
    }
    __syncthreads();
    *n_before = before;
    return carry;
}

// Watterson's theta and Fu & Li's D / D* of one (window, population) from the spectrum's S, xi_1 and xi_{np-1}
__device__ __forceinline__ void pb_sfs_ext(int np, int seg, int xi1, int xin1, bool outg, int32_t *segs, double *theta_w, double *fuli_d,
                                        double *fuli_ds, int32_t *eta_e, int32_t *eta_s) {
    const int ee = np >= 2 ? xi1 : 0, es = np >= 3 ? xi1 + xin1 : ee;
    double thw = nan(""), fd = nan(""), fds = nan("");
    if (np >= 2) {
        double a1 = 0.0, a2 = 0.0;
        for (int j = 1; j < np; ++j) a1 += 1.0 / (double)j;
        for (int j = 1; j < np; ++j) a2 += 1.0 / ((double)j * (double)j);
        thw = (double)seg / a1;
        if (np >= 3 && seg > 0) {
            const double nn = (double)np, Sd = (double)seg, ap = a1 + 1.0 / nn, r = nn / (nn - 1.0);
            const double c = 2.0 * (nn * a1 - 2.0 * (nn - 1.0)) / ((nn - 1.0) * (nn - 2.0));
            const double vd = 1.0 + a1 * a1 / (a2 + a1 * a1) * (c - (nn + 1.0) / (nn - 1.0)), ud = a1 - 1.0 - vd;
            const double d = c + (nn - 2.0) / ((nn - 1.0) * (nn - 1.0)) + 2.0 / (nn - 1.0) * (1.5 - (2.0 * ap - 3.0) / (nn - 2.0) - 1.0 / nn);
            const double vds = (r * r * a2 + a1 * a1 * d - 2.0 * nn * a1 * (a1 + 1.0) / ((nn - 1.0) * (nn - 1.0))) / (a1 * a1 + a2);
            const double uds = r * (a1 - r) - vds;
            if (outg) fd = (Sd - a1 * (double)ee) / sqrt(ud * Sd + vd * Sd * Sd);
            if (np >= 4) fds = (r * Sd - a1 * (double)es) / sqrt(uds * Sd + vds * Sd * Sd);      // n = 3: eta_s = S, 0 / 0
        }
    }
    *segs = seg;
    if (theta_w) *theta_w = thw;
    if (fuli_d) { *fuli_d = fd; *fuli_ds = fds; *eta_e = ee; *eta_s = es; }
}

// ---- F_ST and Snn of every population pair i < j of one window (PB_AN_FST; include/popbam_b200.h, pb_region_fst).
// n1, n2 = pop_nsmpl[i], pop_nsmpl[j]; per segregating site T: c1 = popc(T & pop_mask[i]), c2 = popc(T & pop_mask[j]).
// Hudson (Bhatia et al. 2013), every term scaled by n1 n2 (n1-1) (n2-1):
//   hud_den = sum (n1-1)(n2-1) [c1 (n2-c2) + c2 (n1-c1)],  hud_num = hud_den - sum [c1 (n1-c1) n2 (n2-1) + c2 (n2-c2) n1 (n1-1)]
// Weir & Cockerham's haploid theta (r = 2), scaled by n1 n2 (n1+n2) (n1+n2-2), with G = c1 (n1-c1) n2 + c2 (n2-c2) n1:
//   wc_num = sum (c1 n2 - c2 n1)^2 (n1+n2-2) - G (n1+n2),  wc_den = sum (c1 n2 - c2 n1)^2 (n1+n2-2) + G (2 n1 n2 - n1 - n2)
// Every site term is an integer below 2^31 for n <= 64, so the int64 window sums are exact and independent of the order.
// Snn (Hudson 2000): NN(x) = the other pooled samples at the least diff[x][y]; X_x = |NN(x) & pop(x)| / |NN(x)|;
// Snn = (sum of X_x in ascending sample order, one thread) / (n1 + n2).  All three are NaN if n1 < 2 or n2 < 2.
__device__ __forceinline__ void pb_block_sum_i64x4(long long v[4], long long (*sh)[4] /* [warps][4] */) {
    for (int k = 0; k < 4; ++k)
        for (int o = 16; o > 0; o >>= 1) v[k] += __shfl_xor_sync(0xffffffffu, v[k], o);
    __syncthreads();
    if ((threadIdx.x & 31) == 0)
        for (int k = 0; k < 4; ++k) sh[threadIdx.x >> 5][k] = v[k];
    __syncthreads();
    for (int k = 0; k < 4; ++k) {
        long long t = 0;
        for (int i = 0; i < (int)(blockDim.x >> 5); ++i) t += sh[i][k];
        v[k] = t;
    }
}

__device__ __forceinline__ void pb_fst_pairs(const PbStatArgs &a, int w, const uint64_t *__restrict__ T, int S, const uint16_t *diff) {
    __shared__ long long red[PB_ST_THREADS / 32][4];
    __shared__ double xs[64];
    const int tid = threadIdx.x, n = a.n, P = a.P;
    for (int i = 0; i < P - 1; ++i)
        for (int j = i + 1; j < P; ++j) {
            const uint64_t mi = a.pop_mask[i], mj = a.pop_mask[j], pool = mi | mj;
            const long long n1 = a.pop_nsmpl[i], n2 = a.pop_nsmpl[j];
            const long long hf = (n1 - 1) * (n2 - 1), wa = n1 + n2 - 2, wb = n1 + n2, wc = 2 * n1 * n2 - n1 - n2;
            const size_t x = (size_t)w * P * P + i * P + (j - (i + 1));
            long long v[4] = {0, 0, 0, 0};      // hud_num, hud_den, wc_num, wc_den
            for (int s = tid; s < S; s += PB_ST_THREADS) {
                const uint64_t t = T[s];
                const long long c1 = __popcll(t & mi), c2 = __popcll(t & mj);
                const long long hd = hf * (c1 * (n2 - c2) + c2 * (n1 - c1));
                const long long hw = c1 * (n1 - c1) * n2 * (n2 - 1) + c2 * (n2 - c2) * n1 * (n1 - 1);
                const long long dd = c1 * n2 - c2 * n1, msp = dd * dd * wa, g = c1 * (n1 - c1) * n2 + c2 * (n2 - c2) * n1;
                v[0] += hd - hw; v[1] += hd; v[2] += msp - g * wb; v[3] += msp + g * wc;
            }
            pb_block_sum_i64x4(v, red);
            const bool two = n1 >= 2 && n2 >= 2;
            if (two && tid < n && (pool >> tid & 1)) {
                unsigned mn = 0xffffffffu;
                uint64_t nn = 0;
                for (int y = 0; y < n; ++y) {
                    if (y == tid || !(pool >> y & 1)) continue;
                    const unsigned d = diff[tid * n + y];
                    if (d < mn) { mn = d; nn = 0; }
                    if (d == mn) nn |= 1ULL << y;
                }
                const uint64_t own = (mi >> tid & 1) ? mi : mj;
                xs[tid] = (double)__popcll(nn & own) / (double)__popcll(nn);
                if (a.snn_nn) a.snn_nn[x * n + tid] = nn;
            }
            __syncthreads();
            if (tid == 0) {
                a.hud_num[x] = v[0]; a.hud_den[x] = v[1]; a.wc_num[x] = v[2]; a.wc_den[x] = v[3];
                a.fst_hudson[x] = two && v[1] != 0 ? (double)v[0] / (double)v[1] : nan("");
                a.fst_wc[x] = two && v[3] != 0 ? (double)v[2] / (double)v[3] : nan("");
                double snn = nan("");
                if (two) {
                    double sum = 0.0;
                    for (int y = 0; y < n; ++y)
                        if (pool >> y & 1) sum += xs[y];
                    snn = sum / (double)(n1 + n2);
                }
                a.snn[x] = snn;
            }
            __syncthreads();     // xs and red are reused by the next pair
        }
}

// ---- Snn permutation test (PB_AN_FST with pb_set_snn_perms): grid (window, pair q in dxy order), threads stride over
// the permutations.  NN(x) does not depend on the labels, so a permutation only re-partitions the pool: population i is
// the n1 samples a partial Fisher-Yates shuffle of the pool (ascending sample order) puts first.  snn_ge counts the
// permutations whose Snn >= Snn_obs - 1e-12; snn_p = (1 + snn_ge) / (1 + n_perms).
// Random stream (counter-based, so it does not depend on how a region is cut into windows, shards or GPUs):
//   mix(z)   = splitmix64's finaliser: z = (z ^ z>>30) * 0xbf58476d1ce4e5b9; z = (z ^ z>>27) * 0x94d049bb133111eb; z ^ z>>31
//   key      h = mix(seed + G); then h = mix((h ^ v) + G) for v = tid, win_beg, i, j, permutation index in turn
//            (G = 0x9e3779b97f4a7c15; each v as a 64-bit two's-complement integer)
//   draw k   z_k = mix(h + (k + 1) G), k = 0, 1, ...  (the k-th output of a splitmix64 generator started at h)
//   index    in [0, r): ((z >> 32) * r) >> 32;  shuffle step k swaps slot k with slot k + index(z_k, m - k)
#define PB_GOLDEN64 0x9e3779b97f4a7c15ULL
__device__ __forceinline__ uint64_t pb_mix64(uint64_t z) {
    z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ULL;
    z = (z ^ (z >> 27)) * 0x94d049bb133111ebULL;
    return z ^ (z >> 31);
}

struct PbSnnArgs {
    int n, P, tid;
    uint64_t pop_mask[64];
    uint8_t pop_nsmpl[64];
    const int32_t *win_beg;
    const uint64_t *nn;        // PbStatArgs::snn_nn
    const double *snn;
    double *snn_p;
    int64_t *snn_ge;
    long long n_perms;
    uint64_t seed;
};

__global__ void __launch_bounds__(PB_ST_THREADS) k_snn_perm(const PbSnnArgs a) {
    __shared__ uint64_t nn[64];
    __shared__ unsigned long long red[PB_ST_THREADS / 32];
    const int w = blockIdx.x, P = a.P, n = a.n, tid = threadIdx.x;
    int i = 0, r = blockIdx.y;
    while (r >= P - 1 - i) { r -= P - 1 - i; ++i; }
    const int j = i + 1 + r;
    const size_t x = (size_t)w * P * P + i * P + (j - (i + 1));
    const int n1 = a.pop_nsmpl[i], m = n1 + a.pop_nsmpl[j];
    if (n1 < 2 || a.pop_nsmpl[j] < 2) {
        if (tid == 0) { a.snn_ge[x] = 0; a.snn_p[x] = nan(""); }
        return;
    }
    const uint64_t pool = a.pop_mask[i] | a.pop_mask[j];
    if (tid < n) nn[tid] = a.nn[x * n + tid];
    __syncthreads();
    const double thr = a.snn[x] - 1e-12;
    uint64_t key = pb_mix64(a.seed + PB_GOLDEN64);
    key = pb_mix64((key ^ (uint64_t)(int64_t)a.tid) + PB_GOLDEN64);
    key = pb_mix64((key ^ (uint64_t)(int64_t)a.win_beg[w]) + PB_GOLDEN64);
    key = pb_mix64((key ^ (uint64_t)(int64_t)i) + PB_GOLDEN64);
    key = pb_mix64((key ^ (uint64_t)(int64_t)j) + PB_GOLDEN64);
    unsigned long long ge = 0;
    for (long long k = tid; k < a.n_perms; k += PB_ST_THREADS) {
        const uint64_t h = pb_mix64((key ^ (uint64_t)k) + PB_GOLDEN64);
        uint8_t idx[64];
        {
            uint64_t t = pool;
            for (int c = 0; c < m; ++c) { idx[c] = (uint8_t)(__ffsll((long long)t) - 1); t &= t - 1; }
        }
        uint64_t A = 0;
        for (int c = 0; c < n1; ++c) {
            const uint64_t z = pb_mix64(h + (uint64_t)(c + 1) * PB_GOLDEN64);
            const int rr = c + (int)(((z >> 32) * (uint64_t)(m - c)) >> 32);
            const uint8_t s = idx[rr];
            idx[rr] = idx[c]; idx[c] = s;
            A |= 1ULL << s;
        }
        const uint64_t B = pool & ~A;
        double sum = 0.0;
        for (uint64_t t = pool; t; t &= t - 1) {
            const int y = __ffsll((long long)t) - 1;
            sum += (double)__popcll(nn[y] & ((A >> y & 1) ? A : B)) / (double)__popcll(nn[y]);
        }
        ge += sum / (double)m >= thr;
    }
    for (int o = 16; o > 0; o >>= 1) ge += __shfl_xor_sync(0xffffffffu, ge, o);
    if ((tid & 31) == 0) red[tid >> 5] = ge;
    __syncthreads();
    if (tid == 0) {
        unsigned long long t = 0;
        for (int k = 0; k < PB_ST_THREADS / 32; ++k) t += red[k];
        a.snn_ge[x] = (int64_t)t;
        a.snn_p[x] = (1.0 + (double)t) / (1.0 + (double)a.n_perms);
    }
}

// k_window_stats<true> adds the F_ST pass (PB_AN_FST); k_window_stats<false> compiles to the kernel without it
template <bool FST>
__global__ void __launch_bounds__(PB_ST_THREADS) k_window_stats(const PbStatArgs a) {
    extern __shared__ __align__(16) unsigned char st_smem[];
    uint16_t *diff = reinterpret_cast<uint16_t *>(st_smem);                   // [n*n]
    __shared__ int shi[32];
    __shared__ uint32_t shu[33];
    __shared__ int sfs_s[66];

    const int w = blockIdx.x, tid = threadIdx.x;
    const int n = a.n, P = a.P;
    const int S = a.segsites[w];
    const int64_t so = a.seg_off[w];
    const uint64_t *__restrict__ T = a.seg_type + so;
    const int nwords = (S + 63) >> 6;
    uint64_t *hap = a.hap + (size_t)n * (size_t)(so / 64 + w);
    const uint32_t an = a.analyses;
    const bool outg = (a.flags & PBA_FLAG_OUTGROUP) != 0;

    // ---- haplotype words: bit s of hap[i] = sample i carries the derived allele at segsite s
    if (an & (PBA_NUCDIV | PBA_HAPLO_K | PBA_HAPLO_EHHS | PBA_HAPLO_DXY | PBA_DIVERGE_IND | PBA_TREE | (FST ? PBA_FST : 0u))) {
        for (int idx = tid; idx < n * nwords; idx += PB_ST_THREADS) {
            const int i = idx / nwords, kw = idx - i * nwords;
            uint64_t word = 0;
            const int s0 = kw << 6, s1 = min(S, s0 + 64);
            for (int s = s0; s < s1; ++s) word |= ((T[s] >> i) & 1ULL) << (s - s0);
            hap[(size_t)i * nwords + kw] = word;
        }
        __syncthreads();
    }
    if (an & PBA_DIVERGE_IND) {
        for (int i = tid; i < n; i += PB_ST_THREADS) {
            unsigned d = 0;
            for (int k = 0; k < nwords; ++k) d += __popcll(hap[(size_t)i * nwords + k]);
            a.ind_div[(size_t)w * n + i] = (uint16_t)d;
        }
    }
    // ---- tree: difference matrix with the reference as taxon 0 (pop_tree.cpp:472-494; unsigned short, wraps)
    if (an & PBA_TREE) {
        const int m = n + 1;
        uint16_t *td = a.tree_diff + (size_t)w * m * m;
        for (int pi = tid; pi < m * m; pi += PB_ST_THREADS) {
            const int i = pi / m, j = pi - i * m;
            unsigned d = 0;
            if (i != j) {
                if (i == 0 || j == 0) {
                    const int smp = (i ? i : j) - 1;
                    for (int k = 0; k < nwords; ++k) d += __popcll(hap[(size_t)smp * nwords + k]);
                } else
                    for (int k = 0; k < nwords; ++k) d += __popcll(hap[(size_t)(i - 1) * nwords + k] ^ hap[(size_t)(j - 1) * nwords + k]);
            }
            td[pi] = (uint16_t)d;
        }
    }
    // ---- pairwise difference matrix (unsigned short, wraps)
    if (an & (PBA_NUCDIV | PBA_HAPLO_K | PBA_HAPLO_EHHS | PBA_HAPLO_DXY | (FST ? PBA_FST : 0u))) {
        for (int pi = tid; pi < n * n; pi += PB_ST_THREADS) {
            const int i = pi / n, j = pi - i * n;
            unsigned d = 0;
            if (i != j)
                for (int k = 0; k < nwords; ++k) d += __popcll(hap[(size_t)i * nwords + k] ^ hap[(size_t)j * nwords + k]);
            diff[pi] = (uint16_t)d;
        }
        __syncthreads();
    }
    // ---- nucleotide diversity within / between, minimum dxy
    if (an & (PBA_NUCDIV | PBA_HAPLO_DXY)) {
        for (int pp = tid; pp < P * P; pp += PB_ST_THREADS) {
            const int i = pp / P, j = pp - i * P;
            if (j < i) continue;
            double sum = 0.0;
            unsigned mn = 65535;
            for (int v = 0; v < n - 1; ++v) {
                if (!(a.pop_mask[i] >> v & 1)) continue;
                for (int x = v + 1; x < n; ++x)
                    if (a.pop_mask[j] >> x & 1) { const unsigned d = diff[v * n + x]; sum += (double)d; mn = min(mn, d); }
            }
            if (i == j) {
                double v = sum * (2.0 / (double)(a.pop_nsmpl[i] * (a.pop_nsmpl[i] - 1)));
                if (isnan(v)) v = 0.0;
                a.piw[(size_t)w * P + i] = v;
            } else {
                const size_t x = (size_t)w * P * P + i * P + (j - (i + 1));
                a.pib[x] = sum * (1.0 / (double)(a.pop_nsmpl[i] * a.pop_nsmpl[j]));
                a.min_dxy[x] = (uint16_t)mn;
            }
        }
    }
    // ---- F_ST and Snn of every population pair (extension)
    if constexpr (FST) pb_fst_pairs(a, w, T, S, diff);
    // ---- haplotype count / diversity (literal, within-population ranks index the matrix: SURVEY Q12)
    if (an & (PBA_HAPLO_K | PBA_HAPLO_EHHS)) {
        for (int i = tid; i < P; i += PB_ST_THREADS) {
            const int nelem = a.pop_nsmpl[i];
            int nh = 1; double hd = 1.0;
            if (nelem > 1) {
                int b[64], m = 0;
                for (int j = 0; j < n; ++j) if (a.pop_mask[i] >> j & 1) b[m++] = j;
                for (int j = 0; j < nelem - 1; ++j)
                    for (int k = j + 1; k < nelem; ++k)
                        if (diff[j * n + k] == 0 && b[k] > b[j]) b[k] = j;
                int ff = 0; nh = 0;
                for (int j = 0; j < m; ++j) {
                    int f = 0;
                    for (int k = 0; k < m; ++k) f += b[k] == j;
                    if (f > 0) ++nh;
                    ff += f * f;
                }
                const double sh = (double)ff / (double)(nelem * nelem);
                hd = 1.0 - ((1.0 - sh) * (double)(nelem / (nelem - 1)));
            }
            a.nhaps[(size_t)w * P + i] = nh;
            a.hdiv[(size_t)w * P + i] = hd;
        }
        __syncthreads();   // hdiv visible to the EHHS step of this block
    }

    // ---- per-population passes over the site types
    for (int pi = 0; pi < P; ++pi) {
        const uint64_t mask = a.pop_mask[pi];
        const int np = a.pop_nsmpl[pi];
        const size_t oi = (size_t)w * P + pi;

        if (an & (PBA_SFS | PBA_DIVERGE_POP | PBA_THETA_W | PBA_FULI)) {
            __syncthreads();
            for (int i = tid; i < 66; i += PB_ST_THREADS) sfs_s[i] = 0;
            __syncthreads();
            int seg = 0, fixed = 0;
            for (int s = tid; s < S; s += PB_ST_THREADS) {
                const uint64_t t = T[s];
                int f = __popcll(t & mask);
                if (outg && (t >> a.outidx & 1)) f = np - f;
                if (f >= 0 && f <= np) atomicAdd(&sfs_s[f], 1);
                seg += (f > 0 && f < np);
                fixed += (f == np);
            }
            seg = pb_block_sum_int(seg, shi);
            fixed = pb_block_sum_int(fixed, shi);
            __syncthreads();
            if (tid == 0) {
                if (an & PBA_DIVERGE_POP) { a.div_num_snps[oi] = seg; a.pop_div[oi] = (uint16_t)fixed; }
                if (an & PBA_SFS) {
                    a.sfs_num_snps[oi] = seg;
                    double td = 0.0, fwh = 0.0;
                    const int ns = seg, m = np;
                    if (ns > 0 && m > 1) {
                        double a1 = 0.0, a2 = 0.0, a2n1 = 0.0;
                        for (int j = 1; j < m; ++j) a1 += 1.0 / (double)j;
                        for (int j = 1; j < m; ++j) a2 += 1.0 / (double)(j * j);
                        for (int j = 1; j < m + 1; ++j) a2n1 += 1.0 / (double)(j * j);
                        const double b1 = (m + 1.0) / (3.0 * (m - 1));
                        const double e1 = (b1 - (1.0 / a1)) / a1;
                        const double b2 = (2.0 * ((m * m) + m + 3.0)) / (9.0 * m * (m - 1));
                        const double e2 = (b2 - ((m + 2.0) / (a1 * m)) + (a2 / (a1 * a1))) / ((a1 * a1) + a2);
                        for (int j = 1; j < m; ++j) {
                            td += sfs_s[j] * (((2.0 * j * (m - j)) / (m * (m - 1))) - (1.0 / a1));
                            fwh += sfs_s[j] * ((1.0 / a1) - ((double)j / (m - 1)));
                        }
                        td /= sqrt(e1 * ns + e2 * ns * (ns - 1));
                        fwh /= sqrt(((m - 2) * (ns / a1) / (6.0 * (m - 1))) +
                                    ((ns * (ns - 1) / ((a1 * a1) + a2)) *
                                     (18.0 * (m * m) * (3.0 * m + 2.0) * a2n1 - (88.0 * m * m * m + 9.0 * (m * m) - 13.0 * m + 6.0)) /
                                     (9.0 * m * ((m - 1) * (m - 1)))));
                    } else { td = nan(""); fwh = nan(""); }
                    a.td[oi] = td; a.fwh[oi] = fwh;
                }
                if (an & (PBA_THETA_W | PBA_FULI)) {
                    const bool fl = (an & PBA_FULI) != 0;
                    pb_sfs_ext(np, seg, sfs_s[1], sfs_s[np > 0 ? np - 1 : 0], outg, a.pop_segsites + oi, (an & PBA_THETA_W) ? a.theta_w + oi : nullptr,
                               fl ? a.fuli_d + oi : nullptr, fl ? a.fuli_ds + oi : nullptr, fl ? a.fuli_eta_e + oi : nullptr, fl ? a.fuli_eta_s + oi : nullptr);
                }
            }
        }

        if (an & PBA_HAPLO_EHHS) {
            double e = nan("");
            if (np >= 4) {   // uniform across the block
                uint64_t *lt = a.kt + so + w;
                uint8_t *lm = a.km + so + w;
                int dummy;
                __syncthreads();
                const int L = pb_compact_sites(T, S, mask, [=](uint64_t, int m) { return m > 1 && m < np - 1; }, lt, lm, 0, &dummy, shu);
                __syncthreads();
                // most frequent partition; ties -> smallest value (first in ascending order)
                unsigned long long bm = 0, bt = 0;
                for (int i = tid; i < L; i += PB_ST_THREADS) {
                    const uint64_t t = lt[i];
                    unsigned long long mult = 0;
                    for (int k = 0; k < L; ++k) mult += lt[k] == t;
                    if (mult > bm || (mult == bm && t < bt)) { bm = mult; bt = t; }
                }
                for (int o = 16; o > 0; o >>= 1) {
                    const unsigned long long om = __shfl_xor_sync(0xffffffffu, bm, o), ot = __shfl_xor_sync(0xffffffffu, bt, o);
                    if (om > bm || (om == bm && om > 0 && ot < bt)) { bm = om; bt = ot; }
                }
                __shared__ unsigned long long wm[8], wt[8];
                if ((tid & 31) == 0) { wm[tid >> 5] = bm; wt[tid >> 5] = bt; }
                __syncthreads();
                if (tid == 0) {
                    for (int i = 1; i < PB_ST_THREADS / 32; ++i)
                        if (wm[i] > bm || (wm[i] == bm && wm[i] > 0 && wt[i] < bt)) { bm = wm[i]; bt = wt[i]; }
                    const int f = bm > 0 ? __popcll(bt) : 0;
                    const double sh = (1.0 - ((double)((f * f) + ((np - f) * (np - f))) / (np * np))) * (double)(np / (np - 1));
                    e = a.hdiv[oi] / (1.0 - sh);
                }
            }
            if (tid == 0) a.ehhs[oi] = e;
        }
    }

    // ---- Wall's B and Q: sequential, one `last` shared by all populations (SURVEY Q12)
    if ((an & PBA_LD_WALL) && tid == 0) {
        int ncong[64], npart[64], nsnp[64], nu[64];
        for (int j = 0; j < P; ++j) { ncong[j] = npart[j] = nsnp[j] = nu[j] = 0; }
        uint64_t last = 0;
        for (int i = 0; i < S; ++i) {
            const uint64_t t = T[i];
            for (int j = 0; j < P; ++j) {
                const uint64_t mk = a.pop_mask[j], type = t & mk, comp = ~t & mk;
                if (type > 0 && type < mk) {
                    uint64_t *U = a.wall_u + (size_t)j * a.s_total + so;
                    if (nsnp[j] == 0) { U[nu[j]++] = type; last = type; nsnp[j] = 1; }
                    else {
                        if (type == last || comp == last) {
                            ++ncong[j];
                            bool seen = false;
                            for (int u = 0; u < nu[j] && !seen; ++u) seen = (U[u] == type) || (U[u] == comp);
                            if (!seen) { U[nu[j]++] = type; ++npart[j]; }
                        }
                        ++nsnp[j];
                        last = type;
                    }
                }
            }
        }
        for (int j = 0; j < P; ++j) {
            const size_t oj = (size_t)w * P + j;
            a.wall_num_snps[oj] = S < 1 ? 0 : nsnp[j];
            a.wallb[oj] = S < 1 ? 0.0 : (double)ncong[j] / (double)(nsnp[j] - 1);
            a.wallq[oj] = S < 1 ? 0.0 : (double)(ncong[j] + npart[j]) / nsnp[j];
        }
    }
}
