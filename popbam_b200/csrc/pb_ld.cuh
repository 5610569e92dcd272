// pb_ld.cuh -- pairwise linkage disequilibrium of a window's segregating sites (ld -o 0 / -o 1):
// calc_zns (pop_ld.cpp:201-252) and calc_omegamax (pop_ld.cpp:254-373).
//
// The data: one 64-bit word per SNP (bit i = sample i carries the derived allele), masked by the
// population.  A pair needs popcount(t_j & t_k) and the two marginal counts; with n = samples of the
// population, m = marginal counts, n11 = joint count:
//     r^2 = (x11 - x0 x1)^2 / (x0 (1-x0) x1 (1-x1)) = (n n11 - m_j m_k)^2 / (m_j (n-m_j) m_k (n-m_k))
// i.e. an INTEGER numerator (|.| <= 64*64) times two per-SNP reciprocals.  So the O(S^2) pair loop is
// bit work: AND, POPC, IMAD, one int->double conversion and a double multiply-add per pair -- no
// tensor-core shape anywhere (a 64-bit bitset intersection count is not a dense float contraction),
// operands broadcast from shared memory.  profiles/ has the ncu pipe utilisation of k_ld_rows.
//
//   k_ld_keep    grid (pop x window): ordered compaction of the SNPs with min_freq <= m <= n - min_freq
//                (kept index == the reference's count1/count2 matrix index), S' counting rule (SURVEY Q10)
//   k_ld_rows    grid (row block x pop x window): thread = kept SNP i; tiles of 256 partner SNPs staged in
//                shared memory; Lsum_i = sum_{k<i} r^2, Rsum_i = sum_{k>i} r^2 (ZnS only needs Rsum)
//   k_ld_finish  grid (pop x window): ZnS = 2/(S'(S'-1)) * sum Rsum; omega_max by the running-sum scan
//                of SURVEY Q11 expressed through Lsum/Rsum (no S x S matrix, no O(S^3) loop)
// Extension (no reference counterpart, PB_AN_LD_DPRIME): Lewontin's |D'| = |num| / Dmax over the same kept pairs, with
// num = n n11 - m_j m_k and Dmax = min(m_j (n-m_k), (n-m_j) m_k) if num > 0, else min(m_j m_k, (n-m_j)(n-m_k)): an integer in
// [1, n^2/4] = [1, 1024], so the division is a multiply by a shared-memory table of 1/k.  k_ld_rows<true> adds the sum of
// |D'| and the number of pairs with |num| = Dmax (complete LD) over k > i to every row; k_ld_rows<false> (ZnS / omega only)
// is the kernel without them.
// The summation ORDER differs from the reference's (parallel partial sums; r^2 through reciprocals):
// relative differences ~1e-15, inside the 1e-9 tolerance of the parity contract.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define PB_LD_THREADS 256

struct PbLdArgs {
    int P;
    uint64_t pop_mask[64];
    uint8_t pop_nsmpl[64];
    int min_freq;
    uint32_t analyses;
    const int32_t *segsites;
    const int64_t *seg_off;
    const uint64_t *seg_type;
    int64_t stride;           // per-population stride of the scratch arrays (S_total + 2*NW + 2)
    // scratch [P][stride], window w at offset seg_off[w] + 2*w
    uint64_t *kt;             // kept, masked types
    int32_t *km;              // marginal counts
    double *kinv;             // 1 / (m (n - m))
    double *lsum, *rsum;
    int32_t *kcount;          // [NW][P] kept SNPs
    int32_t *nsnps;           // [NW][P] S' of the reference's counting rule
    double *dpsum;            // per row: sum of |D'| over k > i       (PB_AN_LD_DPRIME)
    int32_t *dpfull;          // per row: pairs k > i in complete LD   (PB_AN_LD_DPRIME)
    // outputs
    int32_t *ld_num_snps;
    double *zns, *omegamax;
    int32_t *ld_kept; double *ld_dprime; int64_t *ld_complete;
};

__global__ void __launch_bounds__(PB_LD_THREADS) k_ld_keep(const PbLdArgs a) {
    __shared__ int wsum[PB_LD_THREADS / 32];
    const int p = (int)(blockIdx.x % a.P), w = (int)(blockIdx.x / a.P), tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int S = a.segsites[w];
    const int64_t so = a.seg_off[w];
    const uint64_t *__restrict__ T = a.seg_type + so;
    const uint64_t mask = a.pop_mask[p];
    const int np = a.pop_nsmpl[p], mf = a.min_freq;
    const size_t base = (size_t)p * a.stride + (size_t)so + 2 * (size_t)w;
    int carry = 0, before = 0;
    for (int b0 = 0; b0 < S; b0 += PB_LD_THREADS) {
        const int s = b0 + tid;
        uint64_t t = 0; int m = 0; bool keep = false;
        if (s < S) { t = T[s] & mask; m = __popcll(t); keep = m >= mf && m <= np - mf; }
        const uint32_t bal = __ballot_sync(0xffffffffu, keep);
        const uint32_t bal_before = __ballot_sync(0xffffffffu, keep && s < S - 1);
        __syncthreads();
        if (lane == 0) wsum[wid] = __popc(bal) | (__popc(bal_before) << 16);
        __syncthreads();
        int pre = 0, tot = 0, totb = 0;
        for (int i = 0; i < PB_LD_THREADS / 32; ++i) { const int v = wsum[i]; if (i < wid) pre += v & 0xffff; tot += v & 0xffff; totb += v >> 16; }
        if (keep) {
            const size_t d = base + carry + pre + __popc(bal & ((1u << lane) - 1u));
            a.kt[d] = t; a.km[d] = m; a.kinv[d] = 1.0 / ((double)m * (double)(np - m));
        }
        carry += tot; before += totb;
    }
    if (tid == 0) {
        a.kcount[(size_t)w * a.P + p] = carry;
        a.nsnps[(size_t)w * a.P + p] = S < 1 ? 0 : before + 1;      // sites 0..S-2 counted when kept, then +1 (SURVEY Q10)
    }
}

// exact int -> double for 0 <= n < 2^32 on the FP64 pipe (exponent-bias trick) instead of a conversion on the
// XU pipe, which the two POPCs of every pair already keep busy (profiles/r1_ld_rows_raw.txt)
__device__ __forceinline__ double pb_u2d(unsigned n) { return __hiloint2double(0x43300000, (int)n) - 4503599627370496.0; }

template <bool DPRIME>
__global__ void __launch_bounds__(PB_LD_THREADS) k_ld_rows(const PbLdArgs a, int need_left, int n_row_blocks) {
    __shared__ uint64_t st[PB_LD_THREADS];
    __shared__ double sinv[PB_LD_THREADS];
    __shared__ int sm[PB_LD_THREADS];
    const int rb = (int)(blockIdx.x % n_row_blocks), pw = (int)(blockIdx.x / n_row_blocks);
    const int p = pw % a.P, w = pw / a.P, tid = threadIdx.x;
    const int K = a.kcount[(size_t)w * a.P + p];
    const int i0 = rb * PB_LD_THREADS;
    if (i0 >= K) return;
    const size_t base = (size_t)p * a.stride + (size_t)a.seg_off[w] + 2 * (size_t)w;
    const int np = a.pop_nsmpl[p];
    const int i = i0 + tid;
    const bool live = i < K;
    const uint64_t ti = live ? a.kt[base + i] : 0;
    const int mi = live ? a.km[base + i] : 0;
    double l = 0.0, r = 0.0;
    double dps = 0.0;      // DPRIME: sum of |D'| over the partners k > i
    int dpf = 0;           //         partners k > i in complete LD
    double *dinv = nullptr;
    if constexpr (DPRIME) {
        __shared__ double dtab[1025];      // 1/k, k = Dmax <= np^2/4 <= 1024
        for (int k = tid; k <= (np * np) / 4; k += PB_LD_THREADS) dtab[k] = k ? 1.0 / (double)k : 0.0;
        dinv = dtab;       // (visible after the first tile's barrier)
    }
    // |D'| of the pair (i, k) from its numerator and the partner's marginal count
    auto dprime = [&](int num, int mk) {
        const int dmax = num > 0 ? min(mi * (np - mk), (np - mi) * mk) : min(mi * mk, (np - mi) * (np - mk));
        const int an = abs(num);
        dps = fma(pb_u2d((unsigned)an), dinv[dmax], dps);
        dpf += an == dmax;
    };
    // partner tiles: all of them for omega (left and right sums), only those at or right of the diagonal for ZnS
    for (int k0 = need_left ? 0 : i0; k0 < K; k0 += PB_LD_THREADS) {
        __syncthreads();
        if (k0 + tid < K) { st[tid] = a.kt[base + k0 + tid]; sinv[tid] = a.kinv[base + k0 + tid]; sm[tid] = a.km[base + k0 + tid]; }
        __syncthreads();
        const int kn = min(PB_LD_THREADS, K - k0);
        if (k0 + kn <= i0) {                       // tile entirely left of every row of this block
#pragma unroll 4
            for (int k = 0; k < kn; ++k) {
                const int num = np * __popcll(ti & st[k]) - mi * sm[k];
                l = fma(pb_u2d((unsigned)(num * num)), sinv[k], l);
            }
        } else if (k0 >= i0 + PB_LD_THREADS) {     // entirely right
#pragma unroll 4
            for (int k = 0; k < kn; ++k) {
                const int num = np * __popcll(ti & st[k]) - mi * sm[k];
                r = fma(pb_u2d((unsigned)(num * num)), sinv[k], r);
                if constexpr (DPRIME) dprime(num, sm[k]);
            }
        } else {                                   // the diagonal tile
            for (int k = 0; k < kn; ++k) {
                const int num = np * __popcll(ti & st[k]) - mi * sm[k];
                const double v = pb_u2d((unsigned)(num * num)) * sinv[k];
                if (k0 + k < i) l += v;
                else if (k0 + k > i) {
                    r += v;
                    if constexpr (DPRIME) dprime(num, sm[k]);
                }
            }
        }
    }
    if (live) {
        const double inv_i = a.kinv[base + i];
        a.rsum[base + i] = r * inv_i;
        if (need_left) a.lsum[base + i] = l * inv_i;
        if constexpr (DPRIME) { a.dpsum[base + i] = dps; a.dpfull[base + i] = dpf; }
    }
}

__global__ void __launch_bounds__(PB_LD_THREADS) k_ld_finish(const PbLdArgs a) {
    __shared__ double sh[PB_LD_THREADS / 32];
    const int p = (int)(blockIdx.x % a.P), w = (int)(blockIdx.x / a.P), tid = threadIdx.x;
    const size_t oi = (size_t)w * a.P + p;
    const int K = a.kcount[oi], ns = a.nsnps[oi], S = a.segsites[w];
    const size_t base = (size_t)p * a.stride + (size_t)a.seg_off[w] + 2 * (size_t)w;
    double part = 0.0;
    for (int i = tid; i < K; i += PB_LD_THREADS) part += a.rsum[base + i];
    for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
    if ((tid & 31) == 0) sh[tid >> 5] = part;
    if (a.analyses & 0x4000u) {                    // PB_AN_LD_DPRIME: mean |D'| and complete pairs over the K(K-1)/2 pairs
        __shared__ double shd[PB_LD_THREADS / 32];
        __shared__ long long shf[PB_LD_THREADS / 32];
        double dp = 0.0;
        long long full = 0;
        for (int i = tid; i < K; i += PB_LD_THREADS) { dp += a.dpsum[base + i]; full += a.dpfull[base + i]; }
        for (int o = 16; o > 0; o >>= 1) { dp += __shfl_xor_sync(0xffffffffu, dp, o); full += __shfl_xor_sync(0xffffffffu, full, o); }
        if ((tid & 31) == 0) { shd[tid >> 5] = dp; shf[tid >> 5] = full; }
        __syncthreads();
        if (tid == 0) {
            dp = 0.0; full = 0;
            for (int i = 0; i < PB_LD_THREADS / 32; ++i) { dp += shd[i]; full += shf[i]; }
            a.ld_kept[oi] = K;
            a.ld_dprime[oi] = K < 2 ? nan("") : dp / ((double)K * (double)(K - 1) / 2.0);
            a.ld_complete[oi] = full;
        }
    }
    __syncthreads();
    if (tid != 0) return;
    double total = 0.0;
    for (int i = 0; i < PB_LD_THREADS / 32; ++i) total += sh[i];
    a.ld_num_snps[oi] = ns;
    if (a.analyses & 0x004u) a.zns[oi] = S < 1 ? 0.0 : total * (2.0 / (double)(ns * (ns - 1)));
    if (a.analyses & 0x008u) {
        double om = 0.0;
        if (S >= 1) {
            double *lsum = a.lsum + base, *rsum = a.rsum + base;
            for (int i = K; i < ns; ++i) { lsum[i] = 0.0; rsum[i] = 0.0; }      // phantom index: last site not kept
            // sl / sb / sr are running totals over the split points (never reset, SURVEY Q11):
            //   wl(i) pairs inside [0,i], x(i) pairs across the split after i, wr(i) pairs inside [i+1, ns)
            // wr(i) as a suffix sum (kinv[] is free by now: scratch), not as "total minus prefix": the subtraction would
            // cancel towards the right end of the window
            double *suf = a.kinv + base;
            { double acc = 0.0; for (int i = ns - 1; i >= 0; --i) { suf[i] = acc; acc += rsum[i]; } }      // suf[i] = sum of rsum over (i, ns)
            double sl = 0.0, sb = 0.0, sr = 0.0, wl = 0.0, pr = 0.0, pl = 0.0;
            for (int i = 0; i < ns - 1; ++i) {
                wl += lsum[i];
                pr += rsum[i]; pl += lsum[i];
                const double x = pr - pl, wr = suf[i];   // pairs across the split after i; pairs whose smaller index is > i
                if (i == 0) continue;
                sl += wl; sb += x; sr += wr;
                const int left = i + 1, right = ns - left;
                double omega = (sl + sr) / (((left * (left - 1)) / 2.0) + ((right * (right - 1)) / 2.0));
                omega *= left * right / sb;
                om = omega > om ? omega : om;
            }
        }
        a.omegamax[oi] = om;
    }
}
