// pb_kernels.cuh -- sm_100a kernels of the pileup -> consensus call -> per-site path.
//
//   k_rebase          batch-relative offsets -> absolute device offsets                      (per read)
//   k_read_prep       bam_plp_push filter + bam_calend, read-start bins                       (per read)
//   k_depth_bound / k_depth_decide    can the raw-depth cap of call_base ever bind?
//   k_qual_mask       which base qualities occur                                              (per base, streaming)
//   k_level_table / k_qual_table / k_need_table / k_rms_table    per-region / per-context lookup tables
//   k_encode          the per-base filter + code of call_base, once per base                  (per base, streaming)
//   k_part_count / k_part_scatter     stable partition of the reads by sample (file order kept), CIGAR -> segments
//   k_pileup_call     pileup, per-(site,sample) call, per-site logic                          (the hot kernel)
//   k_window_sites    order-preserving compaction into num_sites / segregating-site lists
//   k_scan_*          exclusive scans
//
// Reference code these replace: bam_plbuf_push/bam_plp_push/bam_plp_next/resolve_cigar2
// (bam_pileup.c:523,365,283,90), popbamData::call_base (popbam.cpp:186-313), errmod_cal/gl2cns
// (pop_utils.cpp:280-365, :66-100), clean_heterozygotes/segbase/qfilter (pop_utils.cpp:170-201,
// :122-168, :102-120), make_nucdiv and its five clones (pop_nucdiv.cpp:136-204).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "pb_cell.cuh"
#include "pb_walk.cuh"

#define PB_REC_DEAD (1u << 25)    // read fails min_mapQ: it only counts towards the raw-depth cap
#define PB_BIN_SHIFT 7            // read-start bins of the depth bound (128 bp)
#define PB_PART_CHUNK 512         // reads per warp in the sample partition
#define PB_KEY_DROP 0xffu
#define PB_CODE_NONE 0xffu        // base filtered out (quality, N)
#define PB_MAX_SEGS 255           // aligned segments (M/=/X ops) per read

struct PbCounters {               // device-side region counters (one cudaMemcpy back)
    unsigned long long reads_used;
    unsigned long long aligned_bases;
    unsigned long long mapq_mask;     // bit min(mapq,63) for kept reads passing min_mapQ
    unsigned long long qual_mask;     // bit min(baseQ',63) for base qualities passing min_baseQ
    int max_span;                     // max reference span of a kept read
    int unsorted;                     // pos[r] < pos[r-1] seen (bam_pileup.c:384-395)
    int n_levels;
    int too_long;                     // a read spans >= 65536 reference bases or has > 255 aligned segments
    int depth_bound;                  // upper bound of the raw per-sample depth at any position
    int nocap;                        // depth_bound <= max_depth: the raw-depth cap can never bind
    unsigned char qrank[64];          // quality value -> level
    unsigned char qval[64];           // level -> quality value (ascending)
    // counting path (pb_pile.cuh): the cells it hands to k_hard_cells, and the assumptions it verified
    unsigned long long n_cells;       // directory entries written
    unsigned long long n_codes;       // base-code slots reserved in the arena
    int arena_overflow;               // the directory or the code arena was too small: results incomplete
    int spec_fail;                    // launched for a smaller max_span, or the depth cap can bind after all
    int qual_over;                    // a base quality above the assumed ceiling was seen ...
    int qual_max_seen;                // ... and this is the largest (adjusted) one
    int qual_high;                    // a quality byte >= 128 was seen by the kernel variant that assumes there is none
    unsigned int n_records;           // aligned-segment records of the region (all samples)
    int total_bound;                  // upper bound of the reads of ALL samples live at one position (bam_pileup.c:260,375: maxcnt)
    int max_read_bytes;               // most bytes of qual[] one read takes (its padding included)
};

// ------------------------------------------------------------------------------------------------
__global__ void k_rebase(int64_t n, int64_t r0, const uint32_t *__restrict__ cig_off, const uint32_t *__restrict__ base_off,
                         uint64_t cig_base, uint64_t byte_base, uint32_t *__restrict__ cigstart, uint32_t *__restrict__ ncig,
                         uint64_t *__restrict__ base) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    cigstart[r0 + i] = (uint32_t)(cig_base + cig_off[i]);
    ncig[r0 + i] = cig_off[i + 1] - cig_off[i];
    base[r0 + i] = byte_base + base_off[i];
}

// bam_plp_push (bam_pileup.c:371-374): drop flag & 0x704; bam_calend (bam.c:20-70): reference end.
// Also counts the read's aligned segments (M/=/X ops): each becomes one record of the hot kernel.
__global__ void __launch_bounds__(256) k_read_prep(int64_t n, const int32_t *__restrict__ pos, const uint32_t *__restrict__ meta,
                                                   const uint32_t *__restrict__ cigstart, const uint32_t *__restrict__ ncig,
                                                   const uint32_t *__restrict__ cigar, const uint64_t *__restrict__ base, uint64_t n_bytes,
                                                   int n_samples, int min_mapQ, uint8_t *__restrict__ rkey, uint8_t *__restrict__ rnseg,
                                                   int bin_origin, int n_bins, int span_end, uint32_t *__restrict__ bins,
                                                   PbCounters *__restrict__ ctr) {
    unsigned long long used = 0, aligned = 0, mqmask = 0;
    int span = 0, flags = 0, rbytes = 0;     // flags: 1 unsorted, 2 too long
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += (int64_t)gridDim.x * blockDim.x) {
        const uint32_t m = meta[r];
        {
            const uint64_t b0 = base[r], b1 = r + 1 < n ? base[r + 1] : n_bytes;
            rbytes = max(rbytes, b1 >= b0 ? (int)min(b1 - b0, (uint64_t)0x7fffffff) : 0x7fffffff);
        }
        const int p = pos[r];
        const uint32_t c0 = cigstart[r], nc = ncig[r];
        int x = p, al = 0, nseg = 0;
        bool longseg = false;
        // branch-free per operation: M = X consume reference and query (bits 0, 7, 8 of the class masks), D N consume
        // reference (bits 2, 3).  Most reads have one operation, a few have five: the first is taken by all lanes together,
        // the loop behind it runs for the warp's longest list
        {
            const uint32_t c = nc ? __ldg(cigar + c0) : 0u;
            const int op = c & 15, len = (int)(c >> 4);
            const int aln = (0x181 >> op) & 1, ref = (0x18d >> op) & 1;
            x += len & -ref; al = len & -aln; nseg = aln & (len > 0); longseg = (aln & (len > 65535)) != 0;
        }
        for (uint32_t i = 1; i < nc; ++i) {
            const uint32_t c = __ldg(cigar + c0 + i);
            const int op = c & 15, len = (int)(c >> 4);
            const int aln = (0x181 >> op) & 1, ref = (0x18d >> op) & 1;
            x += len & -ref; al += len & -aln; nseg += aln & (len > 0); longseg |= (aln & (len > 65535)) != 0;
        }
        const bool keep = !((m >> 16) & 0x704u) && x > p;
        const uint32_t smp = m & 0xffu;
        const bool listed = keep && smp < (uint32_t)n_samples;
        rkey[r] = listed ? (uint8_t)smp : (uint8_t)PB_KEY_DROP;
        if (listed && (longseg || x - p > 65535 || nseg > PB_MAX_SEGS)) flags |= 2;
        rnseg[r] = (uint8_t)(nseg > PB_MAX_SEGS ? PB_MAX_SEGS : nseg);
        // read starts per (sample, 128 bp bin) for the depth bound; reads that end before the span or start behind it
        // cover none of its positions (bins start 65536 bp before the span: early starts clamp, still an upper bound)
        if (listed && p < span_end && x > bin_origin + 65536) {
            const int b = min(n_bins - 1, max(0, (p - bin_origin) >> PB_BIN_SHIFT));
            atomicAdd(&bins[(size_t)smp * n_bins + b], (uint32_t)(nseg > 0 ? nseg : 1));
        }
        if (keep) {
            used += 1; aligned += (unsigned long long)al; span = max(span, x - p);
            const int mq = (int)((m >> 8) & 0xff);
            if (mq >= min_mapQ) mqmask |= 1ULL << (mq > 63 ? 63 : mq);
        }
        if (r > 0 && p < pos[r - 1]) flags |= 1;
    }
    // warp-aggregate, block-aggregate, then one atomic per counter per block
    for (int o = 16; o > 0; o >>= 1) {
        used += __shfl_xor_sync(0xffffffffu, used, o);
        aligned += __shfl_xor_sync(0xffffffffu, aligned, o);
        mqmask |= __shfl_xor_sync(0xffffffffu, mqmask, o);
        span = max(span, __shfl_xor_sync(0xffffffffu, span, o));
        rbytes = max(rbytes, __shfl_xor_sync(0xffffffffu, rbytes, o));
        flags |= __shfl_xor_sync(0xffffffffu, flags, o);
    }
    __shared__ unsigned long long s_used[8], s_al[8], s_mq[8];
    __shared__ int s_span[8], s_flags[8], s_rb[8];
    const int wid = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0) { s_used[wid] = used; s_al[wid] = aligned; s_mq[wid] = mqmask; s_span[wid] = span; s_flags[wid] = flags; s_rb[wid] = rbytes; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int i = 1; i < (int)(blockDim.x >> 5); ++i) { used += s_used[i]; aligned += s_al[i]; mqmask |= s_mq[i]; span = max(span, s_span[i]); flags |= s_flags[i]; rbytes = max(rbytes, s_rb[i]); }
        if (rbytes) atomicMax(&ctr->max_read_bytes, rbytes);
        if (used) atomicAdd(&ctr->reads_used, used);
        if (aligned) atomicAdd(&ctr->aligned_bases, aligned);
        if (mqmask) atomicOr(&ctr->mapq_mask, mqmask);
        if (span) atomicMax(&ctr->max_span, span);
        if (flags & 1) atomicOr(&ctr->unsorted, 1);
        if (flags & 2) atomicOr(&ctr->too_long, 1);
    }
}

// Upper bound of the raw depth of any (position, sample): the reads covering p start in (p - max_span, p],
// i.e. inside m+1 consecutive 128 bp bins with m = ceil(max_span / 128).  When the bound does not exceed
// max_depth the cap of call_base (popbam.cpp:242-248) can never bind, reads below min_mapQ contribute
// nothing at all, and the hot kernel runs without depth bookkeeping.
__global__ void __launch_bounds__(256) k_depth_bound(const uint32_t *__restrict__ bins, int n_samples, int n_bins, int max_depth,
                                                     const int32_t *__restrict__ pos, int64_t n_reads, PbCounters *__restrict__ ctr) {
    const int m = (ctr->max_span + (1 << PB_BIN_SHIFT) - 1) >> PB_BIN_SHIFT;
    const int64_t total = (int64_t)n_samples * n_bins;
    uint32_t best = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int b = (int)(i % n_bins);
        uint32_t sum = 0;
        for (int d = 0; d <= m && d <= b; ++d) sum += bins[i - d];
        best = max(best, sum);
    }
    for (int o = 16; o > 0; o >>= 1) best = max(best, __shfl_xor_sync(0xffffffffu, best, o));
    if ((threadIdx.x & 31) == 0 && best) atomicMax(&ctr->depth_bound, (int)min(best, 0x7fffffffu));
    // bam_plp_push stops taking reads that start at the current position once more than 8000 nodes are live
    // (bam_pileup.c:260,375; its count includes three bookkeeping nodes); the host refuses a region where that could
    // happen.  Live when read r is pushed: at most the reads that start in (pos[r] - max_span, pos[r]].  One binary
    // search per 256 consecutive reads bounds that for all of them.
    const int ms = ctr->max_span;
    int tbest = 0;
    for (int64_t ch = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; ch * 256 < n_reads; ch += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r0 = ch * 256, r1 = min(n_reads, r0 + 256);
        const int thr = pos[r0] - ms;                      // live reads start after thr
        int64_t lo = 0, hi = r0;
        while (lo < hi) { const int64_t mid = (lo + hi) >> 1; if (pos[mid] > thr) hi = mid; else lo = mid + 1; }
        tbest = max(tbest, (int)min((int64_t)0x7ffffff0, r1 - lo) + 3);
    }
    for (int o = 16; o > 0; o >>= 1) tbest = max(tbest, __shfl_xor_sync(0xffffffffu, tbest, o));
    if ((threadIdx.x & 31) == 0 && tbest) atomicMax(&ctr->total_bound, tbest);
}
__global__ void k_depth_decide(int max_depth, PbCounters *ctr) { ctr->nocap = ctr->depth_bound <= max_depth ? 1 : 0; }

// Which (adjusted) base qualities >= min_baseQ occur anywhere in the batch (superset of what the
// pileup will use: clipped / inserted / padding bytes are included, harmlessly).  Streaming pass over
// qual[]: every byte sets a presence flag in a 256-byte shared-memory table (two instructions per
// byte; equal values hit the same address, so the stores do not conflict), one reduction per block.
__global__ void __launch_bounds__(256) k_qual_mask(const uint8_t *__restrict__ qual, int64_t n_bytes, int illumina, int min_baseQ,
                                                   PbCounters *__restrict__ ctr) {
    __shared__ uint8_t seen[256];
    seen[threadIdx.x] = 0;
    __syncthreads();
    const int64_t nvec = n_bytes >> 4;
    const uint4 *q4 = reinterpret_cast<const uint4 *>(qual);
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += 4 * stride) {
        uint4 v[4];
#pragma unroll
        for (int t = 0; t < 4; ++t) v[t] = i + t * stride < nvec ? __ldg(q4 + i + t * stride) : make_uint4(0, 0, 0, 0);
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            const uint32_t w[4] = {v[t].x, v[t].y, v[t].z, v[t].w};
#pragma unroll
            for (int j = 0; j < 4; ++j)
#pragma unroll
                for (int b = 0; b < 4; ++b) seen[(w[j] >> (8 * b)) & 0xffu] = 1;
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0)
        for (int64_t i = nvec << 4; i < n_bytes; ++i) seen[qual[i]] = 1;
    __syncthreads();
    // one thread per raw quality value: transform, filter, clamp
    unsigned long long mask = 0;
    if (seen[threadIdx.x]) {
        int q = (int)threadIdx.x;
        if (illumina) q = q > 31 ? q - 31 : 0;
        if (q >= min_baseQ) mask = 1ULL << (q > 63 ? 63 : q);
    }
    for (int o = 16; o > 0; o >>= 1) mask |= __shfl_xor_sync(0xffffffffu, mask, o);
    if ((threadIdx.x & 31) == 0 && mask) atomicOr(&ctr->qual_mask, mask);
}

// Distinct values of clamp(min(baseQ, mapQ), 4, 63) (popbam.cpp:279-283) that can occur.
__global__ void k_level_table(PbCounters *ctr) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    const unsigned long long A = ctr->qual_mask, B = ctr->mapq_mask;
    unsigned long long L = 0;
    for (int a = 0; a < 64; ++a) {
        if (!(A >> a & 1)) continue;
        for (int b = 0; b < 64; ++b) {
            if (!(B >> b & 1)) continue;
            int q = a < b ? a : b;
            if (q < 4) q = 4;
            L |= 1ULL << q;
        }
    }
    int nl = 0;
    for (int q = 0; q < 64; ++q) {
        ctr->qrank[q] = (unsigned char)nl;
        if (L >> q & 1) ctr->qval[nl++] = (unsigned char)q;
    }
    ctr->n_levels = nl;
}

// rms_thr[k]: the smallest sum of squared mapping qualities for which call_base's
//     rms = (u64)(sqrtf((float)rmsq / k) + 0.499)           (popbam.cpp:292)
// reaches min_rmsQ with k bases -- every step of that expression is monotone in rmsq, so qfilter's
// rms >= min_rmsQ (pop_utils.cpp:110) is one integer compare for the cells that need nothing else.
__global__ void k_rms_table(int min_rmsQ, int32_t *__restrict__ rms_thr /* [256] */) {
    const int k = threadIdx.x;
    if (k == 0 || min_rmsQ <= 0) { rms_thr[k] = 0; return; }
    auto rms_of = [&](int rmsq) -> uint64_t { return (uint64_t)PB_DADD((double)PB_FSQRT(PB_FDIV((float)rmsq, (float)k)), 0.499); };
    int lo = 0, hi = 255 * 255 * 255 + 1;       // first rmsq with rms >= min_rmsQ (hi: unreachable -> never passes)
    if (rms_of(hi - 1) < (uint64_t)min_rmsQ) { rms_thr[k] = 0x7fffffff; return; }
    while (lo < hi) { const int mid = lo + ((hi - lo) >> 1); if (rms_of(mid) >= (uint64_t)min_rmsQ) hi = mid; else lo = mid + 1; }
    rms_thr[k] = lo;
}

// need[L][k] of pb_need_entry for every level of the region and every depth: one thread per entry.
__global__ void __launch_bounds__(256) k_need_table(const PbCounters *__restrict__ ctr, const double *__restrict__ fk,
                                                    const double *__restrict__ beta, const double *__restrict__ lhet,
                                                    uint8_t *__restrict__ need /* [64][256] */) {
    const int L = blockIdx.x, k = threadIdx.x, nl = ctr->n_levels;
    need[L * 256 + k] = L < nl ? pb_need_entry(L, nl, ctr->qval, k, fk, beta, lhet) : 0;
}

// Quality table of the encode pass: qtab[min(mapQ,63)][raw quality byte] = level(clamp(min(baseQ', mapQ),4,63)) << 2,
// or PB_CODE_NONE when baseQ' < min_baseQ (baseQ' = Illumina-adjusted quality, popbam.cpp:268-283).
__global__ void __launch_bounds__(256) k_qual_table(const PbCounters *__restrict__ ctr, int illumina, int min_baseQ,
                                                    uint8_t *__restrict__ qtab /* [64][256] */) {
    const int m = blockIdx.x, raw = threadIdx.x;
    int bq = raw;
    if (illumina) bq = bq > 31 ? bq - 31 : 0;
    const int qq = max(4, min(63, min(bq, m)));
    qtab[m * 256 + raw] = bq < min_baseQ ? (uint8_t)PB_CODE_NONE : (uint8_t)(ctr->qrank[qq] << 2);
}

// The base filter and code of call_base (popbam.cpp:268-284), once per base and OUTSIDE the
// latency-bound pileup loop:
//   code = level(clamp(min(baseQ', mapQ), 4, 63)) << 2 | nt4      or PB_CODE_NONE when the base is dropped
// (baseQ' < min_baseQ, not A/C/G/T, or the read is dropped / below min_mapQ).  A flat streaming pass
// with persistent CTAs: the 16 KB quality table and a 256-entry sequence-byte table sit in shared
// memory, each thread takes 64 consecutive bytes of qual[] per step (four 16-byte loads, 32 bytes of
// seq4[], four 16-byte stores), i.e. two table lookups and an OR per base.  The read owning a byte is
// found from base[] (reads are laid out back to back in file order) starting from a proportional
// guess, which is exact for equal-length reads.
#define PB_ENC_CHUNK 64
#define PB_QROW 260
__global__ void __launch_bounds__(256) k_encode(int64_t n, const uint32_t *__restrict__ meta, const uint8_t *__restrict__ rkey,
                                                const uint64_t *__restrict__ base, const uint8_t *__restrict__ seq4,
                                                const uint8_t *__restrict__ qual, int64_t n_bytes, double reads_per_byte,
                                                int min_mapQ, const uint8_t *__restrict__ qtab, uint8_t *__restrict__ codes) {
    // row stride 260: a stride of 256 bytes would put equal qualities of different rows in the same bank
    __shared__ __align__(16) uint8_t qtab_s[65 * PB_QROW];   // row 64: all PB_CODE_NONE (reads the pileup never looks at)
    __shared__ uint16_t seq_s[256];       // packed sequence byte -> nt4 of its two bases (0xff: not A/C/G/T), first base low
    for (int i = threadIdx.x; i < 64 * 256 / 4; i += 256) {
        const int row = i >> 6, w = i & 63;
        reinterpret_cast<uint32_t *>(qtab_s + row * PB_QROW)[w] = __ldg(reinterpret_cast<const uint32_t *>(qtab) + i);
    }
    qtab_s[64 * PB_QROW + threadIdx.x] = (uint8_t)PB_CODE_NONE;
    {
        const uint32_t hi = threadIdx.x >> 4, lo = threadIdx.x & 15;
        const uint32_t bh = (uint32_t)((PB_NT16_NT4_LUT >> (hi * 4)) & 0xf), bl = (uint32_t)((PB_NT16_NT4_LUT >> (lo * 4)) & 0xf);
        seq_s[threadIdx.x] = (uint16_t)((bh > 3 ? 0xffu : bh) | (bl > 3 ? 0xffu : bl) << 8);
    }
    __syncthreads();
    // quality-table row of a read: its mapQ row, or the all-NONE row when the read is dropped / below min_mapQ
    auto row_of = [&](int64_t rr) -> uint32_t {
        if (rr >= n || rkey[rr] == PB_KEY_DROP) return 64u * PB_QROW;
        const int mq = (int)((__ldg(meta + rr) >> 8) & 0xffu);
        return mq >= min_mapQ ? (uint32_t)min(mq, 63) * PB_QROW : 64u * PB_QROW;
    };
    const int64_t n_chunks = (n_bytes + PB_ENC_CHUNK - 1) / PB_ENC_CHUNK;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n_chunks; t += (int64_t)gridDim.x * blockDim.x) {
        const uint64_t o = (uint64_t)t * PB_ENC_CHUNK;
        const int nb = (int)min((uint64_t)PB_ENC_CHUNK, (uint64_t)n_bytes - o);
        // owner of byte o: last r with base[r] <= o
        int64_t lo = (int64_t)((double)o * reads_per_byte);
        if (lo >= n) lo = n - 1;
        int64_t hi = lo + 1, step = 1;
        while (lo > 0 && __ldg(base + lo) > o) { hi = lo; lo = max((int64_t)0, lo - step); step <<= 1; }
        step = 1;
        while (hi < n && __ldg(base + hi) <= o) { lo = hi; hi = min(n, hi + step); step <<= 1; }
        while (hi - lo > 1) { const int64_t mid = (lo + hi) >> 1; if (__ldg(base + mid) <= o) lo = mid; else hi = mid; }
        const int64_t r = lo;
        // at most one read boundary inside the chunk is handled without branches: bytes < cut use rowA, the rest rowB
        const uint64_t next = r + 1 < n ? __ldg(base + r + 1) : ~0ULL;
        const uint64_t next2 = r + 2 < n ? __ldg(base + r + 2) : ~0ULL;
        const uint32_t rowA = row_of(r);
        const uint32_t cut = next - o < (uint64_t)PB_ENC_CHUNK ? (uint32_t)(next - o) : (uint32_t)PB_ENC_CHUNK;
        const uint32_t rowB = cut < PB_ENC_CHUNK ? row_of(r + 1) : rowA;
        if (nb == PB_ENC_CHUNK && next2 - o >= (uint64_t)PB_ENC_CHUNK) {
            uint4 qv[4];
            uint4 sv[2];
#pragma unroll
            for (int v = 0; v < 4; ++v) qv[v] = __ldg(reinterpret_cast<const uint4 *>(qual + o) + v);
#pragma unroll
            for (int v = 0; v < 2; ++v) sv[v] = __ldg(reinterpret_cast<const uint4 *>(seq4 + (o >> 1)) + v);
#pragma unroll
            for (int v = 0; v < 4; ++v) {
                const uint32_t qw[4] = {qv[v].x, qv[v].y, qv[v].z, qv[v].w};
                const uint32_t sw[2] = {v & 1 ? sv[v >> 1].z : sv[v >> 1].x, v & 1 ? sv[v >> 1].w : sv[v >> 1].y};
                uint32_t out[4];
#pragma unroll
                for (int g = 0; g < 4; ++g) {
                    const uint32_t q4 = qw[g];
                    const uint32_t sb = sw[g >> 1] >> (16 * (g & 1));
                    const uint32_t b44 = (uint32_t)seq_s[sb & 0xffu] | (uint32_t)seq_s[(sb >> 8) & 0xffu] << 16;
                    const uint32_t i0 = 16 * v + 4 * g;
                    // 0xff in either half stays 0xff after the OR: PB_CODE_NONE
                    const uint32_t l4 = (uint32_t)qtab_s[(i0 + 0 < cut ? rowA : rowB) + (q4 & 0xffu)] |
                                        (uint32_t)qtab_s[(i0 + 1 < cut ? rowA : rowB) + ((q4 >> 8) & 0xffu)] << 8 |
                                        (uint32_t)qtab_s[(i0 + 2 < cut ? rowA : rowB) + ((q4 >> 16) & 0xffu)] << 16 |
                                        (uint32_t)qtab_s[(i0 + 3 < cut ? rowA : rowB) + (q4 >> 24)] << 24;
                    out[g] = l4 | b44;
                }
                reinterpret_cast<uint4 *>(codes + o)[v] = make_uint4(out[0], out[1], out[2], out[3]);
            }
        } else {
            // tail of the array, or reads shorter than the chunk (several boundaries): byte by byte
            int64_t rr = r;
            uint64_t nx = next;
            uint32_t row = rowA;
            for (int i = 0; i < nb; ++i) {
                while (o + i >= nx) {
                    ++rr;
                    nx = rr + 1 < n ? __ldg(base + rr + 1) : ~0ULL;
                    row = row_of(rr);
                }
                const uint32_t sbyte = seq4[(o + i) >> 1];
                const uint32_t b4 = (seq_s[sbyte] >> (8 * (int)((o + i) & 1))) & 0xffu;
                codes[o + i] = (uint8_t)((uint32_t)qtab_s[row + qual[o + i]] | b4);
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Stable partition of the kept reads by sample, expanding every read into its aligned segments.
// One warp owns PB_PART_CHUNK consecutive reads, so the order inside a (chunk, sample) bucket is file
// order; buckets are laid out sample-major, chunk-minor by an exclusive scan of the count matrix.
__global__ void __launch_bounds__(128) k_part_count(int64_t n, const uint8_t *__restrict__ rkey, const uint8_t *__restrict__ rnseg,
                             const uint32_t *__restrict__ meta, int min_mapQ, const PbCounters *__restrict__ ctr, int n_samples,
                             int64_t n_chunks, uint32_t *__restrict__ counts /* [n_samples][n_chunks] */) {
    __shared__ uint32_t cnt_s[4][PB_MAX_SAMPLES];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const bool drop_dead = ctr->nocap != 0;
    const int64_t chunk = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (chunk >= n_chunks) return;
    uint32_t *cnt = cnt_s[wid];                     // segments per sample in this warp's chunk
    cnt[lane] = 0; cnt[lane + 32] = 0;
    __syncwarp();
    const int64_t r0 = chunk * PB_PART_CHUNK;
    for (int i = 0; i < PB_PART_CHUNK; i += 32) {
        const int64_t r = r0 + i + lane;
        uint32_t key = r < n ? rkey[r] : PB_KEY_DROP;
        const uint32_t ns = r < n ? rnseg[r] : 0;
        if (drop_dead && key != PB_KEY_DROP && (int)((meta[r] >> 8) & 0xffu) < min_mapQ) key = PB_KEY_DROP;
        if (key != PB_KEY_DROP && ns) atomicAdd(&cnt[key], ns);
    }
    __syncwarp();
    if (lane < n_samples) counts[(int64_t)lane * n_chunks + chunk] = cnt[lane];
    if (lane + 32 < n_samples) counts[(int64_t)(lane + 32) * n_chunks + chunk] = cnt[lane + 32];
}

// Segment record (16 bytes):
//   x  read start (sort key of the list; all segments of a read carry it)
//   y  segment start (reference coordinate)
//   z  segment length (16 bits) | mapq<<16 | strand<<24 | dead<<25 | (offset bits 32..37)<<26
//   w  low 32 bits of the byte offset of the segment's first base in qual[] / codes[]
__global__ void __launch_bounds__(128) k_part_scatter(int64_t n, const uint8_t *__restrict__ rkey, const uint8_t *__restrict__ rnseg, int n_samples,
                               int64_t n_chunks, const uint32_t *__restrict__ offs /* scanned counts */,
                               const int32_t *__restrict__ pos, const uint32_t *__restrict__ meta, const uint64_t *__restrict__ base,
                               const uint32_t *__restrict__ cigstart, const uint32_t *__restrict__ ncig,
                               const uint32_t *__restrict__ cigar, int min_mapQ, const PbCounters *__restrict__ ctr,
                               int4 *__restrict__ srec) {
    __shared__ uint32_t cur_s[4][PB_MAX_SAMPLES];   // per warp: next free record slot of every sample
    __shared__ uint32_t ns_s[4][32];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const bool drop_dead = ctr->nocap != 0;
    const int64_t chunk = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (chunk >= n_chunks) return;
    uint32_t *cur = cur_s[wid], *nsw = ns_s[wid];
    cur[lane] = lane < n_samples ? offs[(int64_t)lane * n_chunks + chunk] : 0;
    cur[lane + 32] = lane + 32 < n_samples ? offs[(int64_t)(lane + 32) * n_chunks + chunk] : 0;
    const int64_t r0 = chunk * PB_PART_CHUNK;
    for (int i = 0; i < PB_PART_CHUNK; i += 32) {
        const int64_t r = r0 + i + lane;
        uint32_t key = r < n ? rkey[r] : PB_KEY_DROP;
        uint32_t ns = r < n ? rnseg[r] : 0;
        if (drop_dead && key != PB_KEY_DROP && (int)((meta[r] >> 8) & 0xffu) < min_mapQ) key = PB_KEY_DROP;
        if (key == PB_KEY_DROP) ns = 0;
        // my rank: segments of the earlier lanes with my key (file order inside a sample is kept)
        const uint32_t peers = __match_any_sync(0xffffffffu, key);
        nsw[lane] = ns;
        __syncwarp();
        // = number of earlier lanes with my key that emit a record, plus the extra records of the few reads with several
        // segments (a warp-uniform loop over those lanes instead of a per-lane loop over peers)
        const uint32_t lower = peers & ((1u << lane) - 1u);
        uint32_t rank = (uint32_t)__popc(lower & __ballot_sync(0xffffffffu, ns > 0));
        for (uint32_t multi = __ballot_sync(0xffffffffu, ns > 1); multi; multi &= multi - 1) {
            const int j = __ffs(multi) - 1;
            if ((lower >> j) & 1u) rank += nsw[j] - 1;
        }
        const uint32_t mine = key != PB_KEY_DROP ? cur[key] : 0u;
        __syncwarp();
        if (key != PB_KEY_DROP && (peers >> lane) == 1u) cur[key] = mine + rank + ns;     // the group's last lane advances the cursor
        __syncwarp();
        if (key != PB_KEY_DROP && ns) {
            uint32_t dst = mine + rank;
            const uint32_t m = meta[r];
            const int p = pos[r];
            const uint32_t mapq = (m >> 8) & 0xffu;
            const uint32_t zhi = (mapq << 16) | (((m >> 20) & 1u) << 24) | ((int)mapq < min_mapQ ? PB_REC_DEAD : 0u);
            const uint64_t b = base[r];
            const uint32_t cs = cigstart[r], nc = ncig[r];
            int x = p, y = 0;
            uint32_t emitted = 0;
            for (uint32_t ci = 0; ci < nc && emitted < ns; ++ci) {
                const uint32_t c = __ldg(cigar + cs + ci);
                const int op = c & 15, len = (int)(c >> 4);
                if (op == 0 || op == 7 || op == 8) {
                    if (len > 0) {
                        const uint64_t sb = b + (uint64_t)y;
                        int4 rec;
                        rec.x = p;
                        rec.y = x;
                        rec.z = (int)((uint32_t)len | zhi | ((uint32_t)(sb >> 32) << 26));
                        rec.w = (int)(uint32_t)sb;
                        srec[dst++] = rec;
                        ++emitted;
                    }
                    x += len; y += len;
                } else if (op == 2 || op == 3) x += len;
                else if (op == 1 || op == 4) y += len;
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Exclusive scan of uint32 (in place), three kernels; totals fit 32 bits (number of reads).
#define PB_SCAN_ITEMS 8
#define PB_SCAN_THREADS 256
__device__ __forceinline__ uint32_t pb_block_exscan(uint32_t v, uint32_t *total) {
    __shared__ uint32_t wsum[32];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    uint32_t x = v;
    for (int o = 1; o < 32; o <<= 1) { uint32_t y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
    __syncthreads();
    if (lane == 31) wsum[wid] = x;
    __syncthreads();
    if (wid == 0) {
        uint32_t s = lane < nw ? wsum[lane] : 0;
        for (int o = 1; o < 32; o <<= 1) { uint32_t y = __shfl_up_sync(0xffffffffu, s, o); if (lane >= o) s += y; }
        wsum[lane] = s;
    }
    __syncthreads();
    const uint32_t base = wid ? wsum[wid - 1] : 0;
    *total = wsum[nw - 1];
    return base + x - v;
}
__global__ void __launch_bounds__(PB_SCAN_THREADS) k_scan_blocks(uint32_t *data, int64_t n, uint32_t *block_tot) {
    const int64_t b0 = (int64_t)blockIdx.x * PB_SCAN_THREADS * PB_SCAN_ITEMS + (int64_t)threadIdx.x * PB_SCAN_ITEMS;
    uint32_t v[PB_SCAN_ITEMS], s = 0;
#pragma unroll
    for (int i = 0; i < PB_SCAN_ITEMS; ++i) { v[i] = b0 + i < n ? data[b0 + i] : 0; s += v[i]; }
    uint32_t tot;
    uint32_t ex = pb_block_exscan(s, &tot);
#pragma unroll
    for (int i = 0; i < PB_SCAN_ITEMS; ++i) { if (b0 + i < n) data[b0 + i] = ex; ex += v[i]; }
    if (threadIdx.x == 0) block_tot[blockIdx.x] = tot;
}
__global__ void __launch_bounds__(1024) k_scan_totals(uint32_t *block_tot, int64_t nb) {
    __shared__ uint32_t carry_s;
    if (threadIdx.x == 0) carry_s = 0;
    __syncthreads();
    for (int64_t b0 = 0; b0 < nb; b0 += 1024) {
        const int64_t i = b0 + threadIdx.x;
        const uint32_t v = i < nb ? block_tot[i] : 0;
        uint32_t tot;
        const uint32_t ex = pb_block_exscan(v, &tot);
        const uint32_t carry = carry_s;
        if (i < nb) block_tot[i] = carry + ex;
        __syncthreads();
        if (threadIdx.x == 0) carry_s = carry + tot;
        __syncthreads();
    }
}
__global__ void __launch_bounds__(PB_SCAN_THREADS) k_scan_add(uint32_t *data, int64_t n, const uint32_t *__restrict__ block_tot) {
    const int64_t b0 = (int64_t)blockIdx.x * PB_SCAN_THREADS * PB_SCAN_ITEMS + (int64_t)threadIdx.x * PB_SCAN_ITEMS;
    const uint32_t add = block_tot[blockIdx.x];
#pragma unroll
    for (int i = 0; i < PB_SCAN_ITEMS; ++i) if (b0 + i < n) data[b0 + i] += add;
}
// sample start offsets: the count matrix has one extra trailing element, so after the exclusive scan
// offs[s * n_chunks] is the start of sample s for s < n and the total for s == n
__global__ void k_sample_starts(const uint32_t *__restrict__ offs, int n_samples, int64_t n_chunks, uint32_t *__restrict__ sstart,
                                PbCounters *__restrict__ ctr) {
    const int s = threadIdx.x;
    if (s <= n_samples) sstart[s] = offs[(int64_t)s * n_chunks];
    if (s == n_samples) ctr->n_records = offs[(int64_t)s * n_chunks];
}

// ------------------------------------------------------------------------------------------------
struct PbPileArgs {
    // aligned segments of the kept reads, partitioned by sample (file order inside a sample)
    const int4 *srec;
    const uint32_t *sstart;         // [n_samples+1]
    const uint8_t *codes;           // per-base code (k_encode), same offsets as qual[]
    const char *ref;
    int64_t ref_len;
    int span_beg, span_end;
    const int32_t *win_beg, *win_end;
    int n_windows;
    int n_samples;
    int min_depth, max_depth, min_rmsQ, min_snpQ;
    int het_mode;
    const double *fk, *beta, *lhet;
    const PbCounters *ctr;          // max_span, level table
    const uint8_t *need;            // [64][256] walk-free shortcut table (k_need_table)
    const int32_t *rms_thr;         // [256] k_rms_table
    uint64_t *site_type;            // [span]
    uint8_t *site_flag;             // [span]  bit0 used, bit1 segregating
    uint64_t *cb_out;               // [span * n_samples] or null
    uint64_t *acc_cov;              // [span] coverage masks, or null (PB_AN_NUCDIV_MISSING: the counting path's layout in d_acc)
    uint32_t *acc_cnt4;             // [span] derived-base counts, or null with acc_cov
};

#define PB_WCAP 32                // segment records staged per warp and chunk
#define PB_WQ 32                  // deferred (non-unanimous) cells per warp

// Dynamic shared memory of k_pileup_call<TP> for nl quality levels (independent of the sample count).
static inline size_t pb_pile_smem(int tp, int nl) {
    const size_t per_warp = (size_t)PB_WCAP * 32 + (size_t)2 * nl * 32 * 4 + (size_t)PB_WQ * (3 + 2 * nl) * 4 + 32 * 20;
    return (size_t)(tp / 32) * ((per_warp + 15) & ~(size_t)15) + 256 * 8 + 128 * 4 + 256 * 4 + 64 + (size_t)nl * 256 + 64;
}

// One CTA = TP consecutive reference positions x all samples; one WARP = 32 positions, one thread = one
// position.  After a common prologue (tables, the CTA's candidate range per sample) the warps never
// synchronise with each other: every warp owns a slice of shared memory (staged records, one
// histogram column per lane, a queue of deferred cells, the site state of its 32 positions).
//
// Per sample a warp finds, with two ballots over the sorted read starts, the segment records whose
// read starts in (first position - max_span, last position], stages them unpacked into two 16-byte
// halves, and walks them in lock step -- every lane looks at the same record (a broadcast
// shared-memory load), two records per iteration so two code loads are in flight.  Coverage of a
// lane's position is one unsigned compare (p - seg_start < seg_len); the base's pre-digested code
// (k_encode) is one byte load whose address is consecutive across the lanes.  The body is predicated,
// so the warp never splits.  Passing bases are counted in the lane's private (level, strand) x base
// histogram in shared memory (plain read-modify-write, no atomics) and in a packed per-base total.
//
// CAP = true keeps call_base's raw-depth cap ("the first max_depth non-deleted reads in file order,
// before the base filters", popbam.cpp:242-248).  When k_depth_bound proves that no cell can reach
// max_depth the host launches CAP = false: the lists then hold only reads passing min_mapQ and there is
// no depth bookkeeping.
//
// Calls.  After the last record of a sample, cells whose bases all agree (the overwhelming majority)
// are called on the spot: a count test against the need table, else the exact early-exit walk.  The
// others are deferred: the lane moves its histogram into the warp's queue, and the queue is drained
// with one cell per lane when it fills up and after the last sample, so the long general walk
// (pb_call_general) runs on many lanes instead of on the one or two that need it.
//
// Per-site logic (make_X, pop_nucdiv.cpp:148-197) is folded in sample by sample (pb_site_sample): a
// position only keeps its coverage mask, derived-allele mask and derived-base counts (20 bytes of
// shared memory), so nothing per (site, sample) is stored unless the caller asked for the cb words.
template <int TP, bool CAP>
__global__ void __launch_bounds__(TP, TP == 256 ? 5 : 8) k_pileup_call(const PbPileArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int n = a.n_samples;
    const int nl = a.ctr->n_levels;
    const int n_lw = 2 * nl;
    const int qstride = 3 + n_lw;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const size_t per_warp = (((size_t)PB_WCAP * 32 + (size_t)n_lw * 32 * 4 + (size_t)PB_WQ * qstride * 4 + 32 * 20) + 15) & ~(size_t)15;
    unsigned char *wbase = smem_raw + (size_t)wid * per_warp;
    int4 *recA = reinterpret_cast<int4 *>(wbase);                           // [PB_WCAP] {seg start, seg len, D lo, D hi}
    int4 *recB = recA + PB_WCAP;                                            // [PB_WCAP] {strand*32*4, mapq^2, dead, -}
    uint64_t *s_cov = reinterpret_cast<uint64_t *>(recB + PB_WCAP);         // [32]
    uint64_t *s_type = s_cov + 32;                                          // [32]
    uint32_t *s_cnt4 = reinterpret_cast<uint32_t *>(s_type + 32);           // [32]
    uint32_t *hist = s_cnt4 + 32;                                           // [n_lw][32]
    uint32_t *queue = hist + (size_t)n_lw * 32;                             // [PB_WQ][3 + n_lw]
    unsigned char *cbase = smem_raw + (size_t)(TP / 32) * per_warp;         // CTA-wide tables
    double *fk_s = reinterpret_cast<double *>(cbase);                       // [256]
    uint32_t *rng = reinterpret_cast<uint32_t *>(fk_s + 256);               // lo[64], hi[64]
    int32_t *rms_thr_s = reinterpret_cast<int32_t *>(rng + 128);            // [256]
    uint8_t *qval_s = reinterpret_cast<uint8_t *>(rms_thr_s + 256);         // [64]
    uint8_t *need_s = qval_s + 64;                                          // [nl][256]

    const int p0 = a.span_beg + (int)blockIdx.x * TP;
    const int p = p0 + tid;
    const int p_end = min(p0 + TP, a.span_end);
    const bool valid = p < p_end;
    const int max_span = a.ctr->max_span;
    for (int i = tid; i < nl * 64; i += TP) reinterpret_cast<uint32_t *>(need_s)[i] = reinterpret_cast<const uint32_t *>(a.need)[i];
    // the warp's position range
    const int pw0 = p0 + (tid & ~31);
    const int pw1 = min(pw0 + 31, p_end - 1);
    // lanes past the end of the span use a position no segment can cover
    const int pq = valid ? p : 0x7fffffff;

    for (int i = tid; i < 256; i += TP) { fk_s[i] = a.fk[i]; rms_thr_s[i] = a.rms_thr[i]; }
    if (tid < 64) qval_s[tid] = a.ctr->qval[tid];
    for (int lw = 0; lw < n_lw; ++lw) hist[lw * 32 + lane] = 0;
    s_cov[lane] = 0; s_type[lane] = 0; s_cnt4[lane] = 0;
    if (tid < n) {
        // candidate records of sample tid for the whole CTA: read start in (p0 - max_span, p_end)
        const uint32_t s0 = a.sstart[tid], s1 = a.sstart[tid + 1];
        uint32_t lo = s0, hi = s1;
        const int t_lo = p0 - max_span;       // first with start > t_lo
        while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if (a.srec[mid].x > t_lo) hi = mid; else lo = mid + 1; }
        rng[tid] = lo;
        hi = s1;
        uint32_t l2 = lo;                     // first with start >= p_end
        while (l2 < hi) { const uint32_t mid = (l2 + hi) >> 1; if (a.srec[mid].x >= p_end) hi = mid; else l2 = mid + 1; }
        rng[64 + tid] = l2;
    }
    __syncthreads();                          // the only CTA-wide barrier
    if (pw0 >= p_end) return;                 // warp entirely past the end of the span

    const int ref_c = (valid && p >= 0 && p < a.ref_len) ? (int)(unsigned char)a.ref[p] : 'N';
    const int ref_r = pb_iupac_rev(ref_c);

    // fold one called cell into its position's site state.  During the record walk only the owner lane
    // touches a slot; in a drain several lanes may hold cells of the same position (different samples),
    // hence the atomic variant.
    auto fold = [&](int slot, int pos, int refc, int refr, int smp, uint64_t cb, bool atomic) {
        uint32_t d4 = 0;
        bool cov, der;
        cb = pb_site_sample(cb, refc, refr, a.het_mode, a.min_snpQ, a.min_rmsQ, a.min_depth, a.max_depth, &d4, &cov, &der);
        if (atomic) {
            if (d4) atomicAdd(&s_cnt4[slot], d4);
            if (cov) atomicOr(reinterpret_cast<unsigned long long *>(&s_cov[slot]), 1ULL << smp);
            if (der) atomicOr(reinterpret_cast<unsigned long long *>(&s_type[slot]), 1ULL << smp);
        } else {
            s_cnt4[slot] += d4;
            if (cov) s_cov[slot] |= 1ULL << smp;
            if (der) s_type[slot] |= 1ULL << smp;
        }
        if (a.cb_out) a.cb_out[((int64_t)pos - a.span_beg) * n + smp] = cb;
    };
    int qn = 0;                  // cells in the warp's queue (warp-uniform)
    auto drain = [&]() {
        __syncwarp();
        if (lane < qn) {
            const uint32_t *q = queue + (size_t)lane * qstride;
            const int slot = (int)(q[0] & 0xffffu), smp = (int)(q[0] >> 16);
            const int pos = pw0 + slot;
            const int rc = (pos >= 0 && pos < a.ref_len) ? (int)(unsigned char)a.ref[pos] : 'N';
            auto take = [&](int lw) -> uint32_t { return q[3 + lw]; };
            fold(slot, pos, rc, pb_iupac_rev(rc), smp, pb_call_general(take, n_lw, qval_s, q[2], (int)q[1], fk_s, a.beta, a.lhet), true);
        }
        __syncwarp();
        qn = 0;
    };

    uint32_t *const my_hist = hist + lane;
    // one base of this lane's position; `code` was loaded by the caller (PB_CODE_NONE when not taken)
    int depth = 0, rmsq = 0;
    uint32_t tot4 = 0;           // per-base counts of the cell, one byte each
    auto count_base = [&](uint32_t code, const int4 &rb) {
        // branch-free: a filtered base adds 0 to the level-0 word of its strand
        const uint32_t ok = code != PB_CODE_NONE ? 1u : 0u;
        const uint32_t c2 = ok ? code : 0u;
        const uint32_t inc = ok << ((c2 & 3u) << 3);
        // word index (level*2 + strand) * 32  ==  byte offset (code & 0xfc) * 64 + strand*128
        uint32_t *h = reinterpret_cast<uint32_t *>(reinterpret_cast<unsigned char *>(my_hist) + (c2 & 0xfcu) * 64 + rb.x);
        *h += inc;
        tot4 += inc;
        rmsq += (int)ok * rb.y;
    };
    // codes[D + p]: the lane's fixed part of the address
    const uint8_t *const lane_codes = a.codes + (int64_t)pq;

    for (int s = 0; s < n; ++s) {
        // ---- the warp's records of this sample: read start in (pw0 - max_span, pw1], found by ballots over the sorted starts
        const uint32_t lo = rng[s], hi = rng[64 + s];
        uint32_t wlo = lo, whi = lo;
        const int thr = pw0 - max_span;
        for (uint32_t c0 = lo; c0 < hi; c0 += 32) {
            const uint32_t idx = c0 + lane;
            const int x = idx < hi ? a.srec[idx].x : 0x7fffffff;
            wlo += __popc(__ballot_sync(0xffffffffu, x <= thr));
            const uint32_t in = __popc(__ballot_sync(0xffffffffu, x <= pw1));
            whi += in;
            if (in < 32) break;              // sorted: nothing further can start at or before pw1
        }
        for (uint32_t c0 = wlo; c0 < whi; c0 += PB_WCAP) {
            const int cnt = (int)min((uint32_t)PB_WCAP, whi - c0);
            __syncwarp();
            for (int i = lane; i < cnt; i += 32) {
                const int4 r = a.srec[c0 + i];
                const uint32_t z = (uint32_t)r.z, mq = (z >> 16) & 0xffu;
                // D = byte offset of the segment's first code minus the segment start: the code of position p is at
                // codes[D + p], so a lane adds D to its own fixed pointer codes + p
                const int64_t D = (int64_t)(((uint64_t)(z >> 26) << 32) | (uint32_t)r.w) - (int64_t)r.y;
                recA[i] = make_int4(r.y, (int)(z & 0xffffu), (int)(uint32_t)(uint64_t)D, (int)(uint32_t)((uint64_t)D >> 32));
                recB[i] = make_int4((int)(((z >> 24) & 1u) * 128u), (int)(mq * mq), (int)((z >> 25) & 1u), 0);
            }
            __syncwarp();
            int j = 0;
            // four records per iteration: the four code loads are issued before any histogram update, so a
            // warp keeps four global loads in flight (the loop is bound by their latency, see profiles/)
            for (; j + 3 < cnt; j += 4) {
                uint32_t cv[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int4 aq = recA[j + q];                       // same record for every lane: broadcast
                    bool t = (uint32_t)(pq - aq.x) < (uint32_t)aq.y;
                    if (CAP) {                                         // the cap precedes the filters; dead reads count
                        t = t && depth < a.max_depth; depth += t;
                        t = t && !recB[j + q].z;
                    }
                    cv[q] = PB_CODE_NONE;
                    if (t) cv[q] = __ldg(lane_codes + (int64_t)(((uint64_t)(uint32_t)aq.w << 32) | (uint32_t)aq.z));
                }
#pragma unroll
                for (int q = 0; q < 4; ++q) count_base(cv[q], recB[j + q]);
            }
            for (; j < cnt; ++j) {
                const int4 a0 = recA[j], b0 = recB[j];
                bool t0 = (uint32_t)(pq - a0.x) < (uint32_t)a0.y;
                if (CAP) { t0 = t0 && depth < a.max_depth; depth += t0; t0 = t0 && !b0.z; }
                uint32_t c0v = PB_CODE_NONE;
                if (t0) c0v = __ldg(lane_codes + (int64_t)(((uint64_t)(uint32_t)a0.w << 32) | (uint32_t)a0.z));
                count_base(c0v, b0);
            }
        }
        // ---- call the cell.  Raw depth 0, or depth > 0 with every base filtered: errmod_cal(n = 0) + gl2cns give cb = 0
        const bool unan = tot4 != 0 && pb_tot4_unanimous(tot4);
        const bool hard = valid && tot4 != 0 && !unan;
        const uint32_t hard_mask = __ballot_sync(0xffffffffu, hard);
        if (hard_mask && qn + __popc(hard_mask) > PB_WQ) drain();      // warp-uniform
        if (valid) {
            if (tot4 == 0) {
                // cb = 0.  With min_depth > 0 and min_snpQ > 0 such a cell is not covered, not derived and adds no
                // derived-allele count (segbase takes its revert branch): nothing to fold
                if (a.cb_out || a.min_depth <= 0 || a.min_snpQ <= 0) fold(lane, p, ref_c, ref_r, s, 0, false);
            } else if (unan) {
                auto peek = [&](int lw) -> uint32_t { return my_hist[lw * 32]; };
                const int kk = pb_tot4_k(tot4);
                const int bb = (tot4 >> 8 & 255u) ? 1 : (tot4 >> 16 & 255u) ? 2 : (tot4 >> 24) ? 3 : 0;
                // count test against the need table (no error-model arithmetic); exact early-exit walk otherwise
                const bool by_count = pb_unanimous_by_count(peek, nl, need_s, kk, bb);
                if (by_count && !a.cb_out && (int)"ACGT"[bb] == ref_c) {
                    // homozygous reference: clean_heterozygotes and segbase leave the word alone, the site type
                    // bit stays 0; only qfilter's coverage test remains (pop_utils.cpp:102-120)
                    if (rmsq >= rms_thr_s[kk] && kk >= a.min_depth && kk <= a.max_depth) s_cov[lane] |= 1ULL << s;
                } else {
                    const uint64_t cbw = by_count ? pb_unanimous_result(a.lhet, kk, bb, rmsq)
                                                  : pb_call_unanimous(peek, n_lw, qval_s, tot4, rmsq, fk_s, a.beta, a.lhet);
                    fold(lane, p, ref_c, ref_r, s, cbw, false);
                }
                for (int lw = 0; lw < n_lw; ++lw) my_hist[lw * 32] = 0;
            } else {                           // defer: move the histogram into the warp's queue
                const int slot = qn + __popc(hard_mask & ((1u << lane) - 1u));
                uint32_t *q = queue + (size_t)slot * qstride;
                q[0] = (uint32_t)lane | ((uint32_t)s << 16); q[1] = (uint32_t)rmsq; q[2] = tot4;
                for (int lw = 0; lw < n_lw; ++lw) { q[3 + lw] = my_hist[lw * 32]; my_hist[lw * 32] = 0; }
            }
        }
        qn += __popc(hard_mask);
        depth = 0; rmsq = 0; tot4 = 0;
    }
    if (qn) drain();

    // the site: segbase's return value, coverage test, window membership (windows are sorted and disjoint)
    __syncwarp();
    if (valid) {
        const int fq = pb_site_fq(s_cnt4[lane]);
        int lo = 0, hi = a.n_windows;
        while (lo < hi) { const int mid = (lo + hi) >> 1; if (__ldg(a.win_end + mid) > p) hi = mid; else lo = mid + 1; }
        const bool in_win = lo < a.n_windows && __ldg(a.win_beg + lo) <= p;
        const bool used = in_win && __popcll(s_cov[lane]) == n;
        const int64_t o = (int64_t)p - a.span_beg;
        a.site_type[o] = s_type[lane];
        a.site_flag[o] = (uint8_t)((used ? 1 : 0) | ((used && fq > 0) ? 2 : 0));
        if (a.acc_cov) { a.acc_cov[o] = s_cov[lane]; a.acc_cnt4[o] = s_cnt4[lane]; }
    }
}

// ------------------------------------------------------------------------------------------------
// Per window: num_sites, segsites (WRITE = false) and, after the scan of segsites, the ordered list
// of segregating sites (WRITE = true): hap.pos / hap.idx / types / ref / per-sample cb words
// (make_nucdiv tail, pop_nucdiv.cpp:176-199).
template <bool WRITE>
__global__ void __launch_bounds__(256) k_window_sites(int span_beg, const int32_t *__restrict__ win_beg,
                                                      const int32_t *__restrict__ win_end, const uint8_t *__restrict__ site_flag,
                                                      const uint64_t *__restrict__ site_type, const char *__restrict__ ref,
                                                      int64_t ref_len, const uint64_t *__restrict__ cb_all, int n_samples,
                                                      int32_t *__restrict__ num_sites, int32_t *__restrict__ segsites,
                                                      const int64_t *__restrict__ seg_off, uint32_t *__restrict__ seg_pos,
                                                      uint32_t *__restrict__ seg_idx, uint64_t *__restrict__ seg_type,
                                                      uint8_t *__restrict__ seg_ref, uint64_t *__restrict__ seg_cb) {
    const int w = blockIdx.x;
    const int beg = win_beg[w], len = win_end[w] - beg;
    const int64_t off = (int64_t)beg - span_beg;
    uint32_t carry_sites = 0, carry_seg = 0;
    const int64_t so = WRITE ? seg_off[w] : 0;
    // four consecutive positions per thread and step: one block scan per 1024 positions
    for (int b0 = 0; b0 < len; b0 += 1024) {
        const int i0 = b0 + 4 * (int)threadIdx.x;
        uint32_t f[4], v = 0;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            f[q] = i0 + q < len ? site_flag[off + i0 + q] : 0;
            v += (f[q] & 1u) | ((f[q] >> 1 & 1u) << 16);
        }
        uint32_t tot;
        uint32_t ex = pb_block_exscan(v, &tot);
        if (WRITE) {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                if (f[q] & 2u) {
                    const int i = i0 + q;
                    const int64_t d = so + carry_seg + (ex >> 16);
                    seg_pos[d] = (uint32_t)(beg + i);
                    seg_idx[d] = carry_sites + (ex & 0xffffu);
                    seg_type[d] = site_type[off + i];
                    const int64_t rp = (int64_t)beg + i;
                    seg_ref[d] = (rp >= 0 && rp < ref_len) ? (uint8_t)ref[rp] : (uint8_t)'N';
                    if (seg_cb) for (int s = 0; s < n_samples; ++s) seg_cb[d * n_samples + s] = cb_all[(off + i) * n_samples + s];
                }
                ex += (f[q] & 1u) | ((f[q] >> 1 & 1u) << 16);
            }
        }
        carry_sites += tot & 0xffffu;
        carry_seg += tot >> 16;
    }
    if (!WRITE && threadIdx.x == 0) { num_sites[w] = (int32_t)carry_sites; segsites[w] = (int32_t)carry_seg; }
}

// seg_off[w] = exclusive sum of segsites (int64), single block
__global__ void __launch_bounds__(1024) k_scan_windows(const int32_t *__restrict__ segsites, int n_windows, int64_t *__restrict__ seg_off) {
    __shared__ unsigned long long carry_s;
    if (threadIdx.x == 0) carry_s = 0;
    __syncthreads();
    for (int b0 = 0; b0 < n_windows; b0 += 1024) {
        const int i = b0 + (int)threadIdx.x;
        const uint32_t v = i < n_windows ? (uint32_t)segsites[i] : 0;
        uint32_t tot;
        const uint32_t ex = pb_block_exscan(v, &tot);
        const unsigned long long carry = carry_s;
        if (i < n_windows) seg_off[i] = (int64_t)(carry + ex);
        __syncthreads();
        if (threadIdx.x == 0) carry_s = carry + tot;
        __syncthreads();
    }
    if (threadIdx.x == 0) seg_off[n_windows] = (int64_t)carry_s;
}
