// pb_lib.cu -- the C ABI of include/popbam_b200.h: context, device buffers, the kernel pipeline of
// one region, pinned result buffers.  There is no host compute path: every statistic is produced by
// the kernels in pb_kernels.cuh / pb_stats.cuh, and pb_create fails without a CUDA device.
#include <cuda_runtime.h>
#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <future>
#include <string>
#include <vector>

#include "../../include/popbam_b200.h"
#include "pb_kernels.cuh"
#include "pb_fast.cuh"
#include "pb_pile.cuh"
#include "pb_stats.cuh"
#include "pb_ld.cuh"

namespace {

struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    bool listed = false;     // registered in pb_ctx::bufs (done by dev_reserve), so pb_destroy frees every buffer ever allocated
};
struct HostBuf {
    void *p = nullptr;
    size_t cap = 0;
};

std::string g_create_error;

enum RegionState { ST_IDLE = 0, ST_OPEN = 1, ST_LAUNCHED = 2, ST_DONE = 3 };

}  // namespace

// launch shape of k_pile_reads and what it was chosen for
struct PileShape { int spc = 0, warps = 0, tile_q = 0, span32 = 0, qcap = 0, dens16 = 0, tail = 0; bool robust = false; size_t smem = 0; };

struct pb_ctx {
    pb_params prm;
    PileShape pile_shape;
    cudaStream_t stream = nullptr;
    std::string err;
    int64_t launches = 0;
    int n_sms = 148;
    // grids of the persistent (grid-stride) kernels: SM count x resident CTAs per SM, so every launch is one full wave
    int g_encode = 148, g_qual_mask = 148, g_hard_cells = 148, g_read_prep = 148;
    size_t smem_per_sm = 0;
    size_t smem_optin = 0;
    // tables / contig
    DevBuf d_fk, d_beta, d_lhet, d_ref, d_rms_thr;
    int64_t ref_len = 0;
    int32_t ref_tid = -1;
    // region
    int state = ST_IDLE;
    uint32_t analyses = 0;
    int nw = 0;
    int span_beg = 0, span_end = 0;
    std::vector<int32_t> h_wbeg, h_wend;
    DevBuf d_wbeg, d_wend;
    // reads on the device (concatenation of the pushed batches)
    int64_t n_reads = 0, n_cig = 0, n_bytes = 0, n_pushes = 0;
    DevBuf d_pos, d_meta, d_cigstart, d_ncig, d_base, d_cigar, d_seq4, d_qual, d_tmp_cig, d_tmp_base;
    // derived
    DevBuf d_rkey, d_rnseg, d_codes, d_bins, d_need, d_qtab, d_counts, d_blocktot, d_srec, d_sstart, d_ctr;
    DevBuf d_site_type, d_site_flag, d_cb;
    DevBuf d_fastp, d_acc;                      // counting path: PbFastTables, per-position accumulators
    DevBuf d_cells, d_codes16, d_need_raw, d_blk;      // cells left for k_hard_cells (directory, base codes), need_raw[64][256], per-block records of the directory
    DevBuf d_refcode;                           // reference code bytes of the contig (k_ref_codes)
    std::vector<DevBuf *> bufs;            // every device buffer of the context
    bool classic = false;                  // POPBAM_B200_PILEUP=classic: always k_pileup_call (A/B measurements)
    int qual_ceiling = 41;                 // largest quality of a stray base the one-stray-base rule covers (pb_fast.cuh; POPBAM_B200_QCEIL)
    bool qual_robust = false;              // quality bytes >= 128 occur: kernel variant whose packed compares are right for any byte
    int arena_scale = 1;                   // cell arena size factor (raised on overflow)
    int pile_spc = 0, pile_warps = 0;      // POPBAM_B200_PILE=strips,warps: launch shape of k_pile_reads (measurements)
    bool fuse_codes = true;                // POPBAM_B200_CODES=separate: all base codes of the hard cells by k_cell_codes (measurements);
    int codes_skip = 0;                    // =mixed: every other block's (tests: both ways in one region)
    bool need_raw_valid = false;
    bool ran_fast = false;                 // the last pipeline run took the counting path
    int force_classic = 0;                 // the counting path gave up on this region (arena overflow twice): k_pileup_call
    int reruns = 0;                        // regions run again because an assumption of the counting path did not hold
    // what a context has learnt from its earlier regions: with it a region is enqueued without a host round trip
    bool spec_valid = false;
    int spec_span = 0;                     // largest reference span of a read seen so far
    int spec_read_bytes = 0;               // most bytes of qual[] one read takes, seen so far
    bool async_run = false;                // the last run_pipeline left its checks and the segregating-site copy to fill_result
    int async_span = 0;                    // ... and assumed this largest read span
    bool no_async = false;                 // POPBAM_B200_SYNC=1: always take the host round trips (A/B measurements)
    int64_t seg_cap = 0;                   // device layout of the segregating-site arrays (async: sized by the span)
    DevBuf d_seg_type;     // arena of the segregating-site arrays (seg_layout)
    DevBuf d_hap, d_kt, d_km, d_lsum, d_rsum, d_wall_u, d_stats, d_ld_kt, d_ld_km, d_ld_inv, d_ld_cnt, d_ld_dp, d_snn_nn;
    int64_t snn_perms = 0;                 // pb_set_snn_perms: Snn permutations per (window, pair) and the stream's seed
    uint64_t snn_seed = 0;
    int64_t snn_perms_run = 0;             // ... as the last pipeline run used them
    // pinned results
    HostBuf h_ctr, h_small, h_seg, h_span;
    PbCounters ctr_host;
    bool need_valid = false;
    int need_nl = 0;
    unsigned char need_qval[64] = {0};
    int64_t s_total = 0;
    pb_region_result res;
    pb_region_extras ext;
    pb_region_fst fst;
    // bam_fetch_f shim staging (pb_push_record)
    std::vector<int32_t> r_pos;
    std::vector<uint32_t> r_meta, r_cig_off, r_cigar, r_base_off;
    std::vector<uint8_t> r_seq4, r_qual;
    // timing of the last pipeline run
    cudaEvent_t ev[7] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    // second stream: the per-read chain (prep, depth bound, sample partition, strip index) runs beside the per-base
    // chain (quality mask, encode, bit-planes); fk[] = fork / join events (no timing)
    cudaStream_t stream2 = nullptr;
    // k_pile_reads runs on a stream of LOWER priority: the short, latency-bound kernels of other contexts' regions (their
    // per-read chain, hard cells, sites, windows) are scheduled ahead of its remaining CTAs and run beside it
    cudaStream_t stream_lo = nullptr;
    cudaEvent_t fk[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t dbg[4] = {nullptr, nullptr, nullptr, nullptr};   // POPBAM_B200_DEBUG: timeline of the two prep chains
    float ms_prep = 0, ms_pileup = 0, ms_sites = 0, ms_stats = 0;
};

namespace {

int fail(pb_ctx *c, int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (c) c->err = buf; else g_create_error = buf;
    return code;
}

#define PB_CUDA(c, call)                                                                                   \
    do {                                                                                                   \
        cudaError_t e_ = (call);                                                                           \
        if (e_ != cudaSuccess) return fail((c), PB_ERR_CUDA, "%s: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

// grow-only device buffer; `keep` bytes of the old contents are preserved
int dev_reserve(pb_ctx *c, DevBuf &b, size_t bytes, size_t keep = 0) {
    if (bytes <= b.cap) return PB_OK;
    size_t want = std::max(bytes, b.cap + b.cap / 2);
    want = (want + 255) & ~(size_t)255;
    void *np = nullptr;
    cudaError_t e = cudaMalloc(&np, want);
    if (e != cudaSuccess) { cudaGetLastError(); return fail(c, PB_ERR_NOMEM, "cudaMalloc(%zu bytes): %s", want, cudaGetErrorString(e)); }
    if (keep && b.p) {
        e = cudaMemcpyAsync(np, b.p, keep, cudaMemcpyDeviceToDevice, c->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
        if (e != cudaSuccess) { cudaFree(np); return fail(c, PB_ERR_CUDA, "device buffer move: %s", cudaGetErrorString(e)); }
    } else if (b.p) {
        cudaStreamSynchronize(c->stream);   // nothing in flight may still use the old block
    }
    if (b.p) cudaFree(b.p);
    b.p = np; b.cap = want;
    if (!b.listed) { c->bufs.push_back(&b); b.listed = true; }
    return PB_OK;
}
int host_reserve(pb_ctx *c, HostBuf &b, size_t bytes) {
    if (bytes <= b.cap) return PB_OK;
    if (b.p) { cudaStreamSynchronize(c->stream); cudaFreeHost(b.p); b.p = nullptr; b.cap = 0; }
    size_t want = (bytes + 4095) & ~(size_t)4095;
    cudaError_t e = cudaHostAlloc(&b.p, want, cudaHostAllocDefault);
    if (e != cudaSuccess) { cudaGetLastError(); b.p = nullptr; return fail(c, PB_ERR_NOMEM, "cudaHostAlloc(%zu bytes): %s", want, cudaGetErrorString(e)); }
    b.cap = want;
    return PB_OK;
}
#define PB_TRY(x) do { int rc_ = (x); if (rc_ != PB_OK) return rc_; } while (0)

template <class T> T *dp(const DevBuf &b) { return reinterpret_cast<T *>(b.p); }

inline unsigned nblk(int64_t n, int per) { return (unsigned)std::max<int64_t>(1, (n + per - 1) / per); }

// carve `count` elements of T out of a pinned / device arena
struct Carver {
    unsigned char *base;
    size_t off = 0;
    explicit Carver(void *b) : base(reinterpret_cast<unsigned char *>(b)) {}
    template <class T> T *take(size_t count) {
        off = (off + 15) & ~(size_t)15;
        T *r = base ? reinterpret_cast<T *>(base + off) : nullptr;
        off += sizeof(T) * (count ? count : 1);
        return r;
    }
};

// layout of the fixed-size (per window) result arrays, identical on device and pinned host
struct SmallLayout {
    int32_t *num_sites, *segsites; int64_t *seg_off;
    double *piw, *pib; uint16_t *min_dxy;
    int32_t *sfs_num_snps; double *td, *fwh;
    int32_t *ld_num_snps; double *zns, *omegamax;
    int32_t *wall_num_snps; double *wallb, *wallq;
    uint16_t *ind_div, *pop_div; int32_t *div_num_snps;
    int32_t *nhaps; double *hdiv, *ehhs;
    uint16_t *tree_diff;
    int32_t *pop_segsites; double *theta_w, *fuli_d, *fuli_ds; int32_t *fuli_eta_e, *fuli_eta_s;
    int32_t *ld_kept; double *ld_dprime; int64_t *ld_complete;
    int64_t *hud_num, *hud_den, *wc_num, *wc_den; double *fst_hudson, *fst_wc, *snn, *snn_p; int64_t *snn_ge;
    size_t bytes;
};
SmallLayout small_layout(void *base, int NW, int P, int n, bool with_tree, bool with_fst) {
    Carver cv(base);
    SmallLayout L;
    const size_t wp = (size_t)NW * P, wpp = (size_t)NW * P * P, wn = (size_t)NW * n;
    L.num_sites = cv.take<int32_t>(NW); L.segsites = cv.take<int32_t>(NW); L.seg_off = cv.take<int64_t>(NW + 1);
    L.piw = cv.take<double>(wp); L.pib = cv.take<double>(wpp); L.min_dxy = cv.take<uint16_t>(wpp);
    L.sfs_num_snps = cv.take<int32_t>(wp); L.td = cv.take<double>(wp); L.fwh = cv.take<double>(wp);
    L.ld_num_snps = cv.take<int32_t>(wp); L.zns = cv.take<double>(wp); L.omegamax = cv.take<double>(wp);
    L.wall_num_snps = cv.take<int32_t>(wp); L.wallb = cv.take<double>(wp); L.wallq = cv.take<double>(wp);
    L.ind_div = cv.take<uint16_t>(wn); L.pop_div = cv.take<uint16_t>(wp); L.div_num_snps = cv.take<int32_t>(wp);
    L.nhaps = cv.take<int32_t>(wp); L.hdiv = cv.take<double>(wp); L.ehhs = cv.take<double>(wp);
    L.tree_diff = cv.take<uint16_t>(with_tree ? (size_t)NW * (n + 1) * (n + 1) : 1);
    L.pop_segsites = cv.take<int32_t>(wp); L.theta_w = cv.take<double>(wp); L.fuli_d = cv.take<double>(wp); L.fuli_ds = cv.take<double>(wp);
    L.fuli_eta_e = cv.take<int32_t>(wp); L.fuli_eta_s = cv.take<int32_t>(wp);
    L.ld_kept = cv.take<int32_t>(wp); L.ld_dprime = cv.take<double>(wp); L.ld_complete = cv.take<int64_t>(wp);
    L.hud_num = L.hud_den = L.wc_num = L.wc_den = L.snn_ge = nullptr; L.fst_hudson = L.fst_wc = L.snn = L.snn_p = nullptr;
    if (with_fst) {         // the pair arrays of PB_AN_FST (none without it: the arena is what it was before them)
        L.hud_num = cv.take<int64_t>(wpp); L.hud_den = cv.take<int64_t>(wpp); L.wc_num = cv.take<int64_t>(wpp); L.wc_den = cv.take<int64_t>(wpp);
        L.fst_hudson = cv.take<double>(wpp); L.fst_wc = cv.take<double>(wpp); L.snn = cv.take<double>(wpp); L.snn_p = cv.take<double>(wpp);
        L.snn_ge = cv.take<int64_t>(wpp);
    }
    L.bytes = (cv.off + 255) & ~(size_t)255;
    return L;
}
struct SegLayout {
    uint32_t *seg_pos, *seg_idx; uint64_t *seg_type; uint8_t *seg_ref; uint64_t *seg_cb;
    size_t bytes;
};
SegLayout seg_layout(void *base, int64_t S, int n, bool with_cb) {
    Carver cv(base);
    SegLayout L;
    L.seg_type = cv.take<uint64_t>(S); L.seg_cb = with_cb ? cv.take<uint64_t>((size_t)S * n) : nullptr;
    L.seg_pos = cv.take<uint32_t>(S); L.seg_idx = cv.take<uint32_t>(S); L.seg_ref = cv.take<uint8_t>(S);
    L.bytes = (cv.off + 255) & ~(size_t)255;
    return L;
}

int exclusive_scan_u32(pb_ctx *c, uint32_t *data, int64_t n, cudaStream_t st) {
    const int per = PB_SCAN_THREADS * PB_SCAN_ITEMS;
    const int64_t nb = (n + per - 1) / per;
    PB_TRY(dev_reserve(c, c->d_blocktot, sizeof(uint32_t) * (size_t)std::max<int64_t>(nb, 1)));
    k_scan_blocks<<<(unsigned)nb, PB_SCAN_THREADS, 0, st>>>(data, n, dp<uint32_t>(c->d_blocktot));
    k_scan_totals<<<1, 1024, 0, st>>>(dp<uint32_t>(c->d_blocktot), nb);
    k_scan_add<<<(unsigned)nb, PB_SCAN_THREADS, 0, st>>>(data, n, dp<uint32_t>(c->d_blocktot));
    c->launches += 3;
    PB_CUDA(c, cudaGetLastError());
    return PB_OK;
}


int run_pipeline(pb_ctx *c, int attempt = 0, bool allow_async = true) {
    const pb_params &P = c->prm;
    const int n = P.n_samples, NW = c->nw;
    const int64_t N = c->n_reads;
    const int64_t span = (int64_t)c->span_end - c->span_beg;
    cudaStream_t st = c->stream;
    const bool want_cb = (P.flags & PB_FLAG_EMIT_CB) || (c->analyses & PB_AN_SNP);

    PB_CUDA(c, cudaEventRecord(c->ev[0], st));
    // ---- per-read preparation, quality levels, partition by sample
    PB_TRY(dev_reserve(c, c->d_ctr, sizeof(PbCounters)));
    PB_CUDA(c, cudaMemsetAsync(c->d_ctr.p, 0, sizeof(PbCounters), st));
    PB_TRY(dev_reserve(c, c->d_rkey, (size_t)std::max<int64_t>(N, 1) + 8));
    PB_TRY(dev_reserve(c, c->d_rnseg, (size_t)std::max<int64_t>(N, 1)));
    PbCounters *ctr = dp<PbCounters>(c->d_ctr);
    const int illumina = (P.flags & PB_FLAG_ILLUMINA) ? 1 : 0;
    // read-start bins for the depth bound: 128 bp bins from 65536 bp before the span to its end
    const int bin_origin = c->span_beg - 65536;
    const int n_bins = (int)((span + 65536) >> PB_BIN_SHIFT) + 2;
    PB_TRY(dev_reserve(c, c->d_bins, sizeof(uint32_t) * (size_t)n * n_bins));
    PB_CUDA(c, cudaMemsetAsync(c->d_bins.p, 0, sizeof(uint32_t) * (size_t)n * n_bins, st));
    cudaStream_t s2 = c->stream2;
    PB_CUDA(c, cudaEventRecord(c->fk[0], st));
    PB_CUDA(c, cudaStreamWaitEvent(s2, c->fk[0], 0));
    // -- per-read chain on the second stream: flag filter, reference end, depth bound
    if (N > 0) {
        k_read_prep<<<(unsigned)std::min<int64_t>(nblk(N, 256), (int64_t)c->g_read_prep), 256, 0, s2>>>(N, dp<int32_t>(c->d_pos), dp<uint32_t>(c->d_meta), dp<uint32_t>(c->d_cigstart),
                                                 dp<uint32_t>(c->d_ncig), dp<uint32_t>(c->d_cigar), dp<uint64_t>(c->d_base), (uint64_t)c->n_bytes, n, P.min_mapQ,
                                                 dp<uint8_t>(c->d_rkey), dp<uint8_t>(c->d_rnseg), bin_origin, n_bins, c->span_end,
                                                 dp<uint32_t>(c->d_bins), ctr);
        c->launches += 1;
    }
    PB_CUDA(c, cudaEventRecord(c->fk[1], s2));                      // rkey, mapq mask, max_span
    if (c->dbg[0]) cudaEventRecord(c->dbg[0], s2);
    if (N > 0) {
        k_depth_bound<<<c->n_sms * 4, 256, 0, s2>>>(dp<uint32_t>(c->d_bins), n, n_bins, P.max_depth, dp<int32_t>(c->d_pos), N, ctr);
        c->launches += 1;
    }
    k_depth_decide<<<1, 1, 0, s2>>>(P.max_depth, ctr);
    c->launches += 1;
    // The single-kernel path (k_pileup_call) takes the reads as aligned-segment records, stably partitioned by sample; the
    // counting path (pb_pile.cuh) takes the batch as it is, so the partition only runs when that path is not taken.
    auto partition = [&]() -> int {
        PB_TRY(dev_reserve(c, c->d_srec, sizeof(int4) * (size_t)std::max<int64_t>(c->n_cig, 1)));   // one record per M/=/X op at most
        PB_TRY(dev_reserve(c, c->d_sstart, sizeof(uint32_t) * (PB_MAX_SAMPLES + 1)));
        const int64_t n_chunks = std::max<int64_t>(1, (N + PB_PART_CHUNK - 1) / PB_PART_CHUNK);
        const int64_t n_counts = (int64_t)n * n_chunks + 1;
        PB_TRY(dev_reserve(c, c->d_counts, sizeof(uint32_t) * (size_t)n_counts));
        PB_CUDA(c, cudaMemsetAsync(c->d_counts.p, 0, sizeof(uint32_t) * (size_t)n_counts, st));
        const unsigned part_blocks = nblk(n_chunks * 32, 128);
        k_part_count<<<part_blocks, 128, 0, st>>>(N, dp<uint8_t>(c->d_rkey), dp<uint8_t>(c->d_rnseg), dp<uint32_t>(c->d_meta), P.min_mapQ, ctr, n, n_chunks,
                                                 dp<uint32_t>(c->d_counts));
        c->launches += 1;
        PB_TRY(exclusive_scan_u32(c, dp<uint32_t>(c->d_counts), n_counts, st));
        k_sample_starts<<<1, 128, 0, st>>>(dp<uint32_t>(c->d_counts), n, n_chunks, dp<uint32_t>(c->d_sstart), ctr);
        k_part_scatter<<<part_blocks, 128, 0, st>>>(N, dp<uint8_t>(c->d_rkey), dp<uint8_t>(c->d_rnseg), n, n_chunks, dp<uint32_t>(c->d_counts),
                                                   dp<int32_t>(c->d_pos), dp<uint32_t>(c->d_meta), dp<uint64_t>(c->d_base),
                                                   dp<uint32_t>(c->d_cigstart), dp<uint32_t>(c->d_ncig), dp<uint32_t>(c->d_cigar), P.min_mapQ, ctr,
                                                   dp<int4>(c->d_srec));
        c->launches += 2;
        PB_CUDA(c, cudaGetLastError());
        return PB_OK;
    };
    // The counting path is tried when nobody wants the per-cell words and an empty cell is simply "not covered"
    // (min_depth, min_snpQ > 0); whether it can be TAKEN also needs the depth bound from the device.
    const int qoff = illumina ? 31 : 0;
    const bool fast_try = !want_cb && P.min_depth > 0 && P.min_snpQ > 0 && !c->classic && !c->force_classic && N > 0 &&
                          P.min_baseQ + qoff <= 128 && span * n < (int64_t)0x7fffffff;
    const int n_strips = (int)((span + 31) >> 5);
    PB_TRY(dev_reserve(c, c->d_site_type, sizeof(uint64_t) * (size_t)span));
    if (fast_try) PB_TRY(dev_reserve(c, c->d_acc, (size_t)span * 12 + 16));
    PB_CUDA(c, cudaEventRecord(c->fk[2], s2));
    if (c->dbg[1]) cudaEventRecord(c->dbg[1], s2);
    if (c->dbg[2]) cudaEventRecord(c->dbg[2], st);
    // -- quality levels on the main stream.  Bit-sliced path: the RANGE of levels a passing base can have (no pass over
    // the bases).  Single-kernel path: the values present (k_qual_mask), as its per-cell histograms are sized by them.
    auto need_tables = [&](const unsigned char *qval, int nl) -> int {
        // the walk-free shortcut table and the depth ranges only depend on the level set: rebuild them when that changes
        if (c->need_valid && c->need_nl == nl && memcmp(c->need_qval, qval, 64) == 0) return PB_OK;
        PB_TRY(dev_reserve(c, c->d_need, 64 * 256));
        k_need_table<<<std::max(nl, 1), 256, 0, st>>>(ctr, dp<double>(c->d_fk), dp<double>(c->d_beta), dp<double>(c->d_lhet), dp<uint8_t>(c->d_need));
        c->launches += 1;
        PB_CUDA(c, cudaGetLastError());
        c->need_valid = true; c->need_nl = nl; memcpy(c->need_qval, qval, 64);
        return PB_OK;
    };
    auto classic_levels = [&]() -> int {
        if (N > 0) {
            k_qual_mask<<<c->g_qual_mask, 256, 0, st>>>(dp<uint8_t>(c->d_qual), c->n_bytes, illumina, P.min_baseQ, ctr);
            c->launches += 1;
        }
        PB_CUDA(c, cudaStreamWaitEvent(st, c->fk[1], 0));
        k_level_table<<<1, 32, 0, st>>>(ctr);
        c->launches += 1;
        if (N > 0) {
            PB_TRY(dev_reserve(c, c->d_qtab, 64 * 256));
            k_qual_table<<<64, 256, 0, st>>>(ctr, illumina, P.min_baseQ, dp<uint8_t>(c->d_qtab));
            c->launches += 1;
        }
        return PB_OK;
    };
    if (fast_try) {
        // per-context tables of the counting path (pb_fast.cuh): level set {qlo, ..., 63}, need_raw, the per-depth rule tables
        const int qlo = std::max(4, std::min(63, std::min(P.min_baseQ, P.min_mapQ)));
        k_set_levels<<<1, 64, 0, st>>>(ctr, qlo, 63);
        c->launches += 1;
        if (!c->need_raw_valid) {
            PB_TRY(dev_reserve(c, c->d_need_raw, 64 * 256));
            PB_TRY(dev_reserve(c, c->d_fastp, sizeof(PbFastTables)));
            k_need_raw<<<64, 256, 0, st>>>(dp<double>(c->d_fk), dp<double>(c->d_beta), dp<double>(c->d_lhet), dp<uint8_t>(c->d_need_raw));
            k_fast_tables<<<1, 256, 0, st>>>(ctr, dp<uint8_t>(c->d_need_raw), dp<double>(c->d_fk), dp<double>(c->d_beta), dp<double>(c->d_lhet), P.min_depth,
                                            P.min_snpQ, c->qual_ceiling, P.min_mapQ, P.min_rmsQ, dp<int32_t>(c->d_rms_thr), dp<PbFastTables>(c->d_fastp));
            c->launches += 2;
            c->need_raw_valid = true;
        }
    } else {
        PB_TRY(classic_levels());
    }
    // Asynchronous mode: the launch parameters the counting pileup needs from the device (largest read span, most bytes
    // of a read, "the depth cap cannot bind") are taken from the context's earlier regions; the per-read chain then runs
    // BESIDE k_pile_reads instead of in front of it, and fill_result compares what it found with what was assumed (and looks
    // at the sorted / too-long flags) once the region is done.  No host round trip in the middle of the pipeline, so one
    // context keeps a GPU busy.
    const uint32_t sync_bits = PB_AN_SNP | PB_AN_LD_ZNS | PB_AN_LD_OMEGA | PB_AN_LD_DPRIME;          // their buffers / grids are sized by the number of segregating sites
    const bool async = allow_async && !c->no_async && fast_try && c->spec_valid && attempt == 0 && !(c->analyses & sync_bits) && !(P.flags & PB_FLAG_EMIT_CB);
    c->async_run = async;
    if (!async) PB_CUDA(c, cudaStreamWaitEvent(st, c->fk[2], 0));    // join
    if (!fast_try) PB_TRY(partition());
    PB_CUDA(c, cudaGetLastError());
    PB_TRY(host_reserve(c, c->h_ctr, 3 * sizeof(PbCounters) + 64));
    PB_CUDA(c, cudaEventRecord(c->ev[1], st));
    if (async) {
        memset(&c->ctr_host, 0, sizeof c->ctr_host);
        c->ctr_host.max_span = c->spec_span; c->ctr_host.nocap = 1; c->ctr_host.max_read_bytes = c->spec_read_bytes;
        c->async_span = c->spec_span;
    } else {
        PB_CUDA(c, cudaMemcpyAsync(c->h_ctr.p, c->d_ctr.p, sizeof(PbCounters), cudaMemcpyDeviceToHost, st));
        PB_CUDA(c, cudaStreamSynchronize(st));
        c->ctr_host = *reinterpret_cast<PbCounters *>(c->h_ctr.p);
        if (c->ctr_host.unsorted) return fail(c, PB_ERR_UNSORTED, "reads are not sorted by position (bam_pileup.c:384-395)");
        if (c->ctr_host.too_long) return fail(c, PB_ERR_UNSUPPORTED, "a read spans 65536 or more reference bases or has more than 255 aligned segments");
        if (c->ctr_host.total_bound > 8000) return fail(c, PB_ERR_UNSUPPORTED, "up to %d reads may be live at one position: above 8000 the reference's pileup drops reads (bam_pileup.c:260,375), which this library does not reproduce", c->ctr_host.total_bound);
    }

    // ---- the hot kernel
    PB_TRY(dev_reserve(c, c->d_site_flag, (size_t)span));
    if (want_cb) PB_TRY(dev_reserve(c, c->d_cb, sizeof(uint64_t) * (size_t)span * n));
    const bool cap = c->ctr_host.nocap == 0;
    // launch shape of k_pile_reads: strips per CTA and warps per CTA that keep the most warps resident (the counters of all
    // samples, the tiles of all warps and the registers decide), larger blocks first among equals
    PileShape pc;
    if (fast_try && !cap) {
        const int rb = std::max(c->ctr_host.max_read_bytes, 16);
        pc.span32 = (std::max(c->ctr_host.max_span, 1) + 31) & ~31;         // reads of the block before reach that far into a block
        pc.tile_q = std::max(std::min((32 * rb + 32 + 31) & ~31, 8192 + 32), (rb + 16 + 31) & ~31);
        // reads per position of the span; a fifth of a block's reads may have a second aligned segment to queue
        pc.dens16 = (int)std::min<double>(1e6, 16.0 * (double)N / (double)std::max<int64_t>(span, 1)) + 1;
        if (c->pile_shape.spc > 0 && c->pile_shape.span32 == pc.span32 && c->pile_shape.tile_q == pc.tile_q && c->pile_shape.dens16 >= pc.dens16 &&
            c->pile_shape.dens16 <= 2 * pc.dens16 && c->pile_shape.robust == c->qual_robust)
            pc = c->pile_shape;                                            // the same question as for the region before
        else {
            // score: resident warps x the share of a block's reads that start in it (a read that reaches in from the block before
            // is walked twice)
            double best = 0;
            static const int kSpc[] = {64, 48, 32, 24, 16, 14, 12, 8, 6, 4, 3, 2, 1};
            for (int spc : kSpc) {
                const int qcap = std::max(128, std::min(4096, ((int)(0.2 * (32.0 * spc + pc.span32) * pc.dens16 / 16.0) + 63) & ~63));
                for (int warps = 16; warps >= 4; warps >>= 1) {
                    const size_t smem = pb_pile_reads_smem(n, spc, pc.tile_q, warps, qcap);
                    if (smem > c->smem_optin) continue;
                    int per_sm = 0;
                    const cudaError_t e = c->qual_robust ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_pile_reads<true>, warps * 32, smem)
                                                         : cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_pile_reads<false>, warps * 32, smem);
                    if (e != cudaSuccess) { cudaGetLastError(); per_sm = 0; }
                    const double score = (double)per_sm * warps * (32.0 * spc) / (32.0 * spc + c->ctr_host.max_span);
                    if (score > best) { best = score; pc.spc = spc; pc.warps = warps; pc.smem = smem; pc.qcap = qcap; pc.tail = (int)pb_pile_tail_bytes(n, spc, pc.tile_q, warps); }
                }
            }
            if (c->pile_spc > 0 && c->pile_warps > 0) {                      // POPBAM_B200_PILE=spc,warps (measurements)
                const int qcap = std::max(128, std::min(4096, ((int)(0.2 * (32.0 * c->pile_spc + pc.span32) * pc.dens16 / 16.0) + 63) & ~63));
                const size_t smem = pb_pile_reads_smem(n, c->pile_spc, pc.tile_q, c->pile_warps, qcap);
                if (smem <= c->smem_optin) { pc.spc = c->pile_spc; pc.warps = c->pile_warps; pc.smem = smem; pc.qcap = qcap; pc.tail = (int)pb_pile_tail_bytes(n, c->pile_spc, pc.tile_q, c->pile_warps); }
            }
            pc.robust = c->qual_robust;
            c->pile_shape = pc;
        }
    }
    const bool fast = fast_try && !cap && pc.spc > 0;
    if (async && !fast) return run_pipeline(c, attempt, false);          // (cannot happen with the context's own numbers)
    if (fast_try && !fast) {
        // the depth cap can bind (or a read is too long for the counters / tiles): the single-kernel path needs the levels present
        PB_TRY(classic_levels());
        PB_TRY(partition());
        PB_CUDA(c, cudaMemcpyAsync(c->h_ctr.p, c->d_ctr.p, sizeof(PbCounters), cudaMemcpyDeviceToHost, st));
        PB_CUDA(c, cudaStreamSynchronize(st));
        c->ctr_host = *reinterpret_cast<PbCounters *>(c->h_ctr.p);
    }
    const int nl = c->ctr_host.n_levels;
    PbPileArgs pa;
    pa.srec = dp<int4>(c->d_srec); pa.sstart = dp<uint32_t>(c->d_sstart);
    pa.codes = nullptr;
    pa.ref = dp<char>(c->d_ref); pa.ref_len = c->ref_len;
    pa.span_beg = c->span_beg; pa.span_end = c->span_end;
    pa.win_beg = dp<int32_t>(c->d_wbeg); pa.win_end = dp<int32_t>(c->d_wend); pa.n_windows = NW;
    pa.n_samples = n;
    pa.min_depth = P.min_depth; pa.max_depth = P.max_depth; pa.min_rmsQ = P.min_rmsQ; pa.min_snpQ = P.min_snpQ;
    pa.het_mode = (P.flags & PB_FLAG_HETEROZYGOTE) ? 1 : 0;
    pa.fk = dp<double>(c->d_fk); pa.beta = dp<double>(c->d_beta); pa.lhet = dp<double>(c->d_lhet);
    pa.ctr = ctr;
    pa.need = dp<uint8_t>(c->d_need);
    pa.rms_thr = dp<int32_t>(c->d_rms_thr);
    pa.site_type = dp<uint64_t>(c->d_site_type); pa.site_flag = dp<uint8_t>(c->d_site_flag);
    pa.cb_out = want_cb ? dp<uint64_t>(c->d_cb) : nullptr;
    PB_CUDA(c, cudaEventRecord(c->ev[6], st));     // a per-base pass of the single-kernel path (base codes) counts as preparation: ev[6] .. ev[2]
    if (getenv("POPBAM_B200_DEBUG"))
        fprintf(stderr, "[popbam_b200] pileup path: fast=%d cap=%d want_cb=%d min_depth=%d min_snpQ=%d classic=%d N=%lld records=%u nl=%d depth_bound=%d max_span=%d ceiling=%d robust=%d\n",
                (int)fast, (int)cap, (int)want_cb, P.min_depth, P.min_snpQ, (int)c->classic, (long long)N, c->ctr_host.n_records, nl,
                c->ctr_host.depth_bound, c->ctr_host.max_span, c->qual_ceiling, (int)c->qual_robust);
    c->ran_fast = fast;
    if (fast) {
        // arena of the cells left for k_hard_cells: room for one cell in eight and one base in eight (times arena_scale);
        // k_pile_reads reports an overflow, the region is then run again with a larger arena
        const unsigned long long cell_cap = std::max<unsigned long long>(65536, (unsigned long long)span * n / 8 * c->arena_scale);
        const unsigned long long code_cap = std::min<unsigned long long>(0xfffffff0ULL, std::max<unsigned long long>(1 << 20, (unsigned long long)c->n_bytes / 8 * c->arena_scale));
        PB_TRY(dev_reserve(c, c->d_cells, sizeof(uint4) * cell_cap));
        PB_TRY(dev_reserve(c, c->d_codes16, sizeof(uint16_t) * code_cap));
        PB_CUDA(c, cudaEventRecord(c->ev[2], st));
        PbPileReadsArgs fa;
        fa.pos = dp<int32_t>(c->d_pos); fa.meta = dp<uint32_t>(c->d_meta); fa.cigstart = dp<uint32_t>(c->d_cigstart); fa.ncig = dp<uint32_t>(c->d_ncig);
        fa.cigar = dp<uint32_t>(c->d_cigar); fa.base = dp<uint64_t>(c->d_base); fa.n_reads = N; fa.n_bytes = (uint64_t)c->n_bytes;
        fa.qual = dp<uint8_t>(c->d_qual); fa.seq4 = dp<uint8_t>(c->d_seq4);
        fa.refcode = dp<uint32_t>(c->d_refcode); fa.span_beg = c->span_beg; fa.span_end = c->span_end;
        fa.n_samples = n; fa.n_strips = n_strips; fa.spc = pc.spc; fa.asw = pb_pile_asw(pc.spc); fa.tile_q = pc.tile_q; fa.qcap = pc.qcap; fa.tail_bytes = pc.tail;
        fa.max_span = async ? c->async_span : 0;
        fa.min_mapQ = P.min_mapQ; fa.min_rmsQ = P.min_rmsQ; fa.min_baseQ = P.min_baseQ; fa.illumina = illumina;
        fa.qual_ceiling = c->qual_ceiling;
        fa.ctr = ctr; fa.tab = dp<PbFastTables>(c->d_fastp);
        fa.acc_cov = dp<uint64_t>(c->d_acc); fa.acc_cnt4 = reinterpret_cast<uint32_t *>(fa.acc_cov + span); fa.site_type = dp<uint64_t>(c->d_site_type);
        const unsigned n_blocks = (unsigned)((n_strips + pc.spc - 1) / pc.spc);
        PB_TRY(dev_reserve(c, c->d_blk, sizeof(uint4) * (size_t)n_blocks));
        fa.blk = dp<uint4>(c->d_blk); fa.cells = dp<uint4>(c->d_cells); fa.cell_cap = cell_cap; fa.code_cap = code_cap;
        fa.codes = c->fuse_codes ? dp<uint16_t>(c->d_codes16) : nullptr; fa.codes_skip = c->codes_skip;
        if (getenv("POPBAM_B200_DEBUG"))
            fprintf(stderr, "[popbam_b200] k_pile_reads: %u CTAs of %d warps, %d strips per CTA, quality tile %d bytes, %zu bytes of shared memory\n",
                    n_blocks, pc.warps, pc.spc, pc.tile_q, pc.smem);
        PB_CUDA(c, cudaEventRecord(c->fk[3], st));
        PB_CUDA(c, cudaStreamWaitEvent(c->stream_lo, c->fk[3], 0));
        if (c->qual_robust) k_pile_reads<true><<<n_blocks, pc.warps * 32, pc.smem, c->stream_lo>>>(fa);
        else k_pile_reads<false><<<n_blocks, pc.warps * 32, pc.smem, c->stream_lo>>>(fa);
        PB_CUDA(c, cudaEventRecord(c->fk[4], c->stream_lo));
        PB_CUDA(c, cudaStreamWaitEvent(st, c->fk[4], 0));
        PbCellCodesArgs ca;
        ca.pos = fa.pos; ca.meta = fa.meta; ca.cigstart = fa.cigstart; ca.ncig = fa.ncig; ca.cigar = fa.cigar; ca.base = fa.base;
        ca.qual = fa.qual; ca.seq4 = fa.seq4; ca.span_beg = c->span_beg; ca.n_samples = n; ca.spc = pc.spc; ca.max_span = fa.max_span;
        ca.min_mapQ = P.min_mapQ; ca.min_baseQ = P.min_baseQ; ca.illumina = illumina; ca.ctr = ctr;
        ca.blk = fa.blk; ca.cells = fa.cells; ca.codes = dp<uint16_t>(c->d_codes16);
        // room for the reads that can cover a block, three times the region's average (then: the other path)
        ca.lcap = std::min(std::min(65535, (int)((c->smem_optin - pb_cell_codes_smem(n, 0)) / 4) - 64), (int)(3.0 * (32.0 * pc.spc + pc.span32) * pc.dens16 / 16.0) + 256);
        k_cell_codes<<<n_blocks, 256, pb_cell_codes_smem(n, ca.lcap), st>>>(ca);
        PbHardArgs ha;
        ha.cells = fa.cells; ha.codes = ca.codes; ha.ref = pa.ref; ha.ref_len = pa.ref_len;
        ha.span_beg = pa.span_beg; ha.span_end = pa.span_end; ha.win_beg = pa.win_beg; ha.win_end = pa.win_end; ha.n_windows = NW;
        ha.n_samples = n; ha.n_strips = n_strips;
        ha.min_depth = pa.min_depth; ha.max_depth = pa.max_depth; ha.min_rmsQ = pa.min_rmsQ; ha.min_snpQ = pa.min_snpQ;
        ha.het_mode = pa.het_mode; ha.fk = pa.fk; ha.beta = pa.beta; ha.lhet = pa.lhet; ha.ctr = ctr; ha.need_raw = dp<uint8_t>(c->d_need_raw);
        ha.acc_cov = fa.acc_cov; ha.acc_cnt4 = fa.acc_cnt4;
        ha.site_type = pa.site_type; ha.site_flag = pa.site_flag;
        k_hard_cells<<<c->g_hard_cells, PB_HARD_THREADS, pb_hard_smem(), st>>>(ha);
        k_fast_sites<<<nblk(span, 256), 256, 0, st>>>(ha);
        c->launches += 4;
    } else {
        PB_TRY(need_tables(c->ctr_host.qval, nl));
        pa.need = dp<uint8_t>(c->d_need);
        // 256-thread CTAs (40 resident warps per SM) when their shared memory stays small, else 128-thread CTAs
        const bool big = pb_pile_smem(256, nl) <= 46 * 1024;
        const int tp = big ? 256 : 128;
        const size_t smem = pb_pile_smem(tp, nl);
        if (smem > c->smem_optin) return fail(c, PB_ERR_UNSUPPORTED, "shared memory for %d quality levels exceeds %zu bytes", nl, c->smem_optin);
        void (*kern)(const PbPileArgs) = big ? (cap ? k_pileup_call<256, true> : k_pileup_call<256, false>)
                                             : (cap ? k_pileup_call<128, true> : k_pileup_call<128, false>);
        PB_CUDA(c, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        // base codes for k_pileup_call (the counting path reads qual[] / seq4[] directly)
        PB_TRY(dev_reserve(c, c->d_codes, (size_t)std::max<int64_t>(c->n_bytes, 1)));
        pa.codes = dp<uint8_t>(c->d_codes);
        if (N > 0)
            k_encode<<<c->g_encode, 256, 0, st>>>(N, dp<uint32_t>(c->d_meta), dp<uint8_t>(c->d_rkey), dp<uint64_t>(c->d_base),
                                                  dp<uint8_t>(c->d_seq4), dp<uint8_t>(c->d_qual), c->n_bytes,
                                                  (double)N / (double)std::max<int64_t>(c->n_bytes, 1), P.min_mapQ, dp<uint8_t>(c->d_qtab),
                                                  dp<uint8_t>(c->d_codes));
        PB_CUDA(c, cudaEventRecord(c->ev[2], st));
        kern<<<nblk(span, tp), tp, smem, st>>>(pa);
        c->launches += 2;
    }
    PB_CUDA(c, cudaGetLastError());
    PB_CUDA(c, cudaEventRecord(c->ev[3], st));

    // ---- per-window site counts, offsets of the segregating-site lists
    const SmallLayout dl0 = small_layout(nullptr, NW, P.n_pops, n, (c->analyses & PB_AN_TREE) != 0, (c->analyses & PB_AN_FST) != 0);
    PB_TRY(dev_reserve(c, c->d_stats, dl0.bytes));
    PB_TRY(host_reserve(c, c->h_small, dl0.bytes));
    const SmallLayout dl = small_layout(c->d_stats.p, NW, P.n_pops, n, (c->analyses & PB_AN_TREE) != 0, (c->analyses & PB_AN_FST) != 0);
    PB_CUDA(c, cudaMemsetAsync(c->d_stats.p, 0, dl.bytes, st));
    k_window_sites<false><<<NW, 256, 0, st>>>(c->span_beg, pa.win_beg, pa.win_end, pa.site_flag, pa.site_type, pa.ref, pa.ref_len, nullptr, n,
                                             dl.num_sites, dl.segsites, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr);
    k_scan_windows<<<1, 1024, 0, st>>>(dl.segsites, NW, dl.seg_off);
    c->launches += 2;
    PB_CUDA(c, cudaGetLastError());
    int64_t *h_total = reinterpret_cast<int64_t *>(c->h_ctr.p) + (sizeof(PbCounters) + 7) / 8;   // h_ctr has a page
    PB_CUDA(c, cudaMemcpyAsync(h_total, dl.seg_off + NW, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    const SmallLayout hl0 = small_layout(c->h_small.p, NW, P.n_pops, n, (c->analyses & PB_AN_TREE) != 0, (c->analyses & PB_AN_FST) != 0);
    PB_CUDA(c, cudaMemcpyAsync(hl0.segsites, dl.segsites, sizeof(int32_t) * (size_t)NW, cudaMemcpyDeviceToHost, st));
    PbCounters *h_final = reinterpret_cast<PbCounters *>(reinterpret_cast<unsigned char *>(c->h_ctr.p) + 2 * sizeof(PbCounters));
    if (async) PB_CUDA(c, cudaStreamWaitEvent(st, c->fk[2], 0));     // the per-read chain that ran beside the pileup
    PB_CUDA(c, cudaMemcpyAsync(h_final, c->d_ctr.p, sizeof(PbCounters), cudaMemcpyDeviceToHost, st));
    if (!async) PB_CUDA(c, cudaStreamSynchronize(st));
    if (!async && fast && getenv("POPBAM_B200_DEBUG"))
        fprintf(stderr, "[popbam_b200] counting path: %llu of %lld cells left for k_hard_cells (%.2f %%), %llu code slots; overflow %d, quality over ceiling %d (max %d), launch assumptions failed %d\n",
                h_final->n_cells, (long long)(span * n), 100.0 * (double)h_final->n_cells / (double)(span * n), h_final->n_codes,
                h_final->arena_overflow, h_final->qual_over, h_final->qual_max_seen, h_final->spec_fail);
    if (!async && fast && (h_final->arena_overflow || h_final->qual_over || h_final->spec_fail)) {
        // an assumption of the counting path did not hold for this region: nothing of its result is used.  Raise the
        // quality ceiling / the arena size (both stay raised for the context) and run the region again; give up on the
        // counting path for this region after three attempts.
        if (getenv("POPBAM_B200_DEBUG"))
            fprintf(stderr, "[popbam_b200] counting path: run again (arena overflow %d: %llu cells, %llu codes; quality %d above ceiling %d: %d; launch assumptions %d)\n",
                    h_final->arena_overflow, h_final->n_cells, h_final->n_codes, h_final->qual_max_seen, c->qual_ceiling, h_final->qual_over, h_final->spec_fail);
        if (h_final->qual_high) c->qual_robust = true;
        if (h_final->arena_overflow) c->arena_scale *= 4;
        c->reruns += 1;
        if (attempt >= 2 || c->arena_scale > 64) c->force_classic = 1;
        const int rc = run_pipeline(c, attempt + 1, false);
        c->force_classic = 0;
        return rc;
    }
    if (!async && fast) {           // what this region teaches the context
        c->spec_valid = true;
        c->spec_span = std::max(c->spec_span, c->ctr_host.max_span);
        c->spec_read_bytes = std::max(c->spec_read_bytes, c->ctr_host.max_read_bytes);
    }
    // number of segregating sites: known now, or (asynchronous mode) bounded by the span -- the device arrays are laid out
    // for the bound, the kernels read the real offsets from device memory, and fill_result copies what there is
    const int64_t S = async ? span : *h_total;
    c->s_total = async ? -1 : S;
    c->seg_cap = S;
    int s_max = 0;
    if (!async) for (int w = 0; w < NW; ++w) s_max = std::max(s_max, hl0.segsites[w]);

    // ---- segregating-site lists
    const bool with_cb = (c->analyses & PB_AN_SNP) != 0;
    const SegLayout sl0 = seg_layout(nullptr, S, n, with_cb);
    PB_TRY(dev_reserve(c, c->d_seg_type, sl0.bytes));
    if (!async) PB_TRY(host_reserve(c, c->h_seg, sl0.bytes));
    const SegLayout sl = seg_layout(c->d_seg_type.p, S, n, with_cb);
    k_window_sites<true><<<NW, 256, 0, st>>>(c->span_beg, pa.win_beg, pa.win_end, pa.site_flag, pa.site_type, pa.ref, pa.ref_len,
                                            with_cb ? dp<uint64_t>(c->d_cb) : nullptr, n, dl.num_sites, dl.segsites, dl.seg_off,
                                            sl.seg_pos, sl.seg_idx, sl.seg_type, sl.seg_ref, sl.seg_cb);
    c->launches += 1;
    PB_CUDA(c, cudaGetLastError());
    PB_CUDA(c, cudaEventRecord(c->ev[4], st));

    // ---- window statistics
    const uint32_t stat_bits = PB_AN_NUCDIV | PB_AN_SFS | PB_AN_LD_WALL | PB_AN_DIVERGE_IND |
                               PB_AN_DIVERGE_POP | PB_AN_HAPLO_K | PB_AN_HAPLO_EHHS | PB_AN_HAPLO_DXY | PB_AN_TREE |
                               PB_AN_THETA_W | PB_AN_FULI | PB_AN_FST;
    if (c->analyses & stat_bits) {
        PbStatArgs sa;
        memset(&sa, 0, sizeof sa);
        sa.n = n; sa.P = P.n_pops;
        for (int i = 0; i < PB_MAX_SAMPLES; ++i) { sa.pop_mask[i] = P.pop_mask[i]; sa.pop_nsmpl[i] = P.pop_nsmpl[i]; }
        sa.analyses = c->analyses; sa.flags = P.flags; sa.outidx = P.outidx; sa.min_freq = P.min_freq;
        sa.num_sites = dl.num_sites; sa.segsites = dl.segsites; sa.seg_off = dl.seg_off; sa.seg_type = sl.seg_type;
        sa.s_total = S;
        if (c->analyses & (PB_AN_NUCDIV | PB_AN_HAPLO_K | PB_AN_HAPLO_EHHS | PB_AN_HAPLO_DXY | PB_AN_DIVERGE_IND | PB_AN_TREE | PB_AN_FST)) {
            PB_TRY(dev_reserve(c, c->d_hap, sizeof(uint64_t) * (size_t)n * (size_t)(S / 64 + NW + 1)));
            sa.hap = dp<uint64_t>(c->d_hap);
        }
        if (c->analyses & PB_AN_HAPLO_EHHS) {
            PB_TRY(dev_reserve(c, c->d_kt, sizeof(uint64_t) * (size_t)(S + NW + 1)));
            PB_TRY(dev_reserve(c, c->d_km, (size_t)(S + NW + 1)));
            sa.kt = dp<uint64_t>(c->d_kt); sa.km = dp<uint8_t>(c->d_km);
        }
        if (c->analyses & PB_AN_LD_WALL) {
            PB_TRY(dev_reserve(c, c->d_wall_u, sizeof(uint64_t) * (size_t)P.n_pops * (size_t)std::max<int64_t>(S, 1)));
            sa.wall_u = dp<uint64_t>(c->d_wall_u);
        }
        sa.piw = dl.piw; sa.pib = dl.pib; sa.min_dxy = dl.min_dxy;
        sa.sfs_num_snps = dl.sfs_num_snps; sa.td = dl.td; sa.fwh = dl.fwh;
        sa.wall_num_snps = dl.wall_num_snps; sa.wallb = dl.wallb; sa.wallq = dl.wallq;
        sa.ind_div = dl.ind_div; sa.pop_div = dl.pop_div; sa.div_num_snps = dl.div_num_snps; sa.tree_diff = dl.tree_diff;
        sa.nhaps = dl.nhaps; sa.hdiv = dl.hdiv; sa.ehhs = dl.ehhs;
        sa.pop_segsites = dl.pop_segsites; sa.theta_w = dl.theta_w; sa.fuli_d = dl.fuli_d; sa.fuli_ds = dl.fuli_ds;
        sa.fuli_eta_e = dl.fuli_eta_e; sa.fuli_eta_s = dl.fuli_eta_s;
        const int npairs = P.n_pops * (P.n_pops - 1) / 2;
        const bool perms = (c->analyses & PB_AN_FST) && c->snn_perms > 0 && npairs > 0;
        c->snn_perms_run = perms ? c->snn_perms : 0;
        if (c->analyses & PB_AN_FST) {
            sa.hud_num = dl.hud_num; sa.hud_den = dl.hud_den; sa.wc_num = dl.wc_num; sa.wc_den = dl.wc_den;
            sa.fst_hudson = dl.fst_hudson; sa.fst_wc = dl.fst_wc; sa.snn = dl.snn;
            if (perms) {        // nearest-neighbour masks of every (window, pair, sample) for k_snn_perm
                PB_TRY(dev_reserve(c, c->d_snn_nn, sizeof(uint64_t) * (size_t)NW * P.n_pops * P.n_pops * n));
                sa.snn_nn = dp<uint64_t>(c->d_snn_nn);
            }
        }
        ((c->analyses & PB_AN_FST) ? k_window_stats<true> : k_window_stats<false>)<<<NW, PB_ST_THREADS, (size_t)n * n * sizeof(uint16_t), st>>>(sa);
        c->launches += 1;
        PB_CUDA(c, cudaGetLastError());
        if (perms) {
            PbSnnArgs ka;
            memset(&ka, 0, sizeof ka);
            ka.n = n; ka.P = P.n_pops; ka.tid = c->ref_tid;
            for (int i = 0; i < PB_MAX_SAMPLES; ++i) { ka.pop_mask[i] = P.pop_mask[i]; ka.pop_nsmpl[i] = P.pop_nsmpl[i]; }
            ka.win_beg = dp<int32_t>(c->d_wbeg); ka.nn = sa.snn_nn; ka.snn = dl.snn; ka.snn_p = dl.snn_p; ka.snn_ge = dl.snn_ge;
            ka.n_perms = c->snn_perms; ka.seed = c->snn_seed;
            k_snn_perm<<<dim3((unsigned)NW, (unsigned)npairs), PB_ST_THREADS, 0, st>>>(ka);
            c->launches += 1;
            PB_CUDA(c, cudaGetLastError());
        }
    }
    // ---- pairwise LD (ld -o 0 / -o 1, D'): keep list, tiled pair kernel, finish
    if (c->analyses & (PB_AN_LD_ZNS | PB_AN_LD_OMEGA | PB_AN_LD_DPRIME)) {
        PbLdArgs la;
        memset(&la, 0, sizeof la);
        la.P = P.n_pops;
        for (int i = 0; i < PB_MAX_SAMPLES; ++i) { la.pop_mask[i] = P.pop_mask[i]; la.pop_nsmpl[i] = P.pop_nsmpl[i]; }
        la.min_freq = P.min_freq; la.analyses = c->analyses;
        la.segsites = dl.segsites; la.seg_off = dl.seg_off; la.seg_type = sl.seg_type;
        la.stride = S + 2 * (int64_t)NW + 2;
        const size_t cnt = (size_t)P.n_pops * (size_t)la.stride;
        PB_TRY(dev_reserve(c, c->d_ld_kt, sizeof(uint64_t) * cnt));
        PB_TRY(dev_reserve(c, c->d_ld_km, sizeof(int32_t) * cnt));
        PB_TRY(dev_reserve(c, c->d_ld_inv, sizeof(double) * cnt));
        PB_TRY(dev_reserve(c, c->d_lsum, sizeof(double) * cnt));
        PB_TRY(dev_reserve(c, c->d_rsum, sizeof(double) * cnt));
        PB_TRY(dev_reserve(c, c->d_ld_cnt, sizeof(int32_t) * 2 * (size_t)NW * P.n_pops));
        la.kt = dp<uint64_t>(c->d_ld_kt); la.km = dp<int32_t>(c->d_ld_km); la.kinv = dp<double>(c->d_ld_inv);
        la.lsum = dp<double>(c->d_lsum); la.rsum = dp<double>(c->d_rsum);
        la.kcount = dp<int32_t>(c->d_ld_cnt); la.nsnps = la.kcount + (size_t)NW * P.n_pops;
        la.ld_num_snps = dl.ld_num_snps; la.zns = dl.zns; la.omegamax = dl.omegamax;
        la.ld_kept = dl.ld_kept; la.ld_dprime = dl.ld_dprime; la.ld_complete = dl.ld_complete;
        const bool dprime = (c->analyses & PB_AN_LD_DPRIME) != 0;
        if (dprime) {      // per-row |D'| sums (double) and complete-pair counts (int32)
            PB_TRY(dev_reserve(c, c->d_ld_dp, (sizeof(double) + sizeof(int32_t)) * cnt));
            la.dpsum = dp<double>(c->d_ld_dp); la.dpfull = reinterpret_cast<int32_t *>(la.dpsum + cnt);
        }
        const unsigned pw = (unsigned)NW * (unsigned)P.n_pops;
        const int nrb = std::max(1, (s_max + PB_LD_THREADS - 1) / PB_LD_THREADS);
        k_ld_keep<<<pw, PB_LD_THREADS, 0, st>>>(la);
        (dprime ? k_ld_rows<true> : k_ld_rows<false>)<<<pw * (unsigned)nrb, PB_LD_THREADS, 0, st>>>(la, (c->analyses & PB_AN_LD_OMEGA) ? 1 : 0, nrb);
        k_ld_finish<<<pw, PB_LD_THREADS, 0, st>>>(la);
        c->launches += 3;
        PB_CUDA(c, cudaGetLastError());
    }
    PB_CUDA(c, cudaEventRecord(c->ev[5], st));

    // ---- results to pinned host memory
    PB_CUDA(c, cudaMemcpyAsync(c->h_small.p, c->d_stats.p, dl.bytes, cudaMemcpyDeviceToHost, st));
    if (!async && S > 0) PB_CUDA(c, cudaMemcpyAsync(c->h_seg.p, c->d_seg_type.p, sl.bytes, cudaMemcpyDeviceToHost, st));
    if (P.flags & PB_FLAG_EMIT_CB) {
        Carver cv(nullptr);
        cv.take<uint64_t>((size_t)span * n); cv.take<uint64_t>((size_t)span); cv.take<uint8_t>((size_t)span);
        PB_TRY(host_reserve(c, c->h_span, cv.off + 64));
        Carver hv(c->h_span.p);
        uint64_t *hcb = hv.take<uint64_t>((size_t)span * n);
        uint64_t *hty = hv.take<uint64_t>((size_t)span);
        uint8_t *hfl = hv.take<uint8_t>((size_t)span);
        PB_CUDA(c, cudaMemcpyAsync(hcb, c->d_cb.p, sizeof(uint64_t) * (size_t)span * n, cudaMemcpyDeviceToHost, st));
        PB_CUDA(c, cudaMemcpyAsync(hty, c->d_site_type.p, sizeof(uint64_t) * (size_t)span, cudaMemcpyDeviceToHost, st));
        PB_CUDA(c, cudaMemcpyAsync(hfl, c->d_site_flag.p, (size_t)span, cudaMemcpyDeviceToHost, st));
    }
    return PB_OK;
}

int fill_result(pb_ctx *c, pb_region_result *out) {
    const pb_params &P = c->prm;
    const int n = P.n_samples, NW = c->nw;
    PB_CUDA(c, cudaStreamSynchronize(c->stream));
    if (c->async_run) {
        // the region was enqueued on assumptions (run_pipeline): look at what the device found
        const PbCounters fin = *reinterpret_cast<PbCounters *>(reinterpret_cast<unsigned char *>(c->h_ctr.p) + 2 * sizeof(PbCounters));
        if (fin.unsorted) return fail(c, PB_ERR_UNSORTED, "reads are not sorted by position (bam_pileup.c:384-395)");
        if (fin.too_long) return fail(c, PB_ERR_UNSUPPORTED, "a read spans 65536 or more reference bases or has more than 255 aligned segments");
        if (fin.total_bound > 8000) return fail(c, PB_ERR_UNSUPPORTED, "up to %d reads may be live at one position: above 8000 the reference's pileup drops reads (bam_pileup.c:260,375), which this library does not reproduce", fin.total_bound);
        if (getenv("POPBAM_B200_DEBUG"))
            fprintf(stderr, "[popbam_b200] asynchronous region: %llu cells left for k_hard_cells, overflow %d, quality over ceiling %d (max %d), launch assumptions failed %d\n",
                    fin.n_cells, fin.arena_overflow, fin.qual_over, fin.qual_max_seen, fin.spec_fail);
        if (fin.arena_overflow || fin.qual_over || fin.spec_fail || fin.max_span > c->async_span || !fin.nocap) {
            if (fin.qual_high) c->qual_robust = true;
            if (fin.arena_overflow) c->arena_scale *= 4;
            c->reruns += 1;
            PB_TRY(run_pipeline(c, 0, false));          // with the host round trips: learns the span / density / cap again
            PB_CUDA(c, cudaStreamSynchronize(c->stream));
        } else {
            c->spec_span = std::max(c->spec_span, fin.max_span);
            c->spec_read_bytes = std::max(c->spec_read_bytes, fin.max_read_bytes);
            c->ctr_host = fin;
            // the segregating-site arrays: device layout for seg_cap entries, host layout for the S there are
            const int64_t S = *(reinterpret_cast<int64_t *>(c->h_ctr.p) + (sizeof(PbCounters) + 7) / 8);
            c->s_total = S;
            const SegLayout dl = seg_layout(c->d_seg_type.p, c->seg_cap, n, false), hl0 = seg_layout(nullptr, S, n, false);
            PB_TRY(host_reserve(c, c->h_seg, hl0.bytes));
            const SegLayout hl = seg_layout(c->h_seg.p, S, n, false);
            if (S > 0) {
                PB_CUDA(c, cudaMemcpyAsync(hl.seg_type, dl.seg_type, sizeof(uint64_t) * (size_t)S, cudaMemcpyDeviceToHost, c->stream));
                PB_CUDA(c, cudaMemcpyAsync(hl.seg_pos, dl.seg_pos, sizeof(uint32_t) * (size_t)S, cudaMemcpyDeviceToHost, c->stream));
                PB_CUDA(c, cudaMemcpyAsync(hl.seg_idx, dl.seg_idx, sizeof(uint32_t) * (size_t)S, cudaMemcpyDeviceToHost, c->stream));
                PB_CUDA(c, cudaMemcpyAsync(hl.seg_ref, dl.seg_ref, (size_t)S, cudaMemcpyDeviceToHost, c->stream));
                PB_CUDA(c, cudaStreamSynchronize(c->stream));
            }
        }
        c->async_run = false;
    }
    cudaEventElapsedTime(&c->ms_prep, c->ev[0], c->ev[1]);
    { float per_base = 0; cudaEventElapsedTime(&per_base, c->ev[6], c->ev[2]); c->ms_prep += per_base; }
    cudaEventElapsedTime(&c->ms_pileup, c->ev[2], c->ev[3]);
    cudaEventElapsedTime(&c->ms_sites, c->ev[3], c->ev[4]);
    cudaEventElapsedTime(&c->ms_stats, c->ev[4], c->ev[5]);
    const SmallLayout hl = small_layout(c->h_small.p, NW, P.n_pops, n, (c->analyses & PB_AN_TREE) != 0, (c->analyses & PB_AN_FST) != 0);
    const bool with_cb = (c->analyses & PB_AN_SNP) != 0;
    const SegLayout sl = seg_layout(c->h_seg.p, c->s_total, n, with_cb);
    pb_region_result &r = c->res;
    memset(&r, 0, sizeof r);
    r.n_windows = NW; r.n_pops = P.n_pops; r.n_samples = n; r.analyses = c->analyses;
    r.win_beg = c->h_wbeg.data(); r.win_end = c->h_wend.data();
    r.num_sites = hl.num_sites; r.segsites = hl.segsites; r.seg_off = hl.seg_off;
    r.seg_pos = sl.seg_pos; r.seg_idx = sl.seg_idx; r.seg_type = sl.seg_type; r.seg_ref = sl.seg_ref; r.seg_cb = sl.seg_cb;
    const uint32_t an = c->analyses;
    if (an & (PB_AN_NUCDIV | PB_AN_HAPLO_DXY)) { r.piw = hl.piw; r.pib = hl.pib; r.min_dxy = hl.min_dxy; }
    if (an & PB_AN_SFS) { r.sfs_num_snps = hl.sfs_num_snps; r.td = hl.td; r.fwh = hl.fwh; }
    if (an & (PB_AN_LD_ZNS | PB_AN_LD_OMEGA)) { r.ld_num_snps = hl.ld_num_snps; r.zns = hl.zns; r.omegamax = hl.omegamax; }
    if (an & PB_AN_LD_WALL) { r.wall_num_snps = hl.wall_num_snps; r.wallb = hl.wallb; r.wallq = hl.wallq; }
    if (an & PB_AN_DIVERGE_IND) r.ind_div = hl.ind_div;
    if (an & PB_AN_TREE) r.tree_diff = hl.tree_diff;
    pb_region_extras &e = c->ext;
    memset(&e, 0, sizeof e);
    if (an & (PB_AN_THETA_W | PB_AN_FULI)) e.pop_segsites = hl.pop_segsites;
    if (an & PB_AN_THETA_W) e.theta_w = hl.theta_w;
    if (an & PB_AN_FULI) { e.fuli_d = hl.fuli_d; e.fuli_ds = hl.fuli_ds; e.fuli_eta_e = hl.fuli_eta_e; e.fuli_eta_s = hl.fuli_eta_s; }
    if (an & PB_AN_LD_DPRIME) { r.ld_num_snps = hl.ld_num_snps; e.ld_kept = hl.ld_kept; e.ld_dprime = hl.ld_dprime; e.ld_complete = hl.ld_complete; }
    pb_region_fst &f = c->fst;
    memset(&f, 0, sizeof f);
    if (an & PB_AN_FST) {
        f.hud_num = hl.hud_num; f.hud_den = hl.hud_den; f.wc_num = hl.wc_num; f.wc_den = hl.wc_den;
        f.fst_hudson = hl.fst_hudson; f.fst_wc = hl.fst_wc; f.snn = hl.snn;
        if (c->snn_perms_run > 0) { f.snn_p = hl.snn_p; f.snn_ge = hl.snn_ge; }
    }
    if (an & PB_AN_DIVERGE_POP) { r.pop_div = hl.pop_div; r.div_num_snps = hl.div_num_snps; }
    if (an & (PB_AN_HAPLO_K | PB_AN_HAPLO_EHHS)) { r.nhaps = hl.nhaps; r.hdiv = hl.hdiv; }
    if (an & PB_AN_HAPLO_EHHS) r.ehhs = hl.ehhs;
    r.span_beg = c->span_beg; r.span_end = c->span_end;
    if (P.flags & PB_FLAG_EMIT_CB) {
        const size_t span = (size_t)(c->span_end - c->span_beg);
        Carver hv(c->h_span.p);
        r.cb = hv.take<uint64_t>(span * n);
        r.site_type = hv.take<uint64_t>(span);
        r.site_flag = hv.take<uint8_t>(span);
    }
    r.reads_pushed = c->n_reads;
    r.reads_used = (int64_t)c->ctr_host.reads_used;
    r.aligned_bases = (int64_t)c->ctr_host.aligned_bases;
    if (out) *out = r;
    return PB_OK;
}

int flush_records(pb_ctx *c);

}  // namespace

// ================================================================================================
extern "C" {

const char *pb_version(void) { return "popbam_b200 0.1 (sm_100a)"; }

const char *pb_last_error(const pb_ctx *ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

pb_ctx *pb_create(const pb_params *p, const pb_errmod_tables *tables, int *status) {
    auto bail = [&](int code, const char *msg, pb_ctx *c) -> pb_ctx * {
        g_create_error = msg;
        if (c && c->err.size()) g_create_error += std::string(": ") + c->err;
        if (status) *status = code;
        if (c) pb_destroy(c);
        return nullptr;
    };
    if (!p) return bail(PB_ERR_ARG, "null params", nullptr);
    if (p->n_samples < 1 || p->n_samples > PB_MAX_SAMPLES || p->n_pops < 1 || p->n_pops > PB_MAX_SAMPLES)
        return bail(PB_ERR_ARG, "n_samples / n_pops out of range (1..64)", nullptr);
    if (p->max_depth < 1 || p->max_depth > 255)
        return bail(PB_ERR_UNSUPPORTED, "max_depth must be in 1..255 (errmod_cal subsamples above 255, pop_utils.cpp:293)", nullptr);
    // the error-model tables take ~0.25 s of host arithmetic: build them while the CUDA context comes up
    const size_t nb = (size_t)64 * 256 * 256;
    std::vector<double> fk, beta, lhet;
    const bool own_tables = !(tables && tables->fk && tables->beta && tables->lhet);
    std::future<void> table_job;
    if (own_tables) {
        fk.resize(256); beta.resize(nb); lhet.resize(65536);
        table_job = std::async(std::launch::async, [&]() { pb_errmod_tables_cached(fk.data(), beta.data(), lhet.data(), nullptr); });
    }
    struct Joiner { std::future<void> &f; ~Joiner() { if (f.valid()) f.wait(); } } joiner{table_job};
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev < 1) {
        cudaGetLastError();
        return bail(PB_ERR_CUDA, "no CUDA device available (this library has no CPU path)", nullptr);
    }
    if (p->device < 0 || p->device >= ndev) return bail(PB_ERR_ARG, "device ordinal out of range", nullptr);
    if (cudaSetDevice(p->device) != cudaSuccess) return bail(PB_ERR_CUDA, "cudaSetDevice failed", nullptr);
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, p->device) != cudaSuccess) return bail(PB_ERR_CUDA, "cudaGetDeviceProperties failed", nullptr);
    if (prop.major < 10) return bail(PB_ERR_CUDA, "device is not sm_100 class (kernels are built for sm_100a only)", nullptr);
    pb_ctx *c = new pb_ctx();
    c->prm = *p;
    c->n_sms = prop.multiProcessorCount;
    c->smem_optin = prop.sharedMemPerBlockOptin; c->smem_per_sm = prop.sharedMemPerMultiprocessor;
    { const char *e = getenv("POPBAM_B200_PILEUP"); c->classic = e && strcmp(e, "classic") == 0; }
    { const char *e = getenv("POPBAM_B200_SYNC"); c->no_async = e && *e == '1'; }
    { const char *e = getenv("POPBAM_B200_PILE"); if (e) sscanf(e, "%d,%d", &c->pile_spc, &c->pile_warps); }
    { const char *e = getenv("POPBAM_B200_CODES"); if (e && !strcmp(e, "separate")) c->fuse_codes = false; if (e && !strcmp(e, "mixed")) c->codes_skip = 1; }
    { const char *e = getenv("POPBAM_B200_QCEIL"); if (e && atoi(e) >= 4) c->qual_ceiling = std::min(63, atoi(e)); }
    {
        auto wave = [&](auto kern, int threads) {
            int per_sm = 0;
            if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, threads, 0) != cudaSuccess || per_sm < 1) { cudaGetLastError(); per_sm = 1; }
            return c->n_sms * per_sm;
        };
        c->g_encode = wave(k_encode, 256);
        c->g_qual_mask = wave(k_qual_mask, 256);
        c->g_read_prep = wave(k_read_prep, 256);
        {
            int per_sm = 0;
            cudaFuncSetAttribute(k_hard_cells, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pb_hard_smem());
            if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_hard_cells, PB_HARD_THREADS, pb_hard_smem()) != cudaSuccess || per_sm < 1) { cudaGetLastError(); per_sm = 1; }
            c->g_hard_cells = c->n_sms * per_sm;
        }
    }
    // (once per process would do: the attribute belongs to the function, not to the context)
    c->smem_optin -= std::min<size_t>(c->smem_optin, 2048);              // (room for the kernels' static shared memory)
    if (cudaFuncSetAttribute(k_pile_reads<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)c->smem_optin) != cudaSuccess ||
        cudaFuncSetAttribute(k_pile_reads<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)c->smem_optin) != cudaSuccess ||
        cudaFuncSetAttribute(k_cell_codes, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)c->smem_optin) != cudaSuccess) {
        cudaGetLastError();
        return bail(PB_ERR_CUDA, "cudaFuncSetAttribute(shared memory) failed", c);
    }
    {
        int least = 0, greatest = 0;
        if (cudaDeviceGetStreamPriorityRange(&least, &greatest) != cudaSuccess) { cudaGetLastError(); least = greatest = 0; }
        if (cudaStreamCreateWithPriority(&c->stream, cudaStreamNonBlocking, greatest) != cudaSuccess) return bail(PB_ERR_CUDA, "cudaStreamCreate failed", c);
        if (cudaStreamCreateWithPriority(&c->stream2, cudaStreamNonBlocking, greatest) != cudaSuccess) return bail(PB_ERR_CUDA, "cudaStreamCreate failed", c);
        if (cudaStreamCreateWithPriority(&c->stream_lo, cudaStreamNonBlocking, least) != cudaSuccess) return bail(PB_ERR_CUDA, "cudaStreamCreate failed", c);
    }
    for (auto &ev : c->ev)
        if (cudaEventCreate(&ev) != cudaSuccess) return bail(PB_ERR_CUDA, "cudaEventCreate failed", c);
    for (auto &ev : c->fk)
        if (cudaEventCreateWithFlags(&ev, cudaEventDisableTiming) != cudaSuccess) return bail(PB_ERR_CUDA, "cudaEventCreate failed", c);
    if (getenv("POPBAM_B200_DEBUG"))
        for (auto &ev : c->dbg) cudaEventCreate(&ev);
    // error-model tables
    const double *pfk, *pbeta, *plhet;
    if (!own_tables) { pfk = tables->fk; pbeta = tables->beta; plhet = tables->lhet; }
    else {
        table_job.wait();
        pfk = fk.data(); pbeta = beta.data(); plhet = lhet.data();
    }
    if (dev_reserve(c, c->d_fk, 256 * 8) || dev_reserve(c, c->d_beta, nb * 8) || dev_reserve(c, c->d_lhet, 65536 * 8))
        return bail(PB_ERR_NOMEM, "table allocation failed", c);
    if (cudaMemcpy(c->d_fk.p, pfk, 256 * 8, cudaMemcpyHostToDevice) != cudaSuccess ||
        cudaMemcpy(c->d_beta.p, pbeta, nb * 8, cudaMemcpyHostToDevice) != cudaSuccess ||
        cudaMemcpy(c->d_lhet.p, plhet, 65536 * 8, cudaMemcpyHostToDevice) != cudaSuccess)
        return bail(PB_ERR_CUDA, "table upload failed", c);
    if (dev_reserve(c, c->d_rms_thr, 256 * sizeof(int32_t))) return bail(PB_ERR_NOMEM, "table allocation failed", c);
    k_rms_table<<<1, 256, 0, c->stream>>>(p->min_rmsQ, dp<int32_t>(c->d_rms_thr));
    c->launches += 1;
    if (cudaStreamSynchronize(c->stream) != cudaSuccess) return bail(PB_ERR_CUDA, "k_rms_table failed", c);
    if (status) *status = PB_OK;
    return c;
}

void pb_destroy(pb_ctx *c) {
    if (!c) return;
    cudaSetDevice(c->prm.device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    if (c->stream2) cudaStreamSynchronize(c->stream2);
    if (c->stream_lo) cudaStreamSynchronize(c->stream_lo);
    for (DevBuf *b : c->bufs) if (b->p) { cudaFree(b->p); b->p = nullptr; b->cap = 0; }
    HostBuf *hb[] = {&c->h_ctr, &c->h_small, &c->h_seg, &c->h_span};
    for (HostBuf *b : hb) if (b->p) cudaFreeHost(b->p);
    for (auto &ev : c->ev) if (ev) cudaEventDestroy(ev);
    for (auto &ev : c->fk) if (ev) cudaEventDestroy(ev);
    for (auto &ev : c->dbg) if (ev) cudaEventDestroy(ev);
    if (c->stream2) cudaStreamDestroy(c->stream2);
    if (c->stream_lo) cudaStreamDestroy(c->stream_lo);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
}

int pb_set_contig(pb_ctx *c, int32_t tid, const char *ref_bases, int64_t len) {
    if (!c || !ref_bases || len < 0) return fail(c, PB_ERR_ARG, "pb_set_contig: bad argument");
    if (c->state == ST_OPEN || c->state == ST_LAUNCHED) return fail(c, PB_ERR_STATE, "pb_set_contig inside a region");
    PB_CUDA(c, cudaSetDevice(c->prm.device));
    PB_TRY(dev_reserve(c, c->d_ref, (size_t)std::max<int64_t>(len, 1)));
    PB_CUDA(c, cudaMemcpyAsync(c->d_ref.p, ref_bases, (size_t)len, cudaMemcpyHostToDevice, c->stream));
    PB_CUDA(c, cudaStreamSynchronize(c->stream));
    PB_TRY(dev_reserve(c, c->d_refcode, ((size_t)len + PB_REFCODE_PAD) / 8 * 4 + 64));
    k_ref_codes<<<c->n_sms * 4, 256, 0, c->stream>>>(dp<char>(c->d_ref), len, dp<uint32_t>(c->d_refcode));
    c->launches += 1;
    PB_CUDA(c, cudaGetLastError());
    PB_CUDA(c, cudaStreamSynchronize(c->stream));
    c->ref_len = len; c->ref_tid = tid;
    return PB_OK;
}

int pb_region_begin(pb_ctx *c, uint32_t analyses, int32_t n_windows, const int32_t *win_beg, const int32_t *win_end) {
    if (!c || n_windows < 1 || !win_beg || !win_end) return fail(c, PB_ERR_ARG, "pb_region_begin: bad argument");
    if (c->ref_tid < 0 && c->ref_len == 0) return fail(c, PB_ERR_STATE, "pb_region_begin before pb_set_contig");
    for (int i = 0; i < n_windows; ++i) {
        if (win_end[i] < win_beg[i]) return fail(c, PB_ERR_ARG, "window %d has end < begin", i);
        if (i && win_beg[i] < win_end[i - 1]) return fail(c, PB_ERR_ARG, "windows must be sorted and disjoint (window %d)", i);
    }
    if ((int64_t)win_end[n_windows - 1] - win_beg[0] < 1) return fail(c, PB_ERR_ARG, "empty region");
    PB_CUDA(c, cudaSetDevice(c->prm.device));
    PB_CUDA(c, cudaStreamSynchronize(c->stream));
    c->analyses = analyses; c->nw = n_windows;
    c->h_wbeg.assign(win_beg, win_beg + n_windows); c->h_wend.assign(win_end, win_end + n_windows);
    c->span_beg = win_beg[0]; c->span_end = win_end[n_windows - 1];
    PB_TRY(dev_reserve(c, c->d_wbeg, sizeof(int32_t) * (size_t)n_windows));
    PB_TRY(dev_reserve(c, c->d_wend, sizeof(int32_t) * (size_t)n_windows));
    PB_CUDA(c, cudaMemcpyAsync(c->d_wbeg.p, c->h_wbeg.data(), sizeof(int32_t) * (size_t)n_windows, cudaMemcpyHostToDevice, c->stream));
    PB_CUDA(c, cudaMemcpyAsync(c->d_wend.p, c->h_wend.data(), sizeof(int32_t) * (size_t)n_windows, cudaMemcpyHostToDevice, c->stream));
    c->n_reads = c->n_cig = c->n_bytes = c->n_pushes = 0;
    c->r_pos.clear(); c->r_meta.clear(); c->r_cig_off.clear(); c->r_cigar.clear(); c->r_base_off.clear(); c->r_seq4.clear(); c->r_qual.clear();
    c->state = ST_OPEN;
    return PB_OK;
}

int pb_push_batch_async(pb_ctx *c, const pb_read_batch *b) {
    if (!c || !b) return fail(c, PB_ERR_ARG, "pb_push_batch: null argument");
    if (c->state != ST_OPEN) return fail(c, PB_ERR_STATE, "pb_push_batch outside pb_region_begin .. pb_region_launch");
    if (b->n_reads < 0 || b->n_cigar < 0 || b->n_bases < 0 || (b->n_bases & 1)) return fail(c, PB_ERR_ARG, "pb_push_batch: bad counts");
    if (b->n_reads == 0) return PB_OK;
    if (!b->pos || !b->meta || !b->cig_off || !b->cigar || !b->base_off || !b->seq4 || !b->qual) return fail(c, PB_ERR_ARG, "pb_push_batch: null array");
    if ((uint64_t)b->n_bases > 0xffffffffULL || (uint64_t)b->n_cigar > 0xffffffffULL) return fail(c, PB_ERR_ARG, "pb_push_batch: a batch holds at most 2^32 - 1 base bytes / CIGAR operations (its offsets are 32-bit); split it");
    if (b->cig_off[0] != 0 || b->base_off[0] != 0 || (int64_t)b->cig_off[b->n_reads] != b->n_cigar || (int64_t)b->base_off[b->n_reads] != b->n_bases)
        return fail(c, PB_ERR_ARG, "pb_push_batch: cig_off / base_off do not start at 0 or do not end at n_cigar / n_bases");
    if ((uint64_t)(c->n_cig + b->n_cigar) > 0xfffffff0ULL) return fail(c, PB_ERR_UNSUPPORTED, "more than 2^32 CIGAR operations in one region");
    if ((uint64_t)(c->n_reads + b->n_reads) > 0xfffffff0ULL) return fail(c, PB_ERR_UNSUPPORTED, "more than 2^32 reads in one region");
    if ((uint64_t)(c->n_bytes + b->n_bases) >> 36) return fail(c, PB_ERR_UNSUPPORTED, "more than 2^36 base bytes in one region");
    PB_CUDA(c, cudaSetDevice(c->prm.device));
    cudaStream_t st = c->stream;
    const int64_t N0 = c->n_reads, N1 = N0 + b->n_reads;
    PB_TRY(dev_reserve(c, c->d_pos, 4 * (size_t)N1, 4 * (size_t)N0));
    PB_TRY(dev_reserve(c, c->d_meta, 4 * (size_t)N1, 4 * (size_t)N0));
    PB_TRY(dev_reserve(c, c->d_cigstart, 4 * (size_t)N1, 4 * (size_t)N0));
    PB_TRY(dev_reserve(c, c->d_ncig, 4 * (size_t)N1, 4 * (size_t)N0));
    PB_TRY(dev_reserve(c, c->d_base, 8 * (size_t)N1, 8 * (size_t)N0));
    PB_TRY(dev_reserve(c, c->d_cigar, 4 * (size_t)(c->n_cig + b->n_cigar), 4 * (size_t)c->n_cig));
    // 64 zeroed bytes behind the last base: the bulk copies of k_pile_reads round a tile's end up to 16 bytes, its scatter reads a few words past a segment
    PB_TRY(dev_reserve(c, c->d_qual, (size_t)(c->n_bytes + b->n_bases) + 96, (size_t)c->n_bytes));
    PB_TRY(dev_reserve(c, c->d_seq4, (size_t)(c->n_bytes + b->n_bases) / 2 + 96, (size_t)c->n_bytes / 2));
    // batch-relative offsets of every push of the region, one after the other (no push waits for the one before it)
    const size_t t0 = (size_t)N0 + (size_t)c->n_pushes;
    PB_TRY(dev_reserve(c, c->d_tmp_cig, 4 * (t0 + (size_t)b->n_reads + 1), 4 * t0));
    PB_TRY(dev_reserve(c, c->d_tmp_base, 4 * (t0 + (size_t)b->n_reads + 1), 4 * t0));
    PB_CUDA(c, cudaMemcpyAsync(dp<int32_t>(c->d_pos) + N0, b->pos, 4 * (size_t)b->n_reads, cudaMemcpyHostToDevice, st));
    PB_CUDA(c, cudaMemcpyAsync(dp<uint32_t>(c->d_meta) + N0, b->meta, 4 * (size_t)b->n_reads, cudaMemcpyHostToDevice, st));
    PB_CUDA(c, cudaMemcpyAsync(dp<uint32_t>(c->d_tmp_cig) + t0, b->cig_off, 4 * (size_t)(b->n_reads + 1), cudaMemcpyHostToDevice, st));
    PB_CUDA(c, cudaMemcpyAsync(dp<uint32_t>(c->d_tmp_base) + t0, b->base_off, 4 * (size_t)(b->n_reads + 1), cudaMemcpyHostToDevice, st));
    if (b->n_cigar) PB_CUDA(c, cudaMemcpyAsync(dp<uint32_t>(c->d_cigar) + c->n_cig, b->cigar, 4 * (size_t)b->n_cigar, cudaMemcpyHostToDevice, st));
    if (b->n_bases) {
        PB_CUDA(c, cudaMemcpyAsync(dp<uint8_t>(c->d_qual) + c->n_bytes, b->qual, (size_t)b->n_bases, cudaMemcpyHostToDevice, st));
        PB_CUDA(c, cudaMemcpyAsync(dp<uint8_t>(c->d_seq4) + c->n_bytes / 2, b->seq4, (size_t)b->n_bases / 2, cudaMemcpyHostToDevice, st));
    }
    PB_CUDA(c, cudaMemsetAsync(dp<uint8_t>(c->d_qual) + c->n_bytes + b->n_bases, 0, 64, st));
    PB_CUDA(c, cudaMemsetAsync(dp<uint8_t>(c->d_seq4) + (c->n_bytes + b->n_bases) / 2, 0, 64, st));
    k_rebase<<<nblk(b->n_reads, 256), 256, 0, st>>>(b->n_reads, N0, dp<uint32_t>(c->d_tmp_cig) + t0, dp<uint32_t>(c->d_tmp_base) + t0, (uint64_t)c->n_cig,
                                                   (uint64_t)c->n_bytes, dp<uint32_t>(c->d_cigstart), dp<uint32_t>(c->d_ncig), dp<uint64_t>(c->d_base));
    c->launches += 1;
    PB_CUDA(c, cudaGetLastError());
    c->n_reads = N1; c->n_cig += b->n_cigar; c->n_bytes += b->n_bases; c->n_pushes += 1;
    return PB_OK;
}

int pb_region_reserve(pb_ctx *c, int64_t n_reads, int64_t n_cigar, int64_t n_bases) {
    if (!c || n_reads < 0 || n_cigar < 0 || n_bases < 0) return fail(c, PB_ERR_ARG, "pb_region_reserve: bad argument");
    if (c->state != ST_OPEN) return fail(c, PB_ERR_STATE, "pb_region_reserve outside pb_region_begin .. pb_region_launch");
    PB_CUDA(c, cudaSetDevice(c->prm.device));
    const size_t N1 = (size_t)(c->n_reads + n_reads), C1 = (size_t)(c->n_cig + n_cigar), B1 = (size_t)(c->n_bytes + n_bases);
    PB_TRY(dev_reserve(c, c->d_pos, 4 * N1, 4 * (size_t)c->n_reads));
    PB_TRY(dev_reserve(c, c->d_meta, 4 * N1, 4 * (size_t)c->n_reads));
    PB_TRY(dev_reserve(c, c->d_cigstart, 4 * N1, 4 * (size_t)c->n_reads));
    PB_TRY(dev_reserve(c, c->d_ncig, 4 * N1, 4 * (size_t)c->n_reads));
    PB_TRY(dev_reserve(c, c->d_base, 8 * N1, 8 * (size_t)c->n_reads));
    PB_TRY(dev_reserve(c, c->d_cigar, 4 * C1, 4 * (size_t)c->n_cig));
    PB_TRY(dev_reserve(c, c->d_qual, B1 + 96, (size_t)c->n_bytes));
    PB_TRY(dev_reserve(c, c->d_seq4, B1 / 2 + 96, (size_t)c->n_bytes / 2));
    const size_t t0 = (size_t)c->n_reads + (size_t)c->n_pushes;
    PB_TRY(dev_reserve(c, c->d_tmp_cig, 4 * (N1 + (size_t)c->n_pushes + 64), 4 * t0));
    PB_TRY(dev_reserve(c, c->d_tmp_base, 4 * (N1 + (size_t)c->n_pushes + 64), 4 * t0));
    return PB_OK;
}

int pb_push_batch(pb_ctx *c, const pb_read_batch *b) {
    const int rc = pb_push_batch_async(c, b);
    if (rc != PB_OK) return rc;
    PB_CUDA(c, cudaStreamSynchronize(c->stream));                  // the caller may reuse its arrays when this returns
    return PB_OK;
}

int pb_push_record(pb_ctx *c, const void *core32, const void *data, int32_t l_data, int32_t sample) {
    if (!c || !core32 || !data) return fail(c, PB_ERR_ARG, "pb_push_record: null argument");
    if (c->state != ST_OPEN) return fail(c, PB_ERR_STATE, "pb_push_record outside a region");
    // bam1_core_t (bam.h:178-190): tid, pos, bin:16 qual:8 l_qname:8, flag:16 n_cigar:16, l_qseq, mtid, mpos, isize
    const uint32_t *w = reinterpret_cast<const uint32_t *>(core32);
    const int32_t tid = (int32_t)w[0], pos = (int32_t)w[1];
    const uint32_t mapq = (w[2] >> 8) & 0xff, l_qname = w[2] & 0xff, flag = w[3] >> 16, n_cigar = w[3] & 0xffff;
    const int32_t l_qseq = (int32_t)w[4];
    if (l_qseq < 0 || (int64_t)l_qname + 4 * (int64_t)n_cigar + (l_qseq + 1) / 2 + l_qseq > l_data)
        return fail(c, PB_ERR_ARG, "pb_push_record: record shorter than its core says");
    if (tid < 0) return PB_OK;                                       // bam_plp_push drops tid < 0 (bam_pileup.c:371)
    const uint8_t *d = reinterpret_cast<const uint8_t *>(data);
    const uint8_t *cig = d + l_qname, *seq = cig + 4 * n_cigar, *qual = seq + (l_qseq + 1) / 2;
    if (c->r_cig_off.empty()) { c->r_cig_off.push_back(0); c->r_base_off.push_back(0); }
    c->r_pos.push_back(pos);
    c->r_meta.push_back(flag << 16 | mapq << 8 | (uint32_t)(sample >= 0 && sample < 255 ? sample : PB_NO_SAMPLE));
    for (uint32_t i = 0; i < n_cigar; ++i) { uint32_t v; memcpy(&v, cig + 4 * i, 4); c->r_cigar.push_back(v); }
    c->r_cig_off.push_back((uint32_t)c->r_cigar.size());
    const size_t pad = (size_t)(l_qseq + 1) & ~(size_t)1;
    c->r_qual.insert(c->r_qual.end(), qual, qual + l_qseq);
    c->r_qual.resize(c->r_qual.size() + (pad - (size_t)l_qseq), 0);
    c->r_seq4.insert(c->r_seq4.end(), seq, seq + (l_qseq + 1) / 2);
    c->r_base_off.push_back((uint32_t)c->r_qual.size());
    if (c->r_qual.size() > 0x7fffff00u) return flush_records(c);
    return PB_OK;
}

int pb_region_launch(pb_ctx *c) {
    if (!c) return PB_ERR_ARG;
    if (c->state != ST_OPEN) return fail(c, PB_ERR_STATE, "pb_region_launch without an open region");
    PB_CUDA(c, cudaSetDevice(c->prm.device));
    PB_TRY(flush_records(c));
    c->state = ST_IDLE;
    PB_TRY(run_pipeline(c));
    c->state = ST_LAUNCHED;
    return PB_OK;
}

int pb_region_relaunch(pb_ctx *c) {
    if (!c) return PB_ERR_ARG;
    if (c->state != ST_LAUNCHED && c->state != ST_DONE) return fail(c, PB_ERR_STATE, "pb_region_relaunch without a launched region");
    PB_CUDA(c, cudaSetDevice(c->prm.device));
    const int prev = c->state;
    c->state = ST_IDLE;
    PB_TRY(run_pipeline(c));
    c->state = prev == ST_DONE ? ST_LAUNCHED : prev;
    return PB_OK;
}

int pb_region_wait(pb_ctx *c, pb_region_result *out) {
    if (!c) return PB_ERR_ARG;
    if (c->state != ST_LAUNCHED) return fail(c, PB_ERR_STATE, "pb_region_wait without pb_region_launch");
    PB_CUDA(c, cudaSetDevice(c->prm.device));
    PB_TRY(fill_result(c, out));
    c->state = ST_DONE;
    return PB_OK;
}

int pb_region_end(pb_ctx *c, pb_region_result *out) {
    PB_TRY(pb_region_launch(c));
    return pb_region_wait(c, out);
}

int pb_region_get_extras(const pb_ctx *c, pb_region_extras *out) {
    if (!c || !out) return PB_ERR_ARG;
    *out = c->ext;
    return PB_OK;
}

int pb_region_get_fst(const pb_ctx *c, pb_region_fst *out) {
    if (!c || !out) return PB_ERR_ARG;
    *out = c->fst;
    return PB_OK;
}

int pb_set_snn_perms(pb_ctx *c, int64_t n_perms, uint64_t seed) {
    if (!c) return PB_ERR_ARG;
    if (n_perms < 0 || n_perms > 0x7fffffffLL) return fail(c, PB_ERR_ARG, "pb_set_snn_perms: n_perms must be in 0 .. 2^31 - 1");
    c->snn_perms = n_perms; c->snn_seed = seed;
    return PB_OK;
}

void *pb_host_alloc(size_t bytes) {
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}
void pb_host_free(void *p) { if (p) cudaFreeHost(p); }

int pb_region_path(const pb_ctx *c) { return c ? (c->ran_fast ? 1 : 0) : PB_ERR_ARG; }
int pb_region_reruns(const pb_ctx *c) { return c ? c->reruns : PB_ERR_ARG; }
void *pb_stream(pb_ctx *c) { return c ? (void *)c->stream : nullptr; }
int64_t pb_kernel_launches(const pb_ctx *c) { return c ? c->launches : 0; }

int pb_stage_times(const pb_ctx *c, double *ms4) {
    if (!c || !ms4) return PB_ERR_ARG;
    ms4[0] = c->ms_prep; ms4[1] = c->ms_pileup; ms4[2] = c->ms_sites; ms4[3] = c->ms_stats;
    return PB_OK;
}

const pb_params *pb_ctx_params(const pb_ctx *c) { return c ? &c->prm : nullptr; }

}  // extern "C"

namespace {
int flush_records(pb_ctx *c) {
    if (c->r_pos.empty()) return PB_OK;
    pb_read_batch b;
    b.n_reads = (int64_t)c->r_pos.size(); b.n_cigar = (int64_t)c->r_cigar.size(); b.n_bases = (int64_t)c->r_qual.size();
    b.pos = c->r_pos.data(); b.meta = c->r_meta.data(); b.cig_off = c->r_cig_off.data(); b.cigar = c->r_cigar.data();
    b.base_off = c->r_base_off.data(); b.seq4 = c->r_seq4.data(); b.qual = c->r_qual.data();
    static const uint32_t zero = 0;
    if (!b.cigar) b.cigar = &zero;
    const int rc = pb_push_batch(c, &b);
    c->r_pos.clear(); c->r_meta.clear(); c->r_cig_off.clear(); c->r_cigar.clear(); c->r_base_off.clear(); c->r_seq4.clear(); c->r_qual.clear();
    return rc;
}
}  // namespace
