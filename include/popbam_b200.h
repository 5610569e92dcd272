/*
 * popbam_b200.h -- C ABI of the B200-native POPBAM per-window statistics path.
 *
 * This is the drop-in boundary.  In the reference every subcommand's window loop does
 *
 *     buf = bam_plbuf_init(make_X, &t);                       (bam.h:556, bam_pileup.c:505)
 *     bam_fetch(bam, idx, tid, t.beg, t.end, buf, fetch_func); (bam.h:635, bam_index.c:943)
 *     bam_plbuf_push(0, buf);                                  (bam_pileup.c:523)
 *     t.calc_X(); t.print_X(chr);                              (e.g. pop_nucdiv.cpp:102-119)
 *
 * i.e. records enter through `bam_fetch_f` (bam.h:618) and a window result leaves through
 * calc_X/print_X.  The functions below replace exactly that chain: records go in as pinned
 * structure-of-arrays batches (or one at a time through pb_push_record, which has the
 * bam_fetch_f shape), window results come out as plain arrays.  Plain pointers and sizes
 * only; no C++ or torch types.  All functions return PB_OK (0) or a negative pb_status and
 * never call exit() (the reference's fatal_error, pop_utils.cpp:510, is the caller's job).
 *
 * There is NO CPU fallback behind this interface: if no CUDA device is usable the
 * constructor fails with PB_ERR_CUDA.
 */
#ifndef POPBAM_B200_H
#define POPBAM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PB_MAX_SAMPLES 64          /* popbam.1:508 -- site types are 64-bit sample masks */
#define PB_NO_SAMPLE   0xffu       /* read without a usable RG tag (popbam.cpp:227-228)  */

typedef enum pb_status {
    PB_OK = 0,
    PB_ERR_ARG = -1,        /* bad argument / inconsistent batch                         */
    PB_ERR_CUDA = -2,       /* CUDA runtime failure or no device (message: pb_last_error) */
    PB_ERR_STATE = -3,      /* call order violated (e.g. push outside a region)           */
    PB_ERR_NOMEM = -4,      /* host or device allocation failed                           */
    PB_ERR_UNSORTED = -5,   /* reads not coordinate sorted (bam_pileup.c:384-395)         */
    PB_ERR_UNSUPPORTED = -6 /* max_depth > 255 (pop_utils.cpp:293), BAM 'B' cigar op, ... */
} pb_status;

/* option flags: same bit values as the reference (popbam.h:59-94) */
#define PB_FLAG_ILLUMINA     0x02u   /* -i : qualities are Illumina 1.3+ (popbam.cpp:269) */
#define PB_FLAG_SUBSTITUTE   0x10u   /* -t : diverge counts fixed substitutions only      */
#define PB_FLAG_HETEROZYGOTE 0x20u   /* -z : keep heterozygous calls (skip clean_het)     */
#define PB_FLAG_OUTGROUP     0x40u   /* -p : polarise with sample `outidx`                */
#define PB_FLAG_EMIT_CB      0x10000u /* test hook: keep every per-(site,sample) cb word  */

/* analyses computed from one pileup pass (bit mask; several may be requested together) */
#define PB_AN_NUCDIV        0x001u  /* pop_nucdiv.cpp:206  calc_nucdiv                   */
#define PB_AN_SFS           0x002u  /* pop_sfs.cpp:227     calc_sfs (Tajima D, Fay-Wu H)  */
#define PB_AN_LD_ZNS        0x004u  /* pop_ld.cpp:201      calc_zns       (ld -o 0)       */
#define PB_AN_LD_OMEGA      0x008u  /* pop_ld.cpp:254      calc_omegamax  (ld -o 1)       */
#define PB_AN_LD_WALL       0x010u  /* pop_ld.cpp:375      calc_wall      (ld -o 2)       */
#define PB_AN_DIVERGE_IND   0x020u  /* pop_diverge.cpp:226 diverge -o 0                   */
#define PB_AN_DIVERGE_POP   0x040u  /* pop_diverge.cpp:232 diverge -o 1                   */
#define PB_AN_HAPLO_K       0x080u  /* pop_haplo.cpp:208   calc_nhaps     (haplo -o 0)    */
#define PB_AN_HAPLO_EHHS    0x100u  /* pop_haplo.cpp:256   calc_ehhs      (haplo -o 1)    */
#define PB_AN_HAPLO_DXY     0x200u  /* pop_haplo.cpp:325   calc_minDxy    (haplo -o 2)    */
#define PB_AN_SNP           0x400u  /* pop_snp.cpp:148     per-segregating-site rows      */
#define PB_AN_TREE          0x800u  /* pop_tree.cpp:472    difference matrix incl. the reference taxon (tree) */
/* extensions (no counterpart in the reference; each is the companion of one reference bit, --extra-stats)    */
#define PB_AN_THETA_W       0x1000u /* Watterson's theta from the SFS pass             (with nucdiv)          */
#define PB_AN_FULI          0x2000u /* Fu & Li's D (outgroup only) and D*              (with sfs)             */
#define PB_AN_LD_DPRIME     0x4000u /* Lewontin's |D'| over the ZnS pairs              (with ld -o 0)         */
#define PB_AN_FST           0x8000u /* F_ST (Hudson, Weir & Cockerham) and Snn per population pair (with nucdiv) */

/* Run parameters == the fields of popbamData the hot path reads (popbam.h:218-265) plus
 * the population tables assign_pops builds (popbam.cpp:145-171).                           */
typedef struct pb_params {
    int32_t  n_samples;                    /* sm->n                                       */
    int32_t  n_pops;                       /* sm->npops                                   */
    uint64_t pop_mask[PB_MAX_SAMPLES];     /* bit i set: sample i is in population p      */
    uint8_t  pop_nsmpl[PB_MAX_SAMPLES];    /* samples per population                      */
    int32_t  min_depth;                    /* -m, default 3   (popbam.cpp:88)             */
    int32_t  max_depth;                    /* -x, default 255 (popbam.cpp:89), <= 255     */
    int32_t  min_rmsQ;                     /* -q, default 25                              */
    int32_t  min_snpQ;                     /* -s, default 25                              */
    int32_t  min_mapQ;                     /* -a, default 13 (stored as unsigned char)    */
    int32_t  min_baseQ;                    /* -b, default 13 (stored as unsigned char)    */
    uint32_t flags;                        /* PB_FLAG_*                                   */
    int32_t  outidx;                       /* sample index of the outgroup (-p)           */
    int32_t  min_freq;                     /* ld: 1, or 2 with -e (pop_ld.cpp:494)        */
    int32_t  device;                       /* CUDA device ordinal                         */
} pb_params;

/* Error-model tables exactly as errmod_init(1.0-0.83) builds them (pop_utils.cpp:203-266).
 * Pass NULL to pb_create and the library builds them on the host with the same long-double
 * libm calls; pass a table set (e.g. dumped from the reference) to share it bit for bit.   */
typedef struct pb_errmod_tables {
    const double *fk;      /* [256]                                                       */
    const double *beta;    /* [64*256*256]  index q<<16 | n<<8 | k                        */
    const double *lhet;    /* [256*256]     index n<<8 | k                                */
} pb_errmod_tables;

/* One batch of alignment records in FILE ORDER (the order bam_fetch would deliver them),
 * structure-of-arrays, ideally in pinned host memory.  Field provenance:
 *   pos      bam1_core_t.pos                                   (bam.h:178-190)
 *   meta     flag<<16 | mapq<<8 | sample  (core.flag, core.qual; sample = result of
 *            bam_smpl_rg2smid on the RG tag, pop_sample.cpp:228, or PB_NO_SAMPLE)
 *   cig_off  [n_reads+1] first index of the read's ops in cigar[]
 *   cigar    BAM encoding len<<4|op                            (bam.h:225 bam1_cigar)
 *   base_off [n_reads+1] EVEN offset of the read's first base in qual[]; its packed
 *            sequence starts at seq4[base_off/2]               (bam.h:245-258)
 *   seq4     4-bit bases, high nibble first (bam1_seqi)
 *   qual     raw Phred base qualities (bam1_qual)
 * Records whose flag has any of 0x704 set or with tid<0 may be included; they are dropped
 * as bam_plp_push does (bam_pileup.c:371-374).                                             */
typedef struct pb_read_batch {
    int64_t         n_reads;
    int64_t         n_cigar;     /* == cig_off[n_reads]                                   */
    int64_t         n_bases;     /* == base_off[n_reads] (bytes of qual[], padded even)   */
    const int32_t  *pos;
    const uint32_t *meta;
    const uint32_t *cig_off;
    const uint32_t *cigar;
    const uint32_t *base_off;
    const uint8_t  *seq4;
    const uint8_t  *qual;
} pb_read_batch;

/* Results of one region (a run of windows on one contig).  All arrays are owned by the
 * context, live in pinned host memory and stay valid until the next pb_region_begin or
 * pb_destroy.  P = n_pops, n = n_samples, NW = n_windows.  Arrays whose analysis bit was
 * not requested are NULL.  Index conventions follow the reference arrays they replace.     */
typedef struct pb_region_result {
    int32_t  n_windows;
    int32_t  n_pops, n_samples;
    uint32_t analyses;
    const int32_t  *win_beg;      /* [NW] t.beg (0-based)  -- printed +1                   */
    const int32_t  *win_end;      /* [NW] t.end            -- printed +1                   */
    const int32_t  *num_sites;    /* [NW] popbamData::num_sites                            */
    const int32_t  *segsites;     /* [NW] popbamData::segsites                             */
    /* segregating sites of all windows, concatenated; window w owns
     * [seg_off[w], seg_off[w]+segsites[w])                                                */
    const int64_t  *seg_off;      /* [NW+1]                                                */
    const uint32_t *seg_pos;      /* hap.pos  (0-based reference coordinate)               */
    const uint32_t *seg_idx;      /* hap.idx  (rank among the window's aligned sites)      */
    const uint64_t *seg_type;     /* types[hap.idx[s]] : bit i = sample i carries derived  */
    const uint8_t  *seg_ref;      /* raw reference byte at the site                        */
    const uint64_t *seg_cb;       /* [S_total*n] final cb words (PB_AN_SNP): base/snpq/rms/depth */
    /* nucdiv / haplo -o 2 */
    const double   *piw;          /* [NW*P]     not yet divided by num_sites               */
    const double   *pib;          /* [NW*P*P]   index i*P+(j-(i+1)) (pop_nucdiv.cpp:227)   */
    const uint16_t *min_dxy;      /* [NW*P*P]   same indexing (pop_haplo.cpp:336)          */
    /* sfs */
    const int32_t  *sfs_num_snps; /* [NW*P]                                                */
    const double   *td;           /* [NW*P]  NaN == "NA"                                   */
    const double   *fwh;          /* [NW*P]                                                */
    /* ld */
    const int32_t  *ld_num_snps;  /* [NW*P]  (zns/omega counting rule, pop_ld.cpp:219-249) */
    const double   *zns;          /* [NW*P]                                                */
    const double   *omegamax;     /* [NW*P]                                                */
    const int32_t  *wall_num_snps;/* [NW*P]                                                */
    const double   *wallb;        /* [NW*P]                                                */
    const double   *wallq;        /* [NW*P]                                                */
    /* diverge */
    const uint16_t *ind_div;      /* [NW*n]  (unsigned short, wraps; pop_diverge.h)        */
    const uint16_t *pop_div;      /* [NW*P]                                                */
    const int32_t  *div_num_snps; /* [NW*P]                                                */
    /* haplo */
    const int32_t  *nhaps;        /* [NW*P]                                                */
    const double   *hdiv;         /* [NW*P]                                                */
    const double   *ehhs;         /* [NW*P]  NaN == "NA"                                   */
    /* test hook (PB_FLAG_EMIT_CB): cb word of every (position, sample) of the span
     * [span_beg, span_end), position-major, AFTER clean_heterozygotes/segbase/qfilter;
     * plus the per-position record the site kernel produced                               */
    int32_t  span_beg, span_end;
    const uint64_t *cb;           /* [(span_end-span_beg)*n]                               */
    const uint64_t *site_type;    /* [span_end-span_beg]                                   */
    const uint8_t  *site_flag;    /* bit0 used (in a window, all samples covered), bit1 fq>0 */
    /* work counters */
    int64_t  reads_pushed;        /* records received                                      */
    int64_t  reads_used;          /* after the 0x704 / tid / empty-cigar filter            */
    int64_t  aligned_bases;       /* sum of M/=/X lengths of used reads                    */
    /* tree */
    const uint16_t *tree_diff;    /* [NW*(n+1)*(n+1)] treeData::diff_matrix (pop_tree.cpp:472-494), taxon 0 = reference */
} pb_region_result;

/* Extension statistics of the last region (PB_AN_THETA_W, PB_AN_FULI, PB_AN_LD_DPRIME): a struct of its own, so that
 * pb_region_result keeps its size for callers built against the reference-only interface.  Same lifetime as the
 * pb_region_result arrays; an array is NULL unless its bit was requested.  m = pop_nsmpl[p]; xi_j = the window's site
 * frequency spectrum of population p as calc_sfs bins it (outgroup flip with PB_FLAG_OUTGROUP); S = sum xi_j over
 * 0<j<m; a = sum_{i<m} 1/i.  All arrays [NW*P].  (With PB_AN_LD_DPRIME pb_region_result.ld_num_snps is set too.)     */
typedef struct pb_region_extras {
    const int32_t *pop_segsites;  /* S                                                   (THETA_W or FULI)  */
    const double  *theta_w;       /* S / a, not yet divided by num_sites; NaN if m < 2   (THETA_W)          */
    const double  *fuli_d;        /* Fu & Li's D with eta_e; NaN without an outgroup, if m < 3 or S = 0 (FULI) */
    const double  *fuli_ds;       /* Fu & Li's D* with eta_s; NaN if m < 4 (at m = 3 it is 0/0) or S = 0 (FULI) */
    const int32_t *fuli_eta_e;    /* xi_1 (0 if m < 2)                                   (FULI)             */
    const int32_t *fuli_eta_s;    /* xi_1 + xi_{m-1}, counted once when m = 2            (FULI)             */
    const int32_t *ld_kept;       /* K: SNPs with min_freq <= count <= m - min_freq, the ZnS pairs (LD_DPRIME) */
    const double  *ld_dprime;     /* mean |D'| over the K(K-1)/2 pairs; NaN if K < 2     (LD_DPRIME)        */
    const int64_t *ld_complete;   /* pairs with |D'| = 1 (complete LD)                   (LD_DPRIME)        */
} pb_region_extras;

/* Differentiation between the populations of every pair i < j of the last region (PB_AN_FST): a struct of its own,
 * like pb_region_extras.  Same lifetime as the pb_region_result arrays; NULL unless PB_AN_FST was requested (snn_p and
 * snn_ge: unless pb_set_snn_perms asked for permutations too).  All arrays [NW*P*P], index i*P+(j-(i+1)) like pib.
 * n1, n2 = pop_nsmpl[i], pop_nsmpl[j]; for every segregating site of the window, c1 and c2 = the samples of i and j that
 * carry the derived allele.  Calls count as haploid, one per sample, as for pi and dxy (with PB_FLAG_HETEROZYGOTE a
 * heterozygous call counts as derived).  No outgroup flip: every statistic is the same with the allele labels of a site
 * swapped.  The sums are exact integers:
 *   hud_den = sum (n1-1)(n2-1) [c1 (n2-c2) + c2 (n1-c1)]           (= dxy sum * (n1-1)(n2-1))
 *   hud_num = hud_den - sum [c1 (n1-c1) n2 (n2-1) + c2 (n2-c2) n1 (n1-1)]
 *   wc_num  = sum (c1 n2 - c2 n1)^2 (n1+n2-2) - G (n1+n2),           G = c1 (n1-c1) n2 + c2 (n2-c2) n1
 *   wc_den  = sum (c1 n2 - c2 n1)^2 (n1+n2-2) + G (2 n1 n2 - n1 - n2)
 * i.e. Hudson's F_ST as a ratio of averages (Hudson, Slatkin & Maddison 1992; Bhatia et al. 2013) scaled by
 * n1 n2 (n1-1)(n2-1), and Weir & Cockerham's theta for haploid data (Weir 1996, r = 2) scaled by n1 n2 (n1+n2)(n1+n2-2).
 * Snn is Hudson's (2000) nearest-neighbour statistic on the window's pairwise difference matrix (the one nucdiv uses).
 * Every double is NaN if n1 < 2 or n2 < 2; fst_hudson / fst_wc also if their denominator is 0.                        */
typedef struct pb_region_fst {
    const int64_t *hud_num, *hud_den;   /* Hudson's numerator and denominator sums                              */
    const int64_t *wc_num, *wc_den;     /* Weir & Cockerham's                                                  */
    const double  *fst_hudson;          /* hud_num / hud_den                                                   */
    const double  *fst_wc;              /* wc_num / wc_den (1 for a window of fixed differences only)          */
    const double  *snn;                 /* Snn = (1/(n1+n2)) sum_x |NN(x) in pop(x)| / |NN(x)|                  */
    const double  *snn_p;               /* (1 + snn_ge) / (1 + n_perms)                          (permutations) */
    const int64_t *snn_ge;              /* permutations of the pooled labels with Snn >= Snn_obs - 1e-12       */
} pb_region_fst;

typedef struct pb_ctx pb_ctx;

/* ---- life cycle ---------------------------------------------------------------------- */
/* replaces: popbamData ctor + errmod_init + assign_pops (popbam.cpp:79, pop_utils.cpp:257,
 * popbam.cpp:145).  *status receives the error code when NULL is returned.                */
pb_ctx     *pb_create(const pb_params *params, const pb_errmod_tables *tables, int *status);
void        pb_destroy(pb_ctx *ctx);
const char *pb_last_error(const pb_ctx *ctx);   /* ctx may be NULL: last create failure   */
const char *pb_version(void);

/* replaces: faidx_fetch_seq into t.ref_base (pop_nucdiv.cpp:45).  Bytes are kept verbatim
 * (case-sensitive, pop_utils.cpp:139).                                                    */
int pb_set_contig(pb_ctx *ctx, int32_t tid, const char *ref_bases, int64_t len);

/* ---- region = run of windows on the current contig ------------------------------------ */
/* replaces: the per-window init_X/bam_plbuf_init of every main_X window loop.  Windows must
 * be sorted and non-overlapping: win_beg[w] <= pos < win_end[w] (make_X test,
 * pop_nucdiv.cpp:148).  Use pb_window_grid to obtain the reference's grid.                */
int pb_region_begin(pb_ctx *ctx, uint32_t analyses, int32_t n_windows,
                    const int32_t *win_beg, const int32_t *win_end);

/* replaces: bam_fetch(...fetch_func) -> bam_plbuf_push(b, buf) (pop_utils.cpp:500-508).
 * May be called several times per region; batches are concatenated in call order.  The
 * arrays are copied to the device before the call returns (use pinned memory for speed).  */
int pb_push_batch(pb_ctx *ctx, const pb_read_batch *batch);
/* The same without waiting for the copies: the batch arrays (pinned host memory) must stay untouched until
 * pb_region_wait / pb_region_end of this region has returned.  Several pushes and the kernels of the region then
 * queue up behind each other on the context's stream with no host round trip in between.                          */
int pb_push_batch_async(pb_ctx *ctx, const pb_read_batch *batch);
/* Optional: make room on the device for a region's reads before they are pushed (several pb_push_batch calls then do
 * not grow the arrays step by step).  Totals over the pushes to come; more may still be pushed.                      */
int pb_region_reserve(pb_ctx *ctx, int64_t n_reads, int64_t n_cigar, int64_t n_bases);

/* bam_fetch_f-shaped shim (bam.h:618): `b` points at a raw BAM record laid out as bam1_t's
 * core (32 bytes, bam.h:178-190, little endian) followed by its variable-length data
 * (qname, cigar, seq, qual, aux); `sample` is the caller's rg2smid result.                 */
int pb_push_record(pb_ctx *ctx, const void *core32, const void *data, int32_t l_data,
                   int32_t sample);

/* replaces: bam_plbuf_push(0, buf) + calc_X (pop_nucdiv.cpp:112-116).  Runs the kernels,
 * copies the window results back and fills *out.                                          */
int pb_region_end(pb_ctx *ctx, pb_region_result *out);
/* The extension arrays of the region pb_region_end / pb_region_wait returned last.                                  */
int pb_region_get_extras(const pb_ctx *ctx, pb_region_extras *out);
/* The PB_AN_FST arrays of the region pb_region_end / pb_region_wait returned last.                                  */
int pb_region_get_fst(const pb_ctx *ctx, pb_region_fst *out);
/* Permutation test of Snn for the regions that follow (PB_AN_FST): n_perms random re-partitions of each pair's pooled
 * samples (default 0: none), drawn from a counter-based stream keyed on (seed, contig tid, window begin, i, j,
 * permutation), so the result does not depend on how a contig is cut into regions or spread over GPUs.  The generator is
 * written down in popbam_b200/csrc/pb_stats.cuh (k_snn_perm).  PB_ERR_ARG if n_perms < 0 or > 2^31 - 1.                */
int pb_set_snn_perms(pb_ctx *ctx, int64_t n_perms, uint64_t seed);

/* Asynchronous split of pb_region_end for overlap / device timing: launch enqueues every
 * kernel and the result copies on the context's stream; wait blocks and fills *out.       */
int pb_region_launch(pb_ctx *ctx);
int pb_region_wait(pb_ctx *ctx, pb_region_result *out);
/* Re-run the kernels on the reads already resident on the device (bench: kernel-only
 * timing with inputs in HBM).  Valid after pb_region_launch and before the next begin.    */
int pb_region_relaunch(pb_ctx *ctx);
/* Which formulation of the pileup stage the last region took: 1 = the counting pileup (k_pile_reads, the default), 0 = the
 * single-kernel pileup (per-cell words requested, min_depth / min_snpQ of 0, or the raw-depth cap can bind).
 * pb_region_reruns: how many regions of this context were run a second time because an assumption the counting
 * kernels verify on the device (largest base quality, size of the hard-cell arena) did not hold.                */
int pb_region_path(const pb_ctx *ctx);
int pb_region_reruns(const pb_ctx *ctx);
void *pb_stream(pb_ctx *ctx);                   /* cudaStream_t the kernels run on        */
int64_t pb_kernel_launches(const pb_ctx *ctx);  /* kernels launched since pb_create       */
/* CUDA-event durations (ms) of the last region's stages, valid after pb_region_wait:
 * [0] preparation: per-read pass, quality levels, sample partition, and the per-base pass
 *     (bit-planes, or base codes for the single-kernel pileup),
 * [1] the pileup / call / site stage, [2] window compaction, [3] window statistics.        */
int pb_stage_times(const pb_ctx *ctx, double *ms4);

/* ---- helpers that mirror small reference routines ------------------------------------- */
/* window grid of every main_X (pop_nucdiv.cpp:48-78, SURVEY Q14).  win_size==0: one window
 * [beg,end).  Returns the number of windows; fills up to `cap` entries.                   */
int64_t pb_window_grid(int32_t beg, int32_t end, int32_t win_size, int64_t cap,
                       int32_t *win_beg, int32_t *win_end);

/* Host-side table construction == errmod_init(1.0-0.83) (pop_utils.cpp:203-266).  Buffers
 * must hold 256, 64*256*256 and 256*256 doubles.                                          */
int pb_build_errmod_tables(double *fk, double *beta, double *lhet);
/* The same through a cache on disk (SURVEY.md 8(f) rank 3): the tables only depend on the host's libm, so they are
 * computed once per machine.  `cache_dir` NULL: $POPBAM_B200_CACHE_DIR, else $XDG_CACHE_HOME/popbam_b200, else
 * $HOME/.cache/popbam_b200, else /tmp.  The file name carries a fingerprint of the libm calls cal_coef makes; its
 * contents are checksummed; anything that does not verify is rebuilt (and rewritten atomically).  Set
 * POPBAM_B200_NO_TABLE_CACHE=1 to always compute.  Returns PB_OK; *from_cache (may be NULL) says which way.        */
int pb_errmod_tables_cached(double *fk, double *beta, double *lhet, const char *cache_dir);
int pb_errmod_tables_cached_ex(double *fk, double *beta, double *lhet, const char *cache_dir, int *from_cache);

/* Page-locked host memory for pb_read_batch arrays (what pb_push_batch_async wants); NULL when out of memory.     */
void *pb_host_alloc(size_t bytes);
void  pb_host_free(void *p);

/* Text of one window exactly as print_X writes it (pop_nucdiv.cpp:258, pop_sfs.cpp:293,
 * pop_ld.cpp:650, pop_diverge.cpp:496, pop_haplo.cpp:365, pop_snp.cpp:224-303), without
 * touching stdout.  `analysis` is ONE PB_AN_* bit.  opts: min_sites (-k), min_snps (-n),
 * jc (diverge -d jc), snp_output (snp -o 0/1/2).  Returns bytes written (excluding NUL) or
 * the required size if it exceeds cap.                                                    */
typedef struct pb_print_opts {
    const char  *chrom;
    const char *const *pop_names;     /* [P]  sm->popul */
    const char *const *sample_names;  /* [n]  sm->smpl  */
    int32_t min_sites;                /* default 10 */
    int32_t min_snps;                 /* default 10 */
    int32_t jc;
    int32_t snp_output;
    const char *ref_name;             /* tree: treeData::refid, the AS tag of the sequence dictionary (pop_utils.cpp:463) */
} pb_print_opts;
int64_t pb_format_window(const pb_ctx *ctx, const pb_region_result *res, int32_t window,
                         uint32_t analysis, const pb_print_opts *opts, char *buf, int64_t cap);
/* The same, where `analysis` may also be a reference bit OR-ed with its extension (NUCDIV|THETA_W, SFS|FULI,
 * LD_ZNS|LD_DPRIME): the extension's columns (theta[pop]; FuLiD*[pop] and, with PB_FLAG_OUTGROUP, FuLiD[pop];
 * Dp[pop] and Dp1[pop]) then follow the reference's, before the newline.  `ext` may be NULL for reference bits.     */
int64_t pb_format_window_ext(const pb_ctx *ctx, const pb_region_result *res, const pb_region_extras *ext, int32_t window,
                             uint32_t analysis, const pb_print_opts *opts, char *buf, int64_t cap);
/* nucdiv with F_ST: `analysis` is PB_AN_NUCDIV, optionally OR-ed with PB_AN_THETA_W and / or PB_AN_FST.  After the
 * reference's columns and theta[pop] come, per population pair in dxy order, Fst[A-B] (Hudson), FstWC[A-B] and Snn[A-B],
 * plus SnnP[A-B] when permutations ran; NA where the window has fewer than min_sites sites or the value is NaN.
 * `ext` may be NULL without PB_AN_THETA_W, `fst` without PB_AN_FST.                                                   */
int64_t pb_format_window_fst(const pb_ctx *ctx, const pb_region_result *res, const pb_region_extras *ext, const pb_region_fst *fst,
                             int32_t window, uint32_t analysis, const pb_print_opts *opts, char *buf, int64_t cap);

#ifdef __cplusplus
}
#endif
#endif /* POPBAM_B200_H */
