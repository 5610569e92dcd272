/* ext_oracle.c -- TEST INFRASTRUCTURE.  Plain-C restatement of the extension statistics (PB_AN_THETA_W, PB_AN_FULI,
 * PB_AN_LD_DPRIME of include/popbam_b200.h), which the reference never computed.  It works on the result of the
 * reference-pinned oracle (oracle/pb_oracle.c, whose pbo_result has the layout of pb_region_result): the window's
 * segregating-site types and, for the Dp columns, the ZnS site count ld_num_snps.
 *
 *   pbx_extras   the extension arrays of every (window, population), into a pb_region_extras (all nine allocated)
 *   pbx_columns  the text pb_format_window_ext appends to the reference's row for one extension bit
 *
 * Watterson's theta and Fu & Li's D / D* (Fu & Li 1993 with the corrected constants of Simonsen, Churchill & Aquadro
 * 1995) use every expression in the order of pb_stats.cuh and tests/test_extra_stats_host.py; D' is a direct O(K^2) pair
 * loop (no reciprocal table).  Built with -ffp-contract=off so that products and sums round separately.              */
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include "../include/popbam_b200.h"

static int popc64(uint64_t x) { return __builtin_popcountll(x); }

/* one population's spectrum as calc_sfs bins it (outgroup flip), and the closed forms */
static void sfs_ext(const pb_params *p, int pop, const uint64_t *T, int S, int32_t *segs, double *thw, double *fd, double *fds,
                    int32_t *ee, int32_t *es) {
    const int n = p->pop_nsmpl[pop];
    int *sfs = (int *)calloc((size_t)n + 1, sizeof(int));
    int seg = 0;
    for (int s = 0; s < S; ++s) {
        int f = popc64(T[s] & p->pop_mask[pop]);
        if ((p->flags & PB_FLAG_OUTGROUP) && (T[s] >> p->outidx & 1)) f = n - f;
        ++sfs[f];
        if (f > 0 && f < n) ++seg;
    }
    *segs = seg;
    *ee = n >= 2 ? sfs[1] : 0;
    *es = n >= 3 ? sfs[1] + sfs[n - 1] : *ee;
    *thw = NAN; *fd = NAN; *fds = NAN;
    if (n >= 2) {
        double a1 = 0.0, a2 = 0.0;
        for (int j = 1; j < n; ++j) a1 += 1.0 / (double)j;
        for (int j = 1; j < n; ++j) a2 += 1.0 / ((double)j * (double)j);
        *thw = (double)seg / a1;
        if (n >= 3 && seg > 0) {
            const double nn = (double)n, Sd = (double)seg, ap = a1 + 1.0 / nn, r = nn / (nn - 1.0);
            const double c = 2.0 * (nn * a1 - 2.0 * (nn - 1.0)) / ((nn - 1.0) * (nn - 2.0));
            const double vd = 1.0 + a1 * a1 / (a2 + a1 * a1) * (c - (nn + 1.0) / (nn - 1.0)), ud = a1 - 1.0 - vd;
            const double d = c + (nn - 2.0) / ((nn - 1.0) * (nn - 1.0)) + 2.0 / (nn - 1.0) * (1.5 - (2.0 * ap - 3.0) / (nn - 2.0) - 1.0 / nn);
            const double vds = (r * r * a2 + a1 * a1 * d - 2.0 * nn * a1 * (a1 + 1.0) / ((nn - 1.0) * (nn - 1.0))) / (a1 * a1 + a2);
            const double uds = r * (a1 - r) - vds;
            if (p->flags & PB_FLAG_OUTGROUP) *fd = (Sd - a1 * (double)*ee) / sqrt(ud * Sd + vd * Sd * Sd);
            if (n >= 4) *fds = (r * Sd - a1 * (double)*es) / sqrt(uds * Sd + vds * Sd * Sd);      /* n = 3: eta_s = S, 0 / 0 */
        }
    }
    free(sfs);
}

/* Lewontin's D' over the SNPs calc_zns pairs (min_freq <= m <= n - min_freq): num = n*n11 - m1*m2, |D'| = |num| / Dmax,
 * Dmax = min(m1 (n-m2), (n-m1) m2) if num > 0 else min(m1 m2, (n-m1)(n-m2)) */
static void dprime(const pb_params *p, int pop, const uint64_t *T, int S, int32_t *kept, double *dp, int64_t *complete) {
    const int np = p->pop_nsmpl[pop], mf = p->min_freq;
    uint64_t *kt = (uint64_t *)malloc(sizeof(uint64_t) * (size_t)(S > 0 ? S : 1));
    int *km = (int *)malloc(sizeof(int) * (size_t)(S > 0 ? S : 1));
    int K = 0;
    for (int s = 0; s < S; ++s) {
        uint64_t t = T[s] & p->pop_mask[pop]; int m = popc64(t);
        if (m >= mf && m <= np - mf) { kt[K] = t; km[K] = m; ++K; }
    }
    double sum = 0.0; int64_t full = 0;
    for (int j = 0; j < K; ++j) {
        double row = 0.0;      /* per row, then over rows: ~1e-15 relative over the ~10^6 pairs of a dense window */
        for (int k = j + 1; k < K; ++k) {
            const int m1 = km[j], m2 = km[k];
            const int num = np * popc64(kt[j] & kt[k]) - m1 * m2;
            const int dmax = num > 0 ? (m1 * (np - m2) < (np - m1) * m2 ? m1 * (np - m2) : (np - m1) * m2)
                                     : (m1 * m2 < (np - m1) * (np - m2) ? m1 * m2 : (np - m1) * (np - m2));
            const int an = num < 0 ? -num : num;
            row += (double)an / (double)dmax;
            full += an == dmax;
        }
        sum += row;
    }
    *kept = K;
    *dp = K < 2 ? NAN : sum / ((double)K * (double)(K - 1) / 2.0);
    *complete = full;
    free(kt); free(km);
}

int pbx_extras(const pb_params *p, const pb_region_result *r, pb_region_extras *out) {
    const size_t wp = (size_t)r->n_windows * (size_t)r->n_pops, c = wp ? wp : 1;
    int32_t *segs = (int32_t *)calloc(c, 4), *ee = (int32_t *)calloc(c, 4), *es = (int32_t *)calloc(c, 4), *kept = (int32_t *)calloc(c, 4);
    double *thw = (double *)calloc(c, 8), *fd = (double *)calloc(c, 8), *fds = (double *)calloc(c, 8), *dp = (double *)calloc(c, 8);
    int64_t *full = (int64_t *)calloc(c, 8);
    if (!segs || !ee || !es || !kept || !thw || !fd || !fds || !dp || !full) return -4;
    for (int w = 0; w < r->n_windows; ++w) {
        const uint64_t *T = r->seg_type + r->seg_off[w];
        const int S = r->segsites[w];
        for (int i = 0; i < r->n_pops; ++i) {
            const size_t x = (size_t)w * r->n_pops + i;
            sfs_ext(p, i, T, S, segs + x, thw + x, fd + x, fds + x, ee + x, es + x);
            dprime(p, i, T, S, kept + x, dp + x, full + x);
        }
    }
    out->pop_segsites = segs; out->theta_w = thw; out->fuli_d = fd; out->fuli_ds = fds; out->fuli_eta_e = ee; out->fuli_eta_s = es;
    out->ld_kept = kept; out->ld_dprime = dp; out->ld_complete = full;
    return 0;
}

void pbx_free(pb_region_extras *e) {
    free((void *)e->pop_segsites); free((void *)e->theta_w); free((void *)e->fuli_d); free((void *)e->fuli_ds);
    free((void *)e->fuli_eta_e); free((void *)e->fuli_eta_s); free((void *)e->ld_kept); free((void *)e->ld_dprime);
    free((void *)e->ld_complete);
    memset(e, 0, sizeof *e);
}

typedef struct { char *buf; int64_t cap, len; } sbuf;
static void sb_printf(sbuf *s, const char *fmt, ...) __attribute__((format(printf, 2, 3)));
static void sb_printf(sbuf *s, const char *fmt, ...) {
    char tmp[512];
    va_list ap; va_start(ap, fmt);
    int k = vsnprintf(tmp, sizeof tmp, fmt, ap);
    va_end(ap);
    if (k < 0) return;
    if (k >= (int)sizeof tmp) k = (int)sizeof tmp - 1;
    for (int i = 0; i < k; ++i) { if (s->len + 1 < s->cap) s->buf[s->len] = tmp[i]; s->len++; }
    if (s->cap > 0) s->buf[s->len < s->cap ? s->len : s->cap - 1] = 0;
}
static void sb_stat(sbuf *s, const char *name, const char *pop, int ok, double v) {
    if (ok) sb_printf(s, "\t%s[%s]:\t%.5f", name, pop, v);
    else sb_printf(s, "\t%s[%s]:\t%7s", name, pop, "NA");
}

/* the columns one extension bit appends to window w's row (no newline); NA rules of the neighbouring columns:
 * theta like pi (min_sites), Fu & Li like Tajima's D (NaN), Dp like Zns (min_snps on ld_num_snps) and K >= 2 */
int64_t pbx_columns(const pb_params *p, const pb_region_result *r, const pb_region_extras *e, int32_t w, uint32_t ext,
                    const pb_print_opts *o, char *buf, int64_t cap) {
    sbuf s = {buf, cap, 0};
    const int P = r->n_pops, ns = r->num_sites[w];
    if (cap > 0) buf[0] = 0;
    for (int i = 0; i < P; ++i) {
        const size_t x = (size_t)w * P + i;
        if (ext == PB_AN_THETA_W) sb_stat(&s, "theta", o->pop_names[i], ns >= o->min_sites && !isnan(e->theta_w[x]), e->theta_w[x] / ns);
        else if (ext == PB_AN_FULI) {
            sb_stat(&s, "FuLiD*", o->pop_names[i], !isnan(e->fuli_ds[x]), e->fuli_ds[x]);
            if (p->flags & PB_FLAG_OUTGROUP) sb_stat(&s, "FuLiD", o->pop_names[i], !isnan(e->fuli_d[x]), e->fuli_d[x]);
        } else if (ext == PB_AN_LD_DPRIME) {
            const int good = r->ld_num_snps[x] >= o->min_snps && e->ld_kept[x] >= 2;
            sb_stat(&s, "Dp", o->pop_names[i], good, e->ld_dprime[x]);
            if (good) sb_printf(&s, "\tDp1[%s]:\t%lld", o->pop_names[i], (long long)e->ld_complete[x]);
            else sb_printf(&s, "\tDp1[%s]:\t%7s", o->pop_names[i], "NA");
        } else return -1;
    }
    return s.len;
}
