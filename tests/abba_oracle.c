/* abba_oracle.c -- TEST INFRASTRUCTURE.  Plain-C restatement of the PB_AN_ABBA statistics of include/popbam_b200.h
 * (Patterson's D, Martin's f_d and Malinsky's f_dM per window and triple), which the reference never computed.  It works
 * on the result of the reference-pinned oracle (oracle/pb_oracle.c, whose pbo_result has the layout of pb_region_result):
 * the window's segregating-site types.
 *
 *   pba_abba  the arrays of every window and triple, into a pb_region_abba (free with pba_free)
 *   pba_row   the text pb_format_window_abba writes for one window, newline included
 *
 * Per site, with a_k the derived copies in P1, P2, P3, O (k = 1..4) after the outgroup polarisation, m_k = n_k - a_k,
 * and the allele frequencies written as fractions x_k / n_k, the frequency products of Martin et al. (2015) and Malinsky
 * et al. (2015) are taken on the common scale K = n1^2 n2^2 n3^2 n4, on which every one is an integer: a product of
 * four frequencies whose denominators n1, n2, n3 appear at most twice and n4 once is its numerators times K over its
 * denominators.  D, f_d and f_dM are (double) numerator / (double) denominator, NaN where that is 0.
 * Built with -ffp-contract=off.                                                                                     */
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include "../include/popbam_b200.h"

static int popc64(uint64_t x) { return __builtin_popcountll(x); }

/* x1 x2 x3 x4 / (d1 d2 d3 n4) * K, where each d_i is n1, n2 or n3 and (d1, d2, d3) together with n4 divide K */
static int64_t scaled(int64_t K, int64_t x1, int64_t d1, int64_t x2, int64_t d2, int64_t x3, int64_t d3, int64_t x4, int64_t n4) {
    const int64_t den = d1 * d2 * d3 * n4;
    if (K % den) abort();
    return x1 * x2 * x3 * x4 * (K / den);
}

typedef struct { int64_t abba, baba, fd_den, fdm_den; } terms;

/* the four site terms of one triple; c[k] = derived copies (not yet polarised), n[k] = samples, k = 0..3 (O = 3) */
static terms site_terms(const int *c, const int *n) {
    int a[4], m[4];
    const int flip = 2 * c[3] > n[3];
    for (int k = 0; k < 4; ++k) {
        a[k] = flip ? n[k] - c[k] : c[k];
        m[k] = n[k] - a[k];
    }
    const int64_t n1 = n[0], n2 = n[1], n3 = n[2], n4 = n[3];
    const int64_t K = n1 * n1 * n2 * n2 * n3 * n3 * n4;
    terms t;
    /* ABBA = (1-p1) p2 p3 (1-p4), BABA = p1 (1-p2) p3 (1-p4) */
    t.abba = scaled(K, m[0], n1, a[1], n2, a[2], n3, m[3], n4);
    t.baba = scaled(K, a[0], n1, m[1], n2, a[2], n3, m[3], n4);
    /* f_d: S(P1, PD, PD, O) = (1-p1) pD pD (1-p4) - p1 (1-pD) pD (1-p4), pD = max(p2, p3) */
    const int d2 = (int64_t)a[1] * n3 >= (int64_t)a[2] * n2;      /* p2 >= p3 */
    const int aD = d2 ? a[1] : a[2], mD = d2 ? m[1] : m[2];
    const int64_t nD = d2 ? n2 : n3;
    t.fd_den = scaled(K, m[0], n1, aD, nD, aD, nD, m[3], n4) - scaled(K, a[0], n1, mD, nD, aD, nD, m[3], n4);
    /* f_dM: the f_d term where p2 >= p1; otherwise -S(PD, P2, PD, O) with pD = max(p1, p3),
     * S(PD, P2, PD, O) = (1-pD) p2 pD (1-p4) - pD (1-p2) pD (1-p4) */
    if ((int64_t)a[1] * n1 >= (int64_t)a[0] * n2) {
        t.fdm_den = t.fd_den;
    } else {
        const int d1 = (int64_t)a[0] * n3 >= (int64_t)a[2] * n1;  /* p1 >= p3 */
        const int bD = d1 ? a[0] : a[2], lD = d1 ? m[0] : m[2];
        const int64_t kD = d1 ? n1 : n3;
        t.fdm_den = -(scaled(K, lD, kD, a[1], n2, bD, kD, m[3], n4) - scaled(K, bD, kD, m[1], n2, bD, kD, m[3], n4));
    }
    return t;
}

static double ratio(int64_t num, int64_t den) { return den != 0 ? (double)num / (double)den : NAN; }

int pba_abba(const pb_params *p, const pb_region_result *r, int32_t og, int32_t nt, const int32_t *triples, pb_region_abba *out) {
    const size_t cnt = (size_t)r->n_windows * nt ? (size_t)r->n_windows * nt : 1;
    int32_t *tr = malloc(sizeof(int32_t) * 3 * (nt ? nt : 1)), *sites = calloc(cnt, 4);
    int64_t *ab = calloc(cnt, 8), *ba = calloc(cnt, 8), *fd = calloc(cnt, 8), *fm = calloc(cnt, 8);
    double *d = calloc(cnt, 8), *f = calloc(cnt, 8), *g = calloc(cnt, 8);
    if (!tr || !sites || !ab || !ba || !fd || !fm || !d || !f || !g) return -4;
    memcpy(tr, triples, sizeof(int32_t) * 3 * nt);
    for (int w = 0; w < r->n_windows; ++w) {
        const uint64_t *T = r->seg_type + r->seg_off[w];
        for (int t = 0; t < nt; ++t) {
            const int pk[4] = {triples[3 * t], triples[3 * t + 1], triples[3 * t + 2], og};
            int n[4];
            for (int k = 0; k < 4; ++k) n[k] = p->pop_nsmpl[pk[k]];
            int64_t s_ab = 0, s_ba = 0, s_fd = 0, s_fm = 0;
            int s_n = 0;
            for (int s = 0; s < r->segsites[w]; ++s) {
                int c[4];
                for (int k = 0; k < 4; ++k) c[k] = popc64(T[s] & p->pop_mask[pk[k]]);
                const terms x = site_terms(c, n);
                s_ab += x.abba; s_ba += x.baba; s_fd += x.fd_den; s_fm += x.fdm_den;
                s_n += x.abba + x.baba > 0;
            }
            const size_t i = (size_t)w * nt + t;
            sites[i] = s_n; ab[i] = s_ab; ba[i] = s_ba; fd[i] = s_fd; fm[i] = s_fm;
            d[i] = ratio(s_ab - s_ba, s_ab + s_ba);
            f[i] = ratio(s_ab - s_ba, s_fd);
            g[i] = ratio(s_ab - s_ba, s_fm);
        }
    }
    out->n_triples = nt; out->outgroup_pop = og; out->triples = tr; out->sites = sites;
    out->abba = ab; out->baba = ba; out->fd_den = fd; out->fdm_den = fm; out->d = d; out->fd = f; out->fdm = g;
    return 0;
}

void pba_free(pb_region_abba *a) {
    free((void *)a->triples); free((void *)a->sites); free((void *)a->abba); free((void *)a->baba); free((void *)a->fd_den);
    free((void *)a->fdm_den); free((void *)a->d); free((void *)a->fd); free((void *)a->fdm);
    memset(a, 0, sizeof *a);
}

typedef struct { char *buf; int64_t cap, len; } sbuf;
static void sb_printf(sbuf *s, const char *fmt, ...) __attribute__((format(printf, 2, 3)));
static void sb_printf(sbuf *s, const char *fmt, ...) {
    char tmp[1024];
    va_list ap; va_start(ap, fmt);
    int k = vsnprintf(tmp, sizeof tmp, fmt, ap);
    va_end(ap);
    if (k < 0) return;
    if (k >= (int)sizeof tmp) k = (int)sizeof tmp - 1;
    for (int i = 0; i < k; ++i) { if (s->len + 1 < s->cap) s->buf[s->len] = tmp[i]; s->len++; }
    if (s->cap > 0) s->buf[s->len < s->cap ? s->len : s->cap - 1] = 0;
}
static void sb_stat(sbuf *s, const char *name, const char *label, int ok, double v) {
    if (ok) sb_printf(s, "\t%s[%s]:\t%.5f", name, label, v);
    else sb_printf(s, "\t%s[%s]:\t%7s", name, label, "NA");
}

/* the abba row of window w: nucdiv's first four columns, then per triple S, ABBA, BABA, D, fd, fdM */
int64_t pba_row(const pb_params *p, const pb_region_result *r, const pb_region_abba *a, int32_t w, const pb_print_opts *o, char *buf,
                int64_t cap) {
    sbuf s = {buf, cap, 0};
    if (cap > 0) buf[0] = 0;
    const int ns = r->num_sites[w], ok = ns >= o->min_sites;
    sb_printf(&s, "%s\t%d\t%d\t%d", o->chrom, r->win_beg[w] + 1, r->win_end[w] + 1, ns);
    for (int t = 0; t < a->n_triples; ++t) {
        const int32_t *k = a->triples + 3 * t;
        char nm[600];
        snprintf(nm, sizeof nm, "%s-%s-%s", o->pop_names[k[0]], o->pop_names[k[1]], o->pop_names[k[2]]);
        const int64_t n1 = p->pop_nsmpl[k[0]], n2 = p->pop_nsmpl[k[1]], n3 = p->pop_nsmpl[k[2]], n4 = p->pop_nsmpl[a->outgroup_pop];
        const double K = (double)(n1 * n1 * n2 * n2 * n3 * n3 * n4);
        const size_t x = (size_t)w * a->n_triples + t;
        sb_printf(&s, "\tS[%s]:\t%d", nm, a->sites[x]);
        sb_stat(&s, "ABBA", nm, ok, (double)a->abba[x] / K);
        sb_stat(&s, "BABA", nm, ok, (double)a->baba[x] / K);
        sb_stat(&s, "D", nm, ok && !isnan(a->d[x]), a->d[x]);
        sb_stat(&s, "fd", nm, ok && !isnan(a->fd[x]), a->fd[x]);
        sb_stat(&s, "fdM", nm, ok && !isnan(a->fdm[x]), a->fdm[x]);
    }
    sb_printf(&s, "\n");
    return s.len;
}
