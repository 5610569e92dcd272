/* garud_oracle.c -- TEST INFRASTRUCTURE.  Plain-C restatement of the PB_AN_GARUD statistics of include/popbam_b200.h
 * (Garud's H1, H12, H123 and H2/H1 per window and population), which the reference never computed.  It works on the
 * result of the reference-pinned oracle (oracle/pb_oracle.c, whose pbo_result has the layout of pb_region_result): the
 * window's segregating-site types.
 *
 *   pbg_garud    the arrays of every window and population, into a pb_region_garud (free with pbg_free)
 *   pbg_columns  the text pb_format_window_garud appends to a haplo row, without the newline
 *
 * Unlike the kernel (bit-parallel identity masks) it compares the members of a population pairwise, site by site: a
 * member starts a new class unless an earlier member has the same allele at every site, and the class sizes are sorted
 * with qsort.  The doubles are (double) integer / (double) integer, as the header states.                          */
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include "../include/popbam_b200.h"

static int same_haplotype(const uint64_t *T, int S, int i, int j) {
    for (int s = 0; s < S; ++s)
        if (((T[s] >> i) ^ (T[s] >> j)) & 1) return 0;
    return 1;
}

static int by_size_desc(const void *a, const void *b) {
    const int x = *(const int *)a, y = *(const int *)b;
    return (y > x) - (y < x);
}

int pbg_garud(const pb_params *p, const pb_region_result *r, pb_region_garud *out) {
    const int P = r->n_pops, n = r->n_samples;
    const size_t cnt = r->n_windows > 0 && P > 0 ? (size_t)r->n_windows * P : 1;
    int32_t *nh = calloc(cnt, 4), *c1 = calloc(cnt, 4), *c2 = calloc(cnt, 4), *c3 = calloc(cnt, 4), *hh = calloc(cnt, 4);
    double *h1 = calloc(cnt, 8), *h12 = calloc(cnt, 8), *h123 = calloc(cnt, 8), *h2h1 = calloc(cnt, 8);
    if (!nh || !c1 || !c2 || !c3 || !hh || !h1 || !h12 || !h123 || !h2h1) return -4;
    for (int w = 0; w < r->n_windows; ++w) {
        const uint64_t *T = r->seg_type + r->seg_off[w];
        const int S = r->segsites[w];
        for (int k = 0; k < P; ++k) {
            int member[PB_MAX_SAMPLES], size[PB_MAX_SAMPLES], cls[PB_MAX_SAMPLES], m = 0, nc = 0;
            for (int i = 0; i < n; ++i) if (p->pop_mask[k] >> i & 1) member[m++] = i;
            for (int a = 0; a < m; ++a) {
                cls[a] = -1;
                for (int b = 0; b < a && cls[a] < 0; ++b)
                    if (same_haplotype(T, S, member[a], member[b])) cls[a] = cls[b];
                if (cls[a] < 0) { cls[a] = nc; size[nc++] = 0; }
                size[cls[a]] += 1;
            }
            qsort(size, (size_t)nc, sizeof(int), by_size_desc);
            int sq = 0;
            for (int c = 0; c < nc; ++c) sq += size[c] * size[c];
            const int a1 = nc > 0 ? size[0] : 0, a2 = nc > 1 ? size[1] : 0, a3 = nc > 2 ? size[2] : 0;
            const size_t x = (size_t)w * P + k;
            nh[x] = nc; c1[x] = a1; c2[x] = a2; c3[x] = a3; hh[x] = sq;
            const int nk = p->pop_nsmpl[k];
            if (nk < 2) {
                h1[x] = h12[x] = h123[x] = h2h1[x] = NAN;
            } else {
                const double nn = (double)(nk * nk);
                h1[x] = (double)sq / nn;
                h12[x] = (double)(sq + 2 * a1 * a2) / nn;
                h123[x] = (double)(sq + 2 * (a1 * a2 + a1 * a3 + a2 * a3)) / nn;
                h2h1[x] = (double)(sq - a1 * a1) / (double)sq;
            }
        }
    }
    out->n_hap = nh; out->c1 = c1; out->c2 = c2; out->c3 = c3; out->hh = hh;
    out->h1 = h1; out->h12 = h12; out->h123 = h123; out->h2h1 = h2h1;
    return 0;
}

void pbg_free(pb_region_garud *g) {
    free((void *)g->n_hap); free((void *)g->c1); free((void *)g->c2); free((void *)g->c3); free((void *)g->hh);
    free((void *)g->h1); free((void *)g->h12); free((void *)g->h123); free((void *)g->h2h1);
    memset(g, 0, sizeof *g);
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

/* per population: nHap, H1, H12, H123, H2H1; NA below min_sites sites or where the value is NaN */
int64_t pbg_columns(const pb_region_result *r, const pb_region_garud *g, int32_t w, const pb_print_opts *o, char *buf, int64_t cap) {
    sbuf s = {buf, cap, 0};
    if (cap > 0) buf[0] = 0;
    const int ok = r->num_sites[w] >= o->min_sites;
    for (int k = 0; k < r->n_pops; ++k) {
        const size_t x = (size_t)w * r->n_pops + k;
        const char *pn = o->pop_names[k];
        if (ok) sb_printf(&s, "\tnHap[%s]:\t%d", pn, g->n_hap[x]);
        else sb_printf(&s, "\tnHap[%s]:\t%7s", pn, "NA");
        sb_stat(&s, "H1", pn, ok && !isnan(g->h1[x]), g->h1[x]);
        sb_stat(&s, "H12", pn, ok && !isnan(g->h12[x]), g->h12[x]);
        sb_stat(&s, "H123", pn, ok && !isnan(g->h123[x]), g->h123[x]);
        sb_stat(&s, "H2H1", pn, ok && !isnan(g->h2h1[x]), g->h2h1[x]);
    }
    return s.len;
}
