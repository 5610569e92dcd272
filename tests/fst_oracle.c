/* fst_oracle.c -- TEST INFRASTRUCTURE.  Plain-C restatement of the PB_AN_FST statistics of include/popbam_b200.h
 * (Hudson's F_ST, Weir & Cockerham's theta, Hudson's Snn and its permutation test), which the reference never computed.
 * It works on the result of the reference-pinned oracle (oracle/pb_oracle.c, whose pbo_result has the layout of
 * pb_region_result): the window's segregating-site types, from which it builds its own difference matrix.
 *
 *   pbf_fst      the pair arrays of every window, into a pb_region_fst (snn_p / snn_ge only with n_perms > 0)
 *   pbf_columns  the text pb_format_window_fst appends to a nucdiv row (after any theta columns), without the newline
 *
 * Per site the integer terms are those of the header; the window sums are exact.  Snn sums X_x over the pooled samples in
 * ascending order and divides by n1 + n2, as the kernel's thread 0 does.  The permutation stream is splitmix64 (Steele,
 * Lea & Flood 2014) used as a counter-based generator:
 *   mix(z)  = (z ^ z>>30) * 0xbf58476d1ce4e5b9 -> (z ^ z>>27) * 0x94d049bb133111eb -> z ^ z>>31
 *   key     h = mix(seed + G), then h = mix((h ^ v) + G) for v = tid, win_beg, i, j, permutation index (G = 0x9e3779b97f4a7c15)
 *   draw k  mix(h + (k+1) G); index in [0, r) = ((z >> 32) * r) >> 32
 *   shuffle slot k (k < n1) of the pool (ascending sample order) swaps with slot k + index(draw k, m - k); the first n1
 *           slots are population i.
 * Built with -ffp-contract=off so that products and sums round separately.                                            */
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include "../include/popbam_b200.h"

#define GAMMA 0x9e3779b97f4a7c15ULL

static int popc64(uint64_t x) { return __builtin_popcountll(x); }

static uint64_t mix64(uint64_t z) {
    z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ULL;
    z = (z ^ (z >> 27)) * 0x94d049bb133111ebULL;
    return z ^ (z >> 31);
}

uint64_t pbf_key(uint64_t seed, int64_t tid, int64_t win_beg, int64_t i, int64_t j, int64_t perm) {
    const int64_t v[5] = {tid, win_beg, i, j, perm};
    uint64_t h = mix64(seed + GAMMA);
    for (int k = 0; k < 5; ++k) h = mix64((h ^ (uint64_t)v[k]) + GAMMA);
    return h;
}

/* Snn of the partition (A, pool \ A) given every pooled sample's nearest-neighbour mask */
static double snn_of(const uint64_t *nn, uint64_t pool, uint64_t A, int m) {
    const uint64_t B = pool & ~A;
    double sum = 0.0;
    for (int y = 0; y < 64; ++y) {
        if (!(pool >> y & 1)) continue;
        const uint64_t own = (A >> y & 1) ? A : B;
        sum += (double)popc64(nn[y] & own) / (double)popc64(nn[y]);
    }
    return sum / (double)m;
}

/* one (window, pair): sums, ratios, Snn and (n_perms > 0) the permutation count */
static void pair_stats(const pb_params *p, const uint64_t *T, int S, int n, int i, int j, int32_t tid, int32_t win_beg,
                       int64_t n_perms, uint64_t seed, int64_t *hn, int64_t *hd, int64_t *wn, int64_t *wd, double *fh,
                       double *fw, double *snn, double *snn_p, int64_t *snn_ge) {
    const uint64_t mi = p->pop_mask[i], mj = p->pop_mask[j], pool = mi | mj;
    const int64_t n1 = p->pop_nsmpl[i], n2 = p->pop_nsmpl[j];
    int64_t s_hn = 0, s_hd = 0, s_wn = 0, s_wd = 0;
    for (int s = 0; s < S; ++s) {
        const int64_t c1 = popc64(T[s] & mi), c2 = popc64(T[s] & mj);
        const int64_t between = (n1 - 1) * (n2 - 1) * (c1 * (n2 - c2) + c2 * (n1 - c1));
        const int64_t within = c1 * (n1 - c1) * n2 * (n2 - 1) + c2 * (n2 - c2) * n1 * (n1 - 1);
        const int64_t d = c1 * n2 - c2 * n1;
        const int64_t msp = d * d * (n1 + n2 - 2);
        const int64_t g = c1 * (n1 - c1) * n2 + c2 * (n2 - c2) * n1;
        s_hd += between;
        s_hn += between - within;
        s_wn += msp - g * (n1 + n2);
        s_wd += msp + g * (2 * n1 * n2 - n1 - n2);
    }
    *hn = s_hn; *hd = s_hd; *wn = s_wn; *wd = s_wd;
    const int two = n1 >= 2 && n2 >= 2;
    *fh = two && s_hd != 0 ? (double)s_hn / (double)s_hd : NAN;
    *fw = two && s_wd != 0 ? (double)s_wn / (double)s_wd : NAN;
    *snn = NAN;
    if (snn_p) { *snn_p = NAN; *snn_ge = 0; }
    if (!two) return;
    /* nearest neighbours from the window's difference matrix (unsigned short, as the product keeps it) */
    uint64_t nn[64] = {0};
    for (int x = 0; x < n; ++x) {
        if (!(pool >> x & 1)) continue;
        unsigned best = 0xffffffffu;
        for (int y = 0; y < n; ++y) {
            if (y == x || !(pool >> y & 1)) continue;
            int dxy = 0;
            for (int s = 0; s < S; ++s) dxy += (int)((T[s] >> x ^ T[s] >> y) & 1);
            const unsigned dd = (uint16_t)dxy;
            if (dd < best) { best = dd; nn[x] = 0; }
            if (dd == best) nn[x] |= 1ULL << y;
        }
    }
    const int m = (int)(n1 + n2);
    *snn = snn_of(nn, pool, mi, m);
    if (!snn_p) return;
    int slots[64];
    int64_t ge = 0;
    for (int64_t k = 0; k < n_perms; ++k) {
        const uint64_t h = pbf_key(seed, tid, win_beg, i, j, k);
        int c = 0;
        for (int y = 0; y < 64; ++y)
            if (pool >> y & 1) slots[c++] = y;
        uint64_t A = 0;
        for (int t = 0; t < n1; ++t) {
            const uint64_t z = mix64(h + (uint64_t)(t + 1) * GAMMA);
            const int r = t + (int)(((z >> 32) * (uint64_t)(m - t)) >> 32);
            const int sw = slots[r];
            slots[r] = slots[t]; slots[t] = sw;
            A |= 1ULL << sw;
        }
        ge += snn_of(nn, pool, A, m) >= *snn - 1e-12;
    }
    *snn_ge = ge;
    *snn_p = (1.0 + (double)ge) / (1.0 + (double)n_perms);
}

int pbf_fst(const pb_params *p, const pb_region_result *r, int32_t tid, int64_t n_perms, uint64_t seed, pb_region_fst *out) {
    const int P = r->n_pops;
    const size_t c = (size_t)r->n_windows * P * P ? (size_t)r->n_windows * P * P : 1;
    int64_t *hn = calloc(c, 8), *hd = calloc(c, 8), *wn = calloc(c, 8), *wd = calloc(c, 8), *ge = calloc(c, 8);
    double *fh = calloc(c, 8), *fw = calloc(c, 8), *sn = calloc(c, 8), *sp = calloc(c, 8);
    if (!hn || !hd || !wn || !wd || !ge || !fh || !fw || !sn || !sp) return -4;
    for (int w = 0; w < r->n_windows; ++w) {
        const uint64_t *T = r->seg_type + r->seg_off[w];
        for (int i = 0; i < P - 1; ++i)
            for (int j = i + 1; j < P; ++j) {
                const size_t x = (size_t)w * P * P + i * P + (j - (i + 1));
                pair_stats(p, T, r->segsites[w], r->n_samples, i, j, tid, r->win_beg[w], n_perms, seed, hn + x, hd + x, wn + x, wd + x,
                           fh + x, fw + x, sn + x, n_perms > 0 ? sp + x : NULL, n_perms > 0 ? ge + x : NULL);
            }
    }
    out->hud_num = hn; out->hud_den = hd; out->wc_num = wn; out->wc_den = wd;
    out->fst_hudson = fh; out->fst_wc = fw; out->snn = sn;
    if (n_perms > 0) { out->snn_p = sp; out->snn_ge = ge; }
    else { free(sp); free(ge); out->snn_p = NULL; out->snn_ge = NULL; }
    return 0;
}

void pbf_free(pb_region_fst *f) {
    free((void *)f->hud_num); free((void *)f->hud_den); free((void *)f->wc_num); free((void *)f->wc_den);
    free((void *)f->fst_hudson); free((void *)f->fst_wc); free((void *)f->snn); free((void *)f->snn_p); free((void *)f->snn_ge);
    memset(f, 0, sizeof *f);
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
static void sb_stat(sbuf *s, const char *name, const char *pair, int ok, double v) {
    if (ok) sb_printf(s, "\t%s[%s]:\t%.5f", name, pair, v);
    else sb_printf(s, "\t%s[%s]:\t%7s", name, pair, "NA");
}

/* the F_ST columns of window w: per pair in dxy order Fst, FstWC, Snn (+ SnnP); NA like dxy (min_sites) or where NaN */
int64_t pbf_columns(const pb_region_result *r, const pb_region_fst *f, int32_t w, const pb_print_opts *o, char *buf, int64_t cap) {
    sbuf s = {buf, cap, 0};
    const int P = r->n_pops, ok = r->num_sites[w] >= o->min_sites;
    if (cap > 0) buf[0] = 0;
    for (int i = 0; i < P - 1; ++i)
        for (int j = i + 1; j < P; ++j) {
            char nm[600];
            snprintf(nm, sizeof nm, "%s-%s", o->pop_names[i], o->pop_names[j]);
            const size_t x = (size_t)w * P * P + i * P + (j - (i + 1));
            sb_stat(&s, "Fst", nm, ok && !isnan(f->fst_hudson[x]), f->fst_hudson[x]);
            sb_stat(&s, "FstWC", nm, ok && !isnan(f->fst_wc[x]), f->fst_wc[x]);
            sb_stat(&s, "Snn", nm, ok && !isnan(f->snn[x]), f->snn[x]);
            if (f->snn_p) sb_stat(&s, "SnnP", nm, ok && !isnan(f->snn_p[x]), f->snn_p[x]);
        }
    return s.len;
}
