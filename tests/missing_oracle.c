/* missing_oracle.c -- TEST INFRASTRUCTURE.  Plain-C restatement of the PB_AN_NUCDIV_MISSING sums of include/popbam_b200.h
 * (pb_region_nucdiv_missing) and of the lines of `popbam nucdiv --missing`'s two files, which the reference never wrote.
 * Its input is the per-position, per-sample cb words of a span: the reference-pinned oracle's pbo_result.cb from a run
 * with PBO_FLAG_EMIT_CB (oracle/pb_oracle.c), or any raw array.  Per cell: covered = cb & 1, derived = (cb & 3) == 3, and
 * a cell with bit 1 set (segbase called it derived) carries its derived base in bits 10-11.
 *
 *   pbm_sums    the sums and ratios of every window, into a pb_region_nucdiv_missing (free with pbm_free)
 *   pbm_format  one window's lines of PREFIX_pi.txt (pairs = 0) or PREFIX_dxy.txt (pairs = 1)
 *
 * Unlike the kernel (coverage masks, popcounts, stripes, atomics) it walks positions and samples one by one.          */
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include "../include/popbam_b200.h"

int pbm_sums(const pb_params *p, int32_t n_windows, const int32_t *win_beg, const int32_t *win_end, int32_t span_beg,
             const uint64_t *cb, pb_region_nucdiv_missing *out) {
    memset(out, 0, sizeof *out);
    const int n = p->n_samples, P = p->n_pops;
    const size_t wp = (size_t)n_windows * P, wpp = (size_t)n_windows * P * P;
    int32_t *pi_sites = calloc(wp + 1, 4), *dxy_sites = calloc(wpp + 1, 4);
    int64_t *pi_diffs = calloc(wp + 1, 8), *pi_comps = calloc(wp + 1, 8), *pi_missing = calloc(wp + 1, 8);
    int64_t *dxy_diffs = calloc(wpp + 1, 8), *dxy_comps = calloc(wpp + 1, 8), *dxy_missing = calloc(wpp + 1, 8);
    double *pi = calloc(wp + 1, 8), *dxy = calloc(wpp + 1, 8);
    if (!pi_sites || !dxy_sites || !pi_diffs || !pi_comps || !pi_missing || !dxy_diffs || !dxy_comps || !dxy_missing || !pi || !dxy) return -4;
    int pop_of[64];
    for (int s = 0; s < n; ++s) {
        pop_of[s] = -1;
        for (int k = 0; k < P; ++k)
            if ((p->pop_mask[k] >> s) & 1) pop_of[s] = k;
    }
    for (int w = 0; w < n_windows; ++w) {
        for (int x = win_beg[w]; x < win_end[w]; ++x) {
            const uint64_t *c = cb + (size_t)(x - span_beg) * n;
            long long kk[64] = {0}, cc[64] = {0};
            int bases[4] = {0, 0, 0, 0};
            for (int s = 0; s < n; ++s) {
                if (c[s] & 2) bases[(c[s] >> 10) & 3] = 1;
                if (pop_of[s] < 0) continue;
                if (c[s] & 1) kk[pop_of[s]] += 1;
                if ((c[s] & 3) == 3) cc[pop_of[s]] += 1;
            }
            if (bases[0] + bases[1] + bases[2] + bases[3] > 1)          /* fq < 0: the position counts, without differences */
                for (int k = 0; k < P; ++k) cc[k] = 0;
            for (int k = 0; k < P; ++k) {
                if (kk[k] < 2) continue;
                const size_t i = (size_t)w * P + k;
                const long long nk = p->pop_nsmpl[k];
                pi_sites[i] += 1;
                pi_diffs[i] += cc[k] * (kk[k] - cc[k]);
                pi_comps[i] += kk[k] * (kk[k] - 1) / 2;
                pi_missing[i] += nk * (nk - 1) / 2 - kk[k] * (kk[k] - 1) / 2;
            }
            for (int a = 0; a < P; ++a)
                for (int b = a + 1; b < P; ++b) {
                    if (kk[a] < 1 || kk[b] < 1) continue;
                    const size_t i = (size_t)w * P * P + (size_t)a * P + (b - (a + 1));
                    dxy_sites[i] += 1;
                    dxy_diffs[i] += cc[a] * (kk[b] - cc[b]) + cc[b] * (kk[a] - cc[a]);
                    dxy_comps[i] += kk[a] * kk[b];
                    dxy_missing[i] += (long long)p->pop_nsmpl[a] * p->pop_nsmpl[b] - kk[a] * kk[b];
                }
        }
        for (int k = 0; k < P; ++k) {
            const size_t i = (size_t)w * P + k;
            pi[i] = pi_comps[i] ? (double)pi_diffs[i] / (double)pi_comps[i] : NAN;
        }
        for (int a = 0; a < P; ++a)
            for (int b = a + 1; b < P; ++b) {
                const size_t i = (size_t)w * P * P + (size_t)a * P + (b - (a + 1));
                dxy[i] = dxy_comps[i] ? (double)dxy_diffs[i] / (double)dxy_comps[i] : NAN;
            }
    }
    out->pi_sites = pi_sites; out->pi_diffs = pi_diffs; out->pi_comps = pi_comps; out->pi_missing = pi_missing; out->pi = pi;
    out->dxy_sites = dxy_sites; out->dxy_diffs = dxy_diffs; out->dxy_comps = dxy_comps; out->dxy_missing = dxy_missing; out->dxy = dxy;
    return 0;
}

void pbm_free(pb_region_nucdiv_missing *m) {
    free((void *)m->pi_sites); free((void *)m->pi_diffs); free((void *)m->pi_comps); free((void *)m->pi_missing); free((void *)m->pi);
    free((void *)m->dxy_sites); free((void *)m->dxy_diffs); free((void *)m->dxy_comps); free((void *)m->dxy_missing); free((void *)m->dxy);
    memset(m, 0, sizeof *m);
}

static void put(char **o, char *end, const char *fmt, long long a, long long b, long long c, long long d) {
    const int k = snprintf(*o, (size_t)(end - *o), fmt, a, b, c, d);
    *o += k;
}

/* pixy's columns: [pop | pop1 pop2] chromosome window_pos_1 window_pos_2 ratio no_sites count_diffs count_comparisons
 * count_missing; the ratio %.10g, NA without comparisons.  Returns the length; buf must be large enough.                */
int64_t pbm_format(const pb_params *p, const pb_region_nucdiv_missing *m, const int32_t *win_beg, const int32_t *win_end, int32_t w,
                   int32_t pairs, const char *chrom, const char *const *pop_names, char *buf, int64_t cap) {
    const int P = p->n_pops;
    char *o = buf, *end = buf + cap;
    for (int a = 0; a < P; ++a)
        for (int b = pairs ? a + 1 : a; b < (pairs ? P : a + 1); ++b) {
            const size_t i = pairs ? (size_t)w * P * P + (size_t)a * P + (b - (a + 1)) : (size_t)w * P + a;
            const double v = pairs ? m->dxy[i] : m->pi[i];
            const long long comps = pairs ? m->dxy_comps[i] : m->pi_comps[i];
            if (pairs) o += snprintf(o, (size_t)(end - o), "%s\t%s\t", pop_names[a], pop_names[b]);
            else o += snprintf(o, (size_t)(end - o), "%s\t", pop_names[a]);
            o += snprintf(o, (size_t)(end - o), "%s\t%lld\t%lld\t", chrom, (long long)win_beg[w] + 1, (long long)win_end[w]);
            if (comps) o += snprintf(o, (size_t)(end - o), "%.10g", v);
            else o += snprintf(o, (size_t)(end - o), "NA");
            put(&o, end, "\t%lld\t%lld\t%lld\t%lld\n", pairs ? m->dxy_sites[i] : m->pi_sites[i], pairs ? m->dxy_diffs[i] : m->pi_diffs[i], comps,
                pairs ? m->dxy_missing[i] : m->pi_missing[i]);
        }
    return (int64_t)(o - buf);
}
