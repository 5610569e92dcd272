/* spectrum_oracle.c -- TEST INFRASTRUCTURE.  Plain-C restatement of the PB_AN_SPECTRUM site frequency spectra of
 * include/popbam_b200.h (pb_region_spectrum), which the reference never wrote out.  It works on the result of the
 * reference-pinned oracle (oracle/pb_oracle.c, whose pbo_result has the layout of pb_region_result): the window's
 * segregating-site types, num_sites and segsites.
 *
 *   pbs_spectrum  the counts of every window and set, into a pb_region_spectrum (free with pbs_free)
 *
 * Unlike the kernel (groups of sets, warp-aggregated shared-memory histograms) it walks the sites one by one and
 * counts every set's derived alleles sample by sample.                                                               */
#include <stdlib.h>
#include <string.h>
#include "../include/popbam_b200.h"

int pbs_spectrum(const pb_params *p, const pb_region_result *r, int32_t n_sets, const int32_t *sets, pb_region_spectrum *out) {
    memset(out, 0, sizeof *out);
    if (n_sets < 1) return -1;
    int32_t *off = calloc((size_t)n_sets + 1, 4), *cp = malloc(12 * (size_t)n_sets);
    if (!off || !cp) return -4;
    memcpy(cp, sets, 12 * (size_t)n_sets);
    for (int s = 0; s < n_sets; ++s) {
        int b = 1;
        for (int d = 0; d < 3; ++d) {
            const int k = sets[3 * s + d];
            if (k < 0) continue;
            if (k >= r->n_pops) return -1;
            b *= p->pop_nsmpl[k] + 1;
        }
        off[s + 1] = off[s] + b;
    }
    const int B = off[n_sets];
    int32_t *cnt = calloc(r->n_windows > 0 ? (size_t)r->n_windows * B : 1, 4);
    if (!cnt) return -4;
    const int outg = (p->flags & PB_FLAG_OUTGROUP) != 0;
    for (int w = 0; w < r->n_windows; ++w) {
        const uint64_t *T = r->seg_type + r->seg_off[w];
        const int S = r->segsites[w];
        int32_t *x = cnt + (size_t)w * B;
        for (int s = 0; s < n_sets; ++s) {
            x[off[s]] += r->num_sites[w] - S;          /* the sites without a segregating call */
            for (int i = 0; i < S; ++i) {
                const int flip = outg && ((T[i] >> p->outidx) & 1);
                int bin = 0;
                for (int d = 0; d < 3; ++d) {
                    const int k = sets[3 * s + d];
                    if (k < 0) continue;
                    int a = 0;
                    for (int j = 0; j < r->n_samples; ++j)
                        if (((p->pop_mask[k] >> j) & 1) && ((T[i] >> j) & 1)) a += 1;
                    if (flip) a = p->pop_nsmpl[k] - a;
                    bin = bin * (p->pop_nsmpl[k] + 1) + a;
                }
                x[off[s] + bin] += 1;
            }
        }
    }
    out->n_sets = n_sets; out->n_bins = B; out->sets = cp; out->set_off = off; out->counts = cnt;
    return 0;
}

void pbs_free(pb_region_spectrum *s) {
    free((void *)s->sets); free((void *)s->set_off); free((void *)s->counts);
    memset(s, 0, sizeof *s);
}
