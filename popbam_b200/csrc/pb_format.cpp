// pb_format.cpp -- text of one window exactly as the reference's printers write it:
//   print_nucdiv  pop_nucdiv.cpp:258-289     print_sfs     pop_sfs.cpp:293-317
//   print_ld      pop_ld.cpp:650-712         print_diverge pop_diverge.cpp:496-574
//   print_haplo   pop_haplo.cpp:365-442      print_popbam_snp / print_sweep / print_ms  pop_snp.cpp:224-303
//   make_nj / join_tree / print_tree  pop_tree.cpp:208-470  (neighbour joining on the window's difference matrix)
// The reference streams with std::fixed << std::setprecision(5) and prints "NA" through std::setw(7);
// "%.5f" and "%7s" produce the same bytes.  Host-only formatting of results the kernels computed.
#include <cmath>
#include <cstdarg>
#include <algorithm>
#include <cstdio>
#include <cstring>
#include <cfloat>
#include <string>
#include <vector>
#include "../../include/popbam_b200.h"

extern "C" const pb_params *pb_ctx_params(const pb_ctx *c);

namespace {

struct Out {
    std::string s;
    void f(const char *fmt, ...) __attribute__((format(printf, 2, 3))) {
        char tmp[640];
        va_list ap;
        va_start(ap, fmt);
        int k = vsnprintf(tmp, sizeof tmp, fmt, ap);
        va_end(ap);
        if (k > 0) s.append(tmp, (size_t)std::min<int>(k, (int)sizeof tmp - 1));
    }
    // "\tname[label]:\t<value or NA>"
    void stat(const char *name, const char *label, bool ok, double v) {
        if (ok) f("\t%s[%s]:\t%.5f", name, label, v);
        else f("\t%s[%s]:\t%7s", name, label, "NA");
    }
};

// bam_nt16_table followed by bam_nt16_rev_table (popbam.cpp:13-31, bam.h): the letter the reference
// prints for a reference byte / consensus letter
char nt16_roundtrip(int c) {
    static const char rev[17] = "=ACMGRSVTWYHKDBN";
    int code;
    switch (c) {
    case '=': code = 0; break;
    case 'A': case 'a': case '0': code = 1; break;
    case 'C': case 'c': case '1': code = 2; break;
    case 'M': case 'm': code = 3; break;
    case 'G': case 'g': case '2': code = 4; break;
    case 'R': case 'r': code = 5; break;
    case 'S': case 's': code = 6; break;
    case 'V': case 'v': code = 7; break;
    case 'T': case 't': case '3': code = 8; break;
    case 'W': case 'w': code = 9; break;
    case 'Y': case 'y': code = 10; break;
    case 'H': case 'h': code = 11; break;
    case 'K': case 'k': code = 12; break;
    case 'D': case 'd': code = 13; break;
    case 'B': case 'b': code = 14; break;
    default: code = 15; break;
    }
    return rev[code];
}
const char kIupacLetters[17] = "AMRWNCSYNNGKNNNT";   // popbam.cpp iupac[]

inline int popc(uint64_t x) { return __builtin_popcountll(x); }

// Neighbour joining for the tree subcommand (what pop_tree.cpp:208-470 computes: distances :496-515, joining :254-429,
// Newick text :439-470), formulated on a live-cluster list:
//   * D is kept symmetric; r[a] = sum of D(a, b) over the live b in ascending order (the reference accumulates its row
//     sums pair by pair, which adds the same terms to every sum in the same order, and its "distance to everything
//     else" sums of the chosen pair are these row sums again, zeros of merged clusters included);
//   * the pair minimising Q(a, b) = (m - 2) D(a, b) - r[a] - r[b] is searched b-major, a < b, strict "<": the first
//     minimum in that order wins, as in the reference (ties are common with integer difference counts);
//   * the joined cluster keeps the smaller index, D(new, c) = (D(a, c) + D(b, c)) / 2, height[new] = D(a, b) / 2 and the
//     branch lengths are (D(a,b) + (r[a] - D(a,b))/(m-2) - (r[b] - D(a,b))/(m-2)) / 2 - height[a] and D(a,b) - that - height[b],
//     every operation in the reference's order because the printed %.5f digits depend on the rounding.
// Tree: tips 0 .. T-1 (0 = the reference sequence), inner nodes T .. 2T-3 with three ports: port 1 and 2 take the two
// clusters a node joins, port 0 is attached later; the final node joins the last three clusters on ports 0, 1, 2.
// The text starts at the inner node the reference taxon hangs on, lists the subtrees behind its other two ports in port
// order, then the reference taxon; any other node lists the two ports after the one it was entered through.
struct NjNode {
    int peer[3];          // neighbouring node per port
    double len[3];        // branch length per port
};
struct NjForest {
    int T;
    std::vector<NjNode> inner;                    // inner node k is node T + k
    std::vector<int> up;                          // tip -> inner node it hangs on
    std::vector<double> up_len;                   // tip -> its branch length
    const pb_print_opts *names;
    int port_of(int node, int neighbour) const {
        const NjNode &v = inner[node - T];
        return v.peer[0] == neighbour ? 0 : v.peer[1] == neighbour ? 1 : 2;
    }
    void branch(Out &out, double l) const {
        if (l < 0) out.s += ":0.00000"; else out.f(":%.5f", l);
    }
    // the subtree behind `node`, entered from `from`, with the length of the branch it was entered through
    void subtree(Out &out, int node, int from, double l) const {
        if (node < T) out.s += node == 0 ? names->ref_name : names->sample_names[node - 1];
        else {
            const NjNode &v = inner[node - T];
            const int in = port_of(node, from);
            out.s += '(';
            subtree(out, v.peer[(in + 1) % 3], node, v.len[(in + 1) % 3]);
            out.s += ',';
            subtree(out, v.peer[(in + 2) % 3], node, v.len[(in + 2) % 3]);
            out.s += ')';
        }
        branch(out, l);
    }
    void newick(Out &out) const {
        const int root = up[0];
        const NjNode &v = inner[root - T];
        const int in = port_of(root, 0);
        out.s += '(';
        subtree(out, v.peer[(in + 1) % 3], root, v.len[(in + 1) % 3]);
        out.s += ',';
        subtree(out, v.peer[(in + 2) % 3], root, v.len[(in + 2) % 3]);
        out.s += ',';
        subtree(out, 0, root, up_len[0]);
        out.s += ");\n";
    }
};

void nj_newick(Out &out, const uint16_t *diff, int T, int num_sites, const pb_print_opts *o) {
    std::vector<double> dist((size_t)T * T, 0.0), height((size_t)T, 0.0), rowsum((size_t)T, 0.0);
    auto D = [&](int a, int b) -> double & { return dist[(size_t)a * T + b]; };
    for (int a = 0; a < T; ++a)
        for (int b = a + 1; b < T; ++b) {
            double d = (double)diff[a * T + b] / num_sites;                 // p-distance
            if (o->jc) d = -0.75 * log(1.0 - (4.0 * d / 3.0));              // Jukes-Cantor
            D(a, b) = D(b, a) = d;
        }
    NjForest f;
    f.T = T; f.names = o;
    f.inner.resize((size_t)(T - 2));
    f.up.assign((size_t)T, -1); f.up_len.assign((size_t)T, 0.0);
    std::vector<int> top((size_t)T);             // cluster index -> the node at its top (a tip, or the inner node that joined it last)
    std::vector<int> live;                       // cluster indices still to be joined, ascending
    for (int i = 0; i < T; ++i) { top[i] = i; live.push_back(i); }
    // hang `child` (top node of a cluster) on port `port` of inner node `node`
    auto attach = [&](int node, int port, int child, double l) {
        NjNode &v = f.inner[node - T];
        v.peer[port] = child; v.len[port] = l;
        if (child < T) { f.up[child] = node; f.up_len[child] = l; }
        else { NjNode &c = f.inner[child - T]; c.peer[0] = node; c.len[0] = l; }
    };
    int next_node = T;
    while (live.size() > 3) {
        const double m2 = (double)live.size() - 2.0;
        for (int a : live) {
            double r = 0.0;
            for (int b : live) if (b != a) r += D(a, b);
            rowsum[a] = r;
        }
        double best = DBL_MAX;
        int ja = 0, jb = 0;
        for (size_t ib = 1; ib < live.size(); ++ib)
            for (size_t ia = 0; ia < ib; ++ia) {
                const int a = live[ia], b = live[ib];
                const double q = m2 * D(a, b) - rowsum[a] - rowsum[b];
                if (q < best) { best = q; ja = a; jb = b; }
            }
        const double dab = D(ja, jb);
        const double ra = (rowsum[ja] - dab) / m2, rb = (rowsum[jb] - dab) / m2;
        double la = (dab + ra - rb) * 0.5, lb = dab - la;
        la -= height[ja]; lb -= height[jb];
        const int node = next_node++;
        attach(node, 1, top[ja], la);
        attach(node, 2, top[jb], lb);
        top[ja] = node;
        height[ja] = dab * 0.5;
        live.erase(std::find(live.begin(), live.end(), jb));
        for (int c : live)
            if (c != ja) D(ja, c) = D(c, ja) = (D(ja, c) + D(jb, c)) * 0.5;
    }
    const int a = live[0], b = live[1], c = live[2];
    double la = (D(a, b) + D(a, c) - D(b, c)) * 0.5;
    double lb = D(a, b) - la, lc = D(a, c) - la;
    la -= height[a]; lb -= height[b]; lc -= height[c];
    const int node = next_node;
    attach(node, 0, top[a], la); attach(node, 1, top[b], lb); attach(node, 2, top[c], lc);
    f.newick(out);
}

// every printer: one reference bit, optionally with its extension, whose columns follow the reference's, and (nucdiv
// only, checked by pb_format_window_fst) the F_ST columns after those
int64_t format_window(const pb_ctx *ctx, const pb_region_result *r, const pb_region_extras *e, const pb_region_fst *fs, int32_t w,
                      uint32_t an, const pb_print_opts *o, char *buf, int64_t cap) {
    const pb_params *p = pb_ctx_params(ctx);
    if (!p || !r || !o || w < 0 || w >= r->n_windows) return PB_ERR_ARG;
    if ((r->analyses & an) != an) return PB_ERR_ARG;
    const uint32_t ext = an & (PB_AN_THETA_W | PB_AN_FULI | PB_AN_LD_DPRIME);
    const bool with_fst = (an & PB_AN_FST) != 0;
    an &= ~(ext | PB_AN_FST);
    if (ext && (!e || ext != (an == PB_AN_NUCDIV ? PB_AN_THETA_W : an == PB_AN_SFS ? PB_AN_FULI : an == PB_AN_LD_ZNS ? PB_AN_LD_DPRIME : 0u)))
        return PB_ERR_ARG;
    Out out;
    const int P = r->n_pops, n = r->n_samples;
    const int ns = r->num_sites[w];
    const int64_t so = r->seg_off[w];
    const int S = r->segsites[w];
    const size_t wp = (size_t)w * P;
    if (an == PB_AN_SNP) {
        if (!r->seg_cb) return PB_ERR_ARG;
        if (o->snp_output == 0) {                    // print_popbam_snp
            for (int i = 0; i < S; ++i) {
                out.f("%s\t%u\t%c", o->chrom, r->seg_pos[so + i] + 1, nt16_roundtrip(r->seg_ref[so + i]));
                for (int j = 0; j < n; ++j) {
                    const uint64_t cb = r->seg_cb[(size_t)(so + i) * n + j];
                    const unsigned g = (unsigned)((cb >> 8) & 0xff);
                    // g >= 16 only arises from the reference's revert-to-reference arithmetic (SURVEY Q8),
                    // where the reference itself reads iupac[] out of bounds: that letter is undefined
                    const char base = g < 16 ? nt16_roundtrip(kIupacLetters[g]) : '?';
                    out.f("\t%c\t%u\t%u\t%u", base, (unsigned)((cb >> 32) & 0xffff), (unsigned)((cb >> 48) & 0xffff),
                          (unsigned)((cb >> 16) & 0xffff));
                }
                out.f("\n");
            }
        } else if (o->snp_output == 1) {             // print_sweep
            for (int i = 0; i < S; ++i) {
                out.f("%s\t%u", o->chrom, r->seg_pos[so + i] + 1);
                const uint64_t T = r->seg_type[so + i];
                for (int j = 0; j < P; ++j) {
                    const int pn = popc(p->pop_mask[j]);
                    unsigned f = (unsigned)popc(T & p->pop_mask[j]);
                    if ((p->flags & PB_FLAG_OUTGROUP) && (T >> p->outidx & 1)) f = (unsigned)(pn - (int)f) & 0xffff;
                    out.f("\t%u\t%d", f, pn);
                }
                out.f("\n");
            }
        } else {                                     // print_ms
            out.f("//\nsegsites: %d\npositions: ", S);
            for (int i = 0; i < S; ++i)
                out.f("%.8g ", (double)(r->seg_pos[so + i] - (unsigned)r->win_beg[w]) / (r->win_end[w] - r->win_beg[w]));
            out.f("\n");
            for (int i = 0; i < n; ++i) {
                for (int j = 0; j < S; ++j) {
                    const uint64_t T = r->seg_type[so + j];
                    int bit = (int)(T >> i & 1);
                    if ((p->flags & PB_FLAG_OUTGROUP) && (T >> p->outidx & 1)) bit = !bit;
                    out.s.push_back(bit ? '1' : '0');
                }
                out.f("\n");
            }
            out.f("\n");
        }
    } else {
        out.f("%s\t%d\t%d\t%d", o->chrom, r->win_beg[w] + 1, r->win_end[w] + 1, ns);
        const bool ok = ns >= o->min_sites;
        char nm[600];
        if (an == PB_AN_TREE) {      // make_nj (pop_tree.cpp:208-252): the tree ends the row itself
            if (!r->tree_diff || !o->ref_name || n < 2) return PB_ERR_ARG;      // three taxa at least
            if (!ok || S < 1) out.f("\tNA\n");
            else { out.f("\t"); nj_newick(out, r->tree_diff + (size_t)w * (n + 1) * (n + 1), n + 1, ns, o); }
        } else {
        switch (an) {
        case PB_AN_NUCDIV:
            for (int i = 0; i < P; ++i) out.stat("pi", o->pop_names[i], ok, r->piw[wp + i] / ns);
            for (int i = 0; i < P - 1; ++i)
                for (int j = i + 1; j < P; ++j) {
                    snprintf(nm, sizeof nm, "%s-%s", o->pop_names[i], o->pop_names[j]);
                    out.stat("dxy", nm, ok, r->pib[wp * P + i * P + (j - (i + 1))] / ns);
                }
            break;
        case PB_AN_SFS:
            for (int i = 0; i < P; ++i) {
                out.stat("D", o->pop_names[i], !std::isnan(r->td[wp + i]), r->td[wp + i]);
                out.stat("H", o->pop_names[i], !std::isnan(r->fwh[wp + i]), r->fwh[wp + i]);
            }
            break;
        case PB_AN_LD_ZNS: case PB_AN_LD_OMEGA: case PB_AN_LD_WALL:
            for (int i = 0; i < P; ++i) {
                const int nsnp = an == PB_AN_LD_WALL ? r->wall_num_snps[wp + i] : r->ld_num_snps[wp + i];
                out.f("\tS[%s]:\t%d", o->pop_names[i], nsnp);
                const bool good = nsnp >= o->min_snps;
                if (an == PB_AN_LD_ZNS) out.stat("Zns", o->pop_names[i], good, r->zns[wp + i]);
                else if (an == PB_AN_LD_OMEGA) out.stat("omax", o->pop_names[i], good, r->omegamax[wp + i]);
                else { out.stat("B", o->pop_names[i], good, r->wallb[wp + i]); out.stat("Q", o->pop_names[i], good, r->wallq[wp + i]); }
            }
            break;
        case PB_AN_DIVERGE_IND:
            for (int i = 0; i < n; ++i) {
                double d = (double)r->ind_div[(size_t)w * n + i] / ns;
                if (o->jc) d = -0.75 * std::log(1.0 - d * (4.0 / 3.0));
                out.stat("d", o->sample_names[i], ok, d);
            }
            break;
        case PB_AN_DIVERGE_POP:
            for (int i = 0; i < P; ++i) {
                const char *pn = o->pop_names[i];
                if (ok) {
                    const int fx = r->pop_div[wp + i], sg = r->div_num_snps[wp + i];
                    double d = (p->flags & PB_FLAG_SUBSTITUTE) ? (double)fx / ns : (double)(fx + sg) / ns;
                    if (o->jc) d = -0.75 * std::log(1.0 - d * (4.0 / 3.0));
                    out.f("\tFixed[%s]:\t%d\tSeg[%s]:\t%d\td[%s]:\t%.5f", pn, fx, pn, sg, pn, d);
                } else out.f("\tFixed[%s]:\t%7s\tSeg[%s]:\t%7s\td[%s]:\t%7s", pn, "NA", pn, "NA", pn, "NA");
            }
            break;
        case PB_AN_HAPLO_K:
            for (int i = 0; i < P; ++i) {
                const char *pn = o->pop_names[i];
                if (ok) out.f("\tK[%s]:\t%d\tKdiv[%s]:\t%.5f", pn, r->nhaps[wp + i], pn, 1.0 - r->hdiv[wp + i]);
                else out.f("\tK[%s]:\t%7s\tKdiv[%s]:\t%7s", pn, "NA", pn, "NA");
            }
            break;
        case PB_AN_HAPLO_EHHS:
            for (int i = 0; i < P; ++i) out.stat("EHHS", o->pop_names[i], ok && !std::isnan(r->ehhs[wp + i]), r->ehhs[wp + i]);
            break;
        case PB_AN_HAPLO_DXY:
            for (int i = 0; i < P; ++i) out.stat("pi", o->pop_names[i], ok, r->piw[wp + i]);
            for (int i = 0; i < P - 1; ++i)
                for (int j = i + 1; j < P; ++j) {
                    snprintf(nm, sizeof nm, "%s-%s", o->pop_names[i], o->pop_names[j]);
                    const size_t x = wp * P + i * P + (j - (i + 1));
                    if (ok) out.f("\tdxy[%s]:\t%.5f\tmin[%s]:\t%u", nm, r->pib[x], nm, (unsigned)r->min_dxy[x]);
                    else out.f("\tdxy[%s]:\t%7s\tmin[%s]:\t%7s", nm, "NA", nm, "NA");
                }
            break;
        default: return PB_ERR_ARG;
        }
        for (int i = 0; ext && i < P; ++i) {
            const size_t x = wp + i;
            if (ext == PB_AN_THETA_W) out.stat("theta", o->pop_names[i], ok && !std::isnan(e->theta_w[x]), e->theta_w[x] / ns);
            else if (ext == PB_AN_FULI) {
                out.stat("FuLiD*", o->pop_names[i], !std::isnan(e->fuli_ds[x]), e->fuli_ds[x]);
                if (p->flags & PB_FLAG_OUTGROUP) out.stat("FuLiD", o->pop_names[i], !std::isnan(e->fuli_d[x]), e->fuli_d[x]);
            } else {
                const bool good = r->ld_num_snps[x] >= o->min_snps && e->ld_kept[x] >= 2;
                out.stat("Dp", o->pop_names[i], good, e->ld_dprime[x]);
                if (good) out.f("\tDp1[%s]:\t%lld", o->pop_names[i], (long long)e->ld_complete[x]);
                else out.f("\tDp1[%s]:\t%7s", o->pop_names[i], "NA");
            }
        }
        for (int i = 0; with_fst && i < P - 1; ++i)
            for (int j = i + 1; j < P; ++j) {
                snprintf(nm, sizeof nm, "%s-%s", o->pop_names[i], o->pop_names[j]);
                const size_t x = wp * P + i * P + (j - (i + 1));
                out.stat("Fst", nm, ok && !std::isnan(fs->fst_hudson[x]), fs->fst_hudson[x]);
                out.stat("FstWC", nm, ok && !std::isnan(fs->fst_wc[x]), fs->fst_wc[x]);
                out.stat("Snn", nm, ok && !std::isnan(fs->snn[x]), fs->snn[x]);
                if (fs->snn_p) out.stat("SnnP", nm, ok && !std::isnan(fs->snn_p[x]), fs->snn_p[x]);
            }
        out.f("\n");
        }
    }
    const int64_t len = (int64_t)out.s.size();
    if (buf && cap > 0) {
        const int64_t k = std::min<int64_t>(len, cap - 1);
        memcpy(buf, out.s.data(), (size_t)k);
        buf[k] = 0;
    }
    return len;
}

}  // namespace

extern "C" int64_t pb_format_window(const pb_ctx *ctx, const pb_region_result *r, int32_t w, uint32_t an, const pb_print_opts *o,
                                    char *buf, int64_t cap) {
    if (an & (PB_AN_THETA_W | PB_AN_FULI | PB_AN_LD_DPRIME | PB_AN_FST)) return PB_ERR_ARG;
    return format_window(ctx, r, nullptr, nullptr, w, an, o, buf, cap);
}

extern "C" int64_t pb_format_window_ext(const pb_ctx *ctx, const pb_region_result *r, const pb_region_extras *e, int32_t w, uint32_t an,
                                        const pb_print_opts *o, char *buf, int64_t cap) {
    if (an & PB_AN_FST) return PB_ERR_ARG;
    return format_window(ctx, r, e, nullptr, w, an, o, buf, cap);
}

extern "C" int64_t pb_format_window_fst(const pb_ctx *ctx, const pb_region_result *r, const pb_region_extras *e, const pb_region_fst *f,
                                        int32_t w, uint32_t an, const pb_print_opts *o, char *buf, int64_t cap) {
    if ((an & ~(PB_AN_THETA_W | PB_AN_FST)) != PB_AN_NUCDIV) return PB_ERR_ARG;
    if ((an & PB_AN_FST) && (!f || !f->fst_hudson || !f->fst_wc || !f->snn)) return PB_ERR_ARG;
    return format_window(ctx, r, e, f, w, an, o, buf, cap);
}
