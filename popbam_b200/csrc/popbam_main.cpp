// popbam_main.cpp -- the `popbam` command line on the B200 path.
//
// Same command surface and output text as the reference's nucdiv / sfs / ld / diverge / haplo / snp
// subcommands (popbam.cpp:53-77; option tables pop_nucdiv.cpp:297-414, pop_sfs.cpp:319-434,
// pop_ld.cpp:460-584, pop_diverge.cpp:259-396, pop_haplo.cpp:460-580, pop_snp.cpp:319-446), but the
// window loop of every main_X (e.g. pop_nucdiv.cpp:57-124) is replaced by:
//   host threads:  BAI slicing + BGZF inflate + record decode of one region SHARD (a run of whole
//                  windows) into a pb_read_batch                                     (pb_bamio.cpp)
//   GPU threads:   pb_region_begin / pb_push_batch / pb_region_end on their own device, one pb_ctx each
//   main thread:   prints the shards' rows in window order (pb_format_window)
// Shards are independent (every window starts from an empty pileup, SURVEY.md §8(e)), so the GPUs of
// a box each take every G-th shard and no data crosses between them.
//
// Extra options (not in the reference): --gpus N, --shard-mb X, --threads T, and --extra-stats: statistics the
// reference does not compute, as extra columns after its own (nucdiv: Watterson's theta; sfs: Fu & Li's D* and, with
// -p, D; ld -o 0: mean |D'| and the number of SNP pairs in complete LD); for nucdiv only, --fst: F_ST (Hudson, and Weir &
// Cockerham) and Hudson's Snn for every population pair, after the --extra-stats columns, with --snn-perms N: a permutation
// p-value of Snn from N random re-partitions of the pair's samples, drawn from a stream seeded by --seed S (default 0).
#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <future>
#include <mutex>
#include <sstream>
#include <string>
#include <thread>
#include <vector>

#include "../../include/popbam_b200.h"
#include "pb_bamio.h"

namespace {

[[noreturn]] void fatal(const std::string &msg) {
    // fatal_error (pop_utils.cpp:510-519) without the source position of the reference's call site
    fprintf(stderr, "popbam runtime error:\n%s\nExiting program\n", msg.c_str());
    fflush(stdout);
    _Exit(EXIT_FAILURE);       // the table-building thread may still be running: no static destructors
}

struct Options {
    std::string cmd, reffile, headfile, outgroup, dist = "pdist";
    int min_depth = 3, max_depth = 255, min_rmsQ = 25, min_snpQ = 25, min_mapQ = 13, min_baseQ = 13;
    int min_sites = 10, min_snps = 10, win_size = 0, output = 0;
    bool window = false, illumina = false, het = false, min_freq2 = false, substitute = false, has_p = false, has_h = false;
    std::vector<std::string> positional;
    int gpus = 1, threads = 0;
    bool extra_stats = false;
    bool fst = false, snn_opts = false;
    long long snn_perms = 0;
    unsigned long long seed = 0;
    double shard_mb = 2.0;
};

// Option letters that take a value / that are flags, per subcommand (the reference's getopt_pp tables).
struct CmdSpec { const char *name; const char *valued; const char *flags; };
const CmdSpec kCmds[] = {
    {"nucdiv", "fhmxqsabkw", "pin"},   // -p and -n are presence flags here (pop_nucdiv.cpp:326-331, SURVEY Q15)
    {"sfs", "fhmxqpsabkw", "i"},
    {"ld", "fhmxqsaboznwk", "ie"},
    {"diverge", "fhmxqsabkpwod", "nti"},
    {"haplo", "fhomxqsabkw", "i"},
    {"snp", "fhmxqsabozpw", "vi"},
    {"tree", "fhmxqsabkwd", "i"},      // pop_tree.cpp:601-620
};

void usage(const char *cmd) {
    fprintf(stderr,
            "Usage:   popbam %s [options] <in.bam> [region]\n"
            "Options: -f FILE reference fastA   -w INT window (kb)   -m/-x INT min/max depth   -q INT min rms mapQ\n"
            "         -s INT min snpQ   -a/-b INT min mapQ / baseQ   -k INT min sites   -o INT output mode   -p STR outgroup\n"
            "         -i Illumina 1.3+ qualities   --gpus N   --shard-mb X   --threads T\n"
            "         --extra-stats  nucdiv: theta[pop]; sfs: FuLiD*[pop] (and FuLiD[pop] with -p); ld -o 0: Dp[pop], Dp1[pop]\n"
            "         --fst  nucdiv: Fst[A-B] (Hudson), FstWC[A-B] (Weir & Cockerham), Snn[A-B] (Hudson's nearest neighbours)\n"
            "         --snn-perms N  with --fst: SnnP[A-B], p-value of Snn from N permutations   --seed S  their random stream (0)\n", cmd);
}

Options parse(int argc, char **argv) {
    Options o;
    o.cmd = argv[1];
    const CmdSpec *spec = nullptr;
    for (const CmdSpec &c : kCmds) if (o.cmd == c.name) spec = &c;
    if (!spec) { fprintf(stderr, "Error: unrecognized command: %s\n", argv[1]); exit(1); }
    for (int i = 2; i < argc; ++i) {
        const std::string a = argv[i];
        if (a.rfind("--", 0) == 0) {
            auto val = [&]() -> const char * { if (i + 1 >= argc) fatal("missing value for " + a); return argv[++i]; };
            if (a == "--extra-stats") { o.extra_stats = true; continue; }
            if (a == "--fst") { o.fst = true; continue; }
            if (a == "--snn-perms" || a == "--seed") {
                const char *v = val();
                char *end = nullptr;
                if (a == "--seed") o.seed = strtoull(v, &end, 10);
                else o.snn_perms = strtoll(v, &end, 10);
                if (!*v || *end || v[0] == '-' || o.snn_perms > 0x7fffffffLL) fatal("invalid value for " + a + ": " + v);
                o.snn_opts = true;
                continue;
            }
            if (a == "--gpus") o.gpus = atoi(val());
            else if (a == "--shard-mb") o.shard_mb = atof(val());
            else if (a == "--threads") o.threads = atoi(val());
            else fatal("unknown option " + a);
            continue;
        }
        if (a.size() >= 2 && a[0] == '-' && !isdigit((unsigned char)a[1])) {
            // getopt_pp: every character of "-xyz" is an option; a value is the NEXT token, and only if that
            // token is not itself an option (getopt_pp.cpp:81-143, getopt_pp.h:76-84)
            for (size_t ci = 1; ci < a.size(); ++ci) {
                const char c = a[ci];
                const bool last = ci + 1 == a.size();
                if (strchr(spec->valued, c)) {
                    std::string v;
                    bool have = false;
                    if (last && i + 1 < argc) {
                        const char *nx = argv[i + 1];
                        const bool is_opt = nx[0] == '-' && nx[1] != '\0' && !isdigit((unsigned char)nx[1]);
                        if (!is_opt) { v = argv[++i]; have = true; }
                    }
                    if (c == 'z' && o.cmd == "snp") o.het = true;          // OptionPresent('z') (pop_snp.cpp:353)
                    if (c == 'h') o.has_h = true;
                    if (c == 'w') o.window = true;
                    if (c == 'p') o.has_p = true;
                    if (!have) { if (c == 'w') o.win_size *= 1000; continue; }
                    switch (c) {
                    case 'f': o.reffile = v; break;
                    case 'h': o.headfile = v; break;
                    case 'm': o.min_depth = atoi(v.c_str()); break;
                    case 'x': o.max_depth = atoi(v.c_str()); break;
                    case 'q': o.min_rmsQ = atoi(v.c_str()); break;
                    case 's': o.min_snpQ = atoi(v.c_str()); break;
                    // -a / -b are stored in unsigned chars and read with operator>>, i.e. as ONE CHARACTER
                    // (popbam.h:260-261, SURVEY Q13): "-a 20" yields '2' == 50.  Reproduced for drop-in parity.
                    case 'a': if (!v.empty()) o.min_mapQ = (unsigned char)v[0]; break;
                    case 'b': if (!v.empty()) o.min_baseQ = (unsigned char)v[0]; break;
                    case 'k': o.min_sites = atoi(v.c_str()); break;
                    case 'n': o.min_snps = atoi(v.c_str()); break;
                    case 'w': o.win_size = atoi(v.c_str()) * 1000; break;
                    case 'o': o.output = atoi(v.c_str()); break;
                    case 'p': o.outgroup = v; break;
                    case 'd': o.dist = v; break;
                    default: break;      // -z: value parsed and ignored (SURVEY Q15)
                    }
                } else if (strchr(spec->flags, c)) {
                    switch (c) {
                    case 'i': o.illumina = true; break;
                    case 'e': o.min_freq2 = true; break;
                    case 't': o.substitute = true; break;
                    default: break;      // nucdiv -p, -n, -v: dead options
                    }
                } else fatal(std::string("unknown option -") + c);
            }
            continue;
        }
        o.positional.push_back(a);
    }
    if (o.extra_stats && !(o.cmd == "nucdiv" || o.cmd == "sfs" || (o.cmd == "ld" && o.output == 0)))
        fatal("--extra-stats is only available for nucdiv, sfs and ld -o 0");
    if ((o.fst || o.snn_opts) && o.cmd != "nucdiv") fatal("--fst, --snn-perms and --seed are only available for nucdiv");
    if (o.snn_opts && !o.fst) fatal("--snn-perms and --seed go with --fst");
    return o;
}

struct Shard {
    int w0, w1;                 // windows [w0, w1)
    // the shard's reads as one or more batches in file order: PIECES of one bam_fetch (pbio::fetch_piece), decoded by
    // different threads when there are fewer shards than threads (no -w: one window is the whole region) and so that no
    // batch outgrows its 32-bit offsets
    std::vector<pbio::Batch> pieces;
    std::vector<std::pair<int32_t, int32_t>> cuts;     // [lo, hi) of every piece
    int pieces_left = 0;
    std::string text;
    std::string error;
    int state = 0;              // 0 pending, 1 decoded, 2 done
};

struct Run {
    Options opt;
    pbio::BgzfFile bam;
    pbio::BamHeader hdr;
    pbio::SampleTable st;
    pbio::BamIndex idx;
    std::string ref;
    std::string ref_name;       // tree: the AS tag
    int tid = -1, beg = 0, end = 0;
    std::vector<int32_t> wb, we;
    std::vector<Shard> shards;
    pb_params prm;
    uint32_t analysis = 0;
    // error-model tables, built once on the host (while the files are opened) and shared by every context
    std::vector<double> fk, beta, lhet;
    std::shared_future<void> tables_ready;
    std::mutex mu;
    std::condition_variable cv;
    bool pinned = false;
    bool feed_only = false;     // `popbam _feed ...` (test hook, no GPU): the workers print what they were fed instead of results
    std::atomic<double> bases_per_bp{0.0}, reads_per_bp{0.0};      // densest piece decoded so far
    std::atomic<int> next_decode{0};
    std::vector<std::pair<int, int>> items;      // decode work: (shard, piece), shard-major
    int max_ahead = 4;
    int printed = 0;
    // batches (page-locked with POPBAM_B200_PINNED=1, and then expensive to allocate) go back to a pool after use
    std::vector<pbio::Batch> pool;
    pbio::Batch take_batch() {
        std::lock_guard<std::mutex> lk(mu);
        if (pool.empty()) return pbio::Batch();
        pbio::Batch b = std::move(pool.back());
        pool.pop_back();
        return b;
    }
    void give_batch(pbio::Batch &&b) {
        b.clear();
        std::lock_guard<std::mutex> lk(mu);
        pool.push_back(std::move(b));
    }
};

void decode_worker(Run *R) {
    for (;;) {
        const int it = R->next_decode.fetch_add(1);
        if (it >= (int)R->items.size()) return;
        const int s = R->items[it].first, pc = R->items[it].second;
        {   // do not run too far ahead of the printer (bounds host memory)
            std::unique_lock<std::mutex> lk(R->mu);
            R->cv.wait(lk, [&] { return s < R->printed + R->max_ahead; });
        }
        Shard &sh = R->shards[s];
        pbio::Batch b = R->take_batch();
        std::string err;
        const double bp = (double)(sh.cuts[pc].second - sh.cuts[pc].first);
        {
            // room for what pieces of this length held so far (page-locked memory is expensive to grow)
            const double per_bp = R->bases_per_bp.load(), reads_per_bp = R->reads_per_bp.load();
            if (per_bp > 0) {
                const size_t nb = (size_t)(1.25 * per_bp * bp) + 4096, nr = (size_t)(1.25 * reads_per_bp * bp) + 256;
                b.qual.reserve(nb); b.seq4.reserve(nb / 2 + 64); b.pos.reserve(nr); b.meta.reserve(nr); b.cig_off.reserve(nr + 1); b.base_off.reserve(nr + 1);
                b.cigar.reserve(nr + nr / 4);
            }
        }
        try {
            pbio::fetch_piece(R->bam, R->idx, R->st, R->tid, R->wb[sh.w0], R->we[sh.w1 - 1], sh.cuts[pc].first, sh.cuts[pc].second, b);
        } catch (const pbio::Error &e) { err = e.msg; }
        if (bp > 0 && b.n_reads() > 0) {
            double v = (double)b.qual.size() / bp, w = (double)b.n_reads() / bp;
            if (v > R->bases_per_bp.load()) R->bases_per_bp.store(v);
            if (w > R->reads_per_bp.load()) R->reads_per_bp.store(w);
        }
        std::lock_guard<std::mutex> lk(R->mu);
        sh.pieces[pc] = std::move(b);
        if (!err.empty() && sh.error.empty()) sh.error = err;
        if (--sh.pieces_left == 0) { sh.state = 1; R->cv.notify_all(); }
    }
}

// worker w of W takes shards w, w + W, ...; several workers may share a device
void gpu_worker(Run *R, int g, int G, int device) {
    pb_params prm = R->prm;
    prm.device = device;
    int st = 0;
    if (R->feed_only) {
        // what a shard's pieces hold, in a form that does not depend on where the pieces were cut or who decoded them
        for (int s = g; s < (int)R->shards.size(); s += G) {
            Shard &sh = R->shards[s];
            {
                std::unique_lock<std::mutex> lk(R->mu);
                R->cv.wait(lk, [&] { return sh.state >= 1; });
            }
            uint64_t hp = 1469598103934665603ULL, hm = hp, hc = hp, sq = 0, ss = 0;
            int64_t nr = 0, nc = 0;
            auto fnv = [](uint64_t h, const void *v, size_t n) { const unsigned char *b = (const unsigned char *)v; for (size_t i = 0; i < n; ++i) h = (h ^ b[i]) * 1099511628211ULL; return h; };
            for (pbio::Batch &b : sh.pieces) {
                nr += b.n_reads(); nc += (int64_t)b.cigar.size();
                hp = fnv(hp, b.pos.data(), 4 * b.pos.size()); hm = fnv(hm, b.meta.data(), 4 * b.meta.size()); hc = fnv(hc, b.cigar.data(), 4 * b.cigar.size());
                for (size_t i = 0; i < b.qual.size(); ++i) sq += b.qual.data()[i];
                for (size_t i = 0; i < b.seq4.size(); ++i) ss += b.seq4.data()[i];
            }
            char line[256];
            snprintf(line, sizeof line, "%d\t%d\t%lld\t%lld\t%016llx\t%016llx\t%016llx\t%llu\t%llu\n", sh.w0, sh.w1, (long long)nr, (long long)nc,
                     (unsigned long long)hp, (unsigned long long)hm, (unsigned long long)hc, (unsigned long long)sq, (unsigned long long)ss);
            if (sh.error.empty()) sh.text = line;
            for (pbio::Batch &b : sh.pieces) R->give_batch(std::move(b));
            sh.pieces.clear();
            std::lock_guard<std::mutex> lk(R->mu);
            sh.state = 2;
            R->cv.notify_all();
        }
        return;
    }
    R->tables_ready.wait();
    pb_errmod_tables tb;
    tb.fk = R->fk.data(); tb.beta = R->beta.data(); tb.lhet = R->lhet.data();
    pb_ctx *ctx = pb_create(&prm, &tb, &st);
    std::string err;
    if (!ctx) err = std::string("cannot initialise GPU ") + std::to_string(device) + ": " + pb_last_error(nullptr);
    else if (pb_set_contig(ctx, R->tid, R->ref.data(), (int64_t)R->ref.size()) != PB_OK) err = pb_last_error(ctx);
    else if (pb_set_snn_perms(ctx, R->opt.snn_perms, R->opt.seed) != PB_OK) err = pb_last_error(ctx);
    std::vector<const char *> pops, smps;
    for (auto &s : R->st.pops) pops.push_back(s.c_str());
    for (auto &s : R->st.samples) smps.push_back(s.c_str());
    pb_print_opts po;
    po.chrom = R->hdr.names[R->tid].c_str();
    po.pop_names = pops.data(); po.sample_names = smps.data();
    po.min_sites = R->opt.min_sites; po.min_snps = R->opt.min_snps;
    po.jc = R->opt.dist == "jc"; po.snp_output = R->opt.output;
    po.ref_name = R->ref_name.c_str();
    std::vector<char> line(1 << 16);
    for (int s = g; s < (int)R->shards.size(); s += G) {
        Shard &sh = R->shards[s];
        {
            std::unique_lock<std::mutex> lk(R->mu);
            R->cv.wait(lk, [&] { return sh.state >= 1; });
        }
        if (err.empty() && sh.error.empty()) {
            pb_region_result res;
            pb_region_extras ext;
            pb_region_fst fst;
            int rc = pb_region_begin(ctx, R->analysis, sh.w1 - sh.w0, &R->wb[sh.w0], &R->we[sh.w0]);
            {
                int64_t nr = 0, nc = 0, nb = 0;
                for (pbio::Batch &b : sh.pieces) { nr += b.n_reads(); nc += (int64_t)b.cigar.size(); nb += (int64_t)b.qual.size(); }
                if (rc == PB_OK) rc = pb_region_reserve(ctx, nr, nc, nb);        // the device arrays once, not piece by piece
            }
            for (pbio::Batch &b : sh.pieces) {
                // the copies are asynchronous (the batches are page-locked and stay alive until the region is done)
                if (rc != PB_OK || b.n_reads() == 0) continue;
                pb_read_batch rb;
                rb.n_reads = b.n_reads(); rb.n_cigar = (int64_t)b.cigar.size(); rb.n_bases = (int64_t)b.qual.size();
                static const uint32_t zero = 0;
                rb.pos = b.pos.data(); rb.meta = b.meta.data(); rb.cig_off = b.cig_off.data();
                rb.cigar = b.cigar.empty() ? &zero : b.cigar.data();
                rb.base_off = b.base_off.data(); rb.seq4 = b.seq4.data(); rb.qual = b.qual.data();
                rc = R->pinned ? pb_push_batch_async(ctx, &rb) : pb_push_batch(ctx, &rb);
            }
            if (rc == PB_OK) rc = pb_region_end(ctx, &res);
            if (rc == PB_OK) rc = pb_region_get_extras(ctx, &ext);
            if (rc == PB_OK) rc = pb_region_get_fst(ctx, &fst);
            auto format = [&](int w) {
                return (R->analysis & PB_AN_FST) ? pb_format_window_fst(ctx, &res, &ext, &fst, w, R->analysis, &po, line.data(), (int64_t)line.size())
                                                 : pb_format_window_ext(ctx, &res, &ext, w, R->analysis, &po, line.data(), (int64_t)line.size());
            };
            if (rc != PB_OK) sh.error = pb_last_error(ctx);
            else
                for (int w = 0; w < res.n_windows; ++w) {
                    int64_t k = format(w);
                    if (k >= (int64_t)line.size()) { line.resize((size_t)k + 16); k = format(w); }
                    if (k < 0) { sh.error = "formatting failed"; break; }
                    sh.text.append(line.data(), (size_t)k);
                }
        } else if (sh.error.empty()) sh.error = err;
        for (pbio::Batch &b : sh.pieces) R->give_batch(std::move(b));       // (pb_region_end has waited for the copies)
        sh.pieces.clear();
        std::lock_guard<std::mutex> lk(R->mu);
        sh.state = 2;
        R->cv.notify_all();
    }
    if (ctx) pb_destroy(ctx);
}

}  // namespace

int main(int argc, char **argv) {
    if (argc < 2) {
        fprintf(stderr, "Program: popbam (B200 path; %s)\nUsage:   popbam <command> [options] <in.bam> [region]\n"
                        "Commands: snp haplo diverge tree nucdiv ld sfs   (and: index <in.bam>)\n", pb_version());
        return 1;
    }
    if (!strcmp(argv[1], "_fetch")) {
        // test hook (no GPU needed): popbam _fetch <in.bam> <region> <out.bin> dumps the host feeder's batch for the region
        if (argc < 5) return 2;
        try {
            pbio::BgzfFile bam; bam.open(argv[2]);
            pbio::BamHeader hdr = pbio::read_header(bam);
            pbio::SampleTable st = pbio::build_samples(hdr.text, argv[2]);
            pbio::BamIndex idx; idx.load(std::string(argv[2]) + ".bai", hdr.names.size());
            int tid, beg, end;
            if (!pbio::parse_region(hdr, argv[3], &tid, &beg, &end)) fatal(std::string("Bad genome coordinates: ") + argv[3]);
            pbio::Batch b;
            // popbam _fetch <in.bam> <region> <out.bin> [pieces]: with a piece count the region is fetched as that many
            // pieces (pbio::fetch_piece), appended to one batch in order -- it must equal the single fetch
            const int pieces = argc > 5 ? atoi(argv[5]) : 0;
            if (pieces <= 0) pbio::fetch_region(bam, idx, st, tid, beg, end, b);
            else
                for (int i = 0; i < pieces; ++i) {
                    const int32_t lo = (int32_t)(beg + (int64_t)(end - beg) * i / pieces), hi = (int32_t)(beg + (int64_t)(end - beg) * (i + 1) / pieces);
                    if (hi > lo || i == 0) pbio::fetch_piece(bam, idx, st, tid, beg, end, lo, hi, b);
                }
            FILE *f = fopen(argv[4], "wb");
            if (!f) return 2;
            const int64_t hdrv[6] = {b.n_reads(), (int64_t)b.cigar.size(), (int64_t)b.qual.size(), tid, beg, end};
            fwrite(hdrv, 8, 6, f);
            fwrite(b.pos.data(), 4, b.pos.size(), f); fwrite(b.meta.data(), 4, b.meta.size(), f);
            fwrite(b.cig_off.data(), 4, b.cig_off.size(), f); fwrite(b.cigar.data(), 4, b.cigar.size(), f);
            fwrite(b.base_off.data(), 4, b.base_off.size(), f); fwrite(b.seq4.data(), 1, b.seq4.size(), f);
            fwrite(b.qual.data(), 1, b.qual.size(), f);
            fclose(f);
            printf("samples:"); for (auto &x : st.samples) printf(" %s", x.c_str());
            printf("\npops:"); for (size_t i = 0; i < st.pops.size(); ++i) printf(" %s=%llx", st.pops[i].c_str(), (unsigned long long)st.pop_mask[i]);
            printf("\n");
        } catch (const pbio::Error &e) { fatal(e.msg); }
        return 0;
    }
    if (!strcmp(argv[1], "index")) {
        // not a subcommand of the reference's command line (its bam_index_build, bam_index.c:641, is never exposed):
        // popbam index <in.bam> writes <in.bam>.bai, which every analysis needs (popbam.cpp:130)
        if (argc < 3) { fprintf(stderr, "Usage:   popbam index <in.bam>\n"); return 1; }
        try {
            pbio::BgzfFile bam;
            bam.open(argv[2]);
            const long long n = pbio::build_bai(bam, std::string(argv[2]) + ".bai");
            fprintf(stderr, "[popbam index] %lld records\n", n);
        } catch (const pbio::Error &e) { fatal(e.msg); }
        return 0;
    }
    if (!strcmp(argv[1], "_inflate")) {
        // test hook: popbam _inflate <in.bam> <out.bin> writes the concatenated uncompressed BGZF stream
        if (argc < 4) return 2;
        try {
            pbio::BgzfFile bam; bam.open(argv[2]);
            FILE *f = fopen(argv[3], "wb");
            if (!f) return 2;
            std::vector<uint8_t> out;
            uint64_t off = 0;
            for (;;) { const uint32_t c = bam.inflate_block(off, out); if (!c) break; off += c; fwrite(out.data(), 1, out.size(), f); }
            fclose(f);
        } catch (const pbio::Error &e) { fatal(e.msg); }
        return 0;
    }
    Run R;
    if (!strcmp(argv[1], "_feed")) {
        // test hook (no GPU needed): popbam _feed <options and arguments of nucdiv> runs the whole host side -- shards, pieces,
        // decode threads, batch pool, workers in shard order -- and prints one line per shard of what the workers were
        // handed (windows, reads, CIGAR operations, hashes of pos / meta / cigar, byte sums of qual / seq4)
        static char nucdiv[] = "nucdiv";
        argv[1] = nucdiv;
        R.feed_only = true;
    }
    R.opt = parse(argc, argv);
    Options &o = R.opt;
    if (o.positional.size() < 2) { usage(o.cmd.c_str()); fatal("Need to specify BAM file name"); }
    const std::string bamfile = o.positional[0], region = o.positional[1];
    if (o.reffile.empty()) fatal("Need to specify fastA reference file");
    if ((o.cmd == "diverge" || o.cmd == "tree") && o.dist != "pdist" && o.dist != "jc") fatal(o.dist + " is not a valid distance option");
    try {
        { std::ifstream t(bamfile); if (!t) fatal("Specified input file: " + bamfile + " does not exist"); }
        { std::ifstream t(o.reffile); if (!t) fatal("Specified reference file: " + o.reffile + " does not exist"); }
        // the error-model tables take ~0.25 s of host arithmetic: build them while the files are opened and CUDA comes up
        R.fk.resize(256); R.beta.resize((size_t)64 * 256 * 256); R.lhet.resize(65536);
        // (cached on disk after the first run on a machine: pb_errmod_tables_cached)
        if (!R.feed_only) R.tables_ready = std::async(std::launch::async, [&R]() { pb_errmod_tables_cached(R.fk.data(), R.beta.data(), R.lhet.data(), nullptr); }).share();
        R.bam.open(bamfile);
        R.hdr = pbio::read_header(R.bam);
        std::string text = R.hdr.text;
        if (o.has_h) {      // -h: take the header text (sample / population definitions) from a file (popbam.cpp:119-127)
            std::ifstream hin(o.headfile);
            if (!hin) fatal("Cannot read header file " + o.headfile);
            std::stringstream ss; ss << hin.rdbuf(); text = ss.str();
        }
        R.st = pbio::build_samples(text, bamfile);
        if (o.cmd == "tree") {     // get_refid (pop_utils.cpp:463-500): the first AS: tag of the header names the reference taxon
            const size_t at = R.hdr.text.find("AS:");
            if (at == std::string::npos) fatal("Unable to parse reference sequence name\nBe sure the AS tag is defined in the sequence dictionary");
            size_t e = at + 3;
            while (e < R.hdr.text.size() && R.hdr.text[e] && R.hdr.text[e] != '\t' && R.hdr.text[e] != '\n') ++e;
            R.ref_name = R.hdr.text.substr(at + 3, e - (at + 3));
        }
        {
            // <bam>.bai, else <bam without its extension>.bai (bam_index_load_local, bam_index.c:552-560)
            std::string bai = bamfile + ".bai";
            std::ifstream t(bai);
            const size_t dot = bamfile.rfind('.');
            if (!t && dot != std::string::npos && bamfile.compare(dot, std::string::npos, ".bam") == 0) {
                std::ifstream t2(bamfile.substr(0, dot) + ".bai");
                if (t2) bai = bamfile.substr(0, dot) + ".bai";
            }
            R.idx.load(bai, R.hdr.names.size());
        }
        if (!pbio::parse_region(R.hdr, region, &R.tid, &R.beg, &R.end)) fatal("Bad genome coordinates: " + region);
        R.ref = pbio::fetch_contig(o.reffile, R.hdr.names[R.tid]);
    } catch (const pbio::Error &e) { fatal(e.msg); }

    // parameters == the popbamData fields the path reads
    pb_params &p = R.prm;
    memset(&p, 0, sizeof p);
    p.n_samples = (int)R.st.samples.size(); p.n_pops = (int)R.st.pops.size();
    for (int i = 0; i < 64; ++i) { p.pop_mask[i] = R.st.pop_mask[i]; p.pop_nsmpl[i] = R.st.pop_nsmpl[i]; }
    p.min_depth = o.min_depth; p.max_depth = o.max_depth; p.min_rmsQ = o.min_rmsQ; p.min_snpQ = o.min_snpQ;
    p.min_mapQ = o.min_mapQ; p.min_baseQ = o.min_baseQ;
    p.min_freq = o.min_freq2 ? 2 : 1;
    if (o.illumina) p.flags |= PB_FLAG_ILLUMINA;
    if (o.het) p.flags |= PB_FLAG_HETEROZYGOTE;
    if (o.substitute) p.flags |= PB_FLAG_SUBSTITUTE;
    const bool uses_outgroup = o.has_p && (o.cmd == "sfs" || o.cmd == "diverge" || o.cmd == "snp");
    if (uses_outgroup) {
        int found = -1;
        for (int i = 0; i < p.n_samples; ++i) if (R.st.samples[i] == o.outgroup) found = i;   // last match wins, as in the reference
        if (found < 0) fatal("Specified outgroup " + o.outgroup + " not found");
        p.outidx = found; p.flags |= PB_FLAG_OUTGROUP;
    }
    if (o.cmd == "nucdiv") R.analysis = PB_AN_NUCDIV;
    else if (o.cmd == "sfs") R.analysis = PB_AN_SFS;
    else if (o.cmd == "ld") R.analysis = o.output == 1 ? PB_AN_LD_OMEGA : o.output == 2 ? PB_AN_LD_WALL : PB_AN_LD_ZNS;
    else if (o.cmd == "diverge") R.analysis = o.output == 1 ? PB_AN_DIVERGE_POP : PB_AN_DIVERGE_IND;
    else if (o.cmd == "haplo") R.analysis = o.output == 1 ? PB_AN_HAPLO_EHHS : o.output == 2 ? PB_AN_HAPLO_DXY : PB_AN_HAPLO_K;
    else if (o.cmd == "tree") R.analysis = PB_AN_TREE;
    else R.analysis = PB_AN_SNP;
    if (o.output < 0 || o.output > 2) fatal("invalid output option");
    if (o.extra_stats) R.analysis |= o.cmd == "nucdiv" ? PB_AN_THETA_W : o.cmd == "sfs" ? PB_AN_FULI : PB_AN_LD_DPRIME;
    if (o.fst) R.analysis |= PB_AN_FST;

    // window grid of the region, then shards = runs of whole windows
    const int64_t nw = pb_window_grid(R.beg, R.end, o.window ? o.win_size : 0, 0, nullptr, nullptr);
    if (nw < 1) return 0;       // region shorter than one window: the reference's loop does not execute
    R.wb.resize((size_t)nw); R.we.resize((size_t)nw);
    pb_window_grid(R.beg, R.end, o.window ? o.win_size : 0, nw, R.wb.data(), R.we.data());
    const int64_t shard_bp = std::max<int64_t>(1, (int64_t)(o.shard_mb * 1e6));
    for (int w = 0; w < (int)nw;) {
        int e = w + 1;
        while (e < (int)nw && (int64_t)R.we[e] - R.wb[w] <= shard_bp) ++e;
        Shard sh; sh.w0 = w; sh.w1 = e;
        R.shards.push_back(std::move(sh));
        w = e;
    }
    const int G = std::max(1, o.gpus);
    const int D = o.threads > 0 ? o.threads : std::max(2u, std::min(32u, std::thread::hardware_concurrency()));
    // decode work items: every shard in pieces, about four per thread over the region, between 50 kb and 1 Mb long
    {
        const int64_t region_len = std::max<int64_t>(1, (int64_t)R.we.back() - R.wb.front());
        const int64_t piece_bp = std::max<int64_t>(50000, std::min<int64_t>(1000000, region_len / (4 * (int64_t)D)));
        for (size_t si = 0; si < R.shards.size(); ++si) {
            Shard &sh = R.shards[si];
            const int64_t lo = R.wb[sh.w0], hi = R.we[sh.w1 - 1];
            const int np = (int)std::max<int64_t>(1, (hi - lo + piece_bp - 1) / piece_bp);
            for (int i = 0; i < np; ++i) {
                const int32_t a = (int32_t)(lo + (hi - lo) * i / np), b = (int32_t)(lo + (hi - lo) * (i + 1) / np);
                if (b > a || i == 0) { sh.cuts.push_back({a, b}); R.items.push_back({(int)si, (int)sh.cuts.size() - 1}); }
            }
            sh.pieces.resize(sh.cuts.size());
            sh.pieces_left = (int)sh.cuts.size();
        }
    }
    {
        // Page-locked batches (pb_host_alloc) let the copies to the device run asynchronously, but locking the pages costs
        // more than it saves here: measured on the 5 Mb / 1.2 GB BAM of the bench workload, 13.4 s with page-locked batches
        // against 3.1 s with ordinary memory (the command line is bound by inflate + decode at ~1.7 GB/s of batch bytes, far
        // below PCIe).  So they are opt-in: POPBAM_B200_PINNED=1.
        const char *e = getenv("POPBAM_B200_PINNED");
        R.pinned = e && *e == '1';
        if (R.feed_only) R.pinned = false;
        if (R.pinned) pbio::set_batch_allocator(pb_host_alloc, pb_host_free);
    }
    // two contexts (host threads) per GPU: one shard's host->device copy runs beside another shard's kernels
    const int W = 2 * G;
    // every decode thread can have a shard in hand and one waiting (a decoded 50 kb shard of the bench workload is 34 MB)
    R.max_ahead = W + 2;       // shards decoded ahead of the printer (a decoded 2 Mb shard of the bench workload is 1 GB of host memory)

    if (o.cmd == "snp" && o.output == 2) {      // print_ms_header (pop_snp.cpp:305-317)
        printf("ms %d %lld -t 5.0 ", p.n_samples, (long long)nw);
        if (p.n_pops > 1) {
            printf("-I %d ", p.n_pops);
            for (int i = 0; i < p.n_pops; ++i) printf("%d ", (int)p.pop_nsmpl[i]);
        }
        printf("\n1350154902\n\n");
    }

    std::vector<std::thread> th;
    for (int i = 0; i < D; ++i) th.emplace_back(decode_worker, &R);
    for (int w = 0; w < W; ++w) th.emplace_back(gpu_worker, &R, w, W, w % G);
    int rc = 0;
    for (size_t s = 0; s < R.shards.size(); ++s) {
        Shard &sh = R.shards[s];
        {
            std::unique_lock<std::mutex> lk(R.mu);
            R.cv.wait(lk, [&] { return sh.state == 2; });
        }
        if (!sh.error.empty()) { fflush(stdout); fprintf(stderr, "popbam runtime error:\n%s\nExiting program\n", sh.error.c_str()); rc = 1; }
        else fwrite(sh.text.data(), 1, sh.text.size(), stdout);
        sh.text.clear(); sh.text.shrink_to_fit();
        {
            std::lock_guard<std::mutex> lk(R.mu);
            R.printed = (int)s + 1;
            R.cv.notify_all();
        }
        if (rc) { fflush(stdout); _Exit(EXIT_FAILURE); }
    }
    for (auto &t : th) t.join();
    fflush(stdout);
    return rc;
}
