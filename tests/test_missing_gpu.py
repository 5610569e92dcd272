"""pi and dxy over sites with missing calls on the GPU (PB_AN_NUCDIV_MISSING: k_nucdiv_missing) and `popbam nucdiv --missing`
against tests/missing_oracle.c, which tests/test_missing_host.py pins to a numpy restatement of the definition and to the
reference's nucdiv sums.  Integers and doubles exactly, on both pileup paths: the counting path's coverage masks at partly
covered positions are compared with the oracle's here for the first time."""
import os
import subprocess

import numpy as np
import pytest

import pbtest
import popbam_b200
from cases import CASES
from test_abba_host import ABBA, abba_arrays, assert_abba_same, default_triples, regrouped
from test_extra_stats_host import EXE, EXT
from test_fst_host import FST, assert_fst_same, fst_arrays
from test_garud_host import GARUD, assert_garud_same, garud_arrays
from test_gpu_parity import assert_same
from test_missing_host import (ALL_FIXTURES, AN, EMIT_CB, MISSING, VARIANTS, OracleMissing, assert_missing_same, fixture, missing_arrays,
                               oracle_cb)
from test_spectrum_host import SPECTRUM, fixture_sets, spectrum_arrays

pytestmark = pytest.mark.gpu
WINDOWS = [200, 1000, 10000, 0]          # 0: one window over the whole contig (-w 0)


def gpu_missing(ctx):
    return missing_arrays(ctx.nucdiv_missing, ctx.res.n_windows, ctx.res.n_pops)


def want_missing(fx, p, wb, we):
    cb, span_beg, _ = oracle_cb(fx, p, wb, we)
    om = OracleMissing(p, cb, wb, we, span_beg)
    a = om.arrays
    om.close()
    return a


def new_context(p, classic=False):
    if not classic:
        return popbam_b200.Context(p)
    old = os.environ.get("POPBAM_B200_PILEUP")
    os.environ["POPBAM_B200_PILEUP"] = "classic"          # read when the context is created
    try:
        return popbam_b200.Context(p)
    finally:
        if old is None:
            del os.environ["POPBAM_B200_PILEUP"]
        else:
            os.environ["POPBAM_B200_PILEUP"] = old


def run(fx, p, an, wb, we, ctx=None):
    ctx = ctx or popbam_b200.Context(p)
    ctx.set_contig(0, fx.ref())
    ctx.region_begin(an, wb, we)
    ctx.push_batch(fx.batch())
    ctx.region_end()
    return ctx


@pytest.mark.parametrize("variant", list(VARIANTS))
@pytest.mark.parametrize("fxname", ALL_FIXTURES)
def test_counting_path_arrays_match_oracle(fxname, variant):
    fx = fixture(fxname)
    p = fx.params(flags=VARIANTS[variant])
    ctx = popbam_b200.Context(p)
    ctx.set_contig(0, fx.ref())
    for win in WINDOWS:
        wb, we = pbtest.window_grid(0, fx.contig_len, win)
        ctx.region_begin(MISSING | AN["NUCDIV"], wb, we)
        ctx.push_batch(fx.batch())
        ctx.region_end()
        assert ctx.path() == 1, win
        assert_missing_same(gpu_missing(ctx), want_missing(fx, p, wb, we))
    ctx.close()


# the single-kernel pileup, reached three ways: forced, by a depth cap that binds, and by asking for the per-cell words
SINGLE = {"classic": (True, {}), "cap": (False, dict(max_depth=4)), "emit_cb": (False, dict(flags=EMIT_CB))}


@pytest.mark.parametrize("how", list(SINGLE))
@pytest.mark.parametrize("variant", list(VARIANTS))
@pytest.mark.parametrize("fxname", ["c1", "edge", "n64", "wideq", "low4", "low64"])
def test_single_kernel_path_arrays_match_oracle(fxname, variant, how):
    fx = fixture(fxname)
    classic, kw = SINGLE[how]
    kw = dict(kw)
    kw["flags"] = kw.get("flags", 0) | VARIANTS[variant]
    p = fx.params(**kw)
    ctx = new_context(p, classic)
    ctx.set_contig(0, fx.ref())
    for win in (1000, 0):
        wb, we = pbtest.window_grid(0, fx.contig_len, win)
        ctx.region_begin(MISSING, wb, we)
        ctx.push_batch(fx.batch())
        ctx.region_end()
        assert ctx.path() == 0, (how, win)
        assert_missing_same(gpu_missing(ctx), want_missing(fx, p, wb, we))
    ctx.close()


@pytest.mark.parametrize("fxname", ["low4", "n64"])
def test_async_relaunch_and_later_regions_equal_the_first(fxname):
    fx = fixture(fxname)
    p = fx.params()
    wb, we = pbtest.window_grid(0, fx.contig_len, 200)
    want = want_missing(fx, p, wb, we)
    ctx = run(fx, p, MISSING | AN["NUCDIV"], wb, we)
    assert_missing_same(gpu_missing(ctx), want)
    for _ in range(2):      # the context has learnt the region's shape: these are enqueued asynchronously
        ctx.region_begin(MISSING | AN["NUCDIV"], wb, we)
        ctx.push_batch(fx.batch())
        ctx.launch()
        ctx.wait()
        assert_missing_same(gpu_missing(ctx), want)
    for _ in range(2):      # relaunches on the resident reads: the arrays are zeroed again every time
        ctx.relaunch()
        ctx.wait()
        assert_missing_same(gpu_missing(ctx), want)
    ctx.region_begin(AN["NUCDIV"], wb, we)      # a region without the bit returns no arrays
    ctx.push_batch(fx.batch())
    ctx.region_end()
    assert all(len(a) == 0 for a in gpu_missing(ctx).values())
    ctx.close()


@pytest.mark.parametrize("fxname", ["c1", "ld", "n64", "low4"])
def test_one_pass_with_everything_equals_the_bit_alone(fxname):
    fx = fixture(fxname)
    p, _ = regrouped(fx, fxname if fxname in ("c1", "ld", "n64") else "c1", flags=pbtest.FLAG["OUTGROUP"], outidx=fx.n_samples - 1)
    triples = default_triples(p.n_pops, p.n_pops - 1)
    sets = fixture_sets(p.n_pops)
    wb, we = pbtest.window_grid(0, fx.contig_len, 1000)

    def ctx_with_lists():
        c = popbam_b200.Context(p)
        c.set_abba(p.n_pops - 1, triples)
        c.set_spectra(sets)
        return c
    everything = 0xfff | EXT | FST | ABBA | GARUD | SPECTRUM
    one = run(fx, p, everything | MISSING, wb, we, ctx_with_lists())
    rest = run(fx, p, everything, wb, we, ctx_with_lists())
    alone = run(fx, p, MISSING, wb, we)
    assert_same(pbtest.result_arrays(one.res), pbtest.result_arrays(rest.res), list(pbtest.BY_AN))
    assert_fst_same(fst_arrays(one.fst, one.res), fst_arrays(rest.fst, rest.res))
    assert_abba_same(abba_arrays(one.abba, one.res), abba_arrays(rest.abba, rest.res))
    assert_garud_same(garud_arrays(one.garud, one.res), garud_arrays(rest.garud, rest.res))
    assert all(np.array_equal(a, b) for a, b in zip(spectrum_arrays(one.spectrum, one.res), spectrum_arrays(rest.spectrum, rest.res)))
    assert_missing_same(gpu_missing(one), gpu_missing(alone))
    assert_missing_same(gpu_missing(alone), want_missing(fx, p, wb, we))
    for c in (one, rest, alone):
        c.close()


# ---------------------------------------------------------------------------------------------------------------------
# command line

@pytest.fixture(scope="module")
def files(tmp_path_factory):
    d = tmp_path_factory.mktemp("cli_missing_gpu")
    return d, {name: fixture(name).write_files(d / name) for name in ("c1", "low4", "n64")}


PI_HEAD = "pop\tchromosome\twindow_pos_1\twindow_pos_2\tavg_pi\tno_sites\tcount_diffs\tcount_comparisons\tcount_missing\n"
DXY_HEAD = "pop1\tpop2\tchromosome\twindow_pos_1\twindow_pos_2\tavg_dxy\tno_sites\tcount_diffs\tcount_comparisons\tcount_missing\n"


def cli(argv, files, name="c1"):
    d, fs = files
    bam, fa = fs[name]
    r = subprocess.run([str(EXE), "nucdiv"] + argv + ["-f", fa, bam, "chr1"], stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    assert r.returncode == 0, r.stderr.decode()
    return r.stdout.decode()


def read_files(prefix):
    return open(str(prefix) + "_pi.txt").read(), open(str(prefix) + "_dxy.txt").read()


def oracle_files(fx, p, wb, we, chrom="chr1"):
    cb, span_beg, _ = oracle_cb(fx, p, wb, we)
    om = OracleMissing(p, cb, wb, we, span_beg)
    t = PI_HEAD + om.text(0, chrom, fx.pop_names), DXY_HEAD + om.text(1, chrom, fx.pop_names)
    om.close()
    return t


NUCDIV_C1 = [c for c in CASES if c[0] in ("nucdiv_c1", "nucdiv_c1_k", "nucdiv_c1_now")]


@pytest.mark.parametrize("case", NUCDIV_C1, ids=[c[0] for c in NUCDIV_C1])
def test_cli_files_equal_oracle_and_stdout_is_golden(case, files):
    d, _ = files
    fx, p, an, wb, we, _ = pbtest.case_setup(case)
    prefix = d / case[0]
    out = cli(case[2][1:] + ["--missing", str(prefix)], files)
    assert out == pbtest.golden_text(case)
    assert read_files(prefix) == oracle_files(fx, p, wb, we)       # every window, whatever -k says


@pytest.mark.parametrize("name,win", [("low4", "1"), ("n64", "5"), ("low4", None)])
def test_cli_files_on_partly_covered_data(name, win, files):
    d, _ = files
    fx = fixture(name)
    p = fx.params()
    wb, we = pbtest.window_grid(0, fx.contig_len, int(win) * 1000 if win else 0)
    prefix = d / ("%s_%s" % (name, win))
    wargs = ["-w", win] if win else []
    out = cli(wargs + ["--missing", str(prefix)], files, name)
    assert out == cli(wargs, files, name)
    assert read_files(prefix) == oracle_files(fx, p, wb, we)


def test_cli_files_do_not_depend_on_shards_or_threads_and_combine_with_other_options(files):
    d, _ = files
    base = cli(["-w", "1", "--missing", str(d / "base")], files, "low4")
    want = read_files(d / "base")
    for i, extra in enumerate((["--shard-mb", "0.004"], ["--shard-mb", "0.02"], ["--threads", "1"], ["--threads", "3", "--shard-mb", "0.002"])):
        assert cli(["-w", "1", "--missing", str(d / ("v%d" % i))] + extra, files, "low4") == base
        assert read_files(d / ("v%d" % i)) == want, extra
    for extra in (["--fst"], ["--extra-stats"], ["--fst", "--extra-stats", "--snn-perms", "10"]):
        with_missing = cli(["-w", "1", "--missing", str(d / "combo")] + extra, files, "low4")
        assert with_missing == cli(["-w", "1"] + extra, files, "low4"), extra
        assert read_files(d / "combo") == want, extra
