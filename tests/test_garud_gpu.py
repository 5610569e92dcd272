"""Garud's H on the GPU (PB_AN_GARUD: k_garud) against tests/garud_oracle.c, which tests/test_garud_host.py pins to a numpy
restatement of the definition.  Integers exactly, doubles bit for bit."""
import subprocess

import numpy as np
import pytest

import pbtest
import popbam_b200
from cases import CASES, FIXTURES
from test_abba_gpu import run_abba
from test_abba_host import ABBA, abba_arrays, assert_abba_same, default_triples, regrouped
from test_extra_stats_host import EXE, EXT, FLT_EXT, INT_EXT, ext_arrays
from test_fst_host import FST, assert_fst_same, fst_arrays
from test_garud_host import AN, GARUD, assert_garud_same, garud_arrays, oracle_garud, oracle_garud_text
from test_gpu_parity import assert_same

pytestmark = pytest.mark.gpu
VARIANTS = {"plain": 0, "z": pbtest.FLAG["HETEROZYGOTE"]}


def run_region(ctx, fx, an, wb, we):
    ctx.region_begin(an, wb, we)
    ctx.push_batch(fx.batch())
    ctx.region_end()


@pytest.mark.parametrize("variant", list(VARIANTS))
@pytest.mark.parametrize("fxname", list(FIXTURES))
def test_garud_arrays_match_oracle(fxname, variant):
    fx = pbtest.fixture(fxname)
    p = fx.params(flags=VARIANTS[variant])
    ctx = popbam_b200.Context(p)
    ctx.set_contig(0, fx.ref())
    P = p.n_pops
    for win in (200, 1000, 10000):
        wb, we = pbtest.window_grid(0, fx.contig_len, win)
        run_region(ctx, fx, GARUD, wb, we)
        orc = pbtest.OracleRun(p, fx.batch(), fx.ref(), AN["NUCDIV"], wb, we)
        assert np.array_equal(pbtest.result_arrays(ctx.res)["seg_type"], pbtest.result_arrays(orc.res)["seg_type"])
        got, want = garud_arrays(ctx.garud, ctx.res), oracle_garud(p, orc.res)
        assert_garud_same(got, want)
        if win == 200 and fxname not in ("edge", "rg2"):
            # shared haplotypes, so the grouping and the top-three logic are exercised: in both ingroup populations, which
            # for n64 holds samples 32 .. 62 (the second word of each lane)
            n = np.tile([p.pop_nsmpl[k] for k in range(P)], ctx.res.n_windows)
            hit = ((got["n_hap"] < n) & (got["c2"] > 1)).reshape(-1, P).any(axis=0)
            assert hit[0] and hit[1], hit
        orc.close()
    ctx.close()


@pytest.mark.parametrize("fxname", ["c1", "ld", "n64", "ldbig"])
def test_one_pass_with_everything_equals_separate_passes(fxname):
    fx = pbtest.fixture(fxname)
    p, _ = regrouped(fx, fxname)
    og = p.n_pops - 1
    triples = default_triples(p.n_pops, og)
    wb, we = pbtest.window_grid(0, fx.contig_len, 1000)
    one = run_abba(fx, p, 0xfff | EXT | FST | ABBA | GARUD, wb, we, og, triples)
    ref = run_abba(fx, p, 0xfff, wb, we, og, triples)
    assert_same(pbtest.result_arrays(one.res), pbtest.result_arrays(ref.res), list(pbtest.BY_AN))
    ext = run_abba(fx, p, EXT | FST | ABBA, wb, we, og, triples)
    a, b = ext_arrays(one.ext, one.res), ext_arrays(ext.ext, ext.res)
    for k in INT_EXT + FLT_EXT:
        assert a[k].shape == b[k].shape and np.array_equal(np.isnan(a[k]) if k in FLT_EXT else a[k], np.isnan(b[k]) if k in FLT_EXT else b[k]), k
        if k in FLT_EXT:
            assert np.array_equal(a[k][~np.isnan(a[k])], b[k][~np.isnan(b[k])]), k
    assert_fst_same(fst_arrays(one.fst, one.res), fst_arrays(ext.fst, ext.res))
    assert_abba_same(abba_arrays(one.abba, one.res), abba_arrays(ext.abba, ext.res))
    alone = run_abba(fx, p, GARUD, wb, we, og, triples)
    assert_garud_same(garud_arrays(one.garud, one.res), garud_arrays(alone.garud, alone.res))
    orc = pbtest.OracleRun(p, fx.batch(), fx.ref(), AN["NUCDIV"], wb, we)
    assert_garud_same(garud_arrays(alone.garud, alone.res), oracle_garud(p, orc.res))
    # a pass without PB_AN_GARUD returns no Garud arrays
    for c in (ref, ext):
        assert all(v.size == 0 for v in garud_arrays(c.garud, c.res).values())
        assert not c.garud.n_hap and not c.garud.h1
    for c in (one, ref, ext, alone):
        c.close()
    orc.close()


def test_async_relaunch_and_later_regions_equal_the_first():
    fx = pbtest.fixture("n64")
    p = fx.params()
    wb, we = pbtest.window_grid(0, fx.contig_len, 200)
    ctx = popbam_b200.Context(p)
    ctx.set_contig(0, fx.ref())
    run_region(ctx, fx, AN["HAPLO_K"] | GARUD, wb, we)
    first = garud_arrays(ctx.garud, ctx.res)
    orc = pbtest.OracleRun(p, fx.batch(), fx.ref(), AN["NUCDIV"], wb, we)
    assert_garud_same(first, oracle_garud(p, orc.res))
    # second and third regions (the context has learnt the region's shape: these are enqueued asynchronously)
    for _ in range(2):
        ctx.region_begin(AN["HAPLO_K"] | GARUD, wb, we)
        ctx.push_batch(fx.batch())
        ctx.launch()
        ctx.wait()
        assert_garud_same(garud_arrays(ctx.garud, ctx.res), first)
    # relaunches on the resident reads
    for _ in range(2):
        ctx.relaunch()
        ctx.wait()
        assert_garud_same(garud_arrays(ctx.garud, ctx.res), first)
    orc.close(); ctx.close()


# ---------------------------------------------------------------------------------------------------------------------
# command line

@pytest.fixture(scope="module")
def c1_files(tmp_path_factory):
    d = tmp_path_factory.mktemp("cli_garud_gpu")
    return pbtest.fixture("c1").write_files(d / "c1")


def cli(argv, files):
    bam, fa = files
    r = subprocess.run([str(EXE), "haplo", "-w", "1"] + argv + ["-f", fa, bam, "chr1"], stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    assert r.returncode == 0, r.stderr.decode()
    return r.stdout.decode()


@pytest.mark.parametrize("o", [0, 1, 2])
def test_cli_garud_equals_oracle_text(o, c1_files):
    fx = pbtest.fixture("c1")
    an = {0: AN["HAPLO_K"], 1: AN["HAPLO_EHHS"], 2: AN["HAPLO_DXY"]}[o]
    p = fx.params()
    opts = fx.print_opts()
    wb, we = pbtest.window_grid(0, fx.contig_len, 1000)
    orc = pbtest.OracleRun(p, fx.batch(), fx.ref(), an, wb, we)
    got = cli(["-o", str(o), "--garud"], c1_files)
    assert got == oracle_garud_text(orc.text(an, opts), p, orc.res, opts)
    assert "nHap[popA]:" in got and "H2H1[out]:" in got
    # without the option: the reference's rows
    assert cli(["-o", str(o)], c1_files) == orc.text(an, opts)
    orc.close()


@pytest.mark.parametrize("case", [c for c in CASES if c[0] in ("hap0_c1", "hap1_c1", "hap2_c1")], ids=lambda c: c[0])
def test_cli_rows_without_garud_are_golden(case, c1_files):
    bam, fa = c1_files
    r = subprocess.run([str(EXE)] + list(case[2]) + ["-f", fa, bam, "chr1"], stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    assert r.returncode == 0 and r.stdout.decode() == pbtest.golden_text(case)
    with_garud = subprocess.run([str(EXE)] + list(case[2]) + ["--garud", "-f", fa, bam, "chr1"], stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    assert with_garud.returncode == 0
    k = 2 * 5 * pbtest.fixture("c1").n_pops
    assert ["\t".join(r.split("\t")[:-k]) for r in with_garud.stdout.decode().splitlines()] == pbtest.golden_text(case).splitlines()


def test_cli_garud_text_does_not_depend_on_shards_or_threads(c1_files):
    want = cli(["--garud"], c1_files)
    for extra in (["--shard-mb", "0.004"], ["--shard-mb", "0.02"], ["--threads", "1"], ["--threads", "3", "--shard-mb", "0.002"]):
        assert cli(["--garud"] + extra, c1_files) == want, extra
