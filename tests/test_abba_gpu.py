"""ABBA-BABA on the GPU (PB_AN_ABBA: k_abba) against tests/abba_oracle.c, which tests/test_abba_host.py pins to a
Fraction restatement of the published formulas.  Integers exactly, doubles bit for bit."""
import ctypes as C
import subprocess

import numpy as np
import pytest

import pbtest
import popbam_b200
from cases import CASES, FIXTURES
from test_abba_host import (ABBA, AN, EXE, abba_arrays, assert_abba_same, c1_sample_pop, default_triples, oracle_abba,
                            oracle_abba_text, regrouped, regrouped_opts, write_regrouped_header)
from test_extra_stats_host import EXT, FLT_EXT, INT_EXT, ext_arrays
from test_fst_host import FST, assert_fst_same, fst_arrays
from test_gpu_parity import assert_same

pytestmark = pytest.mark.gpu
VARIANTS = {"plain": 0, "z": pbtest.FLAG["HETEROZYGOTE"]}


def run_abba(fx, p, an, wb, we, og, triples):
    ctx = popbam_b200.Context(p)
    ctx.set_contig(0, fx.ref())
    ctx.set_abba(og, triples)
    ctx.region_begin(an, wb, we)
    ctx.push_batch(fx.batch())
    ctx.region_end()
    return ctx


@pytest.mark.parametrize("variant", list(VARIANTS))
@pytest.mark.parametrize("fxname", list(FIXTURES))
def test_abba_arrays_match_oracle(fxname, variant):
    fx = pbtest.fixture(fxname)
    p, _ = regrouped(fx, fxname, flags=VARIANTS[variant])
    og = p.n_pops - 1
    wb, we = pbtest.window_grid(0, fx.contig_len, 10000)
    lists = [default_triples(p.n_pops, og)]
    lists.append(lists[0][::-1])
    lists.append([(t[1], t[0], t[2]) for t in lists[0][1::2]] + lists[0][::3])        # reordered, swapped P1 / P2
    ctx = run_abba(fx, p, ABBA, wb, we, og, lists[0])
    orc = pbtest.OracleRun(p, fx.batch(), fx.ref(), AN["NUCDIV"], wb, we)
    assert np.array_equal(pbtest.result_arrays(ctx.res)["seg_type"], pbtest.result_arrays(orc.res)["seg_type"])
    for k, triples in enumerate(lists):
        if k:
            ctx.set_abba(og, triples)
            ctx.region_begin(ABBA, wb, we)
            ctx.push_batch(fx.batch())
            ctx.region_end()
        assert ctx.abba.n_triples == len(triples) and ctx.abba.outgroup_pop == og
        assert [tuple(ctx.abba.triples[3 * i:3 * i + 3]) for i in range(len(triples))] == [tuple(t) for t in triples]
        want = oracle_abba(p, orc.res, og, triples)
        assert_abba_same(abba_arrays(ctx.abba, ctx.res), want)
        assert int((want["abba"] + want["baba"]).max()) > 0
    orc.close(); ctx.close()


@pytest.mark.parametrize("fxname", ["c1", "ld", "n64", "ldbig"])
def test_one_pass_with_everything_equals_separate_passes(fxname):
    fx = pbtest.fixture(fxname)
    p, _ = regrouped(fx, fxname)
    og = p.n_pops - 1
    triples = default_triples(p.n_pops, og)
    wb, we = pbtest.window_grid(0, fx.contig_len, 5000)
    one = run_abba(fx, p, 0xfff | EXT | FST | ABBA, wb, we, og, triples)
    ref = run_abba(fx, p, 0xfff, wb, we, og, triples)
    assert_same(pbtest.result_arrays(one.res), pbtest.result_arrays(ref.res), list(pbtest.BY_AN))
    ext = run_abba(fx, p, EXT | FST, wb, we, og, triples)
    a, b = ext_arrays(one.ext, one.res), ext_arrays(ext.ext, ext.res)
    for k in INT_EXT + FLT_EXT:
        assert a[k].shape == b[k].shape and np.array_equal(np.isnan(a[k]) if k in FLT_EXT else a[k], np.isnan(b[k]) if k in FLT_EXT else b[k]), k
        if k in FLT_EXT:
            assert np.array_equal(a[k][~np.isnan(a[k])], b[k][~np.isnan(b[k])]), k
    assert_fst_same(fst_arrays(one.fst, one.res), fst_arrays(ext.fst, ext.res))
    alone = run_abba(fx, p, ABBA, wb, we, og, triples)
    assert_abba_same(abba_arrays(one.abba, one.res), abba_arrays(alone.abba, alone.res))
    # a pass without PB_AN_ABBA returns no ABBA arrays
    for c in (ref, ext):
        assert c.abba.n_triples == 0 and all(v.size == 0 for v in abba_arrays(c.abba, c.res).values())
        assert not c.abba.triples and not c.abba.d
    for c in (one, ref, ext, alone):
        c.close()


def test_async_relaunch_and_later_regions_equal_the_first():
    fx = pbtest.fixture("n64")
    p, _ = regrouped(fx, "n64")
    og = p.n_pops - 1
    triples = default_triples(p.n_pops, og)
    wb, we = pbtest.window_grid(0, fx.contig_len, 2000)
    ctx = run_abba(fx, p, AN["NUCDIV"] | ABBA, wb, we, og, triples)
    first = abba_arrays(ctx.abba, ctx.res)
    orc = pbtest.OracleRun(p, fx.batch(), fx.ref(), AN["NUCDIV"], wb, we)
    assert_abba_same(first, oracle_abba(p, orc.res, og, triples))
    # second and third regions (the context has learnt the region's shape: these are enqueued asynchronously)
    for _ in range(2):
        ctx.region_begin(AN["NUCDIV"] | ABBA, wb, we)
        ctx.push_batch(fx.batch())
        ctx.launch()
        ctx.wait()
        assert_abba_same(abba_arrays(ctx.abba, ctx.res), first)
    # relaunches on the resident reads keep the region's triples, even after pb_set_abba
    ctx.set_abba(og, triples[:5])
    for _ in range(2):
        ctx.relaunch()
        ctx.wait()
        assert ctx.abba.n_triples == len(triples)
        assert_abba_same(abba_arrays(ctx.abba, ctx.res), first)
    # a new region takes the new list
    ctx.region_begin(ABBA, wb, we)
    ctx.push_batch(fx.batch())
    ctx.region_end()
    assert ctx.abba.n_triples == 5
    assert_abba_same(abba_arrays(ctx.abba, ctx.res), oracle_abba(p, orc.res, og, triples[:5]))
    orc.close(); ctx.close()


def test_set_abba_checks_its_arguments():
    fx = pbtest.fixture("c1")
    p, _ = regrouped(fx, "c1")
    ctx = popbam_b200.Context(p)
    ctx.set_contig(0, fx.ref())
    wb, we = pbtest.window_grid(0, fx.contig_len, 10000)
    L, h = ctx.L, ctx.h

    def rc(og, triples, n=None):
        flat = (C.c_int32 * max(1, 3 * len(triples)))(*[k for t in triples for k in t])
        return L.pb_set_abba(h, og, len(triples) if n is None else n, flat)
    # no list yet: PB_ERR_STATE
    assert L.pb_region_begin(h, ABBA, len(wb), wb.ctypes.data_as(C.POINTER(C.c_int32)), we.ctypes.data_as(C.POINTER(C.c_int32))) == -3
    assert rc(3, [(0, 1, 4)]) == -1 and rc(3, [(0, -1, 2)]) == -1 and rc(4, [(0, 1, 2)]) == -1
    assert rc(3, [(0, 1, 1)]) == -1 and rc(3, [(0, 1, 3)]) == -1 and rc(2, [(0, 1, 2)]) == -1
    assert rc(3, [(0, 1, 2)], n=-1) == -1 and rc(3, [(0, 1, 2)] * 1025) == -1
    assert rc(3, [(0, 1, 2)] * 1024) == 0
    assert L.pb_region_begin(h, ABBA, len(wb), wb.ctypes.data_as(C.POINTER(C.c_int32)), we.ctypes.data_as(C.POINTER(C.c_int32))) == 0
    ctx.push_batch(fx.batch())
    ctx.region_end()
    assert ctx.abba.n_triples == 1024
    assert rc(3, []) == 0          # cleared
    assert L.pb_region_begin(h, ABBA, len(wb), wb.ctypes.data_as(C.POINTER(C.c_int32)), we.ctypes.data_as(C.POINTER(C.c_int32))) == -3
    ctx.close()


# ---------------------------------------------------------------------------------------------------------------------
# command line

@pytest.fixture(scope="module")
def c1_files(tmp_path_factory):
    d = tmp_path_factory.mktemp("cli_abba_gpu")
    fx = pbtest.fixture("c1")
    bam, fa = fx.write_files(d / "c1")
    return bam, fa, write_regrouped_header(bam, d / "regrouped.sam", c1_sample_pop(fx))


def cli(argv, files, extra=()):
    bam, fa, hdr = files
    r = subprocess.run([str(EXE), "abba", "-w", "10", "-p", "og", "-h", hdr] + argv + list(extra) + ["-f", fa, bam, "chr1"],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    assert r.returncode == 0, r.stderr.decode()
    return r.stdout.decode()


def c1_oracle():
    case = [c for c in CASES if c[0] == "nucdiv_c1"][0]
    fx, _, an, wb, we, _ = pbtest.case_setup(case)
    p, names = regrouped(fx, "c1")
    o = regrouped_opts(fx, names)
    orc = pbtest.OracleRun(p, fx.batch(), fx.ref(), an, wb, we)
    return case, p, names, o, orc


def test_cli_abba_equals_oracle_text(c1_files):
    case, p, names, o, orc = c1_oracle()
    og = p.n_pops - 1
    got = cli([], c1_files)
    assert got == oracle_abba_text(p, orc.res, og, default_triples(p.n_pops, og), o)
    assert "D[P1-P2-P3]:" in got and "fdM[P2-P3-P1]:" in got
    # the first four columns are nucdiv's
    assert ["\t".join(r.split("\t")[:4]) for r in got.splitlines()] == \
        ["\t".join(r.split("\t")[:4]) for r in pbtest.golden_text(case).splitlines()]
    orc.close()


def test_cli_triple_selects_and_orders(c1_files):
    _, p, names, o, orc = c1_oracle()
    got = cli(["--triple", "P3,P1,P2", "--triple", "P2,P1,P3"], c1_files)
    assert got == oracle_abba_text(p, orc.res, p.n_pops - 1, [(2, 0, 1), (1, 0, 2)], o)
    assert got.splitlines()[0].split("\t")[4] == "S[P3-P1-P2]:"
    orc.close()


def test_cli_abba_text_does_not_depend_on_shards_or_threads(c1_files):
    want = cli([], c1_files)
    for extra in (["--shard-mb", "0.01"], ["--shard-mb", "0.02"], ["--threads", "1"]):
        assert cli(extra, c1_files) == want, extra
