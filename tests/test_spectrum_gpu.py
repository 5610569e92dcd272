"""Site frequency spectra on the GPU (PB_AN_SPECTRUM: k_spectrum) and `popbam sfs --jsfs` against tests/spectrum_oracle.c,
which tests/test_spectrum_host.py pins to a numpy restatement of the definition and to the reference's sfs rows.  Counts
exactly."""
import ctypes as C
import subprocess

import numpy as np
import pytest

import pbtest
import popbam_b200
from cases import CASES, FIXTURES
from popbam_b200 import capi
from test_abba_host import ABBA, abba_arrays, assert_abba_same, default_triples, regrouped
from test_extra_stats_host import EXE, EXT
from test_fst_host import FST, assert_fst_same, fst_arrays
from test_garud_host import GARUD, assert_garud_same, garud_arrays
from test_gpu_parity import assert_same
from test_spectrum_host import (AN, SPECTRUM, default_sets, fixture_params, fixture_sets, oracle_spectrum, pad, read_dadi, set_shape,
                                spectrum_arrays, window_sets)

pytestmark = pytest.mark.gpu
VARIANTS = {"plain": 0, "z": pbtest.FLAG["HETEROZYGOTE"]}


def run(fx, p, an, wb, we, sets, triples=None):
    ctx = popbam_b200.Context(p)
    ctx.set_contig(0, fx.ref())
    ctx.set_spectra(sets)
    if triples:
        ctx.set_abba(p.n_pops - 1, triples)
    ctx.region_begin(an, wb, we)
    ctx.push_batch(fx.batch())
    ctx.region_end()
    return ctx


def gpu_spectrum(ctx):
    return spectrum_arrays(ctx.spectrum, ctx.res)


@pytest.mark.parametrize("variant", list(VARIANTS))
@pytest.mark.parametrize("fxname", list(FIXTURES))
def test_spectrum_arrays_match_oracle(fxname, variant):
    fx = pbtest.fixture(fxname)
    for outgroup in (False, True):
        p = fixture_params(fx, outgroup)
        p.flags |= VARIANTS[variant]
        sets = fixture_sets(p.n_pops)
        ctx = popbam_b200.Context(p)
        ctx.set_contig(0, fx.ref())
        ctx.set_spectra(sets)
        for win in (200, 1000, 10000):
            wb, we = pbtest.window_grid(0, fx.contig_len, win)
            ctx.region_begin(SPECTRUM, wb, we)
            ctx.push_batch(fx.batch())
            ctx.region_end()
            orc = pbtest.OracleRun(p, fx.batch(), fx.ref(), AN["NUCDIV"], wb, we)
            assert np.array_equal(pbtest.result_arrays(ctx.res)["seg_type"], pbtest.result_arrays(orc.res)["seg_type"])
            counts, off, got_sets = gpu_spectrum(ctx)
            want, want_off = oracle_spectrum(p, orc.res, sets)
            assert np.array_equal(off, want_off) and np.array_equal(got_sets, [k for s in sets for k in pad(s)])
            assert ctx.spectrum.n_sets == len(sets) and ctx.spectrum.n_bins == want_off[-1]
            assert np.array_equal(counts, want)
            orc.close()
        ctx.close()


def regroup_64(fx):
    """n64's 63 ingroup samples as three populations of 21 (22 x 22 x 22 = 10 648 bins per 3-D set, so (A, B, C) and
    (C, B, A) need a group each) and the outgroup sample alone."""
    p = fx.params(flags=pbtest.FLAG["OUTGROUP"], outidx=63)
    for k in range(64):
        p.pop_mask[k], p.pop_nsmpl[k] = 0, 0
    for g, (s, m) in enumerate([(0, 21), (21, 21), (42, 21), (63, 1)]):
        p.pop_mask[g] = ((1 << m) - 1) << s
        p.pop_nsmpl[g] = m
    p.n_pops = 4
    return p


@pytest.mark.parametrize("fxname", ["n64", "ldbig"])
def test_three_population_sets_over_several_groups(fxname):
    fx = pbtest.fixture(fxname)
    p = regroup_64(fx)
    sets = [(0, 1, 2), (2, 1, 0)] + default_sets(4, 3) + [(1, 2, 0)]
    for win in (1000, 10000):
        wb, we = pbtest.window_grid(0, fx.contig_len, win)
        ctx = run(fx, p, SPECTRUM, wb, we, sets)
        orc = pbtest.OracleRun(p, fx.batch(), fx.ref(), AN["NUCDIV"], wb, we)
        counts, off, _ = gpu_spectrum(ctx)
        want, _ = oracle_spectrum(p, orc.res, sets)
        assert np.array_equal(counts, want)
        for x in window_sets(counts, off, p, sets, ctx.res.n_windows):
            assert np.array_equal(x[1], x[0].transpose(2, 1, 0)) and np.array_equal(x[-1], x[0].transpose(1, 2, 0))
        assert counts.reshape(ctx.res.n_windows, -1)[:, off[0] + 1:off[1]].sum() > 0       # segregating sites in the 3-D bins
        ctx.close(); orc.close()


def test_async_relaunch_and_later_regions_equal_the_first():
    fx = pbtest.fixture("n64")
    p = fixture_params(fx, True)
    sets = fixture_sets(p.n_pops)
    wb, we = pbtest.window_grid(0, fx.contig_len, 200)
    ctx = run(fx, p, AN["SFS"] | SPECTRUM, wb, we, sets)
    first = gpu_spectrum(ctx)
    orc = pbtest.OracleRun(p, fx.batch(), fx.ref(), AN["NUCDIV"], wb, we)
    assert np.array_equal(first[0], oracle_spectrum(p, orc.res, sets)[0])
    for _ in range(2):      # the context has learnt the region's shape: these are enqueued asynchronously
        ctx.region_begin(AN["SFS"] | SPECTRUM, wb, we)
        ctx.push_batch(fx.batch())
        ctx.launch()
        ctx.wait()
        assert all(np.array_equal(a, b) for a, b in zip(gpu_spectrum(ctx), first))
    # a new list applies to the regions that follow: relaunches keep the one their region began with
    ctx.set_spectra([(1, 0)])
    for _ in range(2):
        ctx.relaunch()
        ctx.wait()
        assert all(np.array_equal(a, b) for a, b in zip(gpu_spectrum(ctx), first))
    ctx.region_begin(SPECTRUM, wb, we)
    ctx.push_batch(fx.batch())
    ctx.region_end()
    counts, off, got_sets = gpu_spectrum(ctx)
    assert list(got_sets) == [1, 0, -1] and np.array_equal(counts, oracle_spectrum(p, orc.res, [(1, 0)])[0])
    orc.close(); ctx.close()


@pytest.mark.parametrize("fxname", ["c1", "ld", "n64"])
def test_one_pass_with_everything_equals_the_bit_alone(fxname):
    fx = pbtest.fixture(fxname)
    p, _ = regrouped(fx, fxname, flags=pbtest.FLAG["OUTGROUP"], outidx=fx.n_samples - 1)
    triples = default_triples(p.n_pops, p.n_pops - 1)
    sets = fixture_sets(p.n_pops)
    wb, we = pbtest.window_grid(0, fx.contig_len, 1000)
    one = run(fx, p, 0xfff | EXT | FST | ABBA | GARUD | SPECTRUM, wb, we, sets, triples)
    rest = run(fx, p, 0xfff | EXT | FST | ABBA | GARUD, wb, we, sets, triples)
    alone = run(fx, p, SPECTRUM, wb, we, sets)
    assert_same(pbtest.result_arrays(one.res), pbtest.result_arrays(rest.res), list(pbtest.BY_AN))
    assert_fst_same(fst_arrays(one.fst, one.res), fst_arrays(rest.fst, rest.res))
    assert_abba_same(abba_arrays(one.abba, one.res), abba_arrays(rest.abba, rest.res))
    assert_garud_same(garud_arrays(one.garud, one.res), garud_arrays(rest.garud, rest.res))
    assert all(np.array_equal(a, b) for a, b in zip(gpu_spectrum(one), gpu_spectrum(alone)))
    orc = pbtest.OracleRun(p, fx.batch(), fx.ref(), AN["NUCDIV"], wb, we)
    assert np.array_equal(gpu_spectrum(alone)[0], oracle_spectrum(p, orc.res, sets)[0])
    # a pass without PB_AN_SPECTRUM returns no spectrum
    sp = rest.spectrum
    assert sp.n_sets == 0 and sp.n_bins == 0 and not sp.sets and not sp.set_off and not sp.counts
    for c in (one, rest, alone):
        c.close()
    orc.close()


def test_set_spectra_errors():
    fx = pbtest.fixture("c1")
    p = fx.params()
    ctx = popbam_b200.Context(p)
    ctx.set_contig(0, fx.ref())
    wb, we = pbtest.window_grid(0, fx.contig_len, 10000)
    L = ctx.L

    def set_raw(flat, n=None):
        a = np.ascontiguousarray(flat, dtype=np.int32)
        return L.pb_set_spectra(ctx.h, len(a) // 3 if n is None else n, a.ctypes.data_as(C.POINTER(C.c_int32)))
    with pytest.raises(capi.PopbamError):
        ctx.region_begin(SPECTRUM, wb, we)          # no list yet: PB_ERR_STATE
    for bad in ([-1, -1, -1], [-1, 0, -1], [0, -1, 1], [0, 0, -1], [1, 2, 1], [3, -1, -1], [0, -2, -1], [0, 1, 3]):
        assert set_raw(bad) == -1, bad            # PB_ERR_ARG
    assert set_raw([0, -1, -1], n=-1) == -1
    assert set_raw([2, -1, -1] * 4097) == -1        # more than PB_MAX_SPECTRUM_SETS
    assert set_raw([0, 1, 2] * 5) == 0               # 6 x 6 x 2 = 72 bins per set
    assert set_raw([0, 1, 2] * 910) == 0            # 65 520 bins
    assert set_raw([0, 1, 2] * 911) == -1           # 65 592 bins: more than PB_MAX_SPECTRUM_BINS
    ctx.set_spectra([(0,), (1, 2)])
    ctx.region_begin(SPECTRUM, wb, we)
    ctx.push_batch(fx.batch())
    ctx.region_end()
    assert ctx.spectrum.n_sets == 2 and ctx.spectrum.n_bins == 6 + 12
    ctx.set_spectra([])                              # cleared: PB_ERR_STATE again
    with pytest.raises(capi.PopbamError):
        ctx.region_begin(SPECTRUM, wb, we)
    ctx.close()


# ---------------------------------------------------------------------------------------------------------------------
# command line

@pytest.fixture(scope="module")
def c1_files(tmp_path_factory):
    d = tmp_path_factory.mktemp("cli_spectrum_gpu")
    return d, pbtest.fixture("c1").write_files(d / "c1")


def cli(argv, files, check=True):
    d, (bam, fa) = files
    r = subprocess.run([str(EXE), "sfs"] + argv + ["-f", fa, bam, "chr1"], stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    if check:
        assert r.returncode == 0, r.stderr.decode()
    return r


def summed(p, res, sets):
    counts, off = oracle_spectrum(p, res, sets)
    tot = counts.reshape(res.n_windows, -1).sum(axis=0)
    return [tot[off[i]:off[i + 1]].reshape(set_shape(p, pad(s))) for i, s in enumerate(sets)]


SFS_C1 = {c[0]: c for c in CASES if c[0] in ("sfs_c1", "sfs_c1_og")}


@pytest.mark.parametrize("name", list(SFS_C1))
def test_cli_jsfs_files_equal_the_oracle_sums(name, c1_files):
    case = SFS_C1[name]
    d, _ = c1_files
    fx, p, an, wb, we, _ = pbtest.case_setup(case)
    og = fx.sample_names.index("og") if "-p" in case[2] else -1
    prefix = d / name
    r = cli(case[2][1:] + ["--jsfs", str(prefix)], c1_files)
    assert r.stdout.decode() == pbtest.golden_text(case)
    assert r.stdout.decode() == cli(case[2][1:], c1_files).stdout.decode()
    orc = pbtest.OracleRun(p, fx.batch(), fx.ref(), an, wb, we)
    sets = default_sets(p.n_pops, fx.sample_pop[og] if og >= 0 else -1)
    want = summed(p, orc.res, sets)
    sites = int(pbtest.result_arrays(orc.res)["num_sites"].sum())
    files = sorted(x.name for x in d.glob(name + ".*.fs"))
    names = [".".join([name, "-".join(fx.pop_names[k] for k in s), "fs"]) for s in sets]
    assert files == sorted(names)
    marg = {}
    for s, fn, x in zip(sets, names, want):
        comments, shape, folded, pops, data, mask = read_dadi((d / fn).read_text())
        assert comments == ["popbam sfs chr1:1-%d, %d windows, %d sites, polarised by %s" %
                            (fx.contig_len, len(wb), sites, "og" if og >= 0 else "the reference base")]
        assert shape == x.shape and folded is False and pops == [fx.pop_names[k] for k in s]
        assert np.array_equal(data, x) and int(data.sum()) == sites
        assert mask.flat[0] == 1 and mask.flat[-1] == 1 and int(mask.sum()) == 2
        marg[s] = data
    # the marginals of the 2-D files are the 1-D files
    for s, x in marg.items():
        if len(s) == 2:
            assert np.array_equal(x.sum(axis=1), marg[(s[0],)]) and np.array_equal(x.sum(axis=0), marg[(s[1],)])
    if og >= 0:
        assert "out" not in "".join(files)
    orc.close()


def test_cli_jsfs_files_do_not_depend_on_shards_threads_or_k(c1_files):
    d, _ = c1_files
    cli(["-w", "1", "-p", "og", "--jsfs", str(d / "base")], c1_files)
    want = {x.name.split(".", 1)[1]: x.read_text() for x in d.glob("base.*.fs")}
    assert len(want) == 3
    for i, extra in enumerate((["--shard-mb", "0.004"], ["--shard-mb", "0.02"], ["--threads", "1"], ["--threads", "3", "--shard-mb", "0.002"],
                               ["-k", "9999"])):
        cli(["-w", "1", "-p", "og", "--jsfs", str(d / ("v%d" % i))] + extra, c1_files)
        assert {x.name.split(".", 1)[1]: x.read_text() for x in d.glob("v%d.*.fs" % i)} == want, extra


def test_cli_jsfs_pops_order_and_names(c1_files):
    d, _ = c1_files
    fx = pbtest.fixture("c1")
    p = fx.params(flags=pbtest.FLAG["OUTGROUP"], outidx=10)
    wb, we = pbtest.window_grid(0, fx.contig_len, 10000)
    orc = pbtest.OracleRun(p, fx.batch(), fx.ref(), AN["SFS"], wb, we)
    r = cli(["-w", "10", "-p", "og", "--jsfs", str(d / "named"), "--jsfs-pops", "popB,popA", "--jsfs-pops", "out,popB,popA",
             "--jsfs-pops", "popB"], c1_files)
    assert r.stdout.decode() == pbtest.golden_text(SFS_C1["sfs_c1_og"])
    sets = [(1, 0), (2, 1, 0), (1,)]
    want = summed(p, orc.res, sets)
    assert sorted(x.name for x in d.glob("named.*.fs")) == sorted(["named.popB-popA.fs", "named.out-popB-popA.fs", "named.popB.fs"])
    for fn, s, x in zip(["named.popB-popA.fs", "named.out-popB-popA.fs", "named.popB.fs"], sets, want):
        _, shape, _, pops, data, _ = read_dadi((d / fn).read_text())
        assert pops == [fx.pop_names[k] for k in s] and shape == x.shape and np.array_equal(data, x)
    orc.close()


def test_cli_jsfs_write_failure_is_fatal(c1_files):
    d, _ = c1_files
    r = cli(["-w", "10", "--jsfs", str(d / "missing_dir" / "x")], c1_files, check=False)
    assert r.returncode == 1 and "popbam runtime error:" in r.stderr.decode() and "Cannot write spectrum file" in r.stderr.decode()
    assert r.stdout.decode() == pbtest.golden_text(SFS_C1["sfs_c1"])
