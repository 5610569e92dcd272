"""F_ST and Snn on the GPU (PB_AN_FST: the sums and Snn in k_window_stats, the permutation test in k_snn_perm) against
tests/fst_oracle.c, which tests/test_fst_host.py pins to a numpy restatement, to pi / dxy and to exact p-values.
Integers exactly, F_ST bit for bit, Snn within 1e-12, permutation counts exactly."""
import subprocess

import numpy as np
import pytest

import pbtest
import popbam_b200
from cases import CASES, FIXTURES
from test_extra_stats_host import EXT, INT_EXT, FLT_EXT, OracleExtRun, ext_arrays
from test_fst_host import AN, EXE, FST, INT_FST, assert_fst_same, fst_arrays, oracle_fst, oracle_fst_text
from test_gpu_parity import assert_same

pytestmark = pytest.mark.gpu
N_PERMS = 2000
VARIANTS = {"plain": 0, "og": pbtest.FLAG["OUTGROUP"], "z": pbtest.FLAG["HETEROZYGOTE"]}


def run_fst(fx, p, an, wb, we, n_perms=0, seed=0):
    ctx = popbam_b200.Context(p)
    ctx.set_contig(0, fx.ref())
    ctx.set_snn_perms(n_perms, seed)
    ctx.region_begin(an, wb, we)
    ctx.push_batch(fx.batch())
    ctx.region_end()
    return ctx


def check_against_oracle(got, want):
    assert_fst_same(got, want, INT_FST + ["fst_hudson", "fst_wc", "snn_p"])
    assert_fst_same(got, want, ["snn"], snn_tol=1e-12)


@pytest.mark.parametrize("variant", list(VARIANTS))
@pytest.mark.parametrize("fxname", list(FIXTURES))
def test_fst_arrays_match_oracle(fxname, variant):
    fx = pbtest.fixture(fxname)
    p = fx.params(flags=VARIANTS[variant], outidx=fx.n_samples - 1 if variant == "og" else 0)
    wb, we = pbtest.window_grid(0, fx.contig_len, 10000)
    ctx = run_fst(fx, p, AN["NUCDIV"] | FST, wb, we, N_PERMS, seed=17)
    orc = pbtest.OracleRun(p, fx.batch(), fx.ref(), AN["NUCDIV"], wb, we)
    assert np.array_equal(pbtest.result_arrays(ctx.res)["seg_type"], pbtest.result_arrays(orc.res)["seg_type"])
    got, want = fst_arrays(ctx.fst, ctx.res), oracle_fst(p, orc.res, N_PERMS, 17, 0)
    assert int(want["hud_den"].sum()) > 0 and got["snn_ge"].size
    check_against_oracle(got, want)
    # without permutations there are no permutation arrays, and the rest is the same
    ctx.set_snn_perms(0)
    ctx.relaunch()
    ctx.wait()
    again = fst_arrays(ctx.fst, ctx.res)
    assert again["snn_p"].size == 0 and again["snn_ge"].size == 0
    assert_fst_same(again, got, ["hud_num", "hud_den", "wc_num", "wc_den", "fst_hudson", "fst_wc", "snn"])
    orc.close(); ctx.close()


@pytest.mark.parametrize("fxname", ["c1", "ld", "n64", "ldbig"])
def test_one_pass_with_everything_equals_separate_passes(fxname):
    fx = pbtest.fixture(fxname)
    p = fx.params(flags=pbtest.FLAG["OUTGROUP"], outidx=fx.n_samples - 1)
    wb, we = pbtest.window_grid(0, fx.contig_len, 5000)
    one = run_fst(fx, p, 0xfff | EXT | FST, wb, we, 300, seed=5)
    ref = run_fst(fx, p, 0xfff, wb, we)
    assert_same(pbtest.result_arrays(one.res), pbtest.result_arrays(ref.res), list(pbtest.BY_AN))
    ext = run_fst(fx, p, EXT, wb, we)
    a, b = ext_arrays(one.ext, one.res), ext_arrays(ext.ext, ext.res)
    for k in INT_EXT + FLT_EXT:
        assert a[k].shape == b[k].shape and np.array_equal(np.isnan(a[k]) if k in FLT_EXT else a[k], np.isnan(b[k]) if k in FLT_EXT else b[k]), k
        if k in FLT_EXT:
            assert np.array_equal(a[k][~np.isnan(a[k])], b[k][~np.isnan(b[k])]), k
    alone = run_fst(fx, p, FST, wb, we, 300, seed=5)
    assert_fst_same(fst_arrays(one.fst, one.res), fst_arrays(alone.fst, alone.res))
    # and a pass without PB_AN_FST returns no F_ST arrays
    assert all(v.size == 0 for v in fst_arrays(ref.fst, ref.res).values())
    for c in (one, ref, ext, alone):
        c.close()


def test_second_and_third_region_equal_first():
    fx = pbtest.fixture("c1")
    p = fx.params()
    wb, we = pbtest.window_grid(0, fx.contig_len, 10000)
    ctx = popbam_b200.Context(p)
    ctx.set_contig(0, fx.ref())
    ctx.set_snn_perms(N_PERMS, 3)
    runs = []
    for _ in range(3):
        ctx.region_begin(AN["NUCDIV"] | AN["THETA_W"] | FST, wb, we)
        ctx.push_batch(fx.batch())
        ctx.region_end()
        runs.append(fst_arrays(ctx.fst, ctx.res))
    for r in runs[1:]:
        assert_fst_same(r, runs[0])
    orc = pbtest.OracleRun(p, fx.batch(), fx.ref(), AN["NUCDIV"], wb, we)
    check_against_oracle(runs[-1], oracle_fst(p, orc.res, N_PERMS, 3, 0))
    orc.close(); ctx.close()


@pytest.fixture(scope="module")
def c1_files(tmp_path_factory):
    return pbtest.fixture("c1").write_files(tmp_path_factory.mktemp("cli_fst") / "c1")


def cli(argv, files):
    bam, fa = files
    r = subprocess.run([str(EXE)] + argv + ["-f", fa, bam, "chr1"], stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    assert r.returncode == 0, r.stderr.decode()
    return r.stdout.decode()


@pytest.mark.parametrize("extra", [[], ["--extra-stats"]])
def test_cli_fst_equals_oracle_text(extra, c1_files):
    case = [c for c in CASES if c[0] == "nucdiv_c1"][0]
    fx, p, an, wb, we, o = pbtest.case_setup(case)
    got = cli(["nucdiv", "-w", "10", "--fst", "--snn-perms", "500"] + extra, c1_files)
    ext = AN["THETA_W"] if extra else 0
    orc = OracleExtRun(p, fx.batch(), fx.ref(), an | ext, wb, we)
    assert got == oracle_fst_text(orc.text(an | ext, o), p, orc.res, o, 500, 0, 0)
    # the reference's columns are the golden rows; theta (with --extra-stats) and the F_ST columns follow
    P = fx.n_pops
    k = 2 * (4 * P * (P - 1) // 2 + (P if extra else 0))
    assert ["\t".join(r.split("\t")[:-k]) for r in got.splitlines()] == pbtest.golden_text(case).splitlines()
    # without --fst the output is the golden text
    assert cli(["nucdiv", "-w", "10"], c1_files) == pbtest.golden_text(case)
    orc.close()


def test_cli_fst_text_does_not_depend_on_shards_or_threads(c1_files):
    base = ["nucdiv", "-w", "10", "--fst", "--snn-perms", "500", "--seed", "12345"]
    want = cli(base, c1_files)
    assert "SnnP[" in want
    for extra in (["--shard-mb", "0.01"], ["--shard-mb", "0.02"], ["--threads", "1"], ["--shard-mb", "0.01", "--threads", "1"]):
        assert cli(base + extra, c1_files) == want, extra
