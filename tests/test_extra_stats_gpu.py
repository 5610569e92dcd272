"""The --extra-stats statistics on the GPU (PB_AN_THETA_W and PB_AN_FULI in k_window_stats, PB_AN_LD_DPRIME in
k_ld_rows<true> / k_ld_finish) against the oracle, which tests/test_extra_stats_host.py pins to the closed forms and a
coalescent simulation.  Integers exactly; floating point within 1e-9 relative."""
import subprocess

import numpy as np
import pytest

import pbtest
import popbam_b200
from cases import FIXTURES
from test_extra_stats_host import (AN, EXE, EXT, EXT_OF, FLT_EXT, INT_EXT, TEXT_CASES, OracleExtRun, appended_columns, ext_arrays,
                                   split_extended, variant_params)
from test_gpu_parity import assert_same, run_gpu

pytestmark = pytest.mark.gpu
RTOL = 1e-9


def assert_ext_same(got, want, keys=INT_EXT + FLT_EXT):
    for k in keys:
        if k in INT_EXT:
            assert np.array_equal(got[k], want[k]), k
        else:
            assert np.allclose(got[k], want[k], rtol=RTOL, atol=0.0, equal_nan=True), (k, got[k], want[k])


@pytest.mark.parametrize("variant", ["plain", "og", "mf2"])
@pytest.mark.parametrize("fxname", list(FIXTURES))
def test_extension_arrays_match_oracle(fxname, variant):
    fx = pbtest.fixture(fxname)
    p = variant_params(fx, variant)
    wb, we = pbtest.window_grid(0, fx.contig_len, 10000)
    ctx = run_gpu(fx, p, EXT, wb, we)
    orc = OracleExtRun(p, fx.batch(), fx.ref(), EXT, wb, we)
    got, want = ext_arrays(ctx.ext, ctx.res), orc.arrays()
    assert_ext_same(got, want)
    # ld_num_snps comes with D' alone: the Dp columns are gated by it
    NW, P = ctx.res.n_windows, ctx.res.n_pops
    assert np.array_equal(pbtest.arr(ctx.res.ld_num_snps, NW * P), pbtest.arr(orc.res.ld_num_snps, NW * P))
    orc.close(); ctx.close()


@pytest.mark.parametrize("fxname", ["c1", "ld", "n64", "ldbig"])
def test_one_pass_with_everything_equals_separate_passes(fxname):
    fx = pbtest.fixture(fxname)
    p = fx.params(flags=pbtest.FLAG["OUTGROUP"], outidx=fx.n_samples - 1)
    wb, we = pbtest.window_grid(0, fx.contig_len, 5000)
    all_an = 0xfff | EXT
    one = run_gpu(fx, p, all_an, wb, we)
    got = pbtest.result_arrays(one.res)
    got_ext = ext_arrays(one.ext, one.res)
    for bits in (AN["THETA_W"], AN["FULI"], AN["LD_DPRIME"]):
        sep = run_gpu(fx, p, bits, wb, we)
        want = ext_arrays(sep.ext, sep.res)
        for k in INT_EXT + FLT_EXT:
            if want[k].size:          # the arrays of this bit
                a, b = got_ext[k], want[k]
                assert (np.array_equal(a, b) if k in INT_EXT else np.allclose(a, b, rtol=RTOL, atol=0.0, equal_nan=True)), (bits, k)
        sep.close()
    # and the reference statistics of the same pass are those of a pass without the extensions
    ref = run_gpu(fx, p, 0xfff, wb, we)
    assert_same(got, pbtest.result_arrays(ref.res), list(pbtest.BY_AN))
    one.close(); ref.close()


@pytest.mark.parametrize("an_names", [["NUCDIV", "THETA_W", "SFS", "FULI"], ["LD_ZNS", "LD_DPRIME"]])
def test_second_region_of_a_context_equals_first(an_names):
    """A context's second region is enqueued without host round trips (asynchronous mode) where its analyses allow it."""
    fx = pbtest.fixture("c1")
    p = fx.params(flags=pbtest.FLAG["OUTGROUP"], outidx=fx.n_samples - 1)
    an = 0
    for a in an_names:
        an |= AN[a]
    wb, we = pbtest.window_grid(0, fx.contig_len, 10000)
    ctx = popbam_b200.Context(p)
    ctx.set_contig(0, fx.ref())
    runs = []
    for _ in range(3):
        ctx.region_begin(an, wb, we)
        ctx.push_batch(fx.batch())
        ctx.region_end()
        runs.append(ext_arrays(ctx.ext, ctx.res))
    # the arrays of the requested bits, and only those
    keys = [k for k in INT_EXT + FLT_EXT if runs[0][k].size]
    assert keys == [k for k in INT_EXT + FLT_EXT if (k.startswith("ld_") if "LD_DPRIME" in an_names else not k.startswith("ld_"))]
    for r in runs[1:]:
        assert_ext_same(r, runs[0], keys)
    orc = OracleExtRun(p, fx.batch(), fx.ref(), an, wb, we)
    assert_ext_same(runs[-1], orc.arrays(), keys)
    orc.close(); ctx.close()


@pytest.fixture(scope="module")
def files(tmp_path_factory):
    d = tmp_path_factory.mktemp("cli_ext")
    return {name: pbtest.fixture(name).write_files(d / name) for name in ("c1", "ldbig")}


@pytest.mark.parametrize("case", TEXT_CASES, ids=[c[0] for c in TEXT_CASES])
def test_cli_extra_stats_equals_oracle_text(case, files):
    name, fxname, argv, an_name, _pk, _ok = case
    fx, p, an, wb, we, o = pbtest.case_setup(case)
    bam, fa = files[fxname]
    r = subprocess.run([str(EXE)] + list(argv) + ["--extra-stats", "-f", fa, bam, "chr1"], stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    assert r.returncode == 0, r.stderr.decode()
    got = r.stdout.decode()
    ext = AN[EXT_OF[an_name]]
    orc = OracleExtRun(p, fx.batch(), fx.ref(), an | ext, wb, we)
    assert got == orc.text(an | ext, o)
    rows = split_extended(got, appended_columns(case, p, fx.n_pops), fx.n_pops)
    assert [row for row, _ in rows] == pbtest.golden_text(case).splitlines()
    orc.close()
