"""Garud's H statistics per window and population (PB_AN_GARUD, `popbam haplo --garud`).  The reference never computed
them, so nothing it printed pins them directly.  Instead:
  * a numpy restatement written from the definition (each population's bit columns grouped with np.unique) must equal the
    plain-C restatement (tests/garud_oracle.c) exactly, integers and doubles bit for bit, on synthetic windows and on
    every fixture;
  * hand-made windows and the properties the statistics must have;
  * an anchor to the reference: where its haplotype count is not disturbed by its rank / index quirk (a population whose
    samples are 0 .. m-1), n_hap equals its K and H1 its haplotype homozygosity;
  * the product's printer must write the oracle's rows, whose first columns are the golden haplo rows, and the command
    line must refuse --garud outside haplo.
The GPU path is held to tests/garud_oracle.c in tests/test_garud_gpu.py.

Definitions (include/popbam_b200.h, pb_region_garud): samples i, j of population p share a haplotype iff bit i equals bit
j in every seg_type word of the window; class sizes c1 >= c2 >= c3 >= ..., hh = sum c^2, n = pop_nsmpl[p]:
  h1 = hh / n^2, h12 = (hh + 2 c1 c2) / n^2, h123 = (hh + 2 (c1 c2 + c1 c3 + c2 c3)) / n^2, h2h1 = (hh - c1^2) / hh;
NaN if n < 2."""
import ctypes as C
import subprocess

import numpy as np
import pytest

import pbtest
from cases import CASES, FIXTURES
from popbam_b200 import capi
from test_extra_stats_host import EXE
from test_fst_host import FakeRegion, synth_params

AN = capi.AN
GARUD = AN["GARUD"]
INT_G = ["n_hap", "c1", "c2", "c3", "hh"]
FLT_G = ["h1", "h12", "h123", "h2h1"]

# ---------------------------------------------------------------------------------------------------------------------
# numpy restatement from the definition


def pop_classes(T, mask, n):
    """Sizes of the identity classes of the samples in `mask`, largest first."""
    members = [i for i in range(n) if mask >> i & 1]
    T = np.asarray(T, dtype=np.uint64)
    cols = ((T[:, None] >> np.array(members, dtype=np.uint64)[None, :]) & np.uint64(1)).astype(np.uint8)     # [S, m]
    _, counts = np.unique(cols.T, axis=0, return_counts=True)
    return sorted((int(c) for c in counts), reverse=True)


def expected_garud(windows, params):
    """{key: array [NW*P]} from the definition; windows = list of arrays of seg_type words."""
    P, n = params.n_pops, params.n_samples
    out = {k: [] for k in INT_G + FLT_G}
    for T in windows:
        for p in range(P):
            c = pop_classes(T, int(params.pop_mask[p]), n)
            m = int(params.pop_nsmpl[p])
            assert sum(c) == m
            c1, c2, c3 = (c + [0, 0, 0])[:3]
            hh = sum(x * x for x in c)
            for k, v in zip(INT_G, (len(c), c1, c2, c3, hh)):
                out[k].append(v)
            if m < 2:
                vals = [float("nan")] * 4
            else:       # Python's int / int is the correctly rounded quotient, as (double) a / (double) b in C
                nn = m * m
                vals = [hh / nn, (hh + 2 * c1 * c2) / nn, (hh + 2 * (c1 * c2 + c1 * c3 + c2 * c3)) / nn, (hh - c1 * c1) / hh]
            for k, v in zip(FLT_G, vals):
                out[k].append(v)
    return {k: np.array(v, dtype=np.int32 if k in INT_G else np.float64) for k, v in out.items()}


# ---------------------------------------------------------------------------------------------------------------------
# tests/garud_oracle.c

_garud_oracle = None


def garud_oracle_lib():
    global _garud_oracle
    if _garud_oracle is None:
        so = pbtest.ROOT / "tests" / "_build" / "libpbgoracle.so"
        so.parent.mkdir(exist_ok=True)
        subprocess.check_call(["gcc", "-O2", "-std=c11", "-ffp-contract=off", "-fPIC", "-shared", "-Wall", "-Wextra", "-o", str(so),
                               str(pbtest.ROOT / "tests" / "garud_oracle.c"), "-lm"])
        L = C.CDLL(str(so))
        L.pbg_garud.argtypes = [C.POINTER(capi.Params), C.POINTER(capi.Result), C.POINTER(capi.Garud)]
        L.pbg_free.argtypes = [C.POINTER(capi.Garud)]
        L.pbg_columns.restype = C.c_int64
        L.pbg_columns.argtypes = [C.POINTER(capi.Result), C.POINTER(capi.Garud), C.c_int32, C.POINTER(capi.PrintOpts), C.c_char_p, C.c_int64]
        _garud_oracle = L
    return _garud_oracle


def garud_arrays(g, res):
    """numpy copies of a pb_region_garud (empty where an array is NULL)."""
    n = res.n_windows * res.n_pops
    return {k: pbtest.arr(getattr(g, k), n) for k in INT_G + FLT_G}


def oracle_garud(params, res):
    L = garud_oracle_lib()
    g = capi.Garud()
    assert L.pbg_garud(C.byref(params), C.byref(res), C.byref(g)) == 0
    out = garud_arrays(g, res)
    L.pbg_free(C.byref(g))
    return out


def oracle_garud_text(orc_text, params, res, opts):
    """The oracle's haplo rows followed by the Garud columns of tests/garud_oracle.c."""
    L = garud_oracle_lib()
    g = capi.Garud()
    assert L.pbg_garud(C.byref(params), C.byref(res), C.byref(g)) == 0
    buf = C.create_string_buffer(1 << 16)
    out = []
    for w, row in enumerate(orc_text.splitlines()):
        k = L.pbg_columns(C.byref(res), C.byref(g), w, C.byref(opts), buf, len(buf))
        assert 0 <= k < len(buf)
        out.append(row + buf.raw[:k].decode() + "\n")
    L.pbg_free(C.byref(g))
    return "".join(out)


def assert_garud_same(got, want):
    for k in INT_G + FLT_G:
        a, b = got[k], want[k]
        assert a.shape == b.shape, (k, a.shape, b.shape)
        if k in INT_G:
            assert np.array_equal(a, b), (k, a, b)
        else:       # bit for bit, NaN where NaN
            assert np.array_equal(np.isnan(a), np.isnan(b)) and np.array_equal(a[~np.isnan(a)], b[~np.isnan(b)]), (k, a, b)


def seg_windows(res):
    d = pbtest.result_arrays(res)
    return [d["seg_type"][d["seg_off"][w]:d["seg_off"][w + 1]] for w in range(res.n_windows)]


# ---------------------------------------------------------------------------------------------------------------------
# the two restatements agree

@pytest.mark.parametrize("win", [200, 1000, 10000])
@pytest.mark.parametrize("fxname", list(FIXTURES))
def test_oracle_equals_numpy_on_fixtures(fxname, win):
    fx = pbtest.fixture(fxname)
    p = fx.params()
    wb, we = pbtest.window_grid(0, fx.contig_len, win)
    orc = pbtest.OracleRun(p, fx.batch(), fx.ref(), AN["NUCDIV"], wb, we)
    got = oracle_garud(p, orc.res)
    assert_garud_same(got, expected_garud(seg_windows(orc.res), p))
    orc.close()


def clustered_sites(rng, n, S, k):
    """S site types over n samples that carry k base haplotypes (so many samples share one); about one sample in five
    differs from its base haplotype at one site."""
    base = rng.random((k, S)) < rng.uniform(0.1, 0.9, size=S)[None, :]
    hap = base[rng.integers(0, k, size=n)]
    if S:
        for i in np.flatnonzero(rng.random(n) < 0.2):
            hap[i, rng.integers(0, S)] ^= True
    return (hap.T.astype(np.uint64) << np.arange(n, dtype=np.uint64)[None, :]).sum(axis=1).astype(np.uint64)


def both(windows, sizes):
    p = synth_params(sizes)
    fr = FakeRegion(windows, sum(sizes), len(sizes))
    return oracle_garud(p, fr.res), expected_garud(windows, p), p


SIZES = [[64], [1, 63], [32, 32], [31, 33], [10, 1], [5, 7, 4, 1], [2, 2, 2], [20, 20, 20, 4], [1] * 8, [3, 60, 1], [6]]


@pytest.mark.parametrize("sizes", SIZES, ids=["-".join(map(str, s)) for s in SIZES])
def test_oracle_equals_numpy_on_random_windows(sizes):
    rng = np.random.default_rng(sum(s * 11 ** i for i, s in enumerate(sizes)))
    n = sum(sizes)
    W = [clustered_sites(rng, n, int(rng.integers(1, 300)), int(rng.integers(1, 5))) for _ in range(8)]
    W += [rng.integers(0, 1 << 62, size=40, dtype=np.uint64) & np.uint64((1 << n) - 1 if n < 64 else (1 << 64) - 1), np.zeros(0, np.uint64)]
    got, want, p = both(W, sizes)
    assert_garud_same(got, want)
    # the grouping is exercised: some population has shared haplotypes in some window
    if max(sizes) > 1:
        assert (got["n_hap"] < np.tile(sizes, len(W))).any()


# ---------------------------------------------------------------------------------------------------------------------
# properties

def all_mask(n):
    return (1 << n) - 1


@pytest.mark.parametrize("sizes", [[64], [7, 9, 5], [2, 30, 32], [4, 1, 3]])
def test_bounds_and_order(sizes):
    rng = np.random.default_rng(7 + sum(sizes))
    n = sum(sizes)
    W = [clustered_sites(rng, n, int(rng.integers(0, 200)), int(rng.integers(1, 20))) for _ in range(20)]
    got, _, p = both(W, sizes)
    nn = np.tile(np.array(sizes), len(W))
    big = nn >= 2
    assert (got["c1"] >= got["c2"]).all() and (got["c2"] >= got["c3"]).all() and (got["c3"] >= 0).all()
    assert (got["c1"] + got["c2"] + got["c3"] <= nn).all() and (got["n_hap"] >= 1).all() and (got["n_hap"] <= nn).all()
    h1, h12, h123, h2h1 = (got[k][big] for k in FLT_G)
    assert (h1 >= 1.0 / nn[big]).all() and (h1 <= h12).all() and (h12 <= h123).all() and (h123 <= 1.0).all()
    assert (h2h1 >= 0.0).all() and (h2h1 < 1.0).all()
    assert np.isnan(got["h1"][~big]).all() and np.isnan(got["h2h1"][~big]).all()


@pytest.mark.parametrize("n", [2, 5, 33, 64])
def test_all_samples_identical(n):
    """Every site monomorphic within the population (all carry it or none): one haplotype.  So also for no sites."""
    rng = np.random.default_rng(n)
    T = np.where(rng.random(50) < 0.5, np.uint64(all_mask(n)), np.uint64(0)).astype(np.uint64)
    for W in ([T], [np.zeros(0, np.uint64)]):
        got, want, _ = both(W, [n])
        assert_garud_same(got, want)
        assert got["n_hap"][0] == 1 and got["c1"][0] == n and got["c2"][0] == 0 and got["hh"][0] == n * n
        assert got["h1"][0] == 1.0 and got["h12"][0] == 1.0 and got["h123"][0] == 1.0 and got["h2h1"][0] == 0.0


@pytest.mark.parametrize("n", [2, 3, 17, 64])
def test_all_samples_distinct(n):
    """Sample k alone carries site k: n singleton classes."""
    T = np.array([1 << k for k in range(n)], dtype=np.uint64)
    got, want, _ = both([T], [n])
    assert_garud_same(got, want)
    assert got["n_hap"][0] == n and got["c1"][0] == 1 and got["hh"][0] == n
    assert got["h1"][0] == 1 / n and got["h12"][0] == (n + 2) / (n * n)
    assert got["h2h1"][0] == (n - 1) / n


def test_hand_window():
    """Classes of sizes 4, 3, 2, 1 in a population of 10: hh = 30."""
    n = 10
    groups = [0, 0, 0, 0, 1, 1, 1, 2, 2, 3]
    # site g is carried by group g only (group 0 carries none)
    T = np.array([sum(1 << i for i, x in enumerate(groups) if x == g) for g in (1, 2, 3)], dtype=np.uint64)
    got, want, _ = both([T], [n])
    assert_garud_same(got, want)
    assert [int(got[k][0]) for k in INT_G] == [4, 4, 3, 2, 30]
    assert got["h1"][0] == 30 / 100 and got["h12"][0] == 54 / 100 and got["h123"][0] == 82 / 100 and got["h2h1"][0] == 14 / 30


@pytest.mark.parametrize("sizes", [[12, 20, 1], [64], [3, 3, 3, 3]])
def test_reordering_and_duplicating_sites_change_nothing(sizes):
    rng = np.random.default_rng(3 + sum(sizes))
    n = sum(sizes)
    W = [clustered_sites(rng, n, 120, 6) for _ in range(5)]
    a, _, _ = both(W, sizes)
    W2 = [np.concatenate([t[rng.permutation(len(t))], t[rng.integers(0, len(t), size=40)]]) for t in W]
    b, _, _ = both(W2, sizes)
    assert_garud_same(a, b)


@pytest.mark.parametrize("sizes", [[12, 20, 1], [64], [5, 6]])
def test_complementing_sites_changes_nothing(sizes):
    rng = np.random.default_rng(5 + sum(sizes))
    n = sum(sizes)
    full = np.uint64(all_mask(n)) if n < 64 else np.uint64((1 << 64) - 1)
    W = [clustered_sites(rng, n, 150, 5) for _ in range(5)]
    a, _, _ = both(W, sizes)
    flip = [np.where(rng.random(len(t)) < 0.5, ~t & full, t).astype(np.uint64) for t in W]
    b, _, _ = both(flip, sizes)
    assert_garud_same(a, b)


@pytest.mark.parametrize("sizes", [[12, 20, 1], [30, 34]])
def test_site_monomorphic_within_a_population_changes_nothing_for_it(sizes):
    rng = np.random.default_rng(9 + sum(sizes))
    n, P = sum(sizes), len(sizes)
    p = synth_params(sizes)
    W = [clustered_sites(rng, n, 80, 4) for _ in range(4)]
    a, _, _ = both(W, sizes)
    for k in range(P):
        mk = int(p.pop_mask[k])
        extra = []
        for _ in range(30):
            other = int(rng.integers(0, 1 << 62)) & all_mask(n) & ~mk
            extra.append(other | (mk if rng.random() < 0.5 else 0))
        b, _, _ = both([np.concatenate([t, np.array(extra, dtype=np.uint64)]) for t in W], sizes)
        rows = np.arange(len(W)) * P + k
        assert_garud_same({x: v[rows] for x, v in a.items()}, {x: v[rows] for x, v in b.items()})


def test_permuting_sample_labels_changes_nothing():
    """Samples relabelled by any permutation, the population masks remapped with it."""
    rng = np.random.default_rng(99)
    sizes = [9, 14, 1, 40]
    n = sum(sizes)
    W = [clustered_sites(rng, n, int(rng.integers(0, 150)), 8) for _ in range(6)]
    a, _, p = both(W, sizes)
    perm = rng.permutation(n)

    def relabel(x):
        return sum(((int(x) >> i) & 1) << int(perm[i]) for i in range(n))
    q = synth_params(sizes)
    for k in range(len(sizes)):
        q.pop_mask[k] = relabel(p.pop_mask[k])
    W2 = [np.array([relabel(t) for t in w], dtype=np.uint64) for w in W]
    fr = FakeRegion(W2, n, len(sizes))
    b = oracle_garud(q, fr.res)
    assert_garud_same(a, b)
    assert_garud_same(b, expected_garud(W2, q))


# ---------------------------------------------------------------------------------------------------------------------
# anchor to the reference: popA (samples 0 .. m-1) of every fixture

@pytest.mark.parametrize("win", [200, 1000, 10000])
@pytest.mark.parametrize("fxname", list(FIXTURES))
def test_pop_a_matches_the_reference_haplotype_count(fxname, win):
    fx = pbtest.fixture(fxname)
    p = fx.params()
    m = int(p.pop_nsmpl[0])
    assert int(p.pop_mask[0]) == all_mask(m)
    wb, we = pbtest.window_grid(0, fx.contig_len, win)
    orc = pbtest.OracleRun(p, fx.batch(), fx.ref(), AN["HAPLO_K"], wb, we)
    d = pbtest.result_arrays(orc.res)
    g = oracle_garud(p, orc.res)
    P = p.n_pops
    a = np.arange(orc.res.n_windows) * P           # population 0 of every window
    assert np.array_equal(g["n_hap"][a], d["nhaps"][a])
    if m > 2:       # the reference multiplies by the integer m / (m - 1), which is 1 here: hdiv = 1 - (1 - sum f^2 / m^2)
        assert np.abs(g["h1"][a] - d["hdiv"][a]).max() <= 1e-15
    assert (g["n_hap"][a] < m).any() or win > 200


# ---------------------------------------------------------------------------------------------------------------------
# text: the product's printer against the oracle's rows

HAPLO_CASES = [c for c in CASES if c[0].startswith("hap")]


@pytest.fixture(scope="module")
def fmt():
    so = pbtest.ROOT / "tests" / "_build" / "libfmtharness_garud.so"
    so.parent.mkdir(exist_ok=True)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-o", str(so), str(pbtest.ROOT / "tests" / "fmt_harness.cpp"),
                           str(pbtest.ROOT / "popbam_b200" / "csrc" / "pb_format.cpp")])
    L = C.CDLL(str(so))
    L.fmt_set_params.argtypes = [C.POINTER(capi.Params)]
    L.pb_format_window.restype = C.c_int64
    L.pb_format_window.argtypes = [C.c_void_p, C.POINTER(capi.Result), C.c_int32, C.c_uint32, C.POINTER(capi.PrintOpts), C.c_char_p, C.c_int64]
    L.pb_format_window_ext.restype = C.c_int64
    L.pb_format_window_ext.argtypes = [C.c_void_p, C.POINTER(capi.Result), C.POINTER(capi.Extras), C.c_int32, C.c_uint32, C.POINTER(capi.PrintOpts),
                                       C.c_char_p, C.c_int64]
    L.pb_format_window_fst.restype = C.c_int64
    L.pb_format_window_fst.argtypes = [C.c_void_p, C.POINTER(capi.Result), C.POINTER(capi.Extras), C.POINTER(capi.Fst), C.c_int32, C.c_uint32,
                                       C.POINTER(capi.PrintOpts), C.c_char_p, C.c_int64]
    L.pb_format_window_garud.restype = C.c_int64
    L.pb_format_window_garud.argtypes = [C.c_void_p, C.POINTER(capi.Result), C.POINTER(capi.Garud), C.c_int32, C.c_uint32,
                                         C.POINTER(capi.PrintOpts), C.c_char_p, C.c_int64]
    return L


def split_garud(text, P):
    """Each row -> (the row without the Garud fields, the Garud fields)."""
    k = 2 * 5 * P
    return [("\t".join(r.split("\t")[:-k]), r.split("\t")[-k:]) for r in text.splitlines()]


@pytest.mark.parametrize("min_sites", [None, 9900])
@pytest.mark.parametrize("case", HAPLO_CASES, ids=[c[0] for c in HAPLO_CASES])
def test_product_printer_equals_oracle_rows(fmt, case, min_sites):
    fx, p, an, wb, we, o = pbtest.case_setup(case)
    if min_sites is not None:
        o.min_sites = min_sites
    orc = pbtest.OracleRun(p, fx.batch(), fx.ref(), an, wb, we)
    L = garud_oracle_lib()
    g = capi.Garud()
    assert L.pbg_garud(C.byref(p), C.byref(orc.res), C.byref(g)) == 0
    orc.res.analyses |= GARUD          # as the product's result of a region run with PB_AN_GARUD
    fmt.fmt_set_params(C.byref(p))
    buf = C.create_string_buffer(1 << 16)
    rows = []
    for w in range(orc.res.n_windows):
        k = fmt.pb_format_window_garud(None, C.byref(orc.res), C.byref(g), w, an | GARUD, C.byref(o), buf, len(buf))
        assert 0 <= k < len(buf)
        rows.append(buf.raw[:k].decode())
        assert fmt.pb_format_window_garud(None, C.byref(orc.res), C.byref(g), w, an | GARUD, C.byref(o), buf, 8) == k
    text = "".join(rows)
    assert text == oracle_garud_text(orc.text(an, o), p, orc.res, o)
    parts = split_garud(text, fx.n_pops)
    if min_sites is None:       # the reference's row is the golden row
        assert [r for r, _ in parts] == pbtest.golden_text(case).splitlines()
    assert parts[0][1][::2] == ["%s[%s]:" % (c, pn) for pn in fx.pop_names for c in ("nHap", "H1", "H12", "H123", "H2H1")]
    for w, (_, cols) in enumerate(parts):
        for k in range(fx.n_pops):
            vals = cols[10 * k + 1:10 * k + 10:2]
            if orc.res.num_sites[w] < o.min_sites:
                assert vals == ["     NA"] * 5
            else:           # the doubles of a one-sample population are NaN
                assert vals[0].isdigit() and all((v == "     NA") == (p.pop_nsmpl[k] < 2) for v in vals[1:])
    # the other printers refuse the bit; the Garud printer takes a haplo bit with PB_AN_GARUD and the arrays only
    assert fmt.pb_format_window(None, C.byref(orc.res), 0, an | GARUD, C.byref(o), buf, len(buf)) < 0
    assert fmt.pb_format_window_ext(None, C.byref(orc.res), None, 0, an | GARUD, C.byref(o), buf, len(buf)) < 0
    assert fmt.pb_format_window_fst(None, C.byref(orc.res), None, None, 0, AN["NUCDIV"] | GARUD, C.byref(o), buf, len(buf)) < 0
    assert fmt.pb_format_window_garud(None, C.byref(orc.res), C.byref(g), 0, an, C.byref(o), buf, len(buf)) < 0
    assert fmt.pb_format_window_garud(None, C.byref(orc.res), C.byref(g), 0, AN["NUCDIV"] | GARUD, C.byref(o), buf, len(buf)) < 0
    assert fmt.pb_format_window_garud(None, C.byref(orc.res), None, 0, an | GARUD, C.byref(o), buf, len(buf)) < 0
    # without the bit the reference printer still prints the golden row
    k = fmt.pb_format_window(None, C.byref(orc.res), 0, an, C.byref(o), buf, len(buf))
    assert buf.raw[:k].decode() == orc.text(an, o, [0])
    L.pbg_free(C.byref(g))
    orc.close()


def test_one_sample_population_prints_na():
    """n < 2: the doubles are NaN and print NA; nHap is printed."""
    fx = pbtest.fixture("c1")
    p = fx.params()
    o = fx.print_opts()
    wb, we = pbtest.window_grid(0, fx.contig_len, 10000)
    orc = pbtest.OracleRun(p, fx.batch(), fx.ref(), AN["HAPLO_K"], wb, we)
    text = oracle_garud_text(orc.text(AN["HAPLO_K"], o), p, orc.res, o)
    row = text.splitlines()[0].split("\t")
    i = row.index("nHap[out]:")
    assert row[i + 1] == "1" and row[i + 3:i + 11:2] == ["     NA"] * 4
    orc.close()


# ---------------------------------------------------------------------------------------------------------------------
# command line: refusals before any GPU is touched

@pytest.mark.parametrize("argv", [["nucdiv"], ["sfs"], ["ld", "-o", "0"], ["diverge"], ["snp"], ["tree"], ["abba", "-p", "og"]])
def test_cli_refuses_garud_elsewhere(argv, tmp_path):
    r = subprocess.run([str(EXE)] + argv + ["--garud", "-f", str(tmp_path / "x.fa"), str(tmp_path / "x.bam"), "chr1"],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    assert r.returncode == 1 and "--garud is only available for haplo" in r.stderr


@pytest.mark.parametrize("o", ["0", "1", "2"])
def test_cli_takes_garud_with_haplo(o, tmp_path):
    r = subprocess.run([str(EXE), "haplo", "-o", o, "--garud", "-f", str(tmp_path / "x.fa"), str(tmp_path / "x.bam"), "chr1"],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    assert r.returncode == 1 and "--garud" not in r.stderr and "does not exist" in r.stderr
