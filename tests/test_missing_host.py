"""pi and dxy over sites with missing calls (PB_AN_NUCDIV_MISSING, `popbam nucdiv --missing`).  The reference never computed
them, so nothing it printed pins them directly.  Instead:
  * a numpy restatement written from the definition must equal the plain-C restatement (tests/missing_oracle.c) exactly, on
    random cb matrices and on the reference-pinned oracle's cb words of every fixture and of two low-depth fixtures where
    most positions are partly covered;
  * an anchor to the reference: restricted to the positions where every sample is covered, the sums give the golden nucdiv
    cases' num_sites, piw and pib;
  * properties (full coverage, sample permutations, complementing the derived alleles, one-sample populations, bounds);
  * pb_format_window_nucdiv_missing's text against the C restatement's, and the command line's refusals.
The GPU path is held to tests/missing_oracle.c in tests/test_missing_gpu.py.

Definition (include/popbam_b200.h, pb_region_nucdiv_missing): per position cov = samples with cb & 1, der = samples with
(cb & 3) == 3, cleared where the cells segbase called derived (bit 1) carry two different bases (bits 10-11); per
population k = |cov & m|, c = |der & m|; pi counts positions with k >= 2, dxy positions with k_i, k_j >= 1."""
import ctypes as C
import subprocess

import numpy as np
import pytest

import pbtest
from cases import CASES, FIXTURES
from popbam_b200 import capi
from test_abba_host import run_cli
from test_fst_host import synth_params

AN = capi.AN
MISSING = AN["NUCDIV_MISSING"]
EMIT_CB = pbtest.FLAG["EMIT_CB"]
HET = pbtest.FLAG["HETEROZYGOTE"]
VARIANTS = {"plain": 0, "z": HET}
FIELDS = ["pi_sites", "pi_diffs", "pi_comps", "pi_missing", "pi", "dxy_sites", "dxy_diffs", "dxy_comps", "dxy_missing", "dxy"]

# low-depth fixtures, where most positions are covered in some samples but not all (min_depth is 3)
LOW_DEPTH = {
    "low4": dict(contig_len=20500, n_ingroup=10, has_outgroup=1, depth=4.0, snp_density=0.02, het_frac=0.2, seed=31),
    "low64": dict(contig_len=10500, n_ingroup=63, has_outgroup=1, depth=6.0, snp_density=0.03, seed=32),
}
_low = {}


def fixture(name):
    if name in LOW_DEPTH:
        if name not in _low:
            _low[name] = pbtest.Fixture(**LOW_DEPTH[name])
        return _low[name]
    return pbtest.fixture(name)


ALL_FIXTURES = list(FIXTURES) + list(LOW_DEPTH)

# ---------------------------------------------------------------------------------------------------------------------
# numpy restatement from the definition


def members(p):
    return [[s for s in range(p.n_samples) if int(p.pop_mask[k]) >> s & 1] for k in range(p.n_pops)]


def cov_der(cb):
    """cb [X, n] uint64 -> (cov, der) bool [X, n], der cleared at positions with two different derived bases."""
    cb = np.asarray(cb, dtype=np.uint64)
    cov = (cb & np.uint64(1)) != 0
    der = (cb & np.uint64(3)) == np.uint64(3)
    called = (cb & np.uint64(2)) != 0
    base = (cb >> np.uint64(10)) & np.uint64(3)
    kinds = sum(((called & (base == np.uint64(b))).any(axis=1)).astype(int) for b in range(4))
    der[kinds > 1] = False
    return cov, der


def expected(p, cb, wb, we, span_beg, full_only=False):
    """Every array of pb_region_nucdiv_missing from the definition; cb [span, n]; full_only: only the positions where every
    sample is covered (site_flag bit 0)."""
    n, P, NW = p.n_samples, p.n_pops, len(wb)
    cov, der = cov_der(np.asarray(cb).reshape(-1, n))
    M = members(p)
    K = np.stack([cov[:, m].sum(axis=1) for m in M], axis=1).astype(np.int64)
    Cd = np.stack([der[:, m].sum(axis=1) for m in M], axis=1).astype(np.int64)
    if full_only:
        off = ~cov.all(axis=1)
        K[off] = 0
        Cd[off] = 0
    nn = np.array([int(p.pop_nsmpl[k]) for k in range(P)], dtype=np.int64)
    out = {f: np.zeros(NW * (P if f.startswith("pi") else P * P), dtype=np.float64 if f in ("pi", "dxy") else np.int64) for f in FIELDS}
    for w in range(NW):
        k, c = K[wb[w] - span_beg:we[w] - span_beg], Cd[wb[w] - span_beg:we[w] - span_beg]
        for a in range(P):
            use = k[:, a] >= 2
            ka, ca = k[use, a], c[use, a]
            x = w * P + a
            out["pi_sites"][x] = use.sum()
            out["pi_diffs"][x] = (ca * (ka - ca)).sum()
            out["pi_comps"][x] = (ka * (ka - 1) // 2).sum()
            out["pi_missing"][x] = (nn[a] * (nn[a] - 1) // 2 - ka * (ka - 1) // 2).sum()
            out["pi"][x] = out["pi_diffs"][x] / out["pi_comps"][x] if out["pi_comps"][x] else np.nan
            for b in range(a + 1, P):
                use = (k[:, a] >= 1) & (k[:, b] >= 1)
                ka, ca, kb, cbb = k[use, a], c[use, a], k[use, b], c[use, b]
                x = w * P * P + a * P + (b - (a + 1))
                out["dxy_sites"][x] = use.sum()
                out["dxy_diffs"][x] = (ca * (kb - cbb) + cbb * (ka - ca)).sum()
                out["dxy_comps"][x] = (ka * kb).sum()
                out["dxy_missing"][x] = (nn[a] * nn[b] - ka * kb).sum()
                out["dxy"][x] = out["dxy_diffs"][x] / out["dxy_comps"][x] if out["dxy_comps"][x] else np.nan
    return out


# ---------------------------------------------------------------------------------------------------------------------
# tests/missing_oracle.c

_missing_oracle = None


def missing_oracle_lib():
    global _missing_oracle
    if _missing_oracle is None:
        so = pbtest.ROOT / "tests" / "_build" / "libpbmoracle.so"
        so.parent.mkdir(exist_ok=True)
        subprocess.check_call(["gcc", "-O2", "-std=c11", "-fPIC", "-shared", "-Wall", "-Wextra", "-o", str(so),
                               str(pbtest.ROOT / "tests" / "missing_oracle.c"), "-lm"])
        L = C.CDLL(str(so))
        L.pbm_sums.argtypes = [C.POINTER(capi.Params), C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.c_int32,
                               C.POINTER(C.c_uint64), C.POINTER(capi.NucdivMissing)]
        L.pbm_free.argtypes = [C.POINTER(capi.NucdivMissing)]
        L.pbm_format.restype = C.c_int64
        L.pbm_format.argtypes = [C.POINTER(capi.Params), C.POINTER(capi.NucdivMissing), C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.c_int32,
                                 C.c_int32, C.c_char_p, C.POINTER(C.c_char_p), C.c_char_p, C.c_int64]
        _missing_oracle = L
    return _missing_oracle


def missing_arrays(md, NW, P):
    """Dict of numpy copies of a pb_region_nucdiv_missing (empty where an array is NULL)."""
    return {f: pbtest.arr(getattr(md, f), NW * (P if f.startswith("pi") else P * P)) for f in FIELDS}


class OracleMissing:
    """tests/missing_oracle.c over a cb matrix; keeps the C struct alive for the printer."""

    def __init__(self, p, cb, wb, we, span_beg):
        self.L, self.p = missing_oracle_lib(), p
        self.wb = np.ascontiguousarray(wb, dtype=np.int32)
        self.we = np.ascontiguousarray(we, dtype=np.int32)
        cbc = np.ascontiguousarray(cb, dtype=np.uint64).ravel()
        self.md = capi.NucdivMissing()
        assert self.L.pbm_sums(C.byref(p), len(self.wb), self.wb.ctypes.data_as(C.POINTER(C.c_int32)), self.we.ctypes.data_as(C.POINTER(C.c_int32)),
                               span_beg, cbc.ctypes.data_as(C.POINTER(C.c_uint64)), C.byref(self.md)) == 0
        self.arrays = missing_arrays(self.md, len(self.wb), p.n_pops)

    def text(self, pairs, chrom, pop_names, windows=None):
        names = (C.c_char_p * len(pop_names))(*[x.encode() for x in pop_names])
        buf = C.create_string_buffer(1 << 20)
        out = []
        for w in (range(len(self.wb)) if windows is None else windows):
            k = self.L.pbm_format(C.byref(self.p), C.byref(self.md), self.wb.ctypes.data_as(C.POINTER(C.c_int32)),
                                  self.we.ctypes.data_as(C.POINTER(C.c_int32)), w, pairs, chrom.encode(), names, buf, len(buf))
            out.append(buf.raw[:k].decode())
        return "".join(out)

    def close(self):
        if self.md.pi_sites:
            self.L.pbm_free(C.byref(self.md))

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def assert_missing_same(got, want):
    for f in FIELDS:
        assert got[f].shape == want[f].shape, f
        if f in ("pi", "dxy"):
            assert np.array_equal(got[f], want[f], equal_nan=True), f
        else:
            assert np.array_equal(got[f].astype(np.int64), want[f].astype(np.int64)), f


def oracle_cb(fx, p, wb, we):
    """The reference-pinned oracle's cb words of the region, [span, n], and its result arrays."""
    q = fx.params()
    C.memmove(C.byref(q), C.byref(p), C.sizeof(p))
    q.flags |= EMIT_CB
    orc = pbtest.OracleRun(q, fx.batch(), fx.ref(), AN["NUCDIV"], wb, we)
    d = pbtest.result_arrays(orc.res, want_cb=True)
    span_beg = orc.res.span_beg
    orc.close()
    return d["cb"].reshape(-1, p.n_samples), span_beg, d


def fixture_run(fxname, win, flags=0):
    fx = fixture(fxname)
    p = fx.params(flags=flags)
    wb, we = pbtest.window_grid(0, fx.contig_len, win)
    cb, span_beg, d = oracle_cb(fx, p, wb, we)
    return fx, p, wb, we, cb, span_beg, d


# ---------------------------------------------------------------------------------------------------------------------
# the two restatements agree


def random_cb(rng, X, n, full=False):
    """[X, n] cb words: per position a coverage probability (some all-missing, some all-covered positions), derived cells
    among the covered, segbase's bit 1 on some uncovered cells as well, and bases that make a share of the positions
    carry two different derived bases (fq < 0)."""
    q = rng.choice([0.0, 1.0, 0.3, 0.6, 0.9], size=X)[:, None] if not full else np.ones((X, 1))
    cov = rng.random((X, n)) < q
    called = rng.random((X, n)) < rng.uniform(0, 0.7, size=X)[:, None]
    base = np.where(rng.random((X, 1)) < 0.15, rng.integers(0, 4, size=(X, n)), rng.integers(0, 4, size=(X, 1)))
    cb = (rng.integers(0, 1 << 40, size=(X, n), dtype=np.uint64) << np.uint64(12)) & ~np.uint64(0xc00)
    cb |= cov.astype(np.uint64) | (called.astype(np.uint64) << np.uint64(1)) | (base.astype(np.uint64) << np.uint64(10))
    return cb


def random_windows(rng, X):
    cuts = np.sort(rng.choice(np.arange(1, X), size=min(X - 1, 6), replace=False))
    edges = np.concatenate([[0], cuts, [X]])
    wb, we = edges[:-1].astype(np.int32), edges[1:].astype(np.int32)
    keep = rng.random(len(wb)) < 0.8                # gaps between windows as well
    keep[0] = True
    return wb[keep], we[keep]


SIZES = [[64], [1, 63], [32, 32], [31, 33], [10, 1], [5, 7, 4, 1], [2, 2, 2], [20, 20, 20, 4], [1] * 8, [3, 60, 1], [2] * 32, [1] * 64]


@pytest.mark.parametrize("sizes", SIZES, ids=["-".join(map(str, s)) if len(s) < 9 else "%dx%d" % (len(s), s[0]) for s in SIZES])
def test_oracle_equals_numpy_on_random_cb(sizes):
    rng = np.random.default_rng(sum(s * 7 ** i for i, s in enumerate(sizes)) % (1 << 32))
    n = sum(sizes)
    p = synth_params(sizes)
    X = 1500 if len(sizes) < 20 else 300
    cb = random_cb(rng, X, n)
    wb, we = random_windows(rng, X)
    span_beg = 1000
    om = OracleMissing(p, cb, wb + span_beg, we + span_beg, span_beg)
    assert_missing_same(om.arrays, expected(p, cb, wb + span_beg, we + span_beg, span_beg))
    om.close()


@pytest.mark.parametrize("variant", list(VARIANTS))
@pytest.mark.parametrize("win", [200, 1000, 10000])
@pytest.mark.parametrize("fxname", ALL_FIXTURES)
def test_oracle_equals_numpy_on_fixtures(fxname, win, variant):
    fx, p, wb, we, cb, span_beg, d = fixture_run(fxname, win, VARIANTS[variant])
    om = OracleMissing(p, cb, wb, we, span_beg)
    assert_missing_same(om.arrays, expected(p, cb, wb, we, span_beg))
    om.close()


@pytest.mark.parametrize("fxname", list(LOW_DEPTH))
def test_low_depth_fixtures_exercise_missing_data(fxname):
    for win in (200, 1000, 10000):
        fx, p, wb, we, cb, span_beg, d = fixture_run(fxname, win)
        got = OracleMissing(p, cb, wb, we, span_beg).arrays
        P = p.n_pops
        for w in range(len(wb)):
            for k in range(P):
                if p.pop_nsmpl[k] >= 2:
                    assert got["pi_sites"][w * P + k] > d["num_sites"][w], (win, w, k)
                    assert got["pi_missing"][w * P + k] > 0
        cov, _ = cov_der(cb)
        inwin = np.zeros(len(cov), bool)
        for b, e in zip(wb, we):
            inwin[b - span_beg:e - span_beg] = True
        partly = cov.any(axis=1) & ~cov.all(axis=1)
        assert partly[inwin].mean() > 0.5, partly[inwin].mean()          # most positions are partly covered
        # and they carry differences: pi over the partly covered positions is defined and positive
        assert got["pi_diffs"].sum() > 0 and got["dxy_diffs"].sum() > 0


# ---------------------------------------------------------------------------------------------------------------------
# anchor to the reference: the nucdiv golden cases, restricted to the fully covered positions

NUCDIV_CASES = [c for c in CASES if c[0].startswith("nucdiv")]


@pytest.mark.parametrize("case", NUCDIV_CASES, ids=[c[0] for c in NUCDIV_CASES])
def test_fully_covered_positions_give_the_reference_sums(case):
    fx, p, an, wb, we, o = pbtest.case_setup(case)
    cb, span_beg, d = oracle_cb(fx, p, wb, we)
    full = expected(p, cb, wb, we, span_beg, full_only=True)
    P, NW = p.n_pops, len(wb)
    assert d["num_sites"].sum() > 0
    for w in range(NW):
        for a in range(P):
            na = int(p.pop_nsmpl[a])
            x = w * P + a
            if na >= 2:
                c2 = na * (na - 1) // 2
                assert full["pi_sites"][x] == d["num_sites"][w]
                assert full["pi_comps"][x] == d["num_sites"][w] * c2
                assert abs(full["pi_diffs"][x] - d["piw"][x] * c2) < 1e-6 * max(1, full["pi_diffs"][x])
            else:
                assert full["pi_sites"][x] == 0 and np.isnan(full["pi"][x])
            for b in range(a + 1, P):
                y = w * P * P + a * P + (b - (a + 1))
                assert max(np.nonzero([int(p.pop_mask[a]) >> s & 1 for s in range(64)])[0]) < min(np.nonzero([int(p.pop_mask[b]) >> s & 1 for s in range(64)])[0])
                assert full["dxy_sites"][y] == d["num_sites"][w]
                assert full["dxy_comps"][y] == d["num_sites"][w] * na * int(p.pop_nsmpl[b])
                assert abs(full["dxy_diffs"][y] - d["pib"][y] * na * int(p.pop_nsmpl[b])) < 1e-6 * max(1, full["dxy_diffs"][y])
    # the missing-data sums count more positions than the reference does
    every = expected(p, cb, wb, we, span_beg)
    assert (every["pi_sites"] >= full["pi_sites"]).all() and (every["dxy_sites"] >= full["dxy_sites"]).all()


# ---------------------------------------------------------------------------------------------------------------------
# properties

PROP_SIZES = [[5, 7, 1], [32, 31, 1], [2, 2, 2, 2], [1, 1, 62], [64]]


def run_c(p, cb, wb, we):
    om = OracleMissing(p, cb, wb, we, 0)
    a = om.arrays
    om.close()
    return a


@pytest.mark.parametrize("sizes", PROP_SIZES)
def test_full_coverage_equals_the_full_only_sums(sizes):
    rng = np.random.default_rng(3 + sum(sizes))
    p = synth_params(sizes)
    cb = random_cb(rng, 800, sum(sizes), full=True)
    wb, we = random_windows(rng, 800)
    got = run_c(p, cb, wb, we)
    assert_missing_same(got, expected(p, cb, wb, we, 0, full_only=True))
    P = p.n_pops
    for w in range(len(wb)):
        for a in range(P):
            na = int(p.pop_nsmpl[a])
            assert got["pi_sites"][w * P + a] == (we[w] - wb[w] if na >= 2 else 0) and got["pi_missing"][w * P + a] == 0


@pytest.mark.parametrize("sizes", PROP_SIZES)
def test_permuting_samples_changes_nothing(sizes):
    rng = np.random.default_rng(5 + sum(sizes))
    n = sum(sizes)
    p = synth_params(sizes)
    cb = random_cb(rng, 800, n)
    wb, we = random_windows(rng, 800)
    base = run_c(p, cb, wb, we)
    perm = rng.permutation(n)                   # new sample s is old sample perm[s]
    q = synth_params(sizes)
    for k in range(p.n_pops):
        q.pop_mask[k] = sum(1 << s for s in range(n) if int(p.pop_mask[k]) >> int(perm[s]) & 1)
    assert_missing_same(run_c(q, cb[:, perm], wb, we), base)


@pytest.mark.parametrize("sizes", PROP_SIZES)
def test_complementing_the_derived_alleles_changes_nothing(sizes):
    """Within the covered samples, swapping derived and not derived (at positions whose derived calls share one base, so
    fq >= 0 before and after) leaves every sum as it is: c (k - c) and the dxy term are symmetric under c -> k - c."""
    rng = np.random.default_rng(9 + sum(sizes))
    n = sum(sizes)
    p = synth_params(sizes)
    cb = random_cb(rng, 800, n)
    cb &= ~np.uint64(0xc00)                      # one derived base per position ...
    cb |= (rng.integers(0, 4, size=(800, 1)).astype(np.uint64) << np.uint64(10))
    cov = (cb & np.uint64(1)) != 0
    flip = cov.astype(np.uint64) << np.uint64(1)  # ... and bit 1 toggled in the covered cells
    wb, we = random_windows(rng, 800)
    assert_missing_same(run_c(p, cb ^ flip, wb, we), run_c(p, cb, wb, we))


def test_one_sample_population_has_no_pi_but_has_dxy():
    rng = np.random.default_rng(17)
    p = synth_params([6, 1, 5])
    cb = random_cb(rng, 600, 12)
    wb, we = random_windows(rng, 600)
    got = run_c(p, cb, wb, we)
    for w in range(len(wb)):
        assert got["pi_sites"][w * 3 + 1] == 0 and got["pi_comps"][w * 3 + 1] == 0 and np.isnan(got["pi"][w * 3 + 1])
        assert got["pi_missing"][w * 3 + 1] == 0
    assert (got["dxy_sites"].reshape(-1, 9)[:, [0, 1, 3]] > 0).all()
    assert not np.isnan(got["dxy"].reshape(-1, 9)[:, [0, 1, 3]]).any()


@pytest.mark.parametrize("sizes", SIZES[:8])
def test_bounds(sizes):
    rng = np.random.default_rng(23 + sum(sizes))
    n = sum(sizes)
    p = synth_params(sizes)
    cb = random_cb(rng, 1200, n)
    wb, we = random_windows(rng, 1200)
    got = run_c(p, cb, wb, we)
    P = p.n_pops
    for pre, N in (("pi", len(wb) * P), ("dxy", len(wb) * P * P)):
        d, c, s, m = (got[pre + x] for x in ("_diffs", "_comps", "_sites", "_missing"))
        assert (0 <= d).all() and (d <= c).all() and (m >= 0).all() and (s >= 0).all()
        r = got[pre]
        ok = c > 0
        assert ((r[ok] >= 0) & (r[ok] <= 1)).all()
    for w in range(len(wb)):
        L = we[w] - wb[w]
        for a in range(P):
            na = int(p.pop_nsmpl[a])
            x = w * P + a
            assert got["pi_sites"][x] <= L
            assert got["pi_comps"][x] + got["pi_missing"][x] == got["pi_sites"][x] * (na * (na - 1) // 2)
            for b in range(a + 1, P):
                y = w * P * P + a * P + (b - (a + 1))
                assert got["dxy_comps"][y] + got["dxy_missing"][y] == got["dxy_sites"][y] * na * int(p.pop_nsmpl[b])


# ---------------------------------------------------------------------------------------------------------------------
# pb_format_window_nucdiv_missing through tests/fmt_harness.cpp

@pytest.fixture(scope="module")
def fmt():
    so = pbtest.ROOT / "tests" / "_build" / "libfmtharness_missing.so"
    so.parent.mkdir(exist_ok=True)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-o", str(so), str(pbtest.ROOT / "tests" / "fmt_harness.cpp"),
                           str(pbtest.ROOT / "popbam_b200" / "csrc" / "pb_format.cpp")])
    L = C.CDLL(str(so))
    L.fmt_set_params.argtypes = [C.POINTER(capi.Params)]
    L.pb_format_window_nucdiv_missing.restype = C.c_int64
    L.pb_format_window_nucdiv_missing.argtypes = [C.c_void_p, C.POINTER(capi.Result), C.POINTER(capi.NucdivMissing), C.c_int32, C.c_int32,
                                                  C.POINTER(capi.PrintOpts), C.c_char_p, C.c_int64]
    return L


def product_text(fmt, p, md, wb, we, pairs, chrom, pop_names):
    fmt.fmt_set_params(C.byref(p))
    r = capi.Result()
    wbc, wec = np.ascontiguousarray(wb, dtype=np.int32), np.ascontiguousarray(we, dtype=np.int32)
    r.n_windows, r.n_pops, r.n_samples = len(wb), p.n_pops, p.n_samples
    r.win_beg, r.win_end = wbc.ctypes.data_as(C.POINTER(C.c_int32)), wec.ctypes.data_as(C.POINTER(C.c_int32))
    names = (C.c_char_p * len(pop_names))(*[x.encode() for x in pop_names])
    o = capi.PrintOpts()
    o.chrom, o.pop_names, o.min_sites = chrom.encode(), names, 10 ** 9       # min_sites plays no part
    out = []
    for w in range(len(wb)):
        k = fmt.pb_format_window_nucdiv_missing(None, C.byref(r), C.byref(md), w, pairs, C.byref(o), None, 0)
        assert k >= 0
        buf = C.create_string_buffer(int(k) + 1)
        assert fmt.pb_format_window_nucdiv_missing(None, C.byref(r), C.byref(md), w, pairs, C.byref(o), buf, len(buf)) == k
        if k > 8:       # cap: too small returns the size it needs and writes a NUL-terminated prefix
            small = C.create_string_buffer(8)
            assert fmt.pb_format_window_nucdiv_missing(None, C.byref(r), C.byref(md), w, pairs, C.byref(o), small, 8) == k
            assert small.raw[:7] == buf.raw[:7] and small.raw[7:8] == b"\0"
        out.append(buf.raw[:k].decode())
    return "".join(out)


@pytest.mark.parametrize("fxname", ["c1", "low4", "n64"])
def test_printer_text_equals_the_oracle_text(fmt, fxname):
    fx, p, wb, we, cb, span_beg, d = fixture_run(fxname, 1000)
    om = OracleMissing(p, cb, wb, we, span_beg)
    for pairs in (0, 1):
        got = product_text(fmt, p, om.md, wb, we, pairs, "chr1", fx.pop_names)
        assert got == om.text(pairs, "chr1", fx.pop_names)
        lines = got.splitlines()
        P = p.n_pops
        assert len(lines) == len(wb) * (P * (P - 1) // 2 if pairs else P)
        f = lines[0].split("\t")
        assert len(f) == 9 + pairs and f[1 + pairs] == "chr1" and f[2 + pairs] == str(wb[0] + 1) and f[3 + pairs] == str(we[0])
    # the one-sample outgroup population: NA, no sites
    og = [line for line in om.text(0, "chr1", fx.pop_names).splitlines() if line.startswith(fx.pop_names[-1] + "\t")]
    assert og and all(line.split("\t")[4:7] == ["NA", "0", "0"] for line in og)
    om.close()


def test_printer_ratio_format_and_refusals(fmt):
    p = synth_params([3, 2])
    md_arrays = dict(pi_sites=np.array([4, 0], np.int32), pi_diffs=np.array([1, 0], np.int64), pi_comps=np.array([3, 0], np.int64),
                     pi_missing=np.array([9, 4], np.int64), pi=np.array([1 / 3, np.nan]), dxy_sites=np.array([2, 0, 0, 0], np.int32),
                     dxy_diffs=np.array([5, 0, 0, 0], np.int64), dxy_comps=np.array([7, 0, 0, 0], np.int64),
                     dxy_missing=np.array([5, 0, 0, 0], np.int64), dxy=np.array([5 / 7, 0, 0, 0]))
    md = capi.NucdivMissing()
    for f, a in md_arrays.items():
        setattr(md, f, a.ctypes.data_as(type(getattr(md, f))))
    text = product_text(fmt, p, md, [99], [200], 0, "chrX", ["A", "B"])
    assert text == "A\tchrX\t100\t200\t0.3333333333\t4\t1\t3\t9\nB\tchrX\t100\t200\tNA\t0\t0\t0\t4\n"
    assert product_text(fmt, p, md, [99], [200], 1, "chrX", ["A", "B"]) == "A\tB\tchrX\t100\t200\t0.7142857143\t2\t5\t7\t5\n"
    r = capi.Result()
    r.n_windows = 1
    o = capi.PrintOpts()
    assert fmt.pb_format_window_nucdiv_missing(None, C.byref(r), C.byref(capi.NucdivMissing()), 0, 0, C.byref(o), None, 0) < 0
    assert fmt.pb_format_window_nucdiv_missing(None, C.byref(r), C.byref(md), 0, 2, C.byref(o), None, 0) < 0


# ---------------------------------------------------------------------------------------------------------------------
# command line: refusals before any GPU is touched

@pytest.mark.parametrize("argv", [["sfs"], ["haplo"], ["ld", "-o", "0"], ["diverge"], ["snp"], ["tree"], ["abba", "-p", "og"]])
def test_cli_refuses_missing_elsewhere(argv, tmp_path):
    r = run_cli(argv + ["--missing", str(tmp_path / "m"), "-f", str(tmp_path / "x.fa"), str(tmp_path / "x.bam"), "chr1"])
    assert r.returncode == 1 and "--missing is only available for nucdiv" in r.stderr, r.stderr
    assert not list(tmp_path.glob("m_*"))


def test_cli_refuses_a_missing_or_empty_prefix(tmp_path):
    r = run_cli(["nucdiv", "-w", "10", "-f", str(tmp_path / "x.fa"), str(tmp_path / "x.bam"), "chr1", "--missing"])
    assert r.returncode == 1 and "missing value for --missing" in r.stderr, r.stderr
    r = run_cli(["nucdiv", "-w", "10", "--missing", "", "-f", str(tmp_path / "x.fa"), str(tmp_path / "x.bam"), "chr1"])
    assert r.returncode == 1 and "--missing needs a file name prefix" in r.stderr, r.stderr


def test_cli_refuses_files_it_cannot_open(tmp_path):
    bam, fa = pbtest.fixture("c1").write_files(tmp_path / "c1")
    r = run_cli(["nucdiv", "-w", "10", "--missing", str(tmp_path / "no_such_dir" / "m"), "-f", fa, bam, "chr1"])
    assert r.returncode == 1 and "Cannot write file" in r.stderr and "m_pi.txt" in r.stderr, r.stderr
    assert r.stdout == ""
