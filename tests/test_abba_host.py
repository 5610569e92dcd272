"""ABBA-BABA statistics per window and population triple (PB_AN_ABBA, `popbam abba`).  The reference never computed
them, so nothing it printed pins them.  Instead:
  * a fractions.Fraction restatement written from the published frequency formulas -- Patterson's ABBA / BABA
    (Green et al. 2010, Durand et al. 2011), Martin, Davey & Jiggins (2015) S(P1, P2, P3, O) and f_d, Malinsky et al.
    (2015) f_dM -- must equal the plain-C restatement of the integer sums (tests/abba_oracle.c) exactly, on synthetic
    site sets and on every fixture regrouped into at least three ingroup populations and an outgroup;
  * hand-made windows and the algebraic properties the statistics must have;
  * the product's printer must write the oracle's text, and the command line must refuse bad triples.
The GPU path is held to tests/abba_oracle.c in tests/test_abba_gpu.py.

Definitions (include/popbam_b200.h, pb_region_abba): per site a_k = derived copies of P1, P2, P3, O, n_k = sample counts,
p_k = a_k / n_k after polarising by the outgroup (if p4 > 1/2 every p_k becomes 1 - p_k, ties kept).  On the scale
K = n1^2 n2^2 n3^2 n4:
  abba = sum (1-p1) p2 p3 (1-p4) K, baba = sum p1 (1-p2) p3 (1-p4) K,
  fd_den = sum S(P1, PD, PD, O) K with pD = max(p2, p3),
  fdm_den = sum [S(P1, PD, PD, O) with pD = max(p2, p3) if p2 >= p1, else -S(PD, P2, PD, O) with pD = max(p1, p3)] K,
  S(a, b, c, d) = (1-pa) pb pc (1-pd) - pa (1-pb) pc (1-pd);  sites = #{site: ABBA + BABA > 0};
  D = (abba - baba) / (abba + baba), fd = (abba - baba) / fd_den, fdM = (abba - baba) / fdm_den (NaN where 0)."""
import ctypes as C
import gzip
import os
import re
import struct
import subprocess
from fractions import Fraction
from functools import lru_cache

import numpy as np
import pytest

import pbtest
from cases import FIXTURES
from popbam_b200 import capi
from test_extra_stats_host import EXE
from test_fst_host import FakeRegion, synth_params

AN = capi.AN
ABBA = AN["ABBA"]
INT_ABBA = ["sites", "abba", "baba", "fd_den", "fdm_den"]
FLT_ABBA = ["d", "fd", "fdm"]

# ---------------------------------------------------------------------------------------------------------------------
# Fraction restatement from the frequency formulas


def S(pa, pb, pc, pd):
    """Martin et al. (2015): S(P1, P2, P3, O) = ABBA - BABA of the frequencies."""
    return (1 - pa) * pb * pc * (1 - pd) - pa * (1 - pb) * pc * (1 - pd)


@lru_cache(maxsize=None)
def site_fractions(c, n):
    """(ABBA, BABA, f_d denominator, f_dM denominator) of one site as Fractions; c, n = derived copies and sample counts
    of (P1, P2, P3, O)."""
    p = [Fraction(a, m) for a, m in zip(c, n)]
    if p[3] > Fraction(1, 2):
        p = [1 - x for x in p]
    p1, p2, p3, p4 = p
    abba = (1 - p1) * p2 * p3 * (1 - p4)
    baba = p1 * (1 - p2) * p3 * (1 - p4)
    pd = max(p2, p3)
    fd = S(p1, pd, pd, p4)
    if p2 >= p1:
        fdm = fd
    else:
        pd = max(p1, p3)
        fdm = -S(pd, p2, pd, p4)
    return abba, baba, fd, fdm


def expected_abba(types, params, og, triples):
    """{key: [per window, per triple]} of the Fraction sums (abba, baba, fd_den, fdm_den: over K) and the site counts.
    types = list of windows, each an array of seg_type words."""
    out = {k: [] for k in INT_ABBA}
    for T in types:
        T = np.asarray(T, dtype=np.uint64)
        for t in triples:
            pk = list(t) + [og]
            n = tuple(int(params.pop_nsmpl[k]) for k in pk)
            cnt = np.stack([np.bitwise_count(T & np.uint64(int(params.pop_mask[k]))).astype(np.int64) for k in pk], axis=1) if len(T) else np.zeros((0, 4), np.int64)
            sums = [Fraction(0)] * 4
            sites = 0
            rows, mult = np.unique(cnt, axis=0, return_counts=True) if len(T) else (np.zeros((0, 4), np.int64), [])
            for row, m in zip(rows, mult):
                v = site_fractions(tuple(int(x) for x in row), n)
                sums = [s + int(m) * x for s, x in zip(sums, v)]
                sites += int(m) if v[0] + v[1] > 0 else 0
            out["sites"].append(sites)
            for k, s in zip(["abba", "baba", "fd_den", "fdm_den"], sums):
                out[k].append(s)
    return out


def scale_K(params, og, t):
    n1, n2, n3 = (int(params.pop_nsmpl[k]) for k in t)
    return n1 * n1 * n2 * n2 * n3 * n3 * int(params.pop_nsmpl[og])


def assert_oracle_equals_fractions(got, want, params, og, triples, n_windows):
    NT = len(triples)
    assert np.array_equal(got["sites"], np.array(want["sites"], dtype=np.int32))
    for w in range(n_windows):
        for i, t in enumerate(triples):
            K = scale_K(params, og, t)
            x = w * NT + i
            for k in ("abba", "baba", "fd_den", "fdm_den"):
                assert Fraction(int(got[k][x]), K) == want[k][x], (k, w, t, got[k][x], want[k][x] * K)
            num = int(got["abba"][x]) - int(got["baba"][x])
            for k, den in (("d", int(got["abba"][x]) + int(got["baba"][x])), ("fd", int(got["fd_den"][x])), ("fdm", int(got["fdm_den"][x]))):
                v = got[k][x]
                assert (np.isnan(v) if den == 0 else v == float(num) / float(den)), (k, w, t, v)


# ---------------------------------------------------------------------------------------------------------------------
# tests/abba_oracle.c

_abba_oracle = None


def abba_oracle_lib():
    global _abba_oracle
    if _abba_oracle is None:
        so = pbtest.ROOT / "tests" / "_build" / "libpbaoracle.so"
        so.parent.mkdir(exist_ok=True)
        subprocess.check_call(["gcc", "-O2", "-std=c11", "-ffp-contract=off", "-fPIC", "-shared", "-Wall", "-Wextra", "-o", str(so),
                               str(pbtest.ROOT / "tests" / "abba_oracle.c"), "-lm"])
        L = C.CDLL(str(so))
        L.pba_abba.argtypes = [C.POINTER(capi.Params), C.POINTER(capi.Result), C.c_int32, C.c_int32, C.POINTER(C.c_int32), C.POINTER(capi.Abba)]
        L.pba_free.argtypes = [C.POINTER(capi.Abba)]
        L.pba_row.restype = C.c_int64
        L.pba_row.argtypes = [C.POINTER(capi.Params), C.POINTER(capi.Result), C.POINTER(capi.Abba), C.c_int32, C.POINTER(capi.PrintOpts),
                              C.c_char_p, C.c_int64]
        _abba_oracle = L
    return _abba_oracle


def abba_arrays(ab, res):
    """numpy copies of a pb_region_abba (empty where an array is NULL)."""
    n = res.n_windows * ab.n_triples
    return {k: pbtest.arr(getattr(ab, k), n) for k in INT_ABBA + FLT_ABBA}


def _tri(triples):
    flat = (C.c_int32 * max(1, 3 * len(triples)))(*[k for t in triples for k in t])
    return flat


def oracle_abba(params, res, og, triples):
    L = abba_oracle_lib()
    a = capi.Abba()
    assert L.pba_abba(C.byref(params), C.byref(res), og, len(triples), _tri(triples), C.byref(a)) == 0
    out = abba_arrays(a, res)
    L.pba_free(C.byref(a))
    return out


def oracle_abba_text(params, res, og, triples, opts):
    L = abba_oracle_lib()
    a = capi.Abba()
    assert L.pba_abba(C.byref(params), C.byref(res), og, len(triples), _tri(triples), C.byref(a)) == 0
    buf = C.create_string_buffer(1 << 20)
    out = []
    for w in range(res.n_windows):
        k = L.pba_row(C.byref(params), C.byref(res), C.byref(a), w, C.byref(opts), buf, len(buf))
        assert 0 <= k < len(buf)
        out.append(buf.raw[:k].decode())
    L.pba_free(C.byref(a))
    return "".join(out)


def assert_abba_same(got, want, keys=INT_ABBA + FLT_ABBA):
    for k in keys:
        a, b = got[k], want[k]
        assert a.shape == b.shape, (k, a.shape, b.shape)
        if k in INT_ABBA:
            assert np.array_equal(a, b), (k, a, b)
        else:       # bit for bit, NaN where NaN
            assert np.array_equal(np.isnan(a), np.isnan(b)) and np.array_equal(a[~np.isnan(a)], b[~np.isnan(b)]), (k, a, b)


def default_triples(P, og):
    """Every triple with P1 < P2 and P3 besides them, none the outgroup, in lexicographic order (the command line's list)."""
    return [(i, j, k) for i in range(P) for j in range(i + 1, P) for k in range(P) if og not in (i, j, k) and k not in (i, j)]


# ---------------------------------------------------------------------------------------------------------------------
# fixtures regrouped into >= 3 ingroup populations + the outgroup

N_GROUPS = {"c1": [3, 3, 4], "edge": [2, 2, 2], "rg2": [1, 1, 2], "ld": [6, 6, 6, 5], "n64": [7] * 9, "ldbig": [7] * 9, "wideq": [3, 3, 3]}


def regrouped(fx, fxname, **kw):
    """(params, pop names) with the fixture's first samples split into the groups of N_GROUPS and the last sample alone as
    the outgroup population "out" (the fixtures' own outgroup "og" where they have one)."""
    sizes = N_GROUPS[fxname]
    assert sum(sizes) + 1 == fx.n_samples
    p = fx.params(**kw)
    for k in range(64):
        p.pop_mask[k], p.pop_nsmpl[k] = 0, 0
    s = 0
    for g, m in enumerate(sizes + [1]):
        p.pop_mask[g] = ((1 << m) - 1) << s
        p.pop_nsmpl[g] = m
        s += m
    p.n_pops = len(sizes) + 1
    return p, ["P%d" % (g + 1) for g in range(len(sizes))] + ["out"]


def regrouped_opts(fx, names, **kw):
    o = fx.print_opts(**kw)
    o._names = (C.c_char_p * len(names))(*[s.encode() for s in names])
    o.pop_names = o._names
    return o


@pytest.mark.parametrize("fxname", list(FIXTURES))
def test_oracle_equals_fractions_on_regrouped_fixtures(fxname):
    fx = pbtest.fixture(fxname)
    p, names = regrouped(fx, fxname)
    og = p.n_pops - 1
    wb, we = pbtest.window_grid(0, fx.contig_len, 10000)
    orc = pbtest.OracleRun(p, fx.batch(), fx.ref(), AN["NUCDIV"], wb, we)
    base = pbtest.OracleRun(fx.params(), fx.batch(), fx.ref(), AN["NUCDIV"], wb, we)
    # the site types do not depend on how the samples are grouped
    d = pbtest.result_arrays(orc.res)
    assert np.array_equal(d["seg_type"], pbtest.result_arrays(base.res)["seg_type"])
    triples = default_triples(p.n_pops, og)
    assert len(triples) == {3: 3, 4: 12, 9: 252}[len(N_GROUPS[fxname])]
    got = oracle_abba(p, orc.res, og, triples)
    types = [d["seg_type"][d["seg_off"][w]:d["seg_off"][w + 1]] for w in range(orc.res.n_windows)]
    want = expected_abba(types, p, og, triples)
    assert_oracle_equals_fractions(got, want, p, og, triples, orc.res.n_windows)
    assert int((got["abba"] + got["baba"]).max()) > 0
    orc.close(); base.close()


# ---------------------------------------------------------------------------------------------------------------------
# synthetic site sets

def both(windows, sizes, og, triples):
    """(oracle arrays, Fraction sums) of synthetic windows; populations are consecutive runs of `sizes` samples."""
    p = synth_params(sizes)
    fr = FakeRegion(windows, sum(sizes), len(sizes))
    return oracle_abba(p, fr.res, og, triples), expected_abba(windows, p, og, triples), p


def freq_sites(rng, sizes, count):
    """Site types with a random allele frequency per population (so every a_k from 0 to n_k occurs)."""
    n = sum(sizes)
    out = np.zeros(count, dtype=np.uint64)
    s = 0
    for m in sizes:
        f = rng.uniform(0, 1, size=count)
        bits = rng.random((count, m)) < f[:, None]
        out |= (bits.astype(np.uint64) << np.arange(s, s + m, dtype=np.uint64)).sum(axis=1).astype(np.uint64)
        s += m
    full = np.uint64((1 << n) - 1) if n < 64 else np.uint64((1 << 64) - 1)
    return out[(out != 0) & (out != full)]


@pytest.mark.parametrize("sizes", [[4, 5, 6, 3], [3, 3, 3, 2], [6, 2, 7, 4], [20, 20, 20, 4], [15, 16, 17, 16], [5, 8, 3, 1]])
def test_oracle_equals_fractions_on_random_sites(sizes):
    rng = np.random.default_rng(sum(s * 7 ** i for i, s in enumerate(sizes)))
    P = len(sizes)
    og = P - 1
    triples = [(0, 1, 2), (1, 0, 2), (2, 1, 0), (0, 2, 1)]
    W = [freq_sites(rng, sizes, 400) for _ in range(3)] + [np.zeros(0, np.uint64)]
    got, want, p = both(W, sizes, og, triples)
    assert_oracle_equals_fractions(got, want, p, og, triples, len(W))
    assert np.isnan(got["d"][-1]) and got["abba"][-1] == 0


def _site(sizes, counts):
    """One site type: the first counts[k] samples of population k carry the derived allele."""
    T, s = 0, 0
    for m, c in zip(sizes, counts):
        T |= ((1 << c) - 1) << s
        s += m
    return T


@pytest.mark.parametrize("sizes", [[4, 6, 6, 4], [5, 5, 5, 3], [6, 4, 8, 2]])
def test_ties_match_fractions(sizes):
    """p2 = p3, p1 = p2, p1 = p3 and 2 a4 = n4 (even n4): the tie rules of the integer forms match the max() of the
    frequency formulas."""
    n1, n2, n3, n4 = sizes
    sites = []
    for a1 in range(n1 + 1):
        for a2 in range(n2 + 1):
            for a3 in range(n3 + 1):
                # ties of p1 = p2, p2 = p3, p1 = p3 under these sizes, with every a4 (including n4 / 2)
                if a1 * n2 == a2 * n1 or a2 * n3 == a3 * n2 or a1 * n3 == a3 * n1:
                    for a4 in range(n4 + 1):
                        sites.append(_site(sizes, [a1, a2, a3, a4]))
    T = np.array([t for t in sites if t not in (0, (1 << sum(sizes)) - 1)], dtype=np.uint64)
    triples = [(0, 1, 2), (1, 0, 2)]
    got, want, p = both([T], sizes, 3, triples)
    assert_oracle_equals_fractions(got, want, p, 3, triples, 1)


# ---------------------------------------------------------------------------------------------------------------------
# hand cases

def test_pure_abba_window_gives_d_one_and_fd_one():
    sizes = [4, 5, 5, 3]
    # P1 and O ancestral, P2 and P3 fixed derived: ABBA only, and p2 = p3 with P1 ancestral gives f_d = 1
    W = [np.array([_site(sizes, [0, 5, 5, 0])] * 3 + [_site(sizes, [0, 3, 3, 0])], dtype=np.uint64)]
    got, want, p = both(W, sizes, 3, [(0, 1, 2)])
    assert got["baba"][0] == 0 and got["abba"][0] > 0
    assert got["d"][0] == 1.0 and got["fd"][0] == 1.0 and got["fdm"][0] == 1.0
    assert got["sites"][0] == 4


def test_pure_baba_window_gives_d_minus_one():
    sizes = [4, 5, 5, 3]
    W = [np.array([_site(sizes, [4, 0, 5, 0]), _site(sizes, [2, 1, 3, 1])], dtype=np.uint64)]
    got, want, p = both(W, sizes, 3, [(0, 1, 2)])
    assert got["abba"][0] > 0 and got["baba"][0] > got["abba"][0]
    W = [np.array([_site(sizes, [4, 0, 5, 0])] * 2, dtype=np.uint64)]
    got, _, _ = both(W, sizes, 3, [(0, 1, 2)])
    assert got["abba"][0] == 0 and got["d"][0] == -1.0 and got["fdm"][0] == -1.0


def test_outgroup_monomorphic_derived_site_is_flipped():
    """O carries the non-reference allele in every sample: that allele counts as ancestral, so a site where P1 and O
    carry it and P2, P3 do not is an ABBA site."""
    sizes = [3, 4, 4, 3]
    flipped = _site(sizes, [3, 0, 0, 3])
    got, want, p = both([np.array([flipped], dtype=np.uint64)], sizes, 3, [(0, 1, 2)])
    assert got["abba"][0] == scale_K(p, 3, (0, 1, 2)) and got["baba"][0] == 0 and got["d"][0] == 1.0 and got["sites"][0] == 1
    # ... the same as the explicitly polarised site
    plain = _site(sizes, [0, 4, 4, 0])
    again, _, _ = both([np.array([plain], dtype=np.uint64)], sizes, 3, [(0, 1, 2)])
    assert_abba_same(got, again)


# ---------------------------------------------------------------------------------------------------------------------
# properties

@pytest.mark.parametrize("sizes", [[4, 6, 5, 3], [7, 7, 7, 4], [10, 3, 12, 1]])
def test_swapping_p1_and_p2(sizes):
    rng = np.random.default_rng(31 + sum(sizes))
    W = [freq_sites(rng, sizes, 300) for _ in range(4)]
    got, _, _ = both(W, sizes, 3, [(0, 1, 2), (1, 0, 2)])
    a = {k: v[0::2] for k, v in got.items()}
    b = {k: v[1::2] for k, v in got.items()}
    assert np.array_equal(a["abba"], b["baba"]) and np.array_equal(a["baba"], b["abba"])
    assert np.array_equal(a["fdm_den"], b["fdm_den"]) and np.array_equal(a["sites"], b["sites"])
    assert np.array_equal(a["d"], -b["d"]) and np.array_equal(a["fdm"], -b["fdm"])


@pytest.mark.parametrize("sizes", [[4, 6, 5, 3], [2, 2, 2, 2], [16, 16, 16, 16], [9, 5, 3, 1]])
def test_fdm_bounded(sizes):
    rng = np.random.default_rng(77 + sum(sizes))
    triples = [(0, 1, 2), (1, 0, 2), (2, 0, 1), (0, 2, 1), (1, 2, 0), (2, 1, 0)]
    W = [freq_sites(rng, sizes, 200) for _ in range(5)]
    got, _, _ = both(W, sizes, 3, triples)
    assert (got["fdm_den"] >= 0).all()
    ok = ~np.isnan(got["fdm"])
    assert ok.any() and (np.abs(got["fdm"][ok]) <= 1.0).all()
    # per site too: fdm_den >= |abba - baba| (one-site windows)
    one = [np.array([t], dtype=np.uint64) for t in W[0][:60]]
    g1, _, _ = both(one, sizes, 3, triples)
    assert (g1["fdm_den"] >= np.abs(g1["abba"] - g1["baba"])).all()


@pytest.mark.parametrize("sizes", [[4, 6, 5, 3], [5, 5, 5, 5]])
def test_complementing_sites(sizes):
    """With odd n4 complementing a site's alleles within the four populations changes nothing (with even n4 it can, at
    2 a4 = n4)."""
    rng = np.random.default_rng(5 + sum(sizes))
    n = sum(sizes)
    W = [freq_sites(rng, sizes, 300) for _ in range(3)]
    comp = [(~t) & np.uint64((1 << n) - 1) for t in W]
    triples = [(0, 1, 2), (2, 0, 1)]
    a, _, _ = both(W, sizes, 3, triples)
    b, _, _ = both(comp, sizes, 3, triples)
    assert_abba_same(a, b)


def test_permuting_samples_within_populations():
    sizes = [4, 6, 5, 3]
    rng = np.random.default_rng(99)
    n = sum(sizes)
    W = [freq_sites(rng, sizes, 300) for _ in range(3)]
    perm, s = [], 0
    for m in sizes:
        perm += list(s + rng.permutation(m))
        s += m

    def permute(t):
        bits = [(t >> np.uint64(perm[k])) & np.uint64(1) for k in range(n)]
        return sum(b << np.uint64(k) for k, b in enumerate(bits)).astype(np.uint64)
    triples = default_triples(4, 3)
    a, _, _ = both(W, sizes, 3, triples)
    b, _, _ = both([permute(t) for t in W], sizes, 3, triples)
    assert_abba_same(a, b)


# ---------------------------------------------------------------------------------------------------------------------
# text: the product's printer against the oracle's rows

@pytest.fixture(scope="module")
def fmt():
    so = pbtest.ROOT / "tests" / "_build" / "libfmtharness_abba.so"
    so.parent.mkdir(exist_ok=True)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-o", str(so), str(pbtest.ROOT / "tests" / "fmt_harness.cpp"),
                           str(pbtest.ROOT / "popbam_b200" / "csrc" / "pb_format.cpp")])
    L = C.CDLL(str(so))
    L.fmt_set_params.argtypes = [C.POINTER(capi.Params)]
    L.pb_format_window_abba.restype = C.c_int64
    L.pb_format_window_abba.argtypes = [C.c_void_p, C.POINTER(capi.Result), C.POINTER(capi.Abba), C.c_int32, C.POINTER(capi.PrintOpts),
                                        C.c_char_p, C.c_int64]
    L.pb_format_window.restype = C.c_int64
    L.pb_format_window.argtypes = [C.c_void_p, C.POINTER(capi.Result), C.c_int32, C.c_uint32, C.POINTER(capi.PrintOpts), C.c_char_p, C.c_int64]
    return L


@pytest.mark.parametrize("min_sites", [10, 9900])
@pytest.mark.parametrize("fxname", ["c1", "n64"])
def test_product_printer_equals_oracle_rows(fmt, fxname, min_sites):
    fx = pbtest.fixture(fxname)
    p, names = regrouped(fx, fxname)
    og = p.n_pops - 1
    o = regrouped_opts(fx, names, min_sites=min_sites)
    wb, we = pbtest.window_grid(0, fx.contig_len, 10000)
    orc = pbtest.OracleRun(p, fx.batch(), fx.ref(), AN["NUCDIV"], wb, we)
    triples = default_triples(p.n_pops, og)[::-1][:20]
    L = abba_oracle_lib()
    a = capi.Abba()
    assert L.pba_abba(C.byref(p), C.byref(orc.res), og, len(triples), _tri(triples), C.byref(a)) == 0
    orc.res.analyses |= ABBA          # as the product's result of a region run with PB_AN_ABBA
    fmt.fmt_set_params(C.byref(p))
    buf = C.create_string_buffer(1 << 20)
    rows = []
    for w in range(orc.res.n_windows):
        k = fmt.pb_format_window_abba(None, C.byref(orc.res), C.byref(a), w, C.byref(o), buf, len(buf))
        assert 0 <= k < len(buf)
        rows.append(buf.raw[:k].decode())
        # too small a buffer: the size it needs
        assert fmt.pb_format_window_abba(None, C.byref(orc.res), C.byref(a), w, C.byref(o), buf, 8) == k
    text = "".join(rows)
    assert text == oracle_abba_text(p, orc.res, og, triples, o)
    first = text.splitlines()[0].split("\t")
    assert first[4:16:2] == ["%s[%s-%s-%s]:" % (c, *(names[i] for i in triples[0])) for c in ("S", "ABBA", "BABA", "D", "fd", "fdM")]
    # every floating column is NA in a window with fewer than min_sites sites; S is always printed
    short = 0
    for row in text.splitlines():
        f = row.split("\t")
        floats = [f[4 + 12 * t + c] for t in range(len(triples)) for c in (3, 5, 7, 9, 11)]
        if int(f[3]) < min_sites:
            short += 1
            assert all(v.strip() == "NA" for v in floats) and all(f[5 + 12 * t].isdigit() for t in range(len(triples)))
        else:
            assert any(v.strip() != "NA" for v in floats)
    assert short > 0 if min_sites > 1000 else short < len(rows)
    # the reference printers refuse the bit
    assert fmt.pb_format_window(None, C.byref(orc.res), 0, AN["NUCDIV"] | ABBA, C.byref(o), buf, len(buf)) < 0
    orc.res.analyses &= ~ABBA
    assert fmt.pb_format_window_abba(None, C.byref(orc.res), C.byref(a), 0, C.byref(o), buf, len(buf)) < 0
    L.pba_free(C.byref(a))
    orc.close()


# ---------------------------------------------------------------------------------------------------------------------
# command line: refusals before any GPU is touched

def bam_header_text(bam):
    with gzip.open(bam, "rb") as f:
        assert f.read(4) == b"BAM\1"
        (l_text,) = struct.unpack("<i", f.read(4))
        return f.read(l_text).decode().rstrip("\0")


def write_regrouped_header(bam, path, sample_pop):
    """A header file (-h) whose @RG lines give every sample the population sample_pop[SM]."""
    lines = [ln for ln in bam_header_text(bam).splitlines() if ln.startswith("@RG")]
    out = []
    for ln in lines:
        sm = re.search(r"\tSM:([^\t]*)", ln).group(1)
        out.append(re.sub(r"\tPO:[^\t]*", "\tPO:" + sample_pop[sm], ln))
    path.write_text("\n".join(out) + "\n")
    return str(path)


def c1_sample_pop(fx):
    """c1 regrouped: samples 0-2, 3-5, 6-9 into P1, P2, P3, the outgroup sample og alone in "out"."""
    groups = ["P1"] * 3 + ["P2"] * 3 + ["P3"] * 4 + ["out"]
    return dict(zip(fx.sample_names, groups))


@pytest.fixture(scope="module")
def c1_cli_files(tmp_path_factory):
    d = tmp_path_factory.mktemp("cli_abba")
    fx = pbtest.fixture("c1")
    bam, fa = fx.write_files(d / "c1")
    hdr = write_regrouped_header(bam, d / "regrouped.sam", c1_sample_pop(fx))
    return bam, fa, hdr


def run_cli(argv):
    env = dict(os.environ, POPBAM_B200_NO_TABLE_CACHE="1")
    return subprocess.run([str(EXE)] + argv, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, env=env)


def test_cli_abba_needs_p(tmp_path):
    r = run_cli(["abba", "-w", "10", "-f", str(tmp_path / "x.fa"), str(tmp_path / "x.bam"), "chr1"])
    assert r.returncode == 1 and "abba needs -p SAMPLE" in r.stderr


@pytest.mark.parametrize("argv", [["nucdiv"], ["sfs", "-p", "og"], ["snp"]])
def test_cli_refuses_triple_elsewhere(argv, tmp_path):
    r = run_cli(argv + ["--triple", "P1,P2,P3", "-f", str(tmp_path / "x.fa"), str(tmp_path / "x.bam"), "chr1"])
    assert r.returncode == 1 and "--triple is only available for abba" in r.stderr


@pytest.mark.parametrize("extra,msg", [
    (["--triple", "P1,P2,PX"], "unknown population PX"),
    (["--triple", "P1,P2,P1"], "a population is repeated"),
    (["--triple", "P1,P2,out"], "is the outgroup's"),
    (["--triple", "P1,P2"], "expected three population names"),
    (["-p", "nobody"], "Specified outgroup nobody not found"),
])
def test_cli_refuses_bad_triples(extra, msg, c1_cli_files):
    bam, fa, hdr = c1_cli_files
    argv = ["abba", "-w", "10", "-h", hdr, "-f", fa] + (extra if extra[0] == "-p" else ["-p", "og"] + extra) + [bam, "chr1"]
    r = run_cli(argv)
    assert r.returncode == 1 and msg in r.stderr, r.stderr


def test_cli_refuses_fewer_than_three_ingroup_populations(c1_cli_files):
    bam, fa, _ = c1_cli_files       # the fixture's own grouping: A, B and the outgroup's population
    r = run_cli(["abba", "-w", "10", "-p", "og", "-f", fa, bam, "chr1"])
    assert r.returncode == 1 and "at least three populations besides the outgroup's" in r.stderr


def test_cli_refuses_a_default_list_over_the_limit(tmp_path):
    """20 ingroup populations give C(20, 2) * 18 = 3420 default triples: the message points to --triple."""
    fx = pbtest.fixture("ld")
    bam, fa = fx.write_files(tmp_path / "ld")
    pops = {s: ("Q%d" % (i % 20) if s != "og" else "out") for i, s in enumerate(fx.sample_names)}
    hdr = write_regrouped_header(bam, tmp_path / "h.sam", pops)
    r = run_cli(["abba", "-w", "10", "-p", "og", "-h", hdr, "-f", fa, bam, "chr1"])
    assert r.returncode == 1 and "--triple" in r.stderr and "3420" in r.stderr, r.stderr
