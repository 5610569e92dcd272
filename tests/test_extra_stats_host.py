"""Watterson's theta, Fu & Li's D / D* and Lewontin's D' (the --extra-stats columns; PB_AN_THETA_W, PB_AN_FULI,
PB_AN_LD_DPRIME).  The reference never computed them, so nothing it printed can pin them.  Instead:
  * a numpy restatement of the closed forms is checked against a neutral-coalescent simulation (the numerators have
    mean 0 and the variance the formulas' denominators estimate);
  * a plain-C restatement (tests/ext_oracle.c, on the result of the reference-pinned oracle) must equal that numpy
    restatement on the parity fixtures;
  * the extended text must be the golden row of the reference plus the appended columns.
The GPU path is held to the oracle in tests/test_extra_stats_gpu.py."""
import ctypes as C
import subprocess

import numpy as np
import pytest

import pbtest
from cases import CASES
from popbam_b200 import capi

AN = capi.AN
EXT = AN["THETA_W"] | AN["FULI"] | AN["LD_DPRIME"]
EXE = capi.PKG / "_build" / "popbam"


# ---------------------------------------------------------------------------------------------------------------------
# numpy restatement (same operation order as tests/ext_oracle.c and pb_stats.cuh)

def fuli_constants(n):
    """a1 = sum 1/i, a2 = sum 1/i^2 (i < n) and (u_D, v_D, u_D*, v_D*) of Fu & Li (1993) as corrected by Simonsen,
    Churchill & Aquadro (1995); n >= 3."""
    a1 = 0.0
    for j in range(1, n):
        a1 += 1.0 / j
    a2 = 0.0
    for j in range(1, n):
        a2 += 1.0 / (float(j) * float(j))
    nn = float(n)
    ap = a1 + 1.0 / nn
    r = nn / (nn - 1.0)
    c = 2.0 * (nn * a1 - 2.0 * (nn - 1.0)) / ((nn - 1.0) * (nn - 2.0))
    vd = 1.0 + a1 * a1 / (a2 + a1 * a1) * (c - (nn + 1.0) / (nn - 1.0))
    ud = a1 - 1.0 - vd
    d = c + (nn - 2.0) / ((nn - 1.0) * (nn - 1.0)) + 2.0 / (nn - 1.0) * (1.5 - (2.0 * ap - 3.0) / (nn - 2.0) - 1.0 / nn)
    vds = (r * r * a2 + a1 * a1 * d - 2.0 * nn * a1 * (a1 + 1.0) / ((nn - 1.0) * (nn - 1.0))) / (a1 * a1 + a2)
    uds = r * (a1 - r) - vds
    return a1, a2, ud, vd, uds, vds


def sfs_stats(xi, n, outgroup):
    """(S, theta_W, D, D*, eta_e, eta_s) of one spectrum xi[0..n] of a sample of n."""
    S = int(sum(xi[1:n]))
    ee = int(xi[1]) if n >= 2 else 0
    es = int(xi[1] + xi[n - 1]) if n >= 3 else ee
    thw = fd = fds = np.nan
    if n >= 2:
        a1 = 0.0
        for j in range(1, n):
            a1 += 1.0 / j
        thw = S / a1
        if n >= 3 and S > 0:
            a1, a2, ud, vd, uds, vds = fuli_constants(n)
            Sd, r = float(S), n / (n - 1.0)
            if outgroup:
                fd = (Sd - a1 * ee) / np.sqrt(ud * Sd + vd * Sd * Sd)
            if n >= 4:      # n = 3: eta_s = S and n/(n-1) = a1, so D* is 0 / 0
                fds = (r * Sd - a1 * es) / np.sqrt(uds * Sd + vds * Sd * Sd)
    return S, thw, fd, fds, ee, es


def dprime_stats(types, mask, n, min_freq):
    """(K, mean |D'|, complete pairs) over the SNPs with min_freq <= count <= n - min_freq (the ZnS pairs)."""
    t = np.asarray(types, dtype=np.uint64) & np.uint64(mask)
    m = np.bitwise_count(t).astype(np.int64)
    keep = (m >= min_freq) & (m <= n - min_freq)
    t, m = t[keep], m[keep]
    K = len(t)
    if K < 2:
        return K, np.nan, 0
    bits = ((t[:, None] >> np.arange(64, dtype=np.uint64)[None, :]) & np.uint64(1)).astype(np.int64)
    n11 = bits @ bits.T
    mj, mk = m[:, None], m[None, :]
    num = n * n11 - mj * mk
    dmax = np.where(num > 0, np.minimum(mj * (n - mk), (n - mj) * mk), np.minimum(mj * mk, (n - mj) * (n - mk)))
    iu = np.triu_indices(K, 1)
    a, dm = np.abs(num[iu]), dmax[iu]
    assert dm.min() >= 1 and dm.max() <= n * n // 4
    return K, float(np.sum(a / dm)) / (K * (K - 1) / 2.0), int(np.sum(a == dm))


# ---------------------------------------------------------------------------------------------------------------------
# neutral coalescent: the closed forms against simulated spectra

def coalescent_spectra(n, theta, reps, rng):
    """xi[r, j] = mutations carried by j of n sequences: random lineage pairs merge over n-1 intervals of rate k(k-1)/2;
    each branch receives Poisson(theta * t / 2) mutations into xi[descendants]."""
    desc = np.ones((reps, n), dtype=np.int64)
    xi = np.zeros(reps * (n + 1), dtype=np.int64)
    rows = np.arange(reps)
    for k in range(n, 1, -1):
        t = rng.exponential(2.0 / (k * (k - 1)), size=reps)
        mut = rng.poisson(theta * t[:, None] / 2.0, size=(reps, k))
        xi += np.bincount((rows[:, None] * (n + 1) + desc[:, :k]).ravel(), weights=mut.ravel(), minlength=reps * (n + 1)).astype(np.int64)
        i = rng.integers(0, k, size=reps)
        j = rng.integers(0, k - 1, size=reps)
        j += j >= i
        lo, hi = np.minimum(i, j), np.maximum(i, j)
        desc[rows, lo] += desc[rows, hi]
        desc[rows, hi] = desc[rows, k - 1]
    return xi.reshape(reps, n + 1)


@pytest.mark.parametrize("n", [4, 10, 30])
@pytest.mark.parametrize("theta", [2.0, 10.0])
def test_closed_forms_against_neutral_coalescent(n, theta):
    rng = np.random.default_rng(1000 * n + int(theta))
    reps = 100_000
    xi = coalescent_spectra(n, theta, reps, rng)
    S = xi[:, 1:n].sum(axis=1).astype(float)
    a1, a2, ud, vd, uds, vds = fuli_constants(n)
    # Watterson: E[S] = a1 theta
    assert abs(np.mean(S / a1) / theta - 1.0) < 4 * np.std(S / a1) / np.sqrt(reps) / theta
    for num, u, v in ((S - a1 * xi[:, 1], ud, vd),
                      (n / (n - 1.0) * S - a1 * (xi[:, 1] + xi[:, n - 1]), uds, vds)):
        assert abs(np.mean(num)) < 4 * np.std(num) / np.sqrt(reps)
        ratio = np.var(num) / np.mean(u * S + v * S * S)
        assert abs(ratio - 1.0) < 0.03, ratio


def test_restatement_handles_small_samples():
    xi = np.array([0, 3, 0])
    assert sfs_stats(xi, 2, True)[1] == 3.0 and np.isnan(sfs_stats(xi, 2, True)[2])
    assert sfs_stats(xi, 2, True)[4:] == (3, 3)
    assert np.isnan(sfs_stats(np.array([0, 0]), 1, True)[1])
    assert np.isnan(sfs_stats(np.zeros(6, int), 5, True)[3])


# ---------------------------------------------------------------------------------------------------------------------
# the oracle's arrays against the restatement

def expected_arrays(res, p):
    """The extension arrays of a pb_region_result / pbo_result recomputed from its own seg_type / seg_off."""
    d = pbtest.result_arrays(res)
    NW, P = res.n_windows, res.n_pops
    outg = bool(p.flags & pbtest.FLAG["OUTGROUP"])
    e = {k: [] for k in ("pop_segsites", "theta_w", "fuli_d", "fuli_ds", "fuli_eta_e", "fuli_eta_s", "ld_kept", "ld_dprime", "ld_complete")}
    for w in range(NW):
        T = d["seg_type"][d["seg_off"][w]:d["seg_off"][w + 1]]
        for i in range(P):
            n, mask = int(p.pop_nsmpl[i]), int(p.pop_mask[i])
            f = np.bitwise_count(T & np.uint64(mask)).astype(np.int64)
            if outg:
                flip = ((T >> np.uint64(p.outidx)) & np.uint64(1)).astype(bool)
                f = np.where(flip, n - f, f)
            xi = np.bincount(f, minlength=n + 1)[:n + 1]
            for k, v in zip(("pop_segsites", "theta_w", "fuli_d", "fuli_ds", "fuli_eta_e", "fuli_eta_s"), sfs_stats(xi, n, outg)):
                e[k].append(v)
            for k, v in zip(("ld_kept", "ld_dprime", "ld_complete"), dprime_stats(T, mask, n, p.min_freq)):
                e[k].append(v)
    return {k: np.array(v) for k, v in e.items()}


def ext_arrays(ext, res):
    """numpy copies of a pb_region_extras (empty where an array is NULL)."""
    NW, P = res.n_windows, res.n_pops
    return {k: pbtest.arr(getattr(ext, k), NW * P) for k, _ in capi.Extras._fields_}


_ext_oracle = None


def ext_oracle_lib():
    """tests/ext_oracle.c: the plain-C restatement of the extension statistics on the oracle's result."""
    global _ext_oracle
    if _ext_oracle is None:
        so = pbtest.ROOT / "tests" / "_build" / "libpbxoracle.so"
        so.parent.mkdir(exist_ok=True)
        subprocess.check_call(["gcc", "-O2", "-std=c11", "-ffp-contract=off", "-fPIC", "-shared", "-Wall", "-Wextra", "-o", str(so),
                               str(pbtest.ROOT / "tests" / "ext_oracle.c"), "-lm"])
        L = C.CDLL(str(so))
        L.pbx_extras.argtypes = [C.POINTER(capi.Params), C.POINTER(capi.Result), C.POINTER(capi.Extras)]
        L.pbx_free.argtypes = [C.POINTER(capi.Extras)]
        L.pbx_columns.restype = C.c_int64
        L.pbx_columns.argtypes = [C.POINTER(capi.Params), C.POINTER(capi.Result), C.POINTER(capi.Extras), C.c_int32, C.c_uint32,
                                  C.POINTER(capi.PrintOpts), C.c_char_p, C.c_int64]
        _ext_oracle = L
    return _ext_oracle


COMPANION = {AN["THETA_W"]: AN["NUCDIV"], AN["FULI"]: AN["SFS"], AN["LD_DPRIME"]: AN["LD_ZNS"]}


class OracleExtRun(pbtest.OracleRun):
    """The reference-pinned oracle's region (pbtest.OracleRun; with D' it also runs ZnS for the site count the Dp columns
    are gated by) plus the extension arrays and columns of tests/ext_oracle.c."""

    def __init__(self, params, batch, ref, analyses, win_beg, win_end):
        if analyses & AN["LD_DPRIME"]:
            analyses |= AN["LD_ZNS"]
        super().__init__(params, batch, ref, analyses, win_beg, win_end)
        self.X = ext_oracle_lib()
        self.ext = capi.Extras()
        assert self.X.pbx_extras(C.byref(params), C.byref(self.res), C.byref(self.ext)) == 0

    def text(self, analysis, opts, windows=None):
        ext = analysis & EXT
        an = analysis & ~EXT
        if not ext:
            return super().text(an, opts, windows)
        assert COMPANION[ext] == an
        rows = super().text(an, opts, windows).splitlines()
        buf = C.create_string_buffer(1 << 16)
        out = []
        for row, w in zip(rows, range(self.res.n_windows) if windows is None else windows):
            k = self.X.pbx_columns(C.byref(self.p), C.byref(self.res), C.byref(self.ext), w, ext, C.byref(opts), buf, len(buf))
            assert 0 <= k < len(buf)
            out.append(row + buf.raw[:k].decode() + "\n")
        return "".join(out)

    def arrays(self):
        return ext_arrays(self.ext, self.res)

    def close(self):
        if self.ext.theta_w:
            self.X.pbx_free(C.byref(self.ext))
        super().close()


INT_EXT = ["pop_segsites", "fuli_eta_e", "fuli_eta_s", "ld_kept", "ld_complete"]
FLT_EXT = ["theta_w", "fuli_d", "fuli_ds", "ld_dprime"]

VARIANTS = {"plain": {}, "og": "og", "mf2": dict(min_freq=2)}


def variant_params(fx, variant):
    if variant == "og":
        return fx.params(flags=pbtest.FLAG["OUTGROUP"], outidx=fx.n_samples - 1)
    return fx.params(**VARIANTS[variant])


@pytest.mark.parametrize("variant", list(VARIANTS))
@pytest.mark.parametrize("fxname", ["c1", "edge", "ld", "n64", "ldbig"])
def test_oracle_extension_arrays_equal_restatement(fxname, variant):
    fx = pbtest.fixture(fxname)
    p = variant_params(fx, variant)
    wb, we = pbtest.window_grid(0, fx.contig_len, 10000)
    orc = OracleExtRun(p, fx.batch(), fx.ref(), EXT, wb, we)
    got, want = orc.arrays(), expected_arrays(orc.res, p)
    assert int(want["pop_segsites"].sum()) > 0 and (variant == "mf2" or int(want["ld_kept"].sum()) > 0)
    for k in INT_EXT:
        assert np.array_equal(got[k], want[k].astype(got[k].dtype)), k
    for k in FLT_EXT:
        assert np.allclose(got[k], want[k], rtol=1e-12, atol=0.0, equal_nan=True), (k, got[k], want[k])
    if variant != "og":
        assert np.isnan(got["fuli_d"]).all()
    orc.close()


# ---------------------------------------------------------------------------------------------------------------------
# text: the reference's row, then the extension's columns

EXT_OF = {"NUCDIV": "THETA_W", "SFS": "FULI", "LD_ZNS": "LD_DPRIME"}
TEXT_CASES = [c for c in CASES if c[0] in ("nucdiv_c1", "sfs_c1", "sfs_c1_og", "ld0_c1", "ld0_ldbig")]


def appended_columns(case, p, P):
    """Fields (name/value pairs) the extension appends per population."""
    if case[3] == "NUCDIV":
        return 1
    if case[3] == "SFS":
        return 2 if p.flags & pbtest.FLAG["OUTGROUP"] else 1
    return 2


def split_extended(text, ncols, P):
    """Each row -> (the row without the appended fields, the appended fields)."""
    out = []
    for row in text.splitlines():
        f = row.split("\t")
        k = 2 * ncols * P
        out.append(("\t".join(f[:-k]), f[-k:]))
    return out


@pytest.mark.parametrize("case", TEXT_CASES, ids=[c[0] for c in TEXT_CASES])
def test_oracle_extended_text_is_golden_row_plus_columns(case):
    fx, p, an, wb, we, o = pbtest.case_setup(case)
    ext = AN[EXT_OF[case[3]]]
    orc = OracleExtRun(p, fx.batch(), fx.ref(), an | ext, wb, we)
    text = orc.text(an | ext, o)
    golden = pbtest.golden_text(case).splitlines()
    P = fx.n_pops
    rows = split_extended(text, appended_columns(case, p, P), P)
    assert [r[0] for r in rows] == golden
    d, e = pbtest.result_arrays(orc.res), orc.arrays()
    for w, (_, cols) in enumerate(rows):
        ns = int(d["num_sites"][w])
        for i, name in enumerate(fx.pop_names):
            x = w * P + i
            if case[3] == "NUCDIV":
                want = [("theta[%s]:" % name, "%.5f" % (e["theta_w"][x] / ns) if not np.isnan(e["theta_w"][x]) and ns >= o.min_sites else "%7s" % "NA")]
            elif case[3] == "SFS":
                fmt = lambda v: "%7s" % "NA" if np.isnan(v) else "%.5f" % v  # noqa: E731
                want = [("FuLiD*[%s]:" % name, fmt(e["fuli_ds"][x]))]
                if p.flags & pbtest.FLAG["OUTGROUP"]:
                    want.append(("FuLiD[%s]:" % name, fmt(e["fuli_d"][x])))
            else:
                good = d["ld_num_snps"][x] >= o.min_snps and e["ld_kept"][x] >= 2
                want = [("Dp[%s]:" % name, "%.5f" % e["ld_dprime"][x] if good else "%7s" % "NA"),
                        ("Dp1[%s]:" % name, "%d" % e["ld_complete"][x] if good else "%7s" % "NA")]
            k = len(want)
            assert [tuple(cols[2 * (i * k + j):2 * (i * k + j) + 2]) for j in range(k)] == want
    # without the extension bit the text is unchanged, through both printers
    assert orc.text(an, o) == pbtest.golden_text(case)
    assert pbtest.OracleRun.text(orc, an, o) == pbtest.golden_text(case)
    orc.close()


@pytest.fixture(scope="module")
def fmt():
    so = pbtest.ROOT / "tests" / "_build" / "libfmtharness_ext.so"
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
    return L


@pytest.mark.parametrize("case", TEXT_CASES, ids=[c[0] for c in TEXT_CASES])
def test_product_printer_extended_text_equals_oracle(fmt, case):
    fx, p, an, wb, we, o = pbtest.case_setup(case)
    ext = AN[EXT_OF[case[3]]]
    orc = OracleExtRun(p, fx.batch(), fx.ref(), an | EXT, wb, we)
    fmt.fmt_set_params(C.byref(p))
    buf = C.create_string_buffer(1 << 20)
    out = []
    for w in range(orc.res.n_windows):
        k = fmt.pb_format_window_ext(None, C.byref(orc.res), C.byref(orc.ext), w, an | ext, C.byref(o), buf, len(buf))
        assert 0 <= k < len(buf)
        out.append(buf.raw[:k].decode())
    assert "".join(out) == orc.text(an | ext, o)
    # an extension only goes with its own reference bit, needs the extension arrays, and only through pb_format_window_ext
    other = AN["FULI"] if ext != AN["FULI"] else AN["THETA_W"]
    assert fmt.pb_format_window_ext(None, C.byref(orc.res), C.byref(orc.ext), 0, an | other, C.byref(o), buf, len(buf)) < 0
    assert fmt.pb_format_window_ext(None, C.byref(orc.res), None, 0, an | ext, C.byref(o), buf, len(buf)) < 0
    assert fmt.pb_format_window(None, C.byref(orc.res), 0, an | ext, C.byref(o), buf, len(buf)) < 0
    orc.close()


@pytest.mark.parametrize("argv", [["diverge"], ["ld", "-o", "1"], ["ld", "-o", "2"], ["haplo"], ["snp"], ["tree"]])
def test_cli_refuses_extra_stats_elsewhere(argv, tmp_path):
    r = subprocess.run([str(EXE)] + argv + ["--extra-stats", "-f", str(tmp_path / "x.fa"), str(tmp_path / "x.bam"), "chr1"],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    assert r.returncode == 1 and "--extra-stats is only available for nucdiv, sfs and ld -o 0" in r.stderr
