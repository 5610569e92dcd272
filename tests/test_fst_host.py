"""F_ST (Hudson; Weir & Cockerham) and Hudson's Snn between population pairs (PB_AN_FST, `nucdiv --fst`).  The reference
never computed them, so nothing it printed pins them directly.  Instead:
  * a numpy restatement of the per-site formulas and of the permutation stream must equal the plain-C restatement
    (tests/fst_oracle.c, on the result of the reference-pinned oracle) on every fixture;
  * Hudson's sums must be those the reference-pinned pi and dxy imply;
  * synthetic site sets check fixed differences, allele flips, swapped populations and exchangeable labels;
  * the permutation p-value must converge to the exact one from all C(m, n1) partitions of a small pool.
The GPU path is held to tests/fst_oracle.c in tests/test_fst_gpu.py."""
import ctypes as C
import itertools
import math
import subprocess

import numpy as np
import pytest

import pbtest
from cases import CASES, FIXTURES
from popbam_b200 import capi
from test_extra_stats_host import EXE

AN = capi.AN
FST = AN["FST"]
INT_FST = ["hud_num", "hud_den", "wc_num", "wc_den", "snn_ge"]
FLT_FST = ["fst_hudson", "fst_wc", "snn", "snn_p"]

# ---------------------------------------------------------------------------------------------------------------------
# numpy restatement

M64 = (1 << 64) - 1
GAMMA = 0x9E3779B97F4A7C15


def mix64(z):
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M64
    return z ^ (z >> 31)


def perm_key(seed, tid, win_beg, i, j, k):
    h = mix64((seed + GAMMA) & M64)
    for v in (tid, win_beg, i, j, k):
        h = mix64(((h ^ (v & M64)) + GAMMA) & M64)
    return h


def perm_partition(h, pool, n1):
    """Population i of one permutation: partial Fisher-Yates over the pooled samples in ascending order."""
    slots = list(pool)
    m = len(slots)
    A = 0
    for t in range(n1):
        z = mix64((h + (t + 1) * GAMMA) & M64)
        r = t + (((z >> 32) * (m - t)) >> 32)
        slots[t], slots[r] = slots[r], slots[t]
        A |= 1 << slots[t]
    return A


def site_terms(T, mi, mj, n1, n2):
    """Per-site integer terms (hud_num, hud_den, wc_num, wc_den) of the pair."""
    T = np.asarray(T, dtype=np.uint64)
    c1 = np.bitwise_count(T & np.uint64(mi)).astype(np.int64)
    c2 = np.bitwise_count(T & np.uint64(mj)).astype(np.int64)
    between = (n1 - 1) * (n2 - 1) * (c1 * (n2 - c2) + c2 * (n1 - c1))
    within = c1 * (n1 - c1) * n2 * (n2 - 1) + c2 * (n2 - c2) * n1 * (n1 - 1)
    d = c1 * n2 - c2 * n1
    msp = d * d * (n1 + n2 - 2)
    g = c1 * (n1 - c1) * n2 + c2 * (n2 - c2) * n1
    return between - within, between, msp - g * (n1 + n2), msp + g * (2 * n1 * n2 - n1 - n2)


def nn_masks(T, pool):
    """Nearest-neighbour mask of every pooled sample on the window's difference matrix (unsigned short)."""
    T = np.asarray(T, dtype=np.uint64)
    bits = {x: ((T >> np.uint64(x)) & np.uint64(1)).astype(np.int64) for x in pool}
    nn = {}
    for x in pool:
        d = {y: int(np.sum(bits[x] != bits[y])) & 0xFFFF for y in pool if y != x}
        best = min(d.values())
        nn[x] = sum(1 << y for y, v in d.items() if v == best)
    return nn


def snn_of(nn, pool, A):
    B = sum(1 << y for y in pool) & ~A
    s = 0.0
    for y in pool:
        own = A if A >> y & 1 else B
        s += float(bin(nn[y] & own).count("1")) / float(bin(nn[y]).count("1"))
    return s / float(len(pool))


def pair_stats(T, p, i, j, n_perms=0, seed=0, tid=0, win_beg=0):
    mi, mj = int(p.pop_mask[i]), int(p.pop_mask[j])
    n1, n2 = int(p.pop_nsmpl[i]), int(p.pop_nsmpl[j])
    hn, hd, wn, wd = (int(np.sum(t)) for t in site_terms(T, mi, mj, n1, n2))
    two = n1 >= 2 and n2 >= 2
    out = dict(hud_num=hn, hud_den=hd, wc_num=wn, wc_den=wd,
               fst_hudson=float(hn) / float(hd) if two and hd else np.nan,
               fst_wc=float(wn) / float(wd) if two and wd else np.nan, snn=np.nan, snn_p=np.nan, snn_ge=0)
    if not two:
        return out
    pool = [x for x in range(64) if (mi | mj) >> x & 1]
    nn = nn_masks(T, pool)
    out["snn"] = obs = snn_of(nn, pool, mi)
    if n_perms:
        ge = sum(snn_of(nn, pool, perm_partition(perm_key(seed, tid, win_beg, i, j, k), pool, n1)) >= obs - 1e-12 for k in range(n_perms))
        out["snn_ge"], out["snn_p"] = ge, (1.0 + ge) / (1.0 + n_perms)
    return out


def expected_fst(res, p, n_perms=0, seed=0, tid=0):
    d = pbtest.result_arrays(res)
    NW, P = res.n_windows, res.n_pops
    e = {k: np.zeros(NW * P * P, dtype=np.int64 if k in INT_FST else np.float64) for k in INT_FST + FLT_FST}
    for w in range(NW):
        T = d["seg_type"][d["seg_off"][w]:d["seg_off"][w + 1]]
        for i in range(P - 1):
            for j in range(i + 1, P):
                x = w * P * P + i * P + (j - (i + 1))
                for k, v in pair_stats(T, p, i, j, n_perms, seed, tid, int(d["win_beg"][w])).items():
                    e[k][x] = v
    return e


# ---------------------------------------------------------------------------------------------------------------------
# tests/fst_oracle.c

_fst_oracle = None


def fst_oracle_lib():
    global _fst_oracle
    if _fst_oracle is None:
        so = pbtest.ROOT / "tests" / "_build" / "libpbforacle.so"
        so.parent.mkdir(exist_ok=True)
        subprocess.check_call(["gcc", "-O2", "-std=c11", "-ffp-contract=off", "-fPIC", "-shared", "-Wall", "-Wextra", "-o", str(so),
                               str(pbtest.ROOT / "tests" / "fst_oracle.c"), "-lm"])
        L = C.CDLL(str(so))
        L.pbf_fst.argtypes = [C.POINTER(capi.Params), C.POINTER(capi.Result), C.c_int32, C.c_int64, C.c_uint64, C.POINTER(capi.Fst)]
        L.pbf_free.argtypes = [C.POINTER(capi.Fst)]
        L.pbf_columns.restype = C.c_int64
        L.pbf_columns.argtypes = [C.POINTER(capi.Result), C.POINTER(capi.Fst), C.c_int32, C.POINTER(capi.PrintOpts), C.c_char_p, C.c_int64]
        _fst_oracle = L
    return _fst_oracle


def fst_arrays(fst, res):
    """numpy copies of a pb_region_fst (empty where an array is NULL)."""
    n = res.n_windows * res.n_pops * res.n_pops
    return {k: pbtest.arr(getattr(fst, k), n) for k, _ in capi.Fst._fields_}


def oracle_fst(params, res, n_perms=0, seed=0, tid=0):
    L = fst_oracle_lib()
    f = capi.Fst()
    assert L.pbf_fst(C.byref(params), C.byref(res), tid, n_perms, seed, C.byref(f)) == 0
    out = fst_arrays(f, res)
    L.pbf_free(C.byref(f))
    return out


def oracle_fst_text(orc_text, params, res, opts, n_perms=0, seed=0, tid=0):
    """The oracle's nucdiv rows (with any theta columns) followed by the F_ST columns of tests/fst_oracle.c."""
    L = fst_oracle_lib()
    f = capi.Fst()
    assert L.pbf_fst(C.byref(params), C.byref(res), tid, n_perms, seed, C.byref(f)) == 0
    buf = C.create_string_buffer(1 << 16)
    out = []
    for w, row in enumerate(orc_text.splitlines()):
        k = L.pbf_columns(C.byref(res), C.byref(f), w, C.byref(opts), buf, len(buf))
        assert 0 <= k < len(buf)
        out.append(row + buf.raw[:k].decode() + "\n")
    L.pbf_free(C.byref(f))
    return "".join(out)


def assert_fst_same(got, want, keys=INT_FST + FLT_FST, snn_tol=0.0):
    for k in keys:
        a, b = got[k], want[k]
        assert a.shape == b.shape, (k, a.shape, b.shape)
        if k in INT_FST:
            assert np.array_equal(a, b), (k, a, b)
        elif k == "snn" and snn_tol:
            assert np.allclose(a, b, rtol=0.0, atol=snn_tol, equal_nan=True), (k, a, b)
        else:       # bit for bit, NaN where NaN
            assert np.array_equal(np.isnan(a), np.isnan(b)) and np.array_equal(a[~np.isnan(a)], b[~np.isnan(b)]), (k, a, b)


# ---------------------------------------------------------------------------------------------------------------------
# the oracle against the restatement, and against pi / dxy

@pytest.mark.parametrize("fxname", list(FIXTURES))
def test_oracle_fst_equals_restatement(fxname):
    fx = pbtest.fixture(fxname)
    p = fx.params()
    wb, we = pbtest.window_grid(0, fx.contig_len, 10000)
    orc = pbtest.OracleRun(p, fx.batch(), fx.ref(), AN["NUCDIV"], wb, we)
    got = oracle_fst(p, orc.res, n_perms=40, seed=7, tid=0)
    want = expected_fst(orc.res, p, n_perms=40, seed=7, tid=0)
    assert int(want["hud_den"].sum()) > 0
    assert_fst_same(got, want, INT_FST + ["fst_hudson", "fst_wc", "snn_p"])
    assert_fst_same(got, want, ["snn"], snn_tol=1e-12)
    # the outgroup's one-sample population: every pair with it is NaN
    P = fx.n_pops
    for w in range(orc.res.n_windows):
        for i in range(P - 1):
            for j in range(i + 1, P):
                x = w * P * P + i * P + (j - (i + 1))
                if min(p.pop_nsmpl[i], p.pop_nsmpl[j]) < 2:
                    assert np.isnan(got["snn"][x]) and np.isnan(got["fst_hudson"][x]) and np.isnan(got["fst_wc"][x])
                    assert np.isnan(got["snn_p"][x]) and got["snn_ge"][x] == 0
    orc.close()


@pytest.mark.parametrize("fxname", list(FIXTURES))
def test_hudson_sums_are_those_of_pi_and_dxy(fxname):
    """hud_den = dxy sum (n1-1)(n2-1) and hud_num = hud_den - (within sums), with the sums recovered from the
    reference-pinned piw / pib; so F_ST = 1 - (pi1 + pi2) / (2 dxy)."""
    fx = pbtest.fixture(fxname)
    p = fx.params()
    wb, we = pbtest.window_grid(0, fx.contig_len, 10000)
    orc = pbtest.OracleRun(p, fx.batch(), fx.ref(), AN["NUCDIV"], wb, we)
    f = oracle_fst(p, orc.res)
    d = pbtest.result_arrays(orc.res)
    P = fx.n_pops
    checked = 0
    for w in range(orc.res.n_windows):
        for i in range(P - 1):
            for j in range(i + 1, P):
                x = w * P * P + i * P + (j - (i + 1))
                n1, n2 = int(p.pop_nsmpl[i]), int(p.pop_nsmpl[j])
                between = round(d["pib"][x] * n1 * n2)
                w1 = round(d["piw"][w * P + i] * n1 * (n1 - 1) / 2)
                w2 = round(d["piw"][w * P + j] * n2 * (n2 - 1) / 2)
                assert f["hud_den"][x] == between * (n1 - 1) * (n2 - 1)
                assert f["hud_num"][x] == f["hud_den"][x] - (w1 * n2 * (n2 - 1) + w2 * n1 * (n1 - 1))
                if n1 >= 2 and n2 >= 2 and d["pib"][x] > 0:
                    pi1, pi2 = d["piw"][w * P + i], d["piw"][w * P + j]
                    assert abs(f["fst_hudson"][x] - (1.0 - (pi1 + pi2) / (2.0 * d["pib"][x]))) < 1e-12
                    checked += 1
    assert checked > 0
    orc.close()


# ---------------------------------------------------------------------------------------------------------------------
# synthetic site sets, through both restatements

class FakeRegion:
    """A pb_region_result with only what tests/fst_oracle.c reads: windows of given site types."""

    def __init__(self, windows, n, P, win_beg=None):
        self.types = np.ascontiguousarray(np.concatenate([np.asarray(t, dtype=np.uint64) for t in windows]) if windows else np.zeros(1, np.uint64))
        self.segs = np.array([len(t) for t in windows], dtype=np.int32)
        self.off = np.concatenate([[0], np.cumsum(self.segs)]).astype(np.int64)
        self.wb = np.array(win_beg if win_beg is not None else [100000 * k for k in range(len(windows))], dtype=np.int32)
        self.ns = np.full(len(windows), 10000, dtype=np.int32)
        r = capi.Result()
        r.n_windows, r.n_pops, r.n_samples = len(windows), P, n
        r.seg_type = self.types.ctypes.data_as(C.POINTER(C.c_uint64))
        r.segsites = self.segs.ctypes.data_as(C.POINTER(C.c_int32))
        r.seg_off = self.off.ctypes.data_as(C.POINTER(C.c_int64))
        r.win_beg = self.wb.ctypes.data_as(C.POINTER(C.c_int32))
        r.num_sites = self.ns.ctypes.data_as(C.POINTER(C.c_int32))
        self.res = r


def synth_params(sizes):
    p = capi.Params()
    p.n_samples, p.n_pops = sum(sizes), len(sizes)
    s = 0
    for k, m in enumerate(sizes):
        p.pop_mask[k] = ((1 << m) - 1) << s
        p.pop_nsmpl[k] = m
        s += m
    return p


def both(windows, sizes, n_perms=0, seed=3):
    """(oracle arrays, restatement arrays) of synthetic windows."""
    p = synth_params(sizes)
    fr = FakeRegion(windows, sum(sizes), len(sizes))
    return oracle_fst(p, fr.res, n_perms, seed), expected_fst_fake(fr, p, n_perms, seed)


def expected_fst_fake(fr, p, n_perms, seed):
    P = p.n_pops
    NW = len(fr.segs)
    e = {k: np.zeros(NW * P * P, dtype=np.int64 if k in INT_FST else np.float64) for k in INT_FST + FLT_FST}
    for w in range(NW):
        T = fr.types[fr.off[w]:fr.off[w + 1]]
        for i in range(P - 1):
            for j in range(i + 1, P):
                x = w * P * P + i * P + (j - (i + 1))
                for k, v in pair_stats(T, p, i, j, n_perms, seed, 0, int(fr.wb[w])).items():
                    e[k][x] = v
    if not n_perms:
        e["snn_p"] = np.zeros(0)
        e["snn_ge"] = np.zeros(0, dtype=np.int64)
    return e


def random_windows(rng, sizes, n_windows, sites, structure=0.0):
    """Random site types over the pooled samples; with structure > 0 population 0's allele frequency is pushed away."""
    n = sum(sizes)
    out = []
    for _ in range(n_windows):
        f = rng.uniform(0.05, 0.95, size=sites)
        prob = np.repeat(f[:, None], n, axis=1)
        prob[:, :sizes[0]] = np.clip(prob[:, :sizes[0]] + structure, 0, 1)
        bits = rng.random((sites, n)) < prob
        T = (bits.astype(np.uint64) << np.arange(n, dtype=np.uint64)).sum(axis=1).astype(np.uint64)
        full = np.uint64((1 << n) - 1)
        out.append(T[(T != 0) & (T != full)])
    return out


def test_fixed_differences_give_one():
    sizes = [5, 7, 4]
    p = synth_params(sizes)
    masks = [int(p.pop_mask[k]) for k in range(3)]
    # every site separates one population from the others: fixed between every pair
    T = [masks[0], masks[1], masks[2], masks[0] | masks[1], masks[1], masks[0]]
    got, want = both([T], sizes)
    assert_fst_same(got, want)
    for x in (0, 1, 3):            # (0,1), (0,2), (1,2) at i*P + (j-(i+1))
        assert got["fst_hudson"][x] == 1.0 and got["fst_wc"][x] == 1.0 and got["snn"][x] == 1.0


@pytest.mark.parametrize("sizes", [[4, 6], [8, 8], [3, 10, 2]])
def test_flipping_every_site_changes_nothing(sizes):
    rng = np.random.default_rng(sum(sizes))
    W = random_windows(rng, sizes, 3, 60, structure=0.2)
    full = np.uint64((1 << sum(sizes)) - 1)
    flipped = [(~t) & full for t in W]
    a, ra = both(W, sizes, n_perms=300)
    b, rb = both(flipped, sizes, n_perms=300)
    assert_fst_same(a, ra, INT_FST + ["fst_hudson", "fst_wc", "snn_p"])
    assert_fst_same(b, rb, INT_FST + ["fst_hudson", "fst_wc", "snn_p"])
    assert_fst_same(a, b)


@pytest.mark.parametrize("sizes", [[4, 6], [9, 3]])
def test_swapping_the_populations_changes_nothing(sizes):
    """The statistics are symmetric in i and j (the permutation stream is keyed on (i, j), so snn_ge is not compared)."""
    rng = np.random.default_rng(100 + sum(sizes))
    n = sum(sizes)
    W = random_windows(rng, sizes, 3, 80, structure=0.3)
    # the same samples, population 1 listed first: sample k of the swapped layout is sample (k + sizes[0]) % n
    perm = [(k + sizes[0]) % n for k in range(n)]
    swapped = []
    for t in W:
        bits = [(t >> np.uint64(perm[k])) & np.uint64(1) for k in range(n)]
        swapped.append(sum(b << np.uint64(k) for k, b in enumerate(bits)).astype(np.uint64))
    a, _ = both(W, sizes)
    b, _ = both(swapped, sizes[::-1])
    assert_fst_same(a, b, ["hud_num", "hud_den", "wc_num", "wc_den", "fst_hudson", "fst_wc"])
    assert_fst_same(a, b, ["snn"], snn_tol=1e-12)        # the X_x are summed in another order


@pytest.mark.parametrize("sizes", [[5, 5], [4, 9], [2, 12]])
def test_exchangeable_labels_give_numerators_of_mean_zero(sizes):
    """Identical populations: sample labels exchangeable, so E[hud_num] = E[wc_num] = 0 per site."""
    rng = np.random.default_rng(7 * sizes[0] + sizes[1])
    n1, n2 = sizes
    m = n1 + n2
    reps = 200_000
    k = rng.integers(1, m, size=reps)                           # derived copies in the pool
    keys = rng.random((reps, m))
    rank = np.argsort(np.argsort(keys, axis=1), axis=1)
    carries = rank < k[:, None]                                 # a uniformly random k-subset of the pool
    T = (carries.astype(np.uint64) << np.arange(m, dtype=np.uint64)).sum(axis=1).astype(np.uint64)
    mi, mj = (1 << n1) - 1, ((1 << n2) - 1) << n1
    hn, hd, wn, wd = site_terms(T, mi, mj, n1, n2)
    for num, den in ((hn, hd), (wn, wd)):
        num = num.astype(float)
        assert abs(num.mean()) < 4 * num.std() / math.sqrt(reps), (num.mean(), num.std())
        assert den.mean() > 0
    # with structure the numerators are positive
    W = random_windows(rng, sizes, 1, 5000, structure=0.3)[0]
    hn, hd, wn, wd = site_terms(W, mi, mj, n1, n2)
    assert hn.sum() > 0 and wn.sum() > 0


@pytest.mark.parametrize("sizes,structure", [([4, 5], 0.0), ([4, 5], 0.25), ([3, 6], 0.15), ([5, 5], 0.4)])
def test_permutation_p_value_converges_to_exact(sizes, structure):
    rng = np.random.default_rng(int(1000 * structure) + 10 * sizes[0] + sizes[1])
    W = random_windows(rng, sizes, 2, 40, structure=structure)
    n_perms = 20000
    got, _ = both(W, sizes, n_perms=n_perms, seed=11)
    p = synth_params(sizes)
    n1 = sizes[0]
    pool = list(range(sum(sizes)))
    for w, T in enumerate(W):
        x = w * 4 + 0
        nn = nn_masks(T, pool)
        obs = snn_of(nn, pool, int(p.pop_mask[0]))
        assert got["snn"][x] == obs
        parts = list(itertools.combinations(pool, n1))
        exact = sum(snn_of(nn, pool, sum(1 << s for s in c)) >= obs - 1e-12 for c in parts) / len(parts)
        est = got["snn_ge"][x] / n_perms
        se = math.sqrt(max(exact * (1 - exact), 1.0 / n_perms) / n_perms)
        assert abs(est - exact) <= 3 * se, (est, exact, se)
        assert got["snn_p"][x] == (1.0 + got["snn_ge"][x]) / (1.0 + n_perms)


def test_permutation_stream_is_the_documented_one():
    """The first draws of the documented generator, restated here and in tests/fst_oracle.c, give the same counts."""
    sizes = [6, 7]
    rng = np.random.default_rng(5)
    W = random_windows(rng, sizes, 3, 50, structure=0.1)
    got, want = both(W, sizes, n_perms=500, seed=2024)
    assert_fst_same(got, want, ["snn_ge", "snn_p"])
    assert mix64(0) == 0 and perm_key(0, 0, 0, 0, 0, 0) != perm_key(0, 0, 0, 0, 0, 1)


# ---------------------------------------------------------------------------------------------------------------------
# text: the product's printer against the oracle's columns

NUCDIV_CASES = [c for c in CASES if c[0] in ("nucdiv_c1", "nucdiv_c1_k", "nucdiv_n64", "nucdiv_edge")]


@pytest.fixture(scope="module")
def fmt():
    so = pbtest.ROOT / "tests" / "_build" / "libfmtharness_fst.so"
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
    return L


def split_fst(text, P, perms):
    """Each row -> (the row without the F_ST fields, the F_ST fields)."""
    k = 2 * (4 if perms else 3) * P * (P - 1) // 2
    out = []
    for row in text.splitlines():
        f = row.split("\t")
        out.append(("\t".join(f[:-k]), f[-k:]))
    return out


@pytest.mark.parametrize("perms", [0, 100])
@pytest.mark.parametrize("theta", [False, True])
@pytest.mark.parametrize("case", NUCDIV_CASES, ids=[c[0] for c in NUCDIV_CASES])
def test_product_printer_fst_text_equals_oracle(fmt, case, theta, perms):
    from test_extra_stats_host import OracleExtRun
    fx, p, an, wb, we, o = pbtest.case_setup(case)
    ext = AN["THETA_W"] if theta else 0
    orc = OracleExtRun(p, fx.batch(), fx.ref(), an | ext, wb, we)
    L = fst_oracle_lib()
    f = capi.Fst()
    assert L.pbf_fst(C.byref(p), C.byref(orc.res), 0, perms, 99, C.byref(f)) == 0
    orc.res.analyses |= FST          # as the product's result of a region run with PB_AN_FST
    fmt.fmt_set_params(C.byref(p))
    buf = C.create_string_buffer(1 << 20)
    out = []
    for w in range(orc.res.n_windows):
        k = fmt.pb_format_window_fst(None, C.byref(orc.res), C.byref(orc.ext), C.byref(f), w, an | ext | FST, C.byref(o), buf, len(buf))
        assert 0 <= k < len(buf)
        out.append(buf.raw[:k].decode())
    text = "".join(out)
    assert text == oracle_fst_text(orc.text(an | ext, o), p, orc.res, o, perms, 99, 0)
    # the reference's row, the theta columns, then per pair Fst, FstWC, Snn (+ SnnP)
    rows = split_fst(text, fx.n_pops, perms)
    assert [r for r, _ in rows] == orc.text(an | ext, o).splitlines()
    names = ["Fst", "FstWC", "Snn"] + (["SnnP"] if perms else [])
    pairs = ["%s-%s" % (a, b) for a, b in itertools.combinations(fx.pop_names, 2)]
    assert [c for c in rows[0][1][::2]] == ["%s[%s]:" % (nm, pr) for pr in pairs for nm in names]
    # without FST the new entry point prints what pb_format_window_ext prints
    k = fmt.pb_format_window_fst(None, C.byref(orc.res), C.byref(orc.ext), None, 0, an | ext, C.byref(o), buf, len(buf))
    assert buf.raw[:k].decode() == orc.text(an | ext, o, [0])
    # FST only through pb_format_window_fst, only with nucdiv, and only with the arrays
    assert fmt.pb_format_window_ext(None, C.byref(orc.res), C.byref(orc.ext), 0, an | FST, C.byref(o), buf, len(buf)) < 0
    assert fmt.pb_format_window(None, C.byref(orc.res), 0, an | FST, C.byref(o), buf, len(buf)) < 0
    assert fmt.pb_format_window_fst(None, C.byref(orc.res), C.byref(orc.ext), None, 0, an | FST, C.byref(o), buf, len(buf)) < 0
    L.pbf_free(C.byref(f))
    orc.close()


def test_printer_refuses_fst_with_other_analyses(fmt):
    case = [c for c in CASES if c[0] == "sfs_c1"][0]
    fx, p, an, wb, we, o = pbtest.case_setup(case)
    orc = pbtest.OracleRun(p, fx.batch(), fx.ref(), an | AN["NUCDIV"], wb, we)
    f = capi.Fst()
    L = fst_oracle_lib()
    assert L.pbf_fst(C.byref(p), C.byref(orc.res), 0, 0, 0, C.byref(f)) == 0
    fmt.fmt_set_params(C.byref(p))
    buf = C.create_string_buffer(1 << 16)
    orc.res.analyses = an | AN["NUCDIV"] | FST
    assert fmt.pb_format_window_fst(None, C.byref(orc.res), None, C.byref(f), 0, an | FST, C.byref(o), buf, len(buf)) < 0
    assert fmt.pb_format_window_fst(None, C.byref(orc.res), None, C.byref(f), 0, an | AN["NUCDIV"] | FST, C.byref(o), buf, len(buf)) < 0
    assert fmt.pb_format_window_fst(None, C.byref(orc.res), None, C.byref(f), 0, AN["NUCDIV"] | FST, C.byref(o), buf, len(buf)) > 0
    L.pbf_free(C.byref(f))
    orc.close()


# ---------------------------------------------------------------------------------------------------------------------
# command line

@pytest.mark.parametrize("argv", [["sfs"], ["ld", "-o", "0"], ["diverge"], ["haplo"], ["snp"], ["tree"]])
@pytest.mark.parametrize("opt", [["--fst"], ["--snn-perms", "10"], ["--seed", "5"]])
def test_cli_refuses_fst_elsewhere(argv, opt, tmp_path):
    r = subprocess.run([str(EXE)] + argv + opt + ["-f", str(tmp_path / "x.fa"), str(tmp_path / "x.bam"), "chr1"],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    assert r.returncode == 1 and "--fst, --snn-perms and --seed are only available for nucdiv" in r.stderr


@pytest.mark.parametrize("opt,msg", [(["--snn-perms", "10"], "go with --fst"), (["--fst", "--snn-perms", "-3"], "invalid value"),
                                     (["--fst", "--seed", "x"], "invalid value"), (["--fst", "--snn-perms", "3000000000"], "invalid value")])
def test_cli_checks_permutation_options(opt, msg, tmp_path):
    r = subprocess.run([str(EXE), "nucdiv"] + opt + ["-f", str(tmp_path / "x.fa"), str(tmp_path / "x.bam"), "chr1"],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    assert r.returncode == 1 and msg in r.stderr
