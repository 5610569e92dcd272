"""Site frequency spectra of one to three populations (PB_AN_SPECTRUM, `popbam sfs --jsfs`).  The reference never wrote a
spectrum out, so nothing it printed pins the counts directly.  Instead:
  * a numpy restatement written from the definition (np.histogramdd over the derived-allele counts, plus the sites without
    a segregating call in the all-zero bin) must equal the plain-C restatement (tests/spectrum_oracle.c) exactly, on
    synthetic windows and on every fixture;
  * an anchor to the reference: on the six sfs golden cases the one-population spectra give the reference's number of
    segregating sites, and Tajima's D and Fay & Wu's H recomputed from them print as the golden D[pop] / H[pop] columns;
  * the properties a spectrum must have (sums, marginals, transposition, complementing a site);
  * pb_format_spectrum_dadi's text, read back by a small reader of dadi's format, and the command line's refusals.
The GPU path is held to tests/spectrum_oracle.c in tests/test_spectrum_gpu.py.

Definition (include/popbam_b200.h, pb_region_spectrum): per segregating site a_k = popcount(seg_type & pop_mask[P_k]),
all a_k -> n_k - a_k when PB_FLAG_OUTGROUP is set and sample outidx carries the derived allele; bin (a1, a2, a3) row-major
with the last population fastest; num_sites - segsites more sites in the all-zero bin."""
import ctypes as C
import math
import subprocess

import numpy as np
import pytest

import pbtest
from cases import CASES, FIXTURES
from popbam_b200 import capi
from test_abba_host import run_cli
from test_fst_host import FakeRegion, synth_params

AN = capi.AN
SPECTRUM = AN["SPECTRUM"]
OUTGROUP = pbtest.FLAG["OUTGROUP"]

# ---------------------------------------------------------------------------------------------------------------------
# numpy restatement from the definition


def pad(s):
    return (list(s) + [-1, -1])[:3]


def default_sets(P, og=-1):
    """Every population, then every pair i < j (dxy order), without population og."""
    ks = [i for i in range(P) if i != og]
    return [(i,) for i in ks] + [(i, j) for i in ks for j in ks if i < j]


def set_shape(p, s):
    return tuple(int(p.pop_nsmpl[k]) + 1 for k in s if k >= 0)


def expected_spectrum(windows, num_sites, p, sets):
    """[NW*B] int64 from the definition; windows = list of arrays of seg_type words."""
    n = p.n_samples
    outg = bool(p.flags & OUTGROUP)
    out = []
    for T, ns in zip(windows, num_sites):
        T = np.asarray(T, dtype=np.uint64)
        bits = ((T[:, None] >> np.arange(n, dtype=np.uint64)[None, :]) & np.uint64(1)).astype(np.int64)     # [S, n]
        flip = bits[:, p.outidx].astype(bool) if outg and len(T) else np.zeros(len(T), bool)
        for s in sets:
            ks = [k for k in s if k >= 0]
            cols = []
            for k in ks:
                members = [i for i in range(n) if int(p.pop_mask[k]) >> i & 1]
                a = bits[:, members].sum(axis=1)
                cols.append(np.where(flip, int(p.pop_nsmpl[k]) - a, a))
            shape = set_shape(p, ks)
            h, _ = np.histogramdd(np.stack(cols, axis=1).astype(np.float64) if len(T) else np.zeros((0, len(ks))),
                                  bins=[np.arange(m + 1) - 0.5 for m in shape])
            h = h.astype(np.int64)
            h.flat[0] += int(ns) - len(T)
            out.append(h.ravel())
    return np.concatenate(out) if out else np.zeros(0, np.int64)


# ---------------------------------------------------------------------------------------------------------------------
# tests/spectrum_oracle.c

_spectrum_oracle = None


def spectrum_oracle_lib():
    global _spectrum_oracle
    if _spectrum_oracle is None:
        so = pbtest.ROOT / "tests" / "_build" / "libpbsoracle.so"
        so.parent.mkdir(exist_ok=True)
        subprocess.check_call(["gcc", "-O2", "-std=c11", "-fPIC", "-shared", "-Wall", "-Wextra", "-o", str(so),
                               str(pbtest.ROOT / "tests" / "spectrum_oracle.c")])
        L = C.CDLL(str(so))
        L.pbs_spectrum.argtypes = [C.POINTER(capi.Params), C.POINTER(capi.Result), C.c_int32, C.POINTER(C.c_int32), C.POINTER(capi.Spectrum)]
        L.pbs_free.argtypes = [C.POINTER(capi.Spectrum)]
        _spectrum_oracle = L
    return _spectrum_oracle


def spectrum_arrays(sp, res):
    """(counts [NW*B], set_off [NS+1], sets [3*NS]) of a pb_region_spectrum (empty where an array is NULL)."""
    return (pbtest.arr(sp.counts, res.n_windows * sp.n_bins).astype(np.int64), pbtest.arr(sp.set_off, sp.n_sets + 1 if sp.set_off else 0),
            pbtest.arr(sp.sets, 3 * sp.n_sets))


def oracle_spectrum(params, res, sets):
    L = spectrum_oracle_lib()
    flat = np.ascontiguousarray([k for s in sets for k in pad(s)], dtype=np.int32)
    sp = capi.Spectrum()
    assert L.pbs_spectrum(C.byref(params), C.byref(res), len(sets), flat.ctypes.data_as(C.POINTER(C.c_int32)), C.byref(sp)) == 0
    counts, off, got_sets = spectrum_arrays(sp, res)
    assert np.array_equal(got_sets, flat)
    L.pbs_free(C.byref(sp))
    return counts, off


def window_sets(counts, off, p, sets, NW):
    """counts [NW*B] -> [window][set] arrays of the set's shape."""
    B = int(off[-1])
    return [[counts[w * B + off[i]:w * B + off[i + 1]].reshape(set_shape(p, pad(s))) for i, s in enumerate(sets)] for w in range(NW)]


def seg_windows(res):
    d = pbtest.result_arrays(res)
    return [d["seg_type"][d["seg_off"][w]:d["seg_off"][w + 1]] for w in range(res.n_windows)], d["num_sites"]


def fixture_params(fx, outgroup):
    if outgroup and "og" in fx.sample_names:
        return fx.params(flags=OUTGROUP, outidx=fx.sample_names.index("og"))
    return fx.params()


def fixture_sets(P):
    sets = default_sets(P)
    if P >= 3:
        sets += [(0, 1, 2), (2, 1, 0), (1, 0)]
    return sets


# ---------------------------------------------------------------------------------------------------------------------
# the two restatements agree

@pytest.mark.parametrize("outgroup", [False, True], ids=["ref", "og"])
@pytest.mark.parametrize("win", [200, 1000, 10000])
@pytest.mark.parametrize("fxname", list(FIXTURES))
def test_oracle_equals_numpy_on_fixtures(fxname, win, outgroup):
    fx = pbtest.fixture(fxname)
    p = fixture_params(fx, outgroup)
    wb, we = pbtest.window_grid(0, fx.contig_len, win)
    orc = pbtest.OracleRun(p, fx.batch(), fx.ref(), AN["NUCDIV"], wb, we)
    sets = fixture_sets(p.n_pops)
    got, _ = oracle_spectrum(p, orc.res, sets)
    W, ns = seg_windows(orc.res)
    assert np.array_equal(got, expected_spectrum(W, ns, p, sets))
    orc.close()


SIZES = [[64], [1, 63], [32, 32], [31, 33], [10, 1], [5, 7, 4, 1], [2, 2, 2], [20, 20, 20, 4], [1] * 8, [3, 60, 1], [21, 21, 21, 1]]


def random_sets(rng, P, k):
    out = []
    for _ in range(k):
        d = int(rng.integers(1, min(3, P) + 1))
        out.append(tuple(int(x) for x in rng.permutation(P)[:d]))
    return out


def fake(windows, sizes, outidx=None, num_sites=None):
    p = synth_params(sizes)
    if outidx is not None:
        p.flags, p.outidx = OUTGROUP, outidx
    fr = FakeRegion(windows, sum(sizes), len(sizes))
    if num_sites is not None:
        fr.ns[:] = num_sites
    return p, fr


@pytest.mark.parametrize("outgroup", [False, True], ids=["ref", "og"])
@pytest.mark.parametrize("sizes", SIZES, ids=["-".join(map(str, s)) for s in SIZES])
def test_oracle_equals_numpy_on_random_windows(sizes, outgroup):
    rng = np.random.default_rng(sum(s * 13 ** i for i, s in enumerate(sizes)) + outgroup)
    n, P = sum(sizes), len(sizes)
    full = (1 << n) - 1 if n < 64 else (1 << 64) - 1
    # skewed allele counts as well as uniform ones, 0 to 300 sites
    W = []
    for _ in range(8):
        S = int(rng.integers(0, 301))
        q = rng.uniform(0.01, 0.99, size=S)[:, None]
        bits = rng.random((S, n)) < q
        W.append((bits.astype(np.uint64) << np.arange(n, dtype=np.uint64)[None, :]).sum(axis=1).astype(np.uint64) & np.uint64(full))
    W.append(np.zeros(0, np.uint64))
    sets = default_sets(P) + random_sets(rng, P, 6)
    p, fr = fake(W, sizes, int(rng.integers(0, n)) if outgroup else None)
    got, off = oracle_spectrum(p, fr.res, sets)
    assert np.array_equal(got, expected_spectrum(W, fr.ns, p, sets))
    # every window's set sums to num_sites
    for w in window_sets(got, off, p, sets, len(W)):
        assert all(int(x.sum()) == 10000 for x in w)


# ---------------------------------------------------------------------------------------------------------------------
# anchor to the reference: the sfs golden cases

SFS_CASES = [c for c in CASES if c[0].startswith("sfs")]


def tajima_fay_wu(x, m):
    """Tajima's D and Fay & Wu's H from a one-population spectrum x[0..m], as k_window_stats computes them."""
    ns = int(sum(int(v) for v in x[1:m]))
    if not (ns > 0 and m > 1):
        return float("nan"), float("nan"), ns
    a1 = a2 = a2n1 = 0.0
    for j in range(1, m):
        a1 += 1.0 / j
    for j in range(1, m):
        a2 += 1.0 / (j * j)
    for j in range(1, m + 1):
        a2n1 += 1.0 / (j * j)
    b1 = (m + 1.0) / (3.0 * (m - 1))
    e1 = (b1 - (1.0 / a1)) / a1
    b2 = (2.0 * ((m * m) + m + 3.0)) / (9.0 * m * (m - 1))
    e2 = (b2 - ((m + 2.0) / (a1 * m)) + (a2 / (a1 * a1))) / ((a1 * a1) + a2)
    td = fwh = 0.0
    for j in range(1, m):
        td += int(x[j]) * (((2.0 * j * (m - j)) / (m * (m - 1))) - (1.0 / a1))
        fwh += int(x[j]) * ((1.0 / a1) - (j / (m - 1)))
    with np.errstate(all="ignore"):     # IEEE division and square root, as in C (m = 3 gives 0 / 0)
        td = np.float64(td) / np.sqrt(np.float64(e1 * ns + e2 * ns * (ns - 1)))
        fwh = np.float64(fwh) / np.sqrt(np.float64(((m - 2) * (ns / a1) / (6.0 * (m - 1))) +
                                                   ((ns * (ns - 1) / ((a1 * a1) + a2)) *
                                                    (18.0 * (m * m) * (3.0 * m + 2.0) * a2n1 - (88.0 * m * m * m + 9.0 * (m * m) - 13.0 * m + 6.0)) /
                                                    (9.0 * m * ((m - 1) * (m - 1))))))
    return float(td), float(fwh), ns


def fmt5(v):
    return "%7s" % "NA" if math.isnan(v) else "%.5f" % v


@pytest.mark.parametrize("case", SFS_CASES, ids=[c[0] for c in SFS_CASES])
def test_one_population_spectra_give_the_golden_sfs_rows(case):
    fx, p, an, wb, we, o = pbtest.case_setup(case)
    orc = pbtest.OracleRun(p, fx.batch(), fx.ref(), an, wb, we)
    d = pbtest.result_arrays(orc.res)
    P, NW = p.n_pops, orc.res.n_windows
    sets = [(k,) for k in range(P)]
    counts, off = oracle_spectrum(p, orc.res, sets)
    rows = pbtest.golden_text(case).splitlines()
    assert len(rows) == NW
    for w in range(NW):
        f = rows[w].split("\t")
        assert int(f[3]) == d["num_sites"][w]
        x = window_sets(counts, off, p, sets, NW)[w]
        for k in range(P):
            m = int(p.pop_nsmpl[k])
            td, fwh, ns = tajima_fay_wu(x[k], m)
            assert ns == d["sfs_num_snps"][w * P + k]
            assert f[4 + 4 * k] == "D[%s]:" % fx.pop_names[k] and f[5 + 4 * k] == fmt5(td)
            assert f[6 + 4 * k] == "H[%s]:" % fx.pop_names[k] and f[7 + 4 * k] == fmt5(fwh)
            assert int(x[k].sum()) == d["num_sites"][w]
    assert d["sfs_num_snps"].max() > 0
    orc.close()


# ---------------------------------------------------------------------------------------------------------------------
# properties

def rand_windows(rng, n, k, smax=300):
    full = np.uint64((1 << n) - 1 if n < 64 else (1 << 64) - 1)
    return [rng.integers(0, 1 << 63, size=int(rng.integers(0, smax)), dtype=np.uint64) * np.uint64(2) + rng.integers(0, 2, dtype=np.uint64) & full
            for _ in range(k)]


@pytest.mark.parametrize("outgroup", [False, True], ids=["ref", "og"])
@pytest.mark.parametrize("sizes", [[7, 9, 5], [21, 21, 21, 1], [3, 1, 2], [30, 2, 32]])
def test_marginals_and_transposition(sizes, outgroup):
    rng = np.random.default_rng(sum(sizes) + 5 * outgroup)
    n = sum(sizes)
    W = rand_windows(rng, n, 6)
    sets = [(0,), (1,), (2,), (0, 1), (1, 2), (0, 2), (0, 1, 2), (2, 1, 0), (1, 0), (1, 2, 0)]
    p, fr = fake(W, sizes, n - 1 if outgroup else None, num_sites=[len(t) + 17 * i for i, t in enumerate(W)])
    counts, off = oracle_spectrum(p, fr.res, sets)
    for w, x in enumerate(window_sets(counts, off, p, sets, len(W))):
        a, b, c, ab, bc, ac, abc, cba, ba, bca = x
        assert all(int(v.sum()) == fr.ns[w] for v in x)
        assert np.array_equal(ab.sum(axis=1), a) and np.array_equal(ab.sum(axis=0), b)
        assert np.array_equal(abc.sum(axis=2), ab) and np.array_equal(abc.sum(axis=0), bc) and np.array_equal(abc.sum(axis=1), ac)
        assert np.array_equal(abc.sum(axis=(1, 2)), a)
        assert np.array_equal(ba, ab.T) and np.array_equal(cba, abc.transpose(2, 1, 0)) and np.array_equal(bca, abc.transpose(1, 2, 0))


@pytest.mark.parametrize("sizes", [[64], [12, 20, 1], [5, 6]])
def test_complementing_a_site_maps_a_to_n_minus_a(sizes):
    """Without the outgroup flip, ~t (within the samples) moves a site from bin (a_k) to bin (n_k - a_k).  Only the
    segregating sites are compared: num_sites = segsites, so nothing is added to the all-zero bin."""
    rng = np.random.default_rng(11 + sum(sizes))
    n, P = sum(sizes), len(sizes)
    full = np.uint64((1 << n) - 1 if n < 64 else (1 << 64) - 1)
    W = rand_windows(rng, n, 5)
    sets = default_sets(P) + ([(0, 1, 2)] if P >= 3 else [])
    p, fr = fake(W, sizes, None, num_sites=[len(t) for t in W])
    a, off = oracle_spectrum(p, fr.res, sets)
    Wc = [(~t & full).astype(np.uint64) for t in W]
    p2, fr2 = fake(Wc, sizes, None, num_sites=[len(t) for t in W])
    b, _ = oracle_spectrum(p2, fr2.res, sets)
    for xa, xb in zip(window_sets(a, off, p, sets, len(W)), window_sets(b, off, p, sets, len(W))):
        for u, v in zip(xa, xb):
            assert np.array_equal(u, np.flip(v))
    # the outgroup flip is the complement as seen from the outgroup: a site the outgroup sample carries counts as ~t
    og = n - 1
    q, frq = fake(W, sizes, og, num_sites=[len(t) for t in W])
    c, _ = oracle_spectrum(q, frq.res, sets)
    Wm = [np.where((t >> np.uint64(og)) & np.uint64(1), ~t & full, t).astype(np.uint64) for t in W]
    p3, fr3 = fake(Wm, sizes, None, num_sites=[len(t) for t in W])
    d, _ = oracle_spectrum(p3, fr3.res, sets)
    assert np.array_equal(c, d)


# ---------------------------------------------------------------------------------------------------------------------
# pb_format_spectrum_dadi through tests/fmt_harness.cpp

@pytest.fixture(scope="module")
def fmt():
    so = pbtest.ROOT / "tests" / "_build" / "libfmtharness_spectrum.so"
    so.parent.mkdir(exist_ok=True)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-o", str(so), str(pbtest.ROOT / "tests" / "fmt_harness.cpp"),
                           str(pbtest.ROOT / "popbam_b200" / "csrc" / "pb_format.cpp")])
    L = C.CDLL(str(so))
    L.fmt_set_params.argtypes = [C.POINTER(capi.Params)]
    L.pb_format_spectrum_dadi.restype = C.c_int64
    L.pb_format_spectrum_dadi.argtypes = [C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_int64), C.POINTER(capi.PrintOpts), C.c_char_p,
                                          C.c_char_p, C.c_int64]
    return L


def read_dadi(text):
    """A reader of dadi's spectrum file written from its format: '#' comment lines, then the shape line (dimensions,
    optionally 'folded' / 'unfolded', optionally quoted population names), the data line and an optional mask line."""
    lines = text.split("\n")
    assert lines[-1] == "" and all(ln for ln in lines[:-1])
    lines = lines[:-1]
    comments = [ln[2:] for ln in lines if ln.startswith("#")]
    body = [ln for ln in lines if not ln.startswith("#")]
    assert len(body) == 3
    head = body[0]
    names = []
    if '"' in head:
        q = head.index('"')
        names = head[q:].split('"')[1::2]
        assert head[q:] == " ".join('"%s"' % x for x in names)
        head = head[:q].rstrip()
    tok = head.split(" ")
    folded = None
    if tok[-1] in ("folded", "unfolded"):
        folded = tok.pop() == "folded"
    shape = tuple(int(t) for t in tok)
    assert "  " not in body[1] and "  " not in body[2]
    data = np.array([int(t) for t in body[1].split(" ")], dtype=np.int64).reshape(shape)
    mask = np.array([int(t) for t in body[2].split(" ")], dtype=np.int64).reshape(shape)
    return comments, shape, folded, names, data, mask


@pytest.mark.parametrize("sizes,s", [([5, 5, 1], (0,)), ([5, 5, 1], (1, 0)), ([32, 31, 1], (0, 1)), ([21, 21, 22], (2, 0, 1)),
                                      ([1, 3], (0,)), ([4, 1, 2], (1, 2, 0))])
def test_dadi_text_reads_back(fmt, sizes, s):
    p = synth_params(sizes)
    fmt.fmt_set_params(C.byref(p))
    names = ["pop%c" % chr(65 + i) for i in range(len(sizes))]
    keep = (C.c_char_p * len(sizes))(*[x.encode() for x in names])
    o = capi.PrintOpts()
    o.pop_names = keep
    shape = set_shape(p, pad(s))
    rng = np.random.default_rng(len(shape) + sum(sizes))
    x = rng.integers(0, 1 << 40, size=int(np.prod(shape)), dtype=np.int64)
    s3 = (C.c_int32 * 3)(*pad(s))
    xp = x.ctypes.data_as(C.POINTER(C.c_int64))
    comment = b"popbam sfs chr1:1-30500, 4 windows, 123 sites, polarised by og"
    k = fmt.pb_format_spectrum_dadi(None, s3, xp, C.byref(o), comment, None, 0)
    assert k > 0
    buf = C.create_string_buffer(int(k) + 1)
    assert fmt.pb_format_spectrum_dadi(None, s3, xp, C.byref(o), comment, buf, len(buf)) == k
    text = buf.raw[:k].decode()
    comments, got_shape, folded, got_names, data, mask = read_dadi(text)
    assert comments == [comment.decode()] and got_shape == shape and folded is False
    assert got_names == [names[i] for i in s] and np.array_equal(data.ravel(), x)
    want_mask = np.zeros(shape, np.int64)
    want_mask.flat[0] = 1
    want_mask[tuple(m - 1 for m in shape)] = 1
    assert np.array_equal(mask, want_mask)
    # cap: too small returns the size it needs and writes a NUL-terminated prefix
    small = C.create_string_buffer(16)
    assert fmt.pb_format_spectrum_dadi(None, s3, xp, C.byref(o), comment, small, 16) == k
    assert small.raw[:15] == buf.raw[:15] and small.raw[15:16] == b"\0"
    assert fmt.pb_format_spectrum_dadi(None, s3, xp, C.byref(o), comment, buf, k) == k and buf.raw[k - 1:k] == b"\0"
    # without a comment, and a comment of two lines
    t0 = C.create_string_buffer(int(k) + 1)
    k0 = fmt.pb_format_spectrum_dadi(None, s3, xp, C.byref(o), None, t0, len(t0))
    assert t0.raw[:k0].decode() == text.split("\n", 1)[1]
    k2 = fmt.pb_format_spectrum_dadi(None, s3, xp, C.byref(o), b"one\ntwo", None, 0)
    t2 = C.create_string_buffer(int(k2) + 1)
    fmt.pb_format_spectrum_dadi(None, s3, xp, C.byref(o), b"one\ntwo", t2, len(t2))
    assert read_dadi(t2.raw[:k2].decode())[0] == ["one", "two"]


@pytest.mark.parametrize("bad", [(-1, -1, -1), (-1, 0, -1), (0, -1, 1), (0, 0, -1), (3, -1, -1), (0, 1, 1), (-2, -1, -1)])
def test_dadi_printer_refuses_bad_sets(fmt, bad):
    p = synth_params([5, 5, 1])
    fmt.fmt_set_params(C.byref(p))
    keep = (C.c_char_p * 3)(b"A", b"B", b"C")
    o = capi.PrintOpts()
    o.pop_names = keep
    x = np.zeros(1000, np.int64)
    assert fmt.pb_format_spectrum_dadi(None, (C.c_int32 * 3)(*bad), x.ctypes.data_as(C.POINTER(C.c_int64)), C.byref(o), b"c", None, 0) < 0


# ---------------------------------------------------------------------------------------------------------------------
# command line: refusals before any GPU is touched

@pytest.mark.parametrize("argv", [["nucdiv"], ["haplo"], ["ld", "-o", "0"], ["diverge"], ["snp"], ["tree"], ["abba", "-p", "og"]])
@pytest.mark.parametrize("opt", [["--jsfs", "out/x"], ["--jsfs-pops", "popA"]])
def test_cli_refuses_jsfs_elsewhere(argv, opt, tmp_path):
    r = run_cli(argv + opt + ["-f", str(tmp_path / "x.fa"), str(tmp_path / "x.bam"), "chr1"])
    assert r.returncode == 1 and "--jsfs and --jsfs-pops are only available for sfs" in r.stderr, r.stderr


def test_cli_refuses_jsfs_pops_without_jsfs(tmp_path):
    r = run_cli(["sfs", "--jsfs-pops", "popA", "-f", str(tmp_path / "x.fa"), str(tmp_path / "x.bam"), "chr1"])
    assert r.returncode == 1 and "--jsfs-pops goes with --jsfs" in r.stderr


@pytest.fixture(scope="module")
def cli_files(tmp_path_factory):
    d = tmp_path_factory.mktemp("cli_spectrum")
    c1 = pbtest.fixture("c1").write_files(d / "c1")
    n64 = pbtest.fixture("n64").write_files(d / "n64")
    return d, c1, n64


@pytest.mark.parametrize("extra,msg", [
    (["--jsfs-pops", "popA,popX"], "unknown population popX"),
    (["--jsfs-pops", "popA,popB,popA"], "population popA is repeated"),
    (["--jsfs-pops", "popA,popB,out,popA"], "at most three population names"),
    (["--jsfs-pops", "popA", "--jsfs-pops", ""], "unknown population"),
])
def test_cli_refuses_bad_jsfs_pops(extra, msg, cli_files):
    d, (bam, fa), _ = cli_files
    r = run_cli(["sfs", "-w", "10", "--jsfs", str(d / "x")] + extra + ["-f", fa, bam, "chr1"])
    assert r.returncode == 1 and msg in r.stderr, r.stderr
    assert not list(d.glob("x.*.fs"))


def test_cli_refuses_lists_over_the_abi_limits(cli_files):
    d, _, (bam, fa) = cli_files
    # popA-popB of n64 has 33 x 32 = 1056 bins: 63 of them are 66 528 bins per window
    r = run_cli(["sfs", "-w", "5", "--jsfs", str(d / "y")] + ["--jsfs-pops", "popA,popB"] * 63 + ["-f", fa, bam, "chr1"])
    assert r.returncode == 1 and "66528 bins per window" in r.stderr and "65536" in r.stderr, r.stderr
    r = run_cli(["sfs", "-w", "5", "--jsfs", str(d / "y")] + ["--jsfs-pops", "out"] * 4097 + ["-f", fa, bam, "chr1"])
    assert r.returncode == 1 and "4097 spectrum sets" in r.stderr, r.stderr
