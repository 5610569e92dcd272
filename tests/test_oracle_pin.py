"""Pins the CPU restatement (oracle/pb_oracle.c) against outputs of the UNMODIFIED reference:
the committed goldens (tests/golden/*.txt, kat_*.bin, made by tests/golden/make_goldens.py) and, when the reference
binary is present (oracle/_ref/popbam), a live run on a different seed."""
import ctypes as C
import hashlib
import json

import numpy as np
import pytest

import pbtest
from cases import CASES


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_oracle_text_equals_reference_golden(case):
    fx, p, an, wb, we, o = pbtest.case_setup(case)
    run = pbtest.OracleRun(p, fx.batch(), fx.ref(), an, wb, we)
    got = run.text(an, o)
    if an == pbtest.AN["SNP"] and o.snp_output == 2:
        got = pbtest.ms_header(fx, len(wb)) + got
    ok, why = pbtest.texts_equal(got, pbtest.golden_text(case), snp0=(an == pbtest.AN["SNP"] and o.snp_output == 0))
    assert ok, why
    run.close()


def test_tables_equal_reference_errmod_init():
    kat = json.load(open(pbtest.GOLDEN / "kat_tables.json"))
    t = pbtest.oracle_tables()
    raw = t.fk.tobytes() + t.beta.tobytes() + t.lhet.tobytes()
    assert [float(x).hex() for x in t.fk] == kat["fk"]
    for k, v in kat["beta"].items():
        assert float(t.beta[int(k)]).hex() == v
    for k, v in kat["lhet"].items():
        assert float(t.lhet[int(k)]).hex() == v
    assert hashlib.sha256(raw).hexdigest() == kat["sha256"]


CELL = np.dtype([("k", "<u2"), ("pad", "<u2"), ("rmsq", "<i4"), ("codes", "<u2", 256), ("q", "<f4", 16), ("cb", "<u8")])
SITE = np.dtype([("n", "<i4"), ("min_snpq", "<i4"), ("min_rmsq", "<i4"), ("min_depth", "<i4"), ("max_depth", "<i4"),
                 ("het", "<i4"), ("ref", "u1"), ("pad", "u1", 7), ("cb_in", "<u8", 64), ("cb_out", "<u8", 64),
                 ("fq", "<i4"), ("pad2", "<i4"), ("cov", "<u8")])


def test_cell_call_known_answers():
    """errmod_cal + gl2cns + rms packing vectors dumped from the reference's own objects (oracle/refdump.cpp)."""
    rec = np.fromfile(pbtest.GOLDEN / "kat_cells.bin", dtype=CELL)
    assert len(rec) == 600
    L, t = pbtest.oracle_lib(), pbtest.oracle_tables()
    for r in rec:
        codes = np.array(r["codes"], dtype=np.uint16)
        q = np.zeros(16, dtype=np.float32)
        cb = L.pbo_call_cell(*t.ptrs(), codes.ctypes.data_as(C.POINTER(C.c_uint16)), int(r["k"]), int(r["rmsq"]),
                             q.ctypes.data_as(C.POINTER(C.c_float)))
        assert q.tobytes() == r["q"].tobytes()
        if r["k"] > 0:      # k == 0: NaN -> u64 conversion is the caller's (popbam.cpp:255) never-taken path
            assert cb == int(r["cb"])


def test_site_logic_known_answers():
    rec = np.fromfile(pbtest.GOLDEN / "kat_sites.bin", dtype=SITE)
    assert len(rec) == 300
    L = pbtest.oracle_lib()
    for r in rec:
        p = pbtest.Params()
        p.n_samples, p.n_pops = int(r["n"]), 1
        p.min_snpQ, p.min_rmsQ, p.min_depth, p.max_depth = int(r["min_snpq"]), int(r["min_rmsq"]), int(r["min_depth"]), int(r["max_depth"])
        p.flags = pbtest.FLAG["HETEROZYGOTE"] if r["het"] else 0
        cb = np.array(r["cb_in"], dtype=np.uint64)
        cov, typ = C.c_uint64(), C.c_uint64()
        fq = L.pbo_site_logic(C.byref(p), cb.ctypes.data_as(C.POINTER(C.c_uint64)), bytes([int(r["ref"])]), C.byref(cov), C.byref(typ))
        n = int(r["n"])
        assert fq == int(r["fq"])
        assert cov.value == int(r["cov"])
        assert (cb[:n] == r["cb_out"][:n]).all()


@pytest.mark.skipif(not pbtest.have_ref(), reason="the original POPBAM 0.3 is not built into oracle/_ref/ (make -C oracle ref REF=<its sources>)")
def test_oracle_vs_live_reference(tmp_path):
    fx = pbtest.Fixture(contig_len=20500, n_ingroup=7, has_outgroup=1, depth=16.0, snp_density=0.02, edge_mode=1, seed=977)
    bam, fa = fx.write_files(tmp_path / "live")
    p = fx.params()
    wb, we = pbtest.window_grid(0, fx.contig_len, 10000)
    for argv, an, okw in ((["nucdiv", "-w", "10"], "NUCDIV", {}), (["haplo", "-w", "10", "-o", "2"], "HAPLO_DXY", {}),
                          (["ld", "-w", "10", "-o", "1"], "LD_OMEGA", {})):
        want = pbtest.run_ref(argv + ["-f", fa, bam, "chr1"])
        run = pbtest.OracleRun(p, fx.batch(), fx.ref(), pbtest.AN[an], wb, we)
        assert run.text(pbtest.AN[an], fx.print_opts(**okw)) == want
        run.close()
