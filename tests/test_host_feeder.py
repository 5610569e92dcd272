"""Host feeder of the `popbam` command line (popbam_b200/csrc/pb_bamio.cpp): BGZF inflate, BAM record decode, BAI
region slicing and @RG sample tables, checked on the CPU against the generator's in-memory batch of the same fixture.
(`popbam _fetch` is a test hook that stops before any GPU call.)"""
import subprocess

import numpy as np
import pytest

import pbtest
import popbam_b200

EXE = popbam_b200.capi.PKG / "_build" / "popbam"


def _load(path):
    raw = open(path, "rb").read()
    n, nc, nb, tid, beg, end = np.frombuffer(raw[:48], dtype=np.int64)
    o = 48
    out = {}
    for name, cnt, dt in (("pos", n, np.int32), ("meta", n, np.uint32), ("cig_off", n + 1, np.uint32), ("cigar", nc, np.uint32),
                          ("base_off", n + 1, np.uint32), ("seq4", nb // 2, np.uint8), ("qual", nb, np.uint8)):
        sz = int(cnt) * np.dtype(dt).itemsize
        out[name] = np.frombuffer(raw[o:o + sz], dtype=dt)
        o += sz
    assert o == len(raw)
    return out


def _expected(fx, beg, end):
    """Records of the generator's batch that bam_fetch would deliver for [beg, end) (is_overlap, bam_index.c:729)."""
    b = fx.batch()
    pos = np.ctypeslib.as_array(b.pos, (b.n_reads,)); meta = np.ctypeslib.as_array(b.meta, (b.n_reads,))
    co = np.ctypeslib.as_array(b.cig_off, (b.n_reads + 1,)); bo = np.ctypeslib.as_array(b.base_off, (b.n_reads + 1,))
    cig = np.ctypeslib.as_array(b.cigar, (b.n_cigar,)); qual = np.ctypeslib.as_array(b.qual, (b.n_bases,))
    seq = np.ctypeslib.as_array(b.seq4, (b.n_bases // 2,))
    ops, lens = cig & 15, cig >> 4
    span = np.where(np.isin(ops, [0, 2, 3, 7, 8]), lens, 0)
    cs = np.concatenate([[0], np.cumsum(span)])
    rend = pos + (cs[co[1:]] - cs[co[:-1]])
    keep = (rend > beg) & (pos < end)
    return pos, meta, co, bo, cig, qual, seq, np.nonzero(keep)[0]


@pytest.mark.parametrize("fxname,region,beg,end", [("edge", "chr1", 0, 20500), ("edge", "chr1:5001-9000", 5000, 9000),
                                                    ("rg2", "chr1:12,001-20,500", 12000, 20500), ("c1", "chr1:30000-30400", 29999, 30400)])
def test_fetch_region_equals_generator_batch(tmp_path, fxname, region, beg, end):
    popbam_b200.build()
    fx = pbtest.fixture(fxname)
    bam, fa = fx.write_files(tmp_path / fxname)
    out = tmp_path / "batch.bin"
    r = subprocess.run([str(EXE), "_fetch", bam, region, str(out)], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    assert r.returncode == 0, r.stderr
    # sample / population tables (pop_sample.cpp:15-107, popbam.cpp:145-171)
    lines = r.stdout.splitlines()
    assert lines[0].split()[1:] == fx.sample_names
    masks = fx.params().pop_mask
    assert lines[1].split()[1:] == ["%s=%x" % (nm, masks[i]) for i, nm in enumerate(fx.pop_names)]
    got = _load(out)
    pos, meta, co, bo, cig, qual, seq, idx = _expected(fx, beg, end)
    R = fx.sp.read_len
    assert len(got["pos"]) == len(idx)
    assert np.array_equal(got["pos"], pos[idx])
    assert np.array_equal(got["meta"], meta[idx])          # flag, mapq and the RG -> sample lookup
    assert np.array_equal(np.diff(got["cig_off"].astype(np.int64)), (co[idx + 1] - co[idx]).astype(np.int64))
    assert np.array_equal(got["cigar"], np.concatenate([cig[co[i]:co[i + 1]] for i in idx]) if len(idx) else got["cigar"])
    assert (got["base_off"] % 4 == 0).all()
    for k in list(range(min(50, len(idx)))) + list(range(max(0, len(idx) - 50), len(idx))):
        i = idx[k]
        g0 = int(got["base_off"][k])
        assert np.array_equal(got["qual"][g0:g0 + R], qual[bo[i]:bo[i] + R])
        assert np.array_equal(got["seq4"][g0 // 2:g0 // 2 + (R + 1) // 2], seq[bo[i] // 2:bo[i] // 2 + (R + 1) // 2])


@pytest.mark.parametrize("fxname,region,pieces", [("edge", "chr1", 7), ("edge", "chr1:5001-9000", 3), ("rg2", "chr1:12,001-20,500", 16),
                                                   ("c1", "chr1:30000-30400", 5)])
def test_fetch_in_pieces_equals_one_fetch(tmp_path, fxname, region, pieces):
    """The command line decodes a region as several pieces on different threads (pbio::fetch_piece); appended in order
    they must be the batch of the single bam_fetch (bam_index.c:943-957), byte for byte."""
    popbam_b200.build()
    fx = pbtest.fixture(fxname)
    bam, fa = fx.write_files(tmp_path / fxname)
    one, many = tmp_path / "one.bin", tmp_path / "many.bin"
    for out, extra in ((one, []), (many, [str(pieces)])):
        r = subprocess.run([str(EXE), "_fetch", bam, region, str(out)] + extra, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
        assert r.returncode == 0, r.stderr
    assert one.read_bytes() == many.read_bytes()
    assert len(_load(one)["pos"]) > 0


def _fnv(a):
    h = 1469598103934665603
    for b in np.ascontiguousarray(a).view(np.uint8).tolist():
        h = ((h ^ b) * 1099511628211) & 0xFFFFFFFFFFFFFFFF
    return "%016x" % h


@pytest.mark.parametrize("fxname,region,opts", [("edge", "chr1", ["-w", "1", "--shard-mb", "0.003"]), ("rg2", "chr1", ["-w", "2", "--shard-mb", "0.004"]),
                                                 ("c1", "chr1", [])])
def test_feeder_threads_hand_over_every_shard_whole_and_in_order(tmp_path, fxname, region, opts):
    """`popbam _feed` runs the command line's host side (shards, pieces, decode threads, batch pool, workers) without a
    GPU and prints what each shard's worker was handed.  It must not depend on the number of decode threads or workers,
    and every shard must hold exactly the reads a single bam_fetch of its windows delivers (bam_index.c:943-957)."""
    popbam_b200.build()
    fx = pbtest.fixture(fxname)
    bam, fa = fx.write_files(tmp_path / fxname)
    outs = []
    for extra in (["--threads", "1"], ["--threads", "7", "--gpus", "3"], ["--threads", "16", "--gpus", "2"]):
        r = subprocess.run([str(EXE), "_feed", "-f", fa] + opts + extra + [bam, region], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
        assert r.returncode == 0, r.stderr
        outs.append(r.stdout)
    assert outs[0] == outs[1] == outs[2]
    rows = [ln.split("\t") for ln in outs[0].splitlines()]
    assert len(rows) >= 1 and [int(x[0]) for x in rows] == sorted(int(x[0]) for x in rows)
    win = int(opts[1]) * 1000 if opts else None
    wb, we = pbtest.window_grid(0, fx.contig_len, win) if win else (np.array([0]), np.array([fx.contig_len]))
    for x in rows[:3] + rows[-2:]:
        w0, w1 = int(x[0]), int(x[1])
        out = tmp_path / "shard.bin"
        rr = subprocess.run([str(EXE), "_fetch", bam, "chr1:%d-%d" % (int(wb[w0]) + 1, int(we[w1 - 1])), str(out)], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
        assert rr.returncode == 0, rr.stderr
        got = _load(out)
        assert int(x[2]) == len(got["pos"]) and int(x[3]) == len(got["cigar"])
        assert x[4] == _fnv(got["pos"]) and x[5] == _fnv(got["meta"]) and x[6] == _fnv(got["cigar"])
        assert int(x[7]) == int(got["qual"].astype(np.uint64).sum()) and int(x[8]) == int(got["seq4"].astype(np.uint64).sum())


def test_cli_errors_without_gpu(tmp_path):
    popbam_b200.build()
    r = subprocess.run([str(EXE), "nucdiv", "-f", "nope.fa", str(tmp_path / "missing.bam"), "chr1"], stderr=subprocess.PIPE, text=True)
    assert r.returncode == 1 and "does not exist" in r.stderr
    r = subprocess.run([str(EXE), "frobnicate"], stderr=subprocess.PIPE, text=True)
    assert r.returncode == 1 and "unrecognized command" in r.stderr
    # errors the reference raises before it touches the data (tree: pop_tree.cpp:621-625; all: popbam.cpp:157-166, :130)
    fx = pbtest.fixture("edge")
    bam, fa = fx.write_files(tmp_path / "edge")
    r = subprocess.run([str(EXE), "tree", "-d", "kimura", "-f", fa, bam, "chr1"], stderr=subprocess.PIPE, text=True)
    assert r.returncode == 1 and "kimura is not a valid distance option" in r.stderr
    r = subprocess.run([str(EXE), "nucdiv", "-f", fa, bam, "chrZ"], stderr=subprocess.PIPE, text=True)
    assert r.returncode == 1 and "Bad genome coordinates: chrZ" in r.stderr
    r = subprocess.run([str(EXE), "index"], stderr=subprocess.PIPE, text=True)
    assert r.returncode == 1 and "Usage" in r.stderr
    (tmp_path / "noidx.bam").write_bytes(open(bam, "rb").read())
    r = subprocess.run([str(EXE), "sfs", "-f", fa, str(tmp_path / "noidx.bam"), "chr1"], stderr=subprocess.PIPE, text=True)
    assert r.returncode == 1 and "Index file not available" in r.stderr


def _bgzf_block(payload, level, strategy):
    import struct
    import zlib
    co = zlib.compressobj(level, zlib.DEFLATED, -15, 8, strategy)
    raw = co.compress(payload) + co.flush()
    bsize = len(raw) + 18 + 8
    assert bsize <= 65536
    hdr = b"\x1f\x8b\x08\x04" + b"\0" * 4 + b"\x00\xff" + struct.pack("<H", 6) + b"BC" + struct.pack("<HH", 2, bsize - 1)
    return hdr + raw + struct.pack("<II", zlib.crc32(payload) & 0xffffffff, len(payload))


def test_own_inflate_equals_zlib(tmp_path):
    """The feeder's DEFLATE decoder (pb_inflate.cpp) against zlib: BGZF files built from many kinds of payload at every
    compression level and strategy (stored, fixed and dynamic Huffman blocks, long matches, overlapping copies), and the
    generator's own BAM files."""
    import gzip
    import zlib
    popbam_b200.build()
    rng = np.random.default_rng(7)
    payloads = []
    for n in (0, 1, 2, 3, 7, 8, 9, 10, 11, 15, 16, 17, 100, 4095, 20000, 60000):     # (small ones: the decoder's careful last bytes)
        payloads.append(rng.integers(0, 256, n, dtype=np.uint8).tobytes())                  # incompressible
        payloads.append(rng.integers(0, 4, n, dtype=np.uint8).tobytes())                    # low entropy
        payloads.append((b"ACGTTGCA" * (n // 8 + 1))[:n])                                   # periodic: overlapping copies
        payloads.append(bytes(n))                                                           # one long run
        payloads.append(rng.choice(np.frombuffer(b"!5?DI", dtype=np.uint8), n).tobytes())   # quality-like
    words = [bytes(rng.integers(97, 123, int(rng.integers(2, 12)), dtype=np.uint8)) for _ in range(300)]
    payloads.append(b" ".join(words[int(i)] for i in rng.integers(0, 300, 9000))[:60000])  # text-like, long codes
    # skewed symbol frequencies force maximal code lengths (sub-tables)
    freq = np.array([2.0 ** -(i % 24) for i in range(256)]); freq /= freq.sum()
    payloads.append(rng.choice(256, 60000, p=freq).astype(np.uint8).tobytes())
    blob, want = b"", b""
    for i, pl in enumerate(payloads):
        for level in (0, 1, 6, 9):
            for strat in (zlib.Z_DEFAULT_STRATEGY, zlib.Z_FIXED, zlib.Z_HUFFMAN_ONLY, zlib.Z_RLE, zlib.Z_FILTERED):
                if (i + level + strat) % 3 and len(pl) > 4095:
                    continue                                   # thin the big ones out
                if len(pl) > 60000 and level == 0:
                    continue
                blob += _bgzf_block(pl, level, strat)
                want += pl
    blob += _bgzf_block(b"", 6, zlib.Z_DEFAULT_STRATEGY)        # EOF marker
    src = tmp_path / "mix.bgzf"
    src.write_bytes(blob)
    out = tmp_path / "mix.raw"
    r = subprocess.run([str(EXE), "_inflate", str(src), str(out)], stderr=subprocess.PIPE, text=True)
    assert r.returncode == 0, r.stderr
    assert out.read_bytes() == want
    # corrupt streams are rejected, not mis-decoded silently
    bad = bytearray(_bgzf_block(payloads[4 * 5 + 1] + payloads[13 * 5], 6, zlib.Z_DEFAULT_STRATEGY))
    bad[40] ^= 0x55
    (tmp_path / "bad.bgzf").write_bytes(bytes(bad))
    r = subprocess.run([str(EXE), "_inflate", str(tmp_path / "bad.bgzf"), str(out)], stderr=subprocess.PIPE, text=True)
    assert r.returncode != 0 or out.read_bytes() != payloads[4 * 5 + 1] + payloads[13 * 5]
    # the generator's BAM (level 1) and a level-6 rewrite
    fx = pbtest.fixture("edge")
    for level in (1, 6):
        bam, _ = fx.write_files(tmp_path / ("e%d" % level), level=level)
        r = subprocess.run([str(EXE), "_inflate", bam, str(out)], stderr=subprocess.PIPE, text=True)
        assert r.returncode == 0, r.stderr
        assert out.read_bytes() == gzip.open(bam).read()


def _parse_bai(path):
    d = open(path, "rb").read()
    assert d[:4] == b"BAI\x01"
    o = 4
    nref = int(np.frombuffer(d[o:o + 4], dtype=np.uint32)[0]); o += 4
    refs = []
    for _ in range(nref):
        nbin = int(np.frombuffer(d[o:o + 4], dtype=np.uint32)[0]); o += 4
        bins = {}
        for _b in range(nbin):
            b, nch = np.frombuffer(d[o:o + 8], dtype=np.uint32); o += 8
            bins[int(b)] = np.frombuffer(d[o:o + 16 * int(nch)], dtype=np.uint64).reshape(-1, 2).copy(); o += 16 * int(nch)
        nint = int(np.frombuffer(d[o:o + 4], dtype=np.uint32)[0]); o += 4
        lin = np.frombuffer(d[o:o + 8 * nint], dtype=np.uint64).copy(); o += 8 * nint
        refs.append((bins, lin))
    tail = d[o:]
    return refs, tail


@pytest.mark.parametrize("fxname", ["edge", "rg2", "c1"])
def test_index_builder_serves_the_same_records(tmp_path, fxname):
    """`popbam index` (pbio::build_bai, the restatement of bam_index_build): the index it writes must serve every region
    query exactly as the generator's own index does, cover the same bins with chunks that start where the runs of records
    start, and carry the per-reference record counts in the pseudo-bin."""
    popbam_b200.build()
    fx = pbtest.fixture(fxname)
    bam, fa = fx.write_files(tmp_path / fxname)
    gen_bai = tmp_path / "gen.bai"
    (tmp_path / (fxname + ".bam.bai")).rename(gen_bai) if (tmp_path / (fxname + ".bam.bai")).exists() else None
    bai = str(bam) + ".bai"
    if not gen_bai.exists():            # write_files may name the index differently
        import shutil
        shutil.copy(bai, gen_bai)
    r = subprocess.run([str(EXE), "index", bam], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    assert r.returncode == 0, r.stderr
    n_reads = fx.batch().n_reads
    assert "%d records" % n_reads in r.stderr
    ours, tail = _parse_bai(bai)
    theirs, _ = _parse_bai(gen_bai)
    assert len(tail) == 8 and int(np.frombuffer(tail, dtype=np.uint64)[0]) == 0          # no records without coordinates
    assert len(ours) == len(theirs)
    for (bo, lo), (bt, lt) in zip(ours, theirs):
        meta = bo.pop(37450)
        bt.pop(37450, None)
        assert set(bo) == set(bt)                                                         # the same bins are populated
        assert int(meta[1, 0]) + int(meta[1, 1]) == n_reads                               # mapped + unmapped
        for b in bo:
            # the bin's first chunk starts at the same record; chunk ends may name the same stream position differently
            # (end of one BGZF block == start of the next), so they are checked through the region queries below
            assert bo[b][0, 0] == bt[b][0, 0]
        n = min(len(lo), len(lt))
        assert np.array_equal(lo[:n], lt[:n])                                             # linear index
    # region queries through our index
    rng = np.random.default_rng(3)
    for _ in range(6):
        beg = int(rng.integers(0, fx.contig_len - 200)); end = beg + int(rng.integers(1, 4000))
        end = min(end, fx.contig_len)
        out = tmp_path / "q.bin"
        rr = subprocess.run([str(EXE), "_fetch", bam, "chr1:%d-%d" % (beg + 1, end), str(out)], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
        assert rr.returncode == 0, rr.stderr
        got = _load(out)
        pos, meta_, co, bo_, cig, qual, seq, idx = _expected(fx, beg, end)
        assert np.array_equal(got["pos"], pos[idx])


@pytest.mark.skipif(not pbtest.have_ref(), reason="the original POPBAM 0.3 is not built into oracle/_ref/ (make -C oracle ref REF=<its sources>)")
def test_reference_reads_our_index(tmp_path):
    """The unmodified reference, given the index `popbam index` wrote, prints its golden output."""
    popbam_b200.build()
    fx = pbtest.fixture("c1")
    bam, fa = fx.write_files(tmp_path / "c1")
    r = subprocess.run([str(EXE), "index", bam], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    assert r.returncode == 0, r.stderr
    out = pbtest.run_ref(["nucdiv", "-w", "10", "-f", fa, bam, "chr1"])
    assert out == (pbtest.GOLDEN / "nucdiv_c1.txt").read_text()
