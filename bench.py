#!/usr/bin/env python
"""bench.py -- aligned Gbases/s of the per-window statistics path on B200 (BASELINE.json metric).

Workload (config.workload): by default BASELINE.json configs[1] (--config c2) -- `popbam sfs` (Tajima's D, Fay & Wu's H;
outgroup-polarised) on a 23 Mb X-like contig, 10 samples + outgroup, 30x per sample, 100 bp reads, 10 kb windows,
synthetic data from tools/pbsynth (SURVEY.md §8(d) data model).  --config c1 / c3 / c4 / c5 select the other BASELINE
configurations.  The contig is fed as region shards of --shard-mb (the unit the host feeder hands over in production:
BAM-index chunks of whole windows); ONE STEP = the whole contig = every shard once.

  value      whole-job aligned Gbases/s with every shard's read batch already resident in HBM: the complete device
             pipeline (per-read prep, depth bound, counting pileup, code lists, hard cells, sites, window compaction, window
             statistics, result copy) re-run on resident inputs, timed with CUDA events on the library's streams.
  e2e        same job through the public C ABI from PINNED HOST batches: pb_region_begin / pb_push_batch_async (host->
             device copy inside the timed region) / pb_region_end (device->host result copy inside the timed region).
  roofline   the WHOLE device pipeline: algorithmic bytes of a step / the step's CUDA-event duration (the same region
             `value` is timed on); `dominant_kernel` = the pileup / call / site stage alone; `traffic` = DRAM bytes of all
             kernels of a region from the committed ncu launch list.
  verified   before anything is timed, one window of every distinct shard is compared with the CPU oracle.
  cpu_baseline  the unmodified reference (oracle/_ref/popbam, built from /root/reference by oracle/Makefile) timed on
             one host core on a bounded sample of the same workload; falls back to the oracle port if the binary is absent.
  cli_from_bam  the `popbam` command line of this repo on BAM/BAI/FASTA files (host feeder + GPU), start-up separately.

`--impl reference` times the reference CPU implementation with one process per host core over split regions.
Under torchrun every rank runs its own contig on its own GPU (weak scaling; no collective on the data path).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

import numpy as np  # noqa: E402

# DRAM bytes (read + written) of ALL kernels of one region on a 2.3 Mb shard of configs[1], summed over the committed ncu
# launch list profiles/r2_launches.csv (dram__bytes_read.sum + dram__bytes_write.sum per kernel, one pipeline run)
TRAFFIC_BYTES_PER_SHARD_C2 = 1.77e9
READ_LEN = 100

# BASELINE.json configs[0..4] as c1..c5 (SURVEY.md §8(d) data model).  One STEP = the whole contig = every shard once.
CONFIGS = {
    "c1": dict(label="configs[0]: popbam nucdiv", an=["NUCDIV"], flags=["OUTGROUP"], contig_mb=1.0, shard_mb=1.0, n_ingroup=10, has_outgroup=1,
               rg_per_sample=1, depth=20.0, win=10000, snp=0.01, cli=["nucdiv", "-w", "10", "-p", "og"]),
    "c2": dict(label="configs[1]: popbam sfs -p og", an=["SFS"], flags=["OUTGROUP"], contig_mb=23.0, shard_mb=2.3, n_ingroup=10, has_outgroup=1,
               rg_per_sample=1, depth=30.0, win=10000, snp=0.01, cli=["sfs", "-w", "10", "-p", "og"]),
    "c3": dict(label="configs[2]: popbam ld -o 0 / -o 1 / -o 2 (ZnS, omega_max, Wall B/Q in one pass)", an=["LD_ZNS", "LD_OMEGA", "LD_WALL"], flags=[],
               contig_mb=5.0, shard_mb=0.5, n_ingroup=64, has_outgroup=0, rg_per_sample=1, depth=20.0, win=50000, snp=0.06, cli=["ld", "-w", "50"]),
    "c4": dict(label="configs[3]: popbam diverge -o 0 / -o 1 + haplo -o 0 / -o 1 / -o 2 in one pass, one contig per GPU",
               an=["DIVERGE_IND", "DIVERGE_POP", "HAPLO_K", "HAPLO_EHHS", "HAPLO_DXY"], flags=["OUTGROUP"], contig_mb=24.0, shard_mb=1.0,
               n_ingroup=31, has_outgroup=1, rg_per_sample=1, depth=20.0, win=10000, snp=0.01, cli=["diverge", "-w", "10", "-p", "og"]),
    "c5": dict(label="configs[4]: nucdiv + sfs + ld (ZnS) in one pass, 128 read groups -> 64 samples", an=["NUCDIV", "SFS", "LD_ZNS"], flags=["OUTGROUP"],
               contig_mb=10.0, shard_mb=0.5, n_ingroup=63, has_outgroup=1, rg_per_sample=2, depth=30.0, win=10000, snp=0.01,
               cli=["nucdiv", "-w", "10", "-p", "og"]),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS), help="BASELINE.json configs[0..4] = c1..c5 (default: configs[1], the one the metric is quoted on)")
    ap.add_argument("--contig-mb", type=float, default=0.0, help="0 = the configuration's own")
    ap.add_argument("--shard-mb", type=float, default=0.0, help="0 = the configuration's own")
    ap.add_argument("--threads", type=int, default=0, help="generator threads (0 = auto)")
    ap.add_argument("--inflight", type=int, default=4, help="region shards processed concurrently per GPU (one host thread and one context each)")
    ap.add_argument("--distinct-shards", type=int, default=0,
                    help="generate this many distinct shards and cycle them (0 = auto: all distinct when the host has >= 8 cores per rank)")
    ap.add_argument("--cpu-sample-kb", type=int, default=150)
    ap.add_argument("--quality", default="levels5", choices=["levels5", "wide"],
                    help="base / mapping qualities of the synthetic reads: the five levels of the SURVEY data model (default), or pbsynth's wide spectrum (base qualities 2..41, twenty mapping qualities)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-verify", action="store_true", help="skip the oracle check of one window per distinct shard (outside the timed region)")
    ap.add_argument("--cli-sample-kb", type=int, default=5000, help="BAM sample for the command-line (from-BAM) tier; 0 = skip (one fixture holds at most ~12 Mb of this depth: 32-bit base offsets)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the result arrays of the last timed step (every shard, in shard order; rank 0 under "
                         "torchrun) as float64 DIR/<name>.npy, at most 64 MB in all; every shard then gets its own seeded inputs unless "
                         "--distinct-shards is given, so that runs with the same arguments can be compared output for output")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    a.cfg = dict(CONFIGS[a.config])
    if a.quality == "wide":
        a.cfg["edge_mode"] = 2
        a.cfg["label"] += " [wide quality spectrum: base qualities 2..41, twenty mapping qualities]"
    a.contig_mb = a.contig_mb or a.cfg["contig_mb"]
    a.shard_mb = a.shard_mb or a.cfg["shard_mb"]
    return a


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.stop, self.th = index, [], threading.Event(), None

    def _run(self):
        while not self.stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                     stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self.stop.wait(0.2)

    def __enter__(self):
        self.th = threading.Thread(target=self._run, daemon=True)
        self.th.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.th.join(timeout=6)

    def summary(self):
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(self.rows)}


def shard_plan(args):
    win = args.cfg["win"]
    shard_len = max(1, int(round(args.shard_mb * 1e6 / win))) * win
    n_shards = max(1, int(round(args.contig_mb * 1e6 / shard_len)))
    return shard_len, n_shards


def gen_threads(args, world):
    if args.threads > 0:
        return args.threads
    return max(2, min(32, (os.cpu_count() or 8) // max(1, world)))


def product_window_grid(beg, end, win):
    """The reference's window arithmetic through the PRODUCT's pb_window_grid (pop_nucdiv.cpp:48-78)."""
    import popbam_b200
    L = popbam_b200.lib()
    nw = L.pb_window_grid(beg, end, win, 0, None, None)
    wb = (C.c_int32 * max(nw, 1))(); we = (C.c_int32 * max(nw, 1))()
    L.pb_window_grid(beg, end, win, nw, wb, we)
    return np.array(wb[:nw], dtype=np.int32), np.array(we[:nw], dtype=np.int32)


def algorithmic_bytes(batch, n_cells, n_sites):
    """SURVEY.md §8(d): per read pos 4 + meta 4 + offsets 8 + 4/cigar op + packed seq + qual; per (site,sample) one 8-byte
    consensus word; one reference byte per site."""
    return int(batch.n_reads) * 16 + int(batch.n_cigar) * 4 + int(batch.n_bases) // 2 + int(batch.n_bases) + 8 * n_cells + n_sites


def config_fixture(cfg, length, seed, threads):
    import pbtest
    return pbtest.Fixture(contig_len=length + 1, n_ingroup=cfg["n_ingroup"], has_outgroup=cfg["has_outgroup"], rg_per_sample=cfg["rg_per_sample"],
                          depth=cfg["depth"], read_len=READ_LEN, snp_density=cfg["snp"], seed=seed, n_threads=threads, edge_mode=cfg.get("edge_mode", 0))


def config_params(cfg, fx, device=0):
    import pbtest
    fl = 0
    for f in cfg["flags"]:
        fl |= pbtest.FLAG[f]
    return fx.params(flags=fl, outidx=fx.n_samples - 1 if "OUTGROUP" in cfg["flags"] else 0, device=device)


def verify_shard(sh, res_arrays, an_names, an):
    """One window of the shard against the CPU oracle (TEST INFRASTRUCTURE, outside every timed region): site counts and
    segregating-site types bit for bit, window statistics to 1e-9."""
    import pbtest
    BY_AN = pbtest.BY_AN
    w = len(sh["wb"]) // 2
    orc = pbtest.OracleRun(sh["params"], sh["batch"], sh["ref"], an, sh["wb"][w:w + 1], sh["we"][w:w + 1])
    want = pbtest.result_arrays(orc.res)
    got = res_arrays
    assert int(want["num_sites"][0]) == int(got["num_sites"][w]), "bench self-check: num_sites of window %d" % w
    s0, s1 = int(got["seg_off"][w]), int(got["seg_off"][w + 1])
    assert np.array_equal(want["seg_type"], got["seg_type"][s0:s1]), "bench self-check: segregating-site types of window %d" % w
    assert np.array_equal(want["seg_pos"], got["seg_pos"][s0:s1]), "bench self-check: segregating-site positions of window %d" % w
    NW = len(sh["wb"])
    dev = {}
    for name in an_names:
        ints, flts = BY_AN[name]
        for k in list(ints) + list(flts):
            per = got[k].size // NW
            if per == 0 or k.startswith("seg_"):
                continue
            a, b = want[k][:per], got[k][w * per:(w + 1) * per]
            if k in ints:
                assert np.array_equal(a, b), "bench self-check: %s of window %d" % (k, w)
            else:
                assert np.array_equal(np.isnan(a), np.isnan(b)), "bench self-check: NA pattern of %s, window %d" % (k, w)
                ok = ~np.isnan(a) & (a != 0)
                d = float(np.max(np.abs(a[ok] - b[ok]) / np.abs(a[ok]))) if ok.any() else 0.0
                dev[k] = max(dev.get(k, 0.0), d)
                # omega_max of a window with thousands of kept SNPs: the reference (and the oracle, which restates its loop)
                # adds ~K^3/3 terms one by one into three running sums, whose own rounding noise grows with K^1.5 * 2^-53;
                # tests/test_gpu_parity.py holds omega_max to 1e-9 up to K = 1850
                tol = 5e-8 if k == "omegamax" else 1e-9
                assert d <= tol, "bench self-check: %s of window %d deviates by %.3g (relative)" % (k, w, d)
    orc.close()
    return w, dev


DUMP_BYTES = 64 * 10 ** 6


def dump_outputs(out_dir, per_shard):
    """Result arrays of every shard, concatenated in shard order, as float64 out_dir/<name>.npy; seg_off is rebased to the
    concatenation, and a 64-bit word becomes two columns, its low and high 32 bits (float64 holds those exactly).  Every
    value written is finite: where a statistic is NaN (the reference prints "NA": too few sites or SNPs) or infinite, the
    value is 0 and out_dir/<name>_na.npy holds 1 there (0 elsewhere).  An array too large for its share of DUMP_BYTES is
    cut to a fixed, seeded sample of its rows (the same rows of <name>_na), whose row numbers go to out_dir/<name>_rows.npy."""
    out = {}
    for k in per_shard[0]:
        parts = [r[k] for r in per_shard]
        if k == "seg_off":
            base = np.cumsum([0] + [int(p[-1]) for p in parts])
            parts = [p[:-1] + b for p, b in zip(parts, base[:-1])] + [base[-1:]]
        a = np.concatenate(parts)
        if a.size == 0:
            continue
        if a.dtype == np.uint64:
            a = np.stack([a & np.uint64(0xffffffff), a >> np.uint64(32)], axis=1)
        a = a.astype(np.float64)
        na = ~np.isfinite(a)
        out[k] = {k: np.where(na, 0.0, a), k + "_na": na.astype(np.float64)} if na.any() else {k: a}
    os.makedirs(out_dir, exist_ok=True)
    left = DUMP_BYTES - 3 * 256 * len(out)                   # room for the .npy headers
    for i, (k, g) in enumerate(sorted(out.items(), key=lambda kv: sum(a.nbytes for a in kv[1].values()))):
        share = left // (len(out) - i)
        n, nbytes = len(g[k]), sum(a.nbytes for a in g.values())
        if nbytes > share:
            rows = np.sort(np.random.default_rng(0).choice(n, share // (nbytes // n + 8), replace=False))
            g = {name: a[rows] for name, a in g.items()}
            g[k + "_rows"] = rows.astype(np.float64)
        for name, a in g.items():
            np.save(os.path.join(out_dir, name + ".npy"), a)
            left -= a.nbytes


def run_b200(args):
    import torch
    import pbtest
    import popbam_b200
    rank, world, local = dist_env()
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    cfg = args.cfg
    WIN = cfg["win"]
    shard_len, n_shards = shard_plan(args)
    an = 0
    for a in cfg["an"]:
        an |= pbtest.AN[a]
    shards = []
    t_gen = time.time()
    # a dump must see the same inputs whatever the host's cores and free memory are
    distinct = args.distinct_shards or (n_shards if args.dump_outputs or (os.cpu_count() or 8) // world >= 8 else min(n_shards, 3))
    bytes_per_pos = (cfg["n_ingroup"] + cfg["has_outgroup"]) * cfg["depth"] * 1.75          # pinned bytes per reference position
    try:        # pinned + transient copies of every distinct shard and rank: stay well inside the host's memory
        import psutil
        per_shard = 2.2 * bytes_per_pos * shard_len
        fit = int(psutil.virtual_memory().available * 0.5 / max(1, world) / per_shard)
        if not args.distinct_shards and not args.dump_outputs:
            distinct = max(1, min(distinct, fit))
    except Exception:
        pass
    n = None
    for s in range(n_shards):
        if s >= distinct:       # cycle the generated shards (same shape, same work; each still has its own context and copy in HBM)
            shards.append(shards[s % distinct])
            continue
        fx = config_fixture(cfg, shard_len, 1000 * (rank + 1) + s, gen_threads(args, world))
        n = fx.n_samples
        b = fx.batch()
        # pinned host copies of the batch arrays (what the host feeder fills in production)
        pins, pb = {}, pbtest.Batch()
        pb.n_reads, pb.n_cigar, pb.n_bases = b.n_reads, b.n_cigar, b.n_bases
        for name, cnt, dt, ct in (("pos", b.n_reads, torch.int32, C.c_int32), ("meta", b.n_reads, torch.int32, C.c_uint32),
                                  ("cig_off", b.n_reads + 1, torch.int32, C.c_uint32), ("cigar", b.n_cigar, torch.int32, C.c_uint32),
                                  ("base_off", b.n_reads + 1, torch.int32, C.c_uint32), ("seq4", b.n_bases // 2, torch.uint8, C.c_uint8),
                                  ("qual", b.n_bases, torch.uint8, C.c_uint8)):
            t = torch.empty(int(cnt), dtype=dt, pin_memory=True)
            C.memmove(t.data_ptr(), getattr(b, name), t.numel() * t.element_size())
            pins[name] = t
            setattr(pb, name, C.cast(t.data_ptr(), C.POINTER(ct)))
        wb, we = product_window_grid(0, shard_len + 1, WIN)
        p = config_params(cfg, fx, local)
        shards.append(dict(batch=pb, pins=pins, ref=fx.ref(), wb=wb, we=we, params=p, aligned=fx.aligned_bases(),
                           h2d=sum(t.numel() * t.element_size() for t in pins.values())))
        fx.close()
    t_gen = time.time() - t_gen

    # one context per shard: "value" needs every shard's reads resident in HBM at the same time
    ctxs = []
    for sh in shards:
        ctx = popbam_b200.Context(sh["params"])
        ctx.set_contig(0, sh["ref"])
        ctxs.append(ctx)

    from concurrent.futures import ThreadPoolExecutor
    pool = ThreadPoolExecutor(max_workers=max(1, args.inflight))

    def one_e2e(cs):
        ctx, sh = cs
        ctx.region_begin(an, sh["wb"], sh["we"])
        ctx.push_batch_async(sh["batch"])     # pinned arrays, untouched until region_end returns
        res = ctx.region_end()
        return res.n_windows * (3 * 4 + 8 + 3 * 8 * res.n_pops) + int(res.seg_off[res.n_windows]) * 17

    def e2e_step():
        # shards in flight overlap one shard's host->device copy with another shard's kernels
        return sum(pool.map(one_e2e, zip(ctxs, shards)))

    def one_resident(ctx):
        ctx.relaunch()
        ctx.wait()
        return ctx.stage_times()[1]

    def resident_step():
        return sum(pool.map(one_resident, ctxs))

    def barrier():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        import torch.distributed as dist
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- e2e (also leaves every shard resident for the device-only leg); clocks are sampled over both timed legs
    for _ in range(max(1, args.warmup)):
        d2h = e2e_step()
    # ---- what is about to be timed is checked first: one window per distinct shard against the CPU oracle
    verified = None
    if not args.no_verify and rank == 0:
        t_v = time.time()
        wins = [verify_shard(shards[i], pbtest.result_arrays(ctxs[i].res), cfg["an"], an) for i in range(min(distinct, n_shards))]
        devs = {}
        for _w, dv in wins:
            for k, v in dv.items():
                devs[k] = max(devs.get(k, 0.0), v)
        verified = {"against": "oracle/pb_oracle.c (CPU restatement), outside the timed regions", "windows": len(wins), "max_relative_deviation": devs,
                    "what": "num_sites, segregating-site positions and types bit for bit; window statistics to 1e-9", "seconds": round(time.time() - t_v, 1)}
    paths = [c.path() for c in ctxs]
    barrier()
    clk = ClockSampler(local)
    clk.__enter__()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        d2h = e2e_step()
    barrier()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    # what the copies alone cost: the same pinned arrays to the device, one plain stream per shard in flight, nothing else
    copy_s = None
    try:
        nbuf = max(1, min(args.inflight, len(shards)))
        big = {k: max(sh["pins"][k].numel() for sh in shards) for k in shards[0]["pins"]}
        dev_bufs = [{k: torch.empty(big[k], dtype=shards[0]["pins"][k].dtype, device="cuda") for k in big} for _ in range(nbuf)]
        cstreams = [torch.cuda.Stream() for _ in range(nbuf)]
        barrier()
        t0 = time.perf_counter()
        for i, sh in enumerate(shards):
            with torch.cuda.stream(cstreams[i % nbuf]):
                for k, t in sh["pins"].items():
                    dev_bufs[i % nbuf][k][:t.numel()].copy_(t, non_blocking=True)
        barrier()
        copy_s = max_over_ranks(time.perf_counter() - t0)
        del dev_bufs
    except Exception:      # (memory for the extra buffers: the figure is an extra, not part of the contract)
        copy_s = None

    # ---- device-resident leg, CUDA events around the whole step on the library's stream(s)
    total_aligned = sum(int(c.res.aligned_bases) for c in ctxs)
    for _ in range(args.warmup):
        resident_step()
    launches0 = sum(c.kernel_launches() for c in ctxs)
    pile_ms = 0.0
    barrier()
    e0 = torch.cuda.Event(enable_timing=True)
    e1 = torch.cuda.Event(enable_timing=True)
    ev1 = [torch.cuda.Event() for _ in ctxs]
    streams = [torch.cuda.ExternalStream(c.L.pb_stream(c.h)) for c in ctxs]
    cur = torch.cuda.current_stream()
    step_ms = 0.0
    for _ in range(args.steps):
        # device-side bracket: e0 precedes every library stream's work of this step, e1 follows all of it
        e0.record(cur)
        for st in streams:
            st.wait_event(e0)
        resident_step()
        for i, st in enumerate(streams):
            ev1[i].record(st)
            cur.wait_event(ev1[i])
        e1.record(cur)
        torch.cuda.synchronize()
        step_ms += e0.elapsed_time(e1)
    barrier()
    last_step = [pbtest.result_arrays(c.res) for c in ctxs] if args.dump_outputs and rank == 0 else None
    launches = sum(c.kernel_launches() for c in ctxs) - launches0
    # the stages alone: one more pass with the shards strictly one after the other (library events, pb_stage_times)
    seq_ms = 0.0
    stage_ms = [0.0, 0.0, 0.0, 0.0]
    for ctx, st in zip(ctxs, streams):
        e0.record(st)
        ctx.relaunch()
        ctx.wait()
        e1.record(st)
        e1.synchronize()
        seq_ms += e0.elapsed_time(e1)
        stt = ctx.stage_times()
        pile_ms += stt[1]
        for i in range(4):
            stage_ms[i] += stt[i]
    clk.__exit__(None, None, None)
    dev_s = max_over_ranks(step_ms / 1e3)

    peaks = {}
    try:
        peaks = json.load(open(ROOT / "MEASURED_PEAKS.json"))
    except Exception:
        pass
    peak_gbs = float(peaks.get("hbm_gbs", 6650.0))
    alg_bytes = sum(algorithmic_bytes(s["batch"], int(s["we"][-1] - s["wb"][0]) * n, int(s["we"][-1] - s["wb"][0])) for s in shards)
    step_s = dev_s / args.steps
    achieved = alg_bytes / step_s / 1e9                      # the WHOLE device pipeline of every shard of a step
    n_windows = sum(len(s["wb"]) for s in shards)
    is_c2_shard = args.config == "c2" and abs(shard_len - 2300000) < 1

    line = {
        "metric": "aligned Gbases/s", "value": world * total_aligned / step_s / 1e9, "unit": "Gbases/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": step_s * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8/u64 + f64 (error model)",
        "data": "synthetic (tools/pbsynth, seeded)",
        "config": {"workload": "%s, %.1f Mb contig as %d region shards of %.2f Mb, %d samples%s, %gx per sample, 100 bp reads, %d kb windows" % (
                       cfg["label"], n_shards * shard_len / 1e6, n_shards, shard_len / 1e6, n, " (%d read groups each)" % cfg["rg_per_sample"] if cfg["rg_per_sample"] > 1 else "",
                       cfg["depth"], WIN // 1000),
                   "config": args.config, "per_gpu": "each rank runs its own contig", "windows_per_step": n_windows * world,
                   "windows_per_s": world * n_windows / step_s,
                   "aligned_bases_per_step": world * total_aligned, "l2": "inputs (%.1f GB per step) exceed L2" % (alg_bytes / 1e9),
                   "distinct_shards": distinct, "shards_in_flight": max(1, args.inflight), "generator_s": round(t_gen, 1),
                   "pileup_path": "counting kernels (k_pile_reads + k_cell_codes + k_hard_cells)" if all(p == 1 for p in paths) else "single-kernel pileup on %d of %d shards" % (sum(1 for p in paths if p == 0), len(paths)),
                   "regions_run_twice": sum(c.reruns() for c in ctxs)},
        "e2e": {"value": world * total_aligned / (e2e_s / args.steps) / 1e9, "unit": "Gbases/s",
                "h2d_bytes_per_step": sum(s["h2d"] for s in shards), "d2h_bytes_per_step": int(d2h),
                "windows_per_s": world * n_windows / (e2e_s / args.steps),
                "h2d_copy_only_gbs": (world * sum(s["h2d"] for s in shards) / copy_s / 1e9) if copy_s else None,
                "h2d_achieved_gbs": world * sum(s["h2d"] for s in shards) / (e2e_s / args.steps) / 1e9,
                "note": "h2d_copy_only_gbs = the same pinned arrays copied to the device with nothing else going on (all ranks at once): the ceiling of this tier"},
        "gpu_launches": int(launches),
        "stage_ms_per_shard": {k: v / len(shards) for k, v in zip(["per_read_prep", "pileup_call_site", "window_compaction", "window_stats"], stage_ms)},
        "roofline": {"kernel": "the whole device pipeline of a region: k_read_prep, k_depth_bound, k_pile_reads, k_cell_codes, k_hard_cells, k_fast_sites, window compaction and statistics",
                     "bound": "hbm", "achieved": achieved, "peak": peak_gbs, "unit": "GB/s", "frac": achieved / peak_gbs,
                     "traffic": TRAFFIC_BYTES_PER_SHARD_C2 if is_c2_shard else None,
                     "traffic_source": "sum over ALL kernels of one region of dram__bytes_read.sum + dram__bytes_write.sum, ncu launch list on a 2.3 Mb shard (profiles/r2_launches.csv)",
                     "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback (B200_PROFILING.md)",
                     "algorithmic_bytes_per_step": alg_bytes, "algorithmic_bytes_per_launch": alg_bytes / len(shards),
                     "launch_ms": step_s * 1e3 / len(shards),
                     "timed": "CUDA events around whole steps, %d shards in flight (same region as `value`)" % max(1, args.inflight),
                     "dominant_kernel": {"kernel": "pileup / call / site stage alone: k_pile_reads + k_cell_codes + k_hard_cells + k_fast_sites (library events, shards one after the other)",
                                         "launch_ms": pile_ms / len(shards), "achieved": alg_bytes / (pile_ms / 1e3) / 1e9,
                                         "frac": alg_bytes / (pile_ms / 1e3) / 1e9 / peak_gbs, "share_of_step": pile_ms / max(seq_ms, 1e-9)}},
        "clocks": clk.summary(),
    }
    if verified:
        line["verified"] = verified
    if pbtest.AN["LD_ZNS"] & an or pbtest.AN["LD_OMEGA"] & an:
        # pairwise LD: kept SNP pairs per step (x2 when omega_max needs the sums on both sides) over the statistics stage's time
        pairs = 0
        for c in ctxs:
            k = pbtest.arr(c.res.ld_num_snps, c.res.n_windows * c.res.n_pops).astype(np.int64)
            pairs += int((k * (k - 1) // 2).sum())
        line["ld"] = {"snp_pairs_per_step": pairs, "stats_stage_ms_per_step": stage_ms[3],
                      "pairs_per_s": pairs * (2 if pbtest.AN["LD_OMEGA"] & an else 1) / max(stage_ms[3] / 1e3, 1e-12),
                      "note": "integer popcount work (AND, POPC, IMAD, one DFMA per pair); pipe utilisation from ncu in profiles/"}
    if rank == 0 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline(args, args.cpu_sample_kb * 1000)
        if args.cli_sample_kb != 0:
            cli_len = int(min(args.contig_mb, 5.0) * 1e6) if args.cli_sample_kb < 0 else int(min(args.cli_sample_kb * 1000, args.contig_mb * 1e6))
            line["cli_from_bam"] = cli_from_bam(args, cli_len)
    if last_step:
        dump_outputs(args.dump_outputs, last_step)
    if rank == 0:
        print(json.dumps(line))
    for c in ctxs:
        c.close()
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


def ref_runs(cfg):
    """The reference has one subcommand (and one -o mode) per process: the runs that produce what the configuration's
    single pass produces."""
    w = str(cfg["win"] // 1000)
    og = ["-p", "og"] if "OUTGROUP" in cfg["flags"] else []
    runs = []
    for a in cfg["an"]:
        runs.append({"NUCDIV": ["nucdiv", "-w", w] + og, "SFS": ["sfs", "-w", w] + og, "LD_ZNS": ["ld", "-o", "0", "-w", w], "LD_OMEGA": ["ld", "-o", "1", "-w", w],
                     "LD_WALL": ["ld", "-o", "2", "-w", w], "DIVERGE_IND": ["diverge", "-o", "0", "-w", w] + og, "DIVERGE_POP": ["diverge", "-o", "1", "-w", w] + og,
                     "HAPLO_K": ["haplo", "-o", "0", "-w", w], "HAPLO_EHHS": ["haplo", "-o", "1", "-w", w], "HAPLO_DXY": ["haplo", "-o", "2", "-w", w]}[a])
    return runs


def scaled_sample(cfg, base_len):
    """Sample length with about the work of `base_len` positions of configs[1] (11 samples x 30x), a whole number of windows."""
    scale = (11 * 30.0) / ((cfg["n_ingroup"] + cfg["has_outgroup"]) * cfg["depth"]) / max(1, len(cfg["an"]))
    return max(2, int(round(base_len * scale / cfg["win"]))) * cfg["win"]


def cpu_baseline(args, sample_len):
    """One host core on a bounded sample of the same workload: the unmodified reference binary when it is there
    (kind "reference"), else the oracle port (kind "port")."""
    import pbtest
    cfg = args.cfg
    sample_len = scaled_sample(cfg, sample_len)
    fx = config_fixture(cfg, sample_len, 77, 8)
    aligned = fx.aligned_bases()
    wb, we = product_window_grid(0, fx.contig_len, cfg["win"])
    nwin = len(wb)
    if pbtest.have_ref():
        with tempfile.TemporaryDirectory() as td:
            bam, fa = fx.write_files(Path(td) / "s")
            t0 = time.perf_counter()
            for r in ref_runs(cfg):
                pbtest.run_ref(r + ["-f", fa, bam, "chr1"])
            dt = time.perf_counter() - t0
        kind = "reference"
    else:
        p = config_params(cfg, fx)
        an = 0
        for a in cfg["an"]:
            an |= pbtest.AN[a]
        t0 = time.perf_counter()
        pbtest.OracleRun(p, fx.batch(), fx.ref(), an, wb, we).close()
        dt = time.perf_counter() - t0
        kind = "port"
    fx.close()
    return {"value": aligned / dt / 1e9, "unit": "Gbases/s", "cores": 1, "kind": kind, "windows_per_s": nwin / dt,
            "sample": "%d kb of the same workload (%d windows, %.3f Gbases), %d reference process(es) one after the other, %.1f s" % (
                sample_len // 1000, nwin, aligned / 1e9, len(ref_runs(cfg)), dt)}


def cli_from_bam(args, sample_len):
    """Third timing tier (SURVEY.md §8(d), "E"): the `popbam` command line on BAM/BAI/FASTA files -- BAI slicing, BGZF
    inflate and record decode on host threads into pinned batches, then the GPU path -- wall time of the whole process.
    Start-up (CUDA context, error-model tables, index, FASTA) is measured separately on a one-window region."""
    import pbtest
    import popbam_b200
    cfg = args.cfg
    exe = popbam_b200.capi.PKG / "_build" / "popbam"
    if not exe.exists():
        return {"unavailable": "popbam executable not built"}
    sample_len = max(cfg["win"] * 2, (sample_len // cfg["win"]) * cfg["win"])
    fx = config_fixture(cfg, sample_len, 78, min(32, os.cpu_count() or 4))
    aligned = fx.aligned_bases()
    nwin = len(product_window_grid(0, fx.contig_len, cfg["win"])[0])
    runs = ref_runs(cfg)
    with tempfile.TemporaryDirectory(dir="/dev/shm" if os.path.isdir("/dev/shm") else None) as td:
        bam, fa = fx.write_files(Path(td) / "c")
        bam_bytes = os.path.getsize(bam)
        fx.close()

        def once(region):
            t0 = time.perf_counter()
            rows = 0
            for r in runs:
                q = subprocess.run([str(exe)] + r + ["-f", fa, bam, region], stdout=subprocess.PIPE, stderr=subprocess.PIPE)
                if q.returncode != 0:
                    raise RuntimeError("popbam failed: " + q.stderr.decode()[-300:])
                rows += q.stdout.count(b"\n")
            return time.perf_counter() - t0, rows
        try:
            once("chr1")                                            # page cache, driver
            best, rows = min(once("chr1") for _ in range(2))
            startup = min(once("chr1:1-%d" % (cfg["win"] + 1))[0] for _ in range(2))
        except RuntimeError as e:
            return {"unavailable": str(e)}
    return {"value": aligned / best / 1e9, "unit": "Gbases/s", "windows_per_s": nwin / best, "wall_s": best, "rows": rows,
            "startup_s": startup, "startup_note": "the same command on a one-window region (CUDA context, tables, index, FASTA); in the full run the host threads decode while the context comes up, so the two do not subtract",
            "host_threads": os.cpu_count() or 4, "bam_bytes": bam_bytes,
            "sample": "%.1f Mb BAM of the same workload (%d windows, %.3f Gbases, %.0f MB compressed), %d popbam process(es), whole process incl. CUDA start-up" % (
                sample_len / 1e6, nwin, aligned / 1e9, bam_bytes / 1e6, len(runs))}


def run_reference(args):
    """Reference arm: the reference's CPU implementation with every host core, one `popbam` process per core over
    split regions chr1:a+1-a+mW+1 (BASELINE.md CPU-baseline plan); a step = all regions once (and all the
    configuration's subcommands, one after the other: the reference computes one per process)."""
    import pbtest
    rank, world, _ = dist_env()
    if rank != 0:
        return
    cfg = args.cfg
    WIN = cfg["win"]
    cores = os.cpu_count() or 1
    procs = min(cores, 64)
    win_per_proc = max(1, scaled_sample(cfg, 4 * 10000) // WIN)
    length = procs * win_per_proc * WIN
    fx = config_fixture(cfg, length, 77, min(32, cores))
    aligned = fx.aligned_bases()
    use_ref = pbtest.have_ref()
    runs = ref_runs(cfg)
    with tempfile.TemporaryDirectory() as td:
        if use_ref:
            bam, fa = fx.write_files(Path(td) / "r")
            regions = ["chr1:%d-%d" % (i * win_per_proc * WIN + 1, (i + 1) * win_per_proc * WIN + 1) for i in range(procs)]

            def step():
                for r in runs:
                    ps = [subprocess.Popen([str(pbtest.REF_BIN)] + r + ["-f", fa, bam, reg], stdout=subprocess.DEVNULL,
                                           stderr=subprocess.DEVNULL) for reg in regions]
                    for q in ps:
                        if q.wait() != 0:
                            raise RuntimeError("reference popbam failed")
            kind = "reference"
        else:
            p = config_params(cfg, fx)
            an = 0
            for a in cfg["an"]:
                an |= pbtest.AN[a]
            b, ref = fx.batch(), fx.ref()
            grids = [product_window_grid(i * win_per_proc * WIN, (i + 1) * win_per_proc * WIN + 1, WIN) for i in range(procs)]

            def one(i):
                pbtest.OracleRun(p, b, ref, an, grids[i][0], grids[i][1]).close()

            def step():
                th = [threading.Thread(target=one, args=(i,)) for i in range(procs)]     # ctypes releases the GIL
                [t.start() for t in th]
                [t.join() for t in th]
            kind = "port"
        for _ in range(args.warmup):
            step()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            step()
        dt = (time.perf_counter() - t0) / args.steps
    value = aligned / dt / 1e9
    nwin = procs * win_per_proc
    sample = "%d regions of %d kb (%d windows, %.3f Gbases) of the same workload per step, one process per core%s" % (
        procs, win_per_proc * WIN // 1000, nwin, aligned / 1e9, ", %d subcommands one after the other" % len(runs) if len(runs) > 1 else "")
    print(json.dumps({
        "impl": "reference", "metric": "aligned Gbases/s", "value": value, "unit": "Gbases/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8/u64 + f64 (error model)", "data": "synthetic (tools/pbsynth, seeded)",
        "config": {"workload": "%s, %d samples, %gx, 100 bp reads, %d kb windows; bounded sample: %s" % (cfg["label"], fx.n_samples, cfg["depth"], WIN // 1000, sample),
                   "config": args.config, "windows_per_s": nwin / dt},
        "cpu_baseline": {"value": value, "unit": "Gbases/s", "cores": procs, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "Gbases/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
    fx.close()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
