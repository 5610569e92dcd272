"""Cost of the site frequency spectra (PB_AN_SPECTRUM, k_spectrum) in the window stage: pb_stage_times [3] (CUDA events
around the window statistics) and [1] (the pileup stage) of one region with `sfs -p` alone (PB_AN_SFS with the outgroup
flip) and with PB_AN_SFS | PB_AN_SPECTRUM, in interleaved relaunches on reads resident on the device.  Shapes:
  * the shape of BASELINE.json configs[1] (10 ingroup samples in two populations of 5 + an outgroup, 30x, 100 bp reads,
    SNP density 0.01, one 2.3 Mb shard) with 10 kb and with 1 kb windows; the command line's default sets (popA, popB,
    popA-popB);
  * a dense 64-sample shape: 63 ingroup samples regrouped into three populations of 21 + the outgroup, 30x, so that most
    sites have every sample covered (at 10x almost none has, and a bench there would measure the launch only); the default
    sets (three 1-D, three 2-D) plus the 3-D set (A, B, C) of 22 x 22 x 22 bins.
The spectra of the first and the last region are checked against the numpy restatement of the definition
(tests/test_spectrum_host.py) on the same segregating sites.  Prints one JSON line (and writes it to --out).

    python tools/spectrum_bench.py [--reps 30] [--out FILE]
"""
import argparse
import json
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
import pbtest  # noqa: E402
import popbam_b200  # noqa: E402
from popbam_b200 import capi  # noqa: E402
from test_spectrum_host import default_sets, expected_spectrum, seg_windows, spectrum_arrays  # noqa: E402

AN = capi.AN
C1 = dict(contig_len=2300001, n_ingroup=10, has_outgroup=1, depth=30.0, read_len=100, snp_density=0.01, seed=41)
DENSE = dict(contig_len=500001, n_ingroup=63, has_outgroup=1, depth=30.0, read_len=100, snp_density=0.01, seed=47)
SHAPES = {
    "c1_2.3mb_10kb": dict(fx=C1, win=10000, groups=None),
    "c1_2.3mb_1kb": dict(fx=C1, win=1000, groups=None),
    "dense64_0.5mb_5kb": dict(fx=DENSE, win=5000, groups=[21, 21, 21]),
}


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=60)
        return q.stdout.strip()
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def shape_params(fx, groups):
    """The fixture's populations, or its ingroup samples regrouped; the outgroup sample (the last) polarises."""
    p = fx.params(flags=pbtest.FLAG["OUTGROUP"], outidx=fx.n_samples - 1)
    if groups:
        for k in range(64):
            p.pop_mask[k], p.pop_nsmpl[k] = 0, 0
        s = 0
        for g, m in enumerate(groups + [1]):
            p.pop_mask[g] = ((1 << m) - 1) << s
            p.pop_nsmpl[g] = m
            s += m
        p.n_pops = len(groups) + 1
    return p


def check(ctx, p, sets):
    counts, _, _ = spectrum_arrays(ctx.spectrum, ctx.res)
    W, ns = seg_windows(ctx.res)
    assert np.array_equal(counts, expected_spectrum(W, ns, p, sets))


def measure(fx, shape, reps):
    p = shape_params(fx, shape["groups"])
    P = p.n_pops
    og = P - 1
    sets = default_sets(P, og) + ([(0, 1, 2)] if shape["groups"] else [])
    wb, we = pbtest.window_grid(0, fx.contig_len, shape["win"])
    variants = {"off": AN["SFS"], "on": AN["SFS"] | AN["SPECTRUM"]}
    ctxs = {}
    for name, an in variants.items():
        c = popbam_b200.Context(p)
        c.set_contig(0, fx.ref())
        c.set_spectra(sets)
        c.region_begin(an, wb, we)
        c.push_batch(fx.batch())
        c.region_end()
        ctxs[name] = c
    NW = len(wb)
    on = ctxs["on"]
    assert np.array_equal(pbtest.arr(ctxs["off"].res.td, NW * P), pbtest.arr(on.res.td, NW * P), equal_nan=True)
    check(on, p, sets)
    segs = int(pbtest.arr(on.res.segsites, NW).sum())
    sites = int(pbtest.arr(on.res.num_sites, NW).sum())
    stats = {k: [] for k in variants}
    pile = {k: [] for k in variants}
    for rep in range(reps + 3):                      # 3 warm-up rounds, then interleaved
        for k, c in ctxs.items():
            c.relaunch()
            c.wait()
            if rep >= 3:
                t = c.stage_times()
                stats[k].append(t[3])
                pile[k].append(t[1])
    check(on, p, sets)
    out = {"workload": "pbsynth contig %d kb, %d samples in %d populations (%s), %.0fx, 100 bp reads, SNP density 0.01, %d windows of %d kb, "
                       "%d sites with every sample covered, %d segregating sites, %d spectrum sets, %d bins per window"
                       % (fx.contig_len // 1000, fx.n_samples, P, "/".join(str(int(p.pop_nsmpl[i])) for i in range(P)),
                          shape["fx"]["depth"], NW, shape["win"] // 1000, sites, segs, len(sets), on.spectrum.n_bins)}
    for k in variants:
        a, b = np.array(stats[k]), np.array(pile[k])
        out[k] = {"window_stage_ms_median": float(np.median(a)), "ms_min": float(a.min()), "ms_max": float(a.max()),
                  "pileup_stage_ms_median": float(np.median(b))}
    out["added_ms"] = out["on"]["window_stage_ms_median"] - out["off"]["window_stage_ms_median"]
    out["added_share_of_pileup"] = out["added_ms"] / out["off"]["pileup_stage_ms_median"]
    for c in ctxs.values():
        c.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--shapes", default=",".join(SHAPES))
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    out = {"tool": "tools/spectrum_bench.py", "gpu": gpu_info(), "reps": args.reps,
           "timed": "pb_stage_times [3] (CUDA events around the window statistics: k_window_stats, k_spectrum) and [1] (the pileup stage), "
                    "relaunches on resident reads, sfs -p alone ('off') and sfs -p + PB_AN_SPECTRUM ('on') alternating"}
    fixtures = {}
    for name in args.shapes.split(","):
        key = json.dumps(SHAPES[name]["fx"], sort_keys=True)
        if key not in fixtures:
            fixtures[key] = pbtest.Fixture(**SHAPES[name]["fx"])
        out[name] = measure(fixtures[key], SHAPES[name], args.reps)
    for fx in fixtures.values():
        fx.close()
    line = json.dumps(out)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
