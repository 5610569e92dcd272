"""Cost of Garud's H (PB_AN_GARUD, k_garud) in the window stage: pb_stage_times [3] (CUDA events around the window
statistics) and [1] (the pileup stage) of one region with `haplo -o 0` alone (PB_AN_HAPLO_K) and with PB_AN_HAPLO_K |
PB_AN_GARUD, in interleaved relaunches on reads resident on the device.  Shapes:
  * the shape of BASELINE.json configs[1] (10 ingroup samples in two populations of 5 + an outgroup, 30x, 100 bp reads,
    SNP density 0.01, one 2.3 Mb shard) with 10 kb windows and with 1 kb windows (ten times the CTAs, a tenth of the
    sites each);
  * 63 ingroup samples in populations of 32 and 31 + an outgroup, 1 Mb at 10x, 10 kb windows.  At 10x few sites have every
    one of 64 samples covered, so this shape measures the launch over 64-sample populations more than the per-site work.
The Garud arrays of the first region are checked against a numpy restatement of the definition (tests/test_garud_host.py)
on the same segregating sites.  Prints one JSON line (and writes it to --out).

    python tools/garud_bench.py [--reps 30] [--out FILE]
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
from test_garud_host import assert_garud_same, expected_garud, garud_arrays, seg_windows  # noqa: E402

AN = capi.AN
C1 = dict(contig_len=2300001, n_ingroup=10, has_outgroup=1, depth=30.0, read_len=100, snp_density=0.01, seed=41)
SHAPES = {
    "c1_2.3mb_10kb": dict(fx=C1, win=10000),
    "c1_2.3mb_1kb": dict(fx=C1, win=1000),
    "n64_1mb_10kb": dict(fx=dict(contig_len=1000001, n_ingroup=63, has_outgroup=1, depth=10.0, read_len=100, snp_density=0.01, seed=43),
                         win=10000),
}


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=60)
        return q.stdout.strip()
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def measure(fx, shape, reps):
    p = fx.params()
    P = p.n_pops
    wb, we = pbtest.window_grid(0, fx.contig_len, shape["win"])
    variants = {"off": AN["HAPLO_K"], "on": AN["HAPLO_K"] | AN["GARUD"]}
    ctxs = {}
    for name, an in variants.items():
        c = popbam_b200.Context(p)
        c.set_contig(0, fx.ref())
        c.region_begin(an, wb, we)
        c.push_batch(fx.batch())
        c.region_end()
        ctxs[name] = c
    NW = len(wb)
    on = ctxs["on"]
    assert np.array_equal(pbtest.arr(ctxs["off"].res.nhaps, NW * P), pbtest.arr(on.res.nhaps, NW * P))
    assert_garud_same(garud_arrays(on.garud, on.res), expected_garud(seg_windows(on.res), p))
    segs = int(pbtest.arr(on.res.segsites, NW).sum())
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
    assert_garud_same(garud_arrays(on.garud, on.res), expected_garud(seg_windows(on.res), p))
    out = {"workload": "pbsynth contig %d kb, %d samples in %d populations (%s), %.0fx, 100 bp reads, SNP density 0.01, %d windows of %d kb, "
                       "%d segregating sites" % (fx.contig_len // 1000, fx.n_samples, P, "/".join(str(int(p.pop_nsmpl[i])) for i in range(P)),
                                                 shape["fx"]["depth"], NW, shape["win"] // 1000, segs)}
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
    out = {"tool": "tools/garud_bench.py", "gpu": gpu_info(), "reps": args.reps,
           "timed": "pb_stage_times [3] (CUDA events around the window statistics: k_window_stats, k_garud) and [1] (the pileup stage), "
                    "relaunches on resident reads, haplo -o 0 alone ('off') and haplo -o 0 + PB_AN_GARUD ('on') alternating"}
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
