"""Cost of the ABBA-BABA pass (PB_AN_ABBA, k_abba) in the window stage: pb_stage_times [3] (CUDA events around the
window statistics) and [1] (the pileup stage) of one region with nucdiv alone and with nucdiv + ABBA, in interleaved
relaunches on reads resident on the device.  Two shapes:
  * the shape of BASELINE.json configs[1] (10 ingroup samples + an outgroup, 30x, 100 bp reads, SNP density 0.01, 10 kb
    windows, one 2.3 Mb shard), the ingroup regrouped 3 / 3 / 4: 3 triples;
  * 63 ingroup samples + an outgroup in nine populations of 7, 1 Mb at 10x, 10 kb windows: 252 triples.  At 10x few sites
    have every one of 64 samples covered, so this shape measures the cost of the 252-triple launch more than the per-site
    work.
Prints one JSON line (and writes it to --out).

    python tools/abba_bench.py [--reps 30] [--out FILE]
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

AN = capi.AN
SHAPES = {
    "c1_2.3mb": dict(fx=dict(contig_len=2300001, n_ingroup=10, has_outgroup=1, depth=30.0, read_len=100, snp_density=0.01, seed=41),
                     groups=[3, 3, 4]),
    "n64_1mb": dict(fx=dict(contig_len=1000001, n_ingroup=63, has_outgroup=1, depth=10.0, read_len=100, snp_density=0.01, seed=43),
                    groups=[7] * 9),
}


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=60)
        return q.stdout.strip()
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def regroup(fx, groups):
    """pb_params with the ingroup samples in consecutive populations of `groups` and the outgroup sample alone, last."""
    p = fx.params()
    for k in range(64):
        p.pop_mask[k], p.pop_nsmpl[k] = 0, 0
    s = 0
    for g, m in enumerate(groups + [1]):
        p.pop_mask[g], p.pop_nsmpl[g] = ((1 << m) - 1) << s, m
        s += m
    p.n_pops = len(groups) + 1
    return p


def measure(shape, reps):
    fx = pbtest.Fixture(**shape["fx"])
    p = regroup(fx, shape["groups"])
    P, og = p.n_pops, p.n_pops - 1
    triples = [(i, j, k) for i in range(P) for j in range(i + 1, P) for k in range(P) if og not in (i, j, k) and k not in (i, j)]
    wb, we = pbtest.window_grid(0, fx.contig_len, 10000)
    variants = {"off": AN["NUCDIV"], "on": AN["NUCDIV"] | AN["ABBA"]}
    ctxs = {}
    for name, an in variants.items():
        c = popbam_b200.Context(p)
        c.set_contig(0, fx.ref())
        c.set_abba(og, triples)
        c.region_begin(an, wb, we)
        c.push_batch(fx.batch())
        c.region_end()
        ctxs[name] = c
    NW = len(wb)
    assert np.array_equal(pbtest.arr(ctxs["off"].res.piw, NW * P), pbtest.arr(ctxs["on"].res.piw, NW * P))
    segs = int(pbtest.arr(ctxs["off"].res.segsites, NW).sum())
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
    out = {"workload": "pbsynth contig %d kb, %d samples in %d populations (%s), %.0fx, 100 bp reads, SNP density 0.01, %d windows of 10 kb, "
                       "%d segregating sites" % (fx.contig_len // 1000, fx.n_samples, P, "/".join(str(int(p.pop_nsmpl[i])) for i in range(P)),
                                                 shape["fx"]["depth"], NW, segs),
           "triples": len(triples)}
    for k in variants:
        a, b = np.array(stats[k]), np.array(pile[k])
        out[k] = {"window_stage_ms_median": float(np.median(a)), "ms_min": float(a.min()), "ms_max": float(a.max()),
                  "pileup_stage_ms_median": float(np.median(b))}
    out["added_ms"] = out["on"]["window_stage_ms_median"] - out["off"]["window_stage_ms_median"]
    out["added_share_of_pileup"] = out["added_ms"] / out["off"]["pileup_stage_ms_median"]
    out["site_triples_per_s"] = segs * len(triples) / (out["added_ms"] / 1e3) if out["added_ms"] > 0 else None
    for c in ctxs.values():
        c.close()
    fx.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--shapes", default=",".join(SHAPES))
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    out = {"tool": "tools/abba_bench.py", "gpu": gpu_info(), "reps": args.reps,
           "timed": "pb_stage_times [3] (CUDA events around the window statistics: k_window_stats, k_abba) and [1] (the pileup stage), "
                    "relaunches on resident reads, nucdiv alone ('off') and nucdiv + PB_AN_ABBA ('on') alternating"}
    for name in args.shapes.split(","):
        out[name] = measure(SHAPES[name], args.reps)
    line = json.dumps(out)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
