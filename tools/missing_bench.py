"""Cost of pi and dxy over sites with missing calls (PB_AN_NUCDIV_MISSING, k_nucdiv_missing) in the window stage:
pb_stage_times [3] (CUDA events around the window statistics) and [1] (the pileup stage) of one region with nucdiv alone
(PB_AN_NUCDIV) and with PB_AN_NUCDIV | PB_AN_NUCDIV_MISSING, in interleaved relaunches on reads resident on the device.
Shapes:
  * the shape of BASELINE.json configs[1] (10 ingroup samples in two populations of 5 + an outgroup, 30x, 100 bp reads,
    SNP density 0.01, one 2.3 Mb shard) with 10 kb windows, 1 kb windows and one window over the shard (-w 0);
  * a 64-sample shape at 10x, where most positions are covered in some samples but not all (63 ingroup samples regrouped
    into three populations of 21 + the outgroup, 0.5 Mb, 5 kb windows).
The arrays of the first and the last region are checked against the numpy restatement of the definition
(tests/test_missing_host.py), fed with the per-cell words of the same region from a run with PB_FLAG_EMIT_CB.  Prints one
JSON line (and writes it to --out).

    python tools/missing_bench.py [--reps 30] [--out FILE]
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
from test_missing_host import assert_missing_same, expected, missing_arrays  # noqa: E402

AN = capi.AN
C1 = dict(contig_len=2300001, n_ingroup=10, has_outgroup=1, depth=30.0, read_len=100, snp_density=0.01, seed=41)
LOW64 = dict(contig_len=500001, n_ingroup=63, has_outgroup=1, depth=10.0, read_len=100, snp_density=0.01, seed=53)
SHAPES = {
    "c1_2.3mb_10kb": dict(fx=C1, win=10000, groups=None),
    "c1_2.3mb_1kb": dict(fx=C1, win=1000, groups=None),
    "c1_2.3mb_w0": dict(fx=C1, win=0, groups=None),
    "low64_0.5mb_5kb": dict(fx=LOW64, win=5000, groups=[21, 21, 21]),
}


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=60)
        return q.stdout.strip()
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def shape_params(fx, groups, flags=0):
    """The fixture's populations, or its ingroup samples regrouped with the outgroup sample (the last) alone."""
    p = fx.params(flags=flags)
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


def restated(fx, shape, wb, we):
    """The numpy restatement over the per-cell words of a PB_FLAG_EMIT_CB run of the same region (single-kernel path)."""
    p = shape_params(fx, shape["groups"], pbtest.FLAG["EMIT_CB"])
    c = popbam_b200.Context(p)
    c.set_contig(0, fx.ref())
    c.region_begin(AN["NUCDIV_MISSING"], wb, we)
    c.push_batch(fx.batch())
    c.region_end()
    res = c.res
    cb = pbtest.arr(res.cb, (res.span_end - res.span_beg) * p.n_samples).reshape(-1, p.n_samples)
    want = expected(p, cb, wb, we, res.span_beg)
    assert_missing_same(missing_arrays(c.nucdiv_missing, res.n_windows, p.n_pops), want)
    partly = ((cb & np.uint64(1)) != 0).sum(axis=1)
    share = float(((partly > 0) & (partly < p.n_samples)).mean())
    c.close()
    return want, share


def measure(fx, shape, reps):
    p = shape_params(fx, shape["groups"])
    P = p.n_pops
    wb, we = pbtest.window_grid(0, fx.contig_len, shape["win"])
    want, partly = restated(fx, shape, wb, we)
    variants = {"off": AN["NUCDIV"], "on": AN["NUCDIV"] | AN["NUCDIV_MISSING"]}
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
    assert on.path() == 1
    assert np.array_equal(pbtest.arr(ctxs["off"].res.piw, NW * P), pbtest.arr(on.res.piw, NW * P), equal_nan=True)
    assert_missing_same(missing_arrays(on.nucdiv_missing, NW, P), want)           # the first region
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
    assert_missing_same(missing_arrays(on.nucdiv_missing, NW, P), want)           # the last region
    sites = int(pbtest.arr(on.res.num_sites, NW).sum())
    pi_sites = want["pi_sites"].reshape(NW, P)
    out = {"workload": "pbsynth contig %d kb, %d samples in %d populations (%s), %.0fx, 100 bp reads, SNP density 0.01, %d windows of %s, "
                       "%d positions with every sample covered, %.3f of the positions partly covered, pi positions per population %s"
                       % (fx.contig_len // 1000, fx.n_samples, P, "/".join(str(int(p.pop_nsmpl[i])) for i in range(P)),
                          shape["fx"]["depth"], NW, "%d kb" % (shape["win"] // 1000) if shape["win"] else "the whole shard", sites, partly,
                          "/".join(str(int(x)) for x in pi_sites.sum(axis=0)))}
    for k in variants:
        a, b = np.array(stats[k]), np.array(pile[k])
        out[k] = {"window_stage_ms_median": float(np.median(a)), "ms_min": float(a.min()), "ms_max": float(a.max()),
                  "pileup_stage_ms_median": float(np.median(b))}
    out["added_ms"] = out["on"]["window_stage_ms_median"] - out["off"]["window_stage_ms_median"]
    out["added_share_of_pileup"] = out["added_ms"] / out["off"]["pileup_stage_ms_median"]
    out["pileup_on_minus_off_ms"] = out["on"]["pileup_stage_ms_median"] - out["off"]["pileup_stage_ms_median"]
    for c in ctxs.values():
        c.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--shapes", default=",".join(SHAPES))
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    out = {"tool": "tools/missing_bench.py", "gpu": gpu_info(), "reps": args.reps,
           "timed": "pb_stage_times [3] (CUDA events around the window statistics: k_window_stats, k_nucdiv_missing, k_nucdiv_missing_ratio) "
                    "and [1] (the pileup stage), relaunches on resident reads, nucdiv alone ('off') and nucdiv + PB_AN_NUCDIV_MISSING ('on') "
                    "alternating"}
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
