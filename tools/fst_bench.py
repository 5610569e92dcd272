"""Cost of F_ST and Snn (PB_AN_FST) in the window stage: pb_stage_times [3] (CUDA events around k_window_stats and, with
permutations, k_snn_perm) of one region in four configurations -- nucdiv alone, nucdiv + F_ST, and nucdiv + F_ST with
1 000 and with 10 000 Snn permutations per (window, pair) -- in interleaved relaunches on reads resident on the device.
The pileup stage (pb_stage_times [1], k_pile_reads) of the same relaunches is reported beside it.  Data: the shape of
BASELINE.json configs[1] (10 samples in two populations + an outgroup, 30x, 100 bp reads, SNP density 0.01, 10 kb
windows), one 2.3 Mb shard.  Prints one JSON line (and writes it to --out).

    python tools/fst_bench.py [--reps 30] [--out FILE]
    python tools/fst_bench.py --variants off      (from a checkout of an earlier commit: its window stage without F_ST)
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
VARIANTS = {"off": (AN["NUCDIV"], 0), "on": (AN["NUCDIV"] | AN.get("FST", 0), 0),
            "perm1000": (AN["NUCDIV"] | AN.get("FST", 0), 1000), "perm10000": (AN["NUCDIV"] | AN.get("FST", 0), 10000)}


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=60)
        return q.stdout.strip()
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--contig-kb", type=int, default=2300)
    ap.add_argument("--variants", default=",".join(VARIANTS))
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    names = args.variants.split(",")
    fx = pbtest.Fixture(contig_len=args.contig_kb * 1000 + 1, n_ingroup=10, has_outgroup=1, depth=30.0, read_len=100, snp_density=0.01, seed=41)
    p = fx.params(flags=pbtest.FLAG["OUTGROUP"], outidx=fx.n_samples - 1)
    wb, we = pbtest.window_grid(0, fx.contig_len, 10000)
    ctxs = {}
    for name in names:
        an, perms = VARIANTS[name]
        c = popbam_b200.Context(p)
        c.set_contig(0, fx.ref())
        if perms:
            c.set_snn_perms(perms, 1)
        c.region_begin(an, wb, we)
        c.push_batch(fx.batch())
        c.region_end()
        ctxs[name] = c
    NW, P = len(wb), fx.n_pops
    # the same windows, the same pi / dxy, the same F_ST whatever else runs
    piw = {k: pbtest.arr(c.res.piw, NW * P) for k, c in ctxs.items()}
    assert all(np.array_equal(v, piw[names[0]]) for v in piw.values())
    fst = {k: pbtest.arr(c.fst.fst_hudson, NW * P * P) for k, c in ctxs.items() if k != "off"}
    assert all(np.array_equal(v, next(iter(fst.values())), equal_nan=True) for v in fst.values())
    segs = int(pbtest.arr(ctxs[names[0]].res.segsites, NW).sum())
    stats = {k: [] for k in names}
    pile = {k: [] for k in names}
    for rep in range(args.reps + 3):                      # 3 warm-up rounds, then interleaved
        for k, c in ctxs.items():
            c.relaunch()
            c.wait()
            if rep >= 3:
                t = c.stage_times()
                stats[k].append(t[3])
                pile[k].append(t[1])
    pairs = P * (P - 1) // 2
    pairs_snn = sum(1 for i in range(P) for j in range(i + 1, P) if p.pop_nsmpl[i] >= 2 and p.pop_nsmpl[j] >= 2)
    out = {"tool": "tools/fst_bench.py", "gpu": gpu_info(),
           "workload": "pbsynth contig %d kb, %d samples in %d populations (%s), 30x, 100 bp reads, SNP density 0.01, %d windows of 10 kb, "
                       "%d segregating sites" % (args.contig_kb, fx.n_samples, P, "/".join(str(int(p.pop_nsmpl[i])) for i in range(P)), NW, segs),
           "pairs": pairs, "pairs_with_snn": pairs_snn, "reps": args.reps,
           "timed": "pb_stage_times [3] (CUDA events around k_window_stats + k_snn_perm) and [1] (the pileup stage), relaunches on resident reads, "
                    "the variants alternating"}
    for k in names:
        a, b = np.array(stats[k]), np.array(pile[k])
        out[k] = {"window_stage_ms_median": float(np.median(a)), "ms_min": float(a.min()), "ms_max": float(a.max()),
                  "pileup_stage_ms_median": float(np.median(b))}
        if VARIANTS[k][1]:
            out[k]["permutations_per_s"] = VARIANTS[k][1] * NW * pairs_snn / (float(np.median(a)) / 1e3)
    if "off" in out:
        for k in names:
            if k != "off":
                out[k]["over_off_ms"] = out[k]["window_stage_ms_median"] - out["off"]["window_stage_ms_median"]
                out[k]["over_off_share_of_pileup"] = out[k]["over_off_ms"] / out["off"]["pileup_stage_ms_median"]
    line = json.dumps(out)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")
    for c in ctxs.values():
        c.close()


if __name__ == "__main__":
    main()
