"""Cost of Lewontin's D' (PB_AN_LD_DPRIME) on top of ZnS: the statistics stage (pb_stage_times [3]: k_ld_keep, k_ld_rows,
k_ld_finish) of one region with LD_ZNS against LD_ZNS | LD_DPRIME, in interleaved relaunches on reads resident on the
device.  Data: the shape of the ld configuration (BASELINE.json configs[2]: 64 samples, 20x, dense SNPs, 50 kb windows),
one 0.5 Mb shard.  Prints one JSON line (and writes it to --out).

    python tools/ext_stats_bench.py [--reps 40] [--out FILE]
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
from popbam_b200.capi import AN  # noqa: E402


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=60)
        return q.stdout.strip()
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=40)
    ap.add_argument("--contig-kb", type=int, default=500)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    fx = pbtest.Fixture(contig_len=args.contig_kb * 1000 + 500, n_ingroup=64, has_outgroup=0, depth=20.0, snp_density=0.06, seed=31)
    p = fx.params()
    wb, we = pbtest.window_grid(0, fx.contig_len, 50000)
    variants = {"zns": AN["LD_ZNS"], "zns+dprime": AN["LD_ZNS"] | AN["LD_DPRIME"]}
    ctxs = {}
    for name, an in variants.items():
        c = popbam_b200.Context(p)
        c.set_contig(0, fx.ref())
        c.region_begin(an, wb, we)
        c.push_batch(fx.batch())
        c.region_end()
        ctxs[name] = c
    # the same windows, the same ZnS
    nwp = len(wb) * fx.n_pops
    z = {k: pbtest.arr(c.res.zns, nwp) for k, c in ctxs.items()}
    assert np.array_equal(z["zns"], z["zns+dprime"])
    kept = pbtest.arr(ctxs["zns+dprime"].ext.ld_kept, nwp).astype(np.int64)
    pairs = int((kept * (kept - 1) // 2).sum())
    ms = {k: [] for k in variants}
    for rep in range(args.reps + 3):                      # 3 warm-up rounds, then interleaved
        for k, c in ctxs.items():
            c.relaunch()
            c.wait()
            if rep >= 3:
                ms[k].append(c.stage_times()[3])
    out = {"tool": "tools/ext_stats_bench.py", "gpu": gpu_info(),
           "workload": "pbsynth contig %d kb, 64 samples in %d population(s), 20x, SNP density 0.06, %d windows of 50 kb" % (args.contig_kb, fx.n_pops, len(wb)),
           "kept_snps_per_window": [int(x) for x in kept], "snp_pairs": pairs, "reps": args.reps,
           "timed": "pb_stage_times [3] (CUDA events around k_ld_keep + k_ld_rows + k_ld_finish), relaunches on resident reads, the two analyses alternating"}
    for k, v in ms.items():
        a = np.array(v)
        out[k] = {"stats_stage_ms_median": float(np.median(a)), "ms_min": float(a.min()), "ms_max": float(a.max()),
                  "pairs_per_s_median": pairs / (float(np.median(a)) / 1e3)}
    out["dprime_cost_ratio_median"] = out["zns+dprime"]["stats_stage_ms_median"] / out["zns"]["stats_stage_ms_median"]
    line = json.dumps(out)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")
    for c in ctxs.values():
        c.close()


if __name__ == "__main__":
    main()
