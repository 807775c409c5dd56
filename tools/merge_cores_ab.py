"""A/B of the contracted d3 r8 chain (`merge_cores`, DESIGN.md §4.15) on one GPU.

    python tools/merge_cores_ab.py --out DIR [--levels 0,1,2] [--reps 3] [--steps 10] [--warmup 3] [--configs 3,9]
                                   [--dump-configs 3,9,4]

1. Card name, power limit and SM clocks (nvidia-smi), read in the same run as the timings.
2. `bench.py --configs <configs> --no-cpu-baseline` with TTRNN_MERGE_CORES = each of `--levels`, rotated, `--reps` runs
   each: ms_per_step per config and the per-variant k_rnn_fwd / k_rnn_bwd times of every run.
3. `bench.py --configs <dump-configs> --dump-outputs` once per level, and the largest relative difference of every
   dumped array against the first level (norm-wise and element-wise).
Everything goes to DIR/summary.json (and is printed); the raw bench lines to DIR/bench_*.json.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def card_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        res = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=60)
        return {"query": q, "value": res.stdout.strip()}
    except Exception as e:                      # reported, not fatal: the timings still stand with the bench's own record
        return {"query": q, "error": str(e)}


def bench(mc, args, extra, tag):
    env = dict(os.environ, TTRNN_MERGE_CORES=str(mc))
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--no-cpu-baseline"] + extra
    res = subprocess.run(cmd, capture_output=True, text=True, env=env, cwd=ROOT)
    if res.returncode != 0:
        raise SystemExit("bench failed (%s):\n%s" % (" ".join(cmd), res.stderr[-4000:]))
    line = json.loads(res.stdout.strip().splitlines()[-1])
    with open(os.path.join(args.out, "bench_%s.json" % tag), "w") as f:
        json.dump(line, f)
    return line


def per_config(line):
    out = {}
    for rec in line.get("all_configs", []):
        variants = [{k: v[k] for k in ("kernel", "rows_per_cta", "ctas", "rows", "ms_per_launch", "ms_per_step")}
                    for v in (rec.get("roofline") or {}).get("recurrent_variants", [])]
        out[str(rec["id"])] = {"ms_per_step": rec["ms_per_step"], "recurrent_variants": variants,
                               "recurrent_us_per_layer_step": (rec.get("roofline") or {}).get("recurrent_us_per_layer_step")}
    return out


def compare_dumps(d0, d1):
    rows = {}
    for name in sorted(os.listdir(d0)):
        if not name.endswith(".npy"):
            continue
        a, b = np.load(os.path.join(d0, name)).astype(np.float64), np.load(os.path.join(d1, name)).astype(np.float64)
        den = np.linalg.norm(a)
        rows[name] = {"identical": bool(np.array_equal(a, b)),
                      "rel_norm": float(np.linalg.norm(a - b) / den) if den > 0 else float(np.linalg.norm(a - b)),
                      "max_abs_over_max": float(np.max(np.abs(a - b)) / max(np.max(np.abs(a)), 1e-30))}
    return rows


def worst_per_config(cmp):
    worst = {}
    for name, v in cmp.items():
        w = worst.setdefault(name.split("_")[0], {"max_rel_norm": 0.0, "worst_array": None, "all_identical": True})
        if v["rel_norm"] >= w["max_rel_norm"]:
            w["max_rel_norm"], w["worst_array"] = v["rel_norm"], name
        w["all_identical"] = w["all_identical"] and v["identical"]
    return worst


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--levels", default="0,1,2", help="merge_cores values; the first is the reference")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--configs", default="3,9")
    ap.add_argument("--dump-configs", default="3,9,4")
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    levels = [int(v) for v in args.levels.split(",")]
    summary = {"card_before": card_info(), "runs": {str(mc): [] for mc in levels}}
    timing = ["--configs", args.configs, "--steps", str(args.steps), "--warmup", str(args.warmup)]
    for rep in range(args.reps):
        for k in range(len(levels)):
            mc = levels[(k + rep) % len(levels)]
            summary["runs"][str(mc)].append(per_config(bench(mc, args, timing, "mc%d_rep%d" % (mc, rep))))
    summary["card_after"] = card_info()
    stats = {}
    for cid in args.configs.split(","):
        s = {}
        for mc in levels:
            v = [r[cid]["ms_per_step"] for r in summary["runs"][str(mc)]]
            s["merge_cores=%d" % mc] = {"ms_per_step": v, "median": statistics.median(v),
                                        "spread_pct": 100.0 * (max(v) - min(v)) / statistics.median(v)}
        for mc in levels[1:]:
            s["speedup_median_%d" % mc] = s["merge_cores=%d" % levels[0]]["median"] / s["merge_cores=%d" % mc]["median"]
        stats[cid] = s
    summary["stats"] = stats
    if args.dump_configs:
        dirs = {}
        for mc in levels:
            d = os.path.join(args.out, "dump_mc%d" % mc)
            bench(mc, args, ["--configs", args.dump_configs, "--steps", "2", "--warmup", "1", "--dump-outputs", d],
                  "dump_mc%d" % mc)
            dirs[mc] = d
        summary["dump_compare"], summary["dump_worst"] = {}, {}
        for mc in levels[1:]:
            cmp = compare_dumps(dirs[levels[0]], dirs[mc])
            summary["dump_compare"][str(mc)] = cmp
            summary["dump_worst"][str(mc)] = worst_per_config(cmp)
    with open(os.path.join(args.out, "summary.json"), "w") as f:
        json.dump(summary, f, indent=1)
    print(json.dumps({"card": summary["card_before"], "stats": stats, "dump_worst": summary.get("dump_worst")}, indent=1))


if __name__ == "__main__":
    main()
