"""A/B timing of the fused random rollout between two built trees of this repository.

    python tools/ab_rollout.py --base DIR --new DIR [--rounds 5] [--steps 100] [--out FILE]

`bench.py` measures the tree it lives in, so each build is run as `python DIR/bench.py ...`.  The two trees take turns, config
by config and round by round, so that a drift of the card or of other work on the host falls on both alike.  Configurations:
the headline (65,536 two-player games, `k_rollout_rotate`), `--players 3` and `--players 4` (rotating as well) and
`--games 262144` (`k_rollout_random`).  Prints every run's `value` (env steps/s) and `kernel_ms_min`, then per build the median
and the min-max spread, with the card's name, power limit and maximum SM clock read in the same call."""
import argparse
import json
import os
import statistics
import subprocess
import sys

CONFIGS = [("headline", []), ("players3", ["--players", "3"]), ("players4", ["--players", "4"]), ("games262144", ["--games", "262144"])]


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()
    return out[0] if out else "unknown"


def run(tree, extra, steps):
    cmd = [sys.executable, os.path.join(tree, "bench.py"), "--no-extras", "--no-cpu-baseline", "--pyref-seconds", "0",
           "--steps", str(steps)] + extra
    p = subprocess.run(cmd, capture_output=True, text=True)
    if p.returncode != 0:
        raise RuntimeError("%s failed (%d):\n%s" % (" ".join(cmd), p.returncode, p.stderr[-2000:]))
    line = json.loads(p.stdout.strip().splitlines()[-1])
    roof = line.get("roofline") or {}
    return line["value"], roof.get("kernel_ms_min", line.get("kernel_ms_min")), roof.get("kernel")


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--base", required=True, help="tree of the reference build (already built)")
    ap.add_argument("--new", required=True, help="tree of the build under test (already built)")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--out", default=None, help="also write the runs and the summary as JSON here")
    args = ap.parse_args()
    trees = {"base": os.path.abspath(args.base), "new": os.path.abspath(args.new)}
    gpu = card()
    print("card (name, power limit, max SM clock):", gpu, flush=True)
    runs = {c: {b: [] for b in trees} for c, _ in CONFIGS}
    for r in range(args.rounds):
        for c, extra in CONFIGS:
            order = list(trees) if r % 2 == 0 else list(trees)[::-1]
            for b in order:
                value, kms, kernel = run(trees[b], extra, args.steps)
                runs[c][b].append({"value": value, "kernel_ms_min": kms, "kernel": kernel})
                print("round %d %-12s %-4s value %.4e  kernel_ms_min %.4f  %s" % (r, c, b, value, kms, kernel), flush=True)
    summary = {}
    print("\n%-12s %-4s %12s %12s %12s %9s" % ("config", "build", "median", "min", "max", "vs base"))
    for c, _ in CONFIGS:
        summary[c] = {}
        for b in trees:
            v = [x["value"] for x in runs[c][b]]
            summary[c][b] = {"median": statistics.median(v), "min": min(v), "max": max(v),
                             "spread": max(v) - min(v), "kernel_ms_min": min(x["kernel_ms_min"] for x in runs[c][b])}
        for b in trees:
            s = summary[c][b]
            print("%-12s %-4s %12.4e %12.4e %12.4e %+8.2f%%" % (c, b, s["median"], s["min"], s["max"],
                                                                100.0 * (s["median"] / summary[c]["base"]["median"] - 1.0)))
    if args.out:
        with open(args.out, "w") as f:
            json.dump({"card": gpu, "rounds": args.rounds, "steps": args.steps, "runs": runs, "summary": summary}, f, indent=1)


if __name__ == "__main__":
    main()
