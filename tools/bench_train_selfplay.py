"""One training batch (rollout + tensor-core update + Adam, one CUDA graph replay) against the random agent and in two-seat
self-play, timed with CUDA events.

    python tools/bench_train_selfplay.py [--games 16384] [--reps 10] [--out FILE]

Per arm: SelfPlayTrainer(games) (random opponent) and SelfPlayTrainer(games, self_play=True).  Two eager batches and the
capture come first, then ``--reps`` graph replays, each timed alone (events around the replay, then a synchronise).
Reported: ms per batch (mean, min, max), episodes/s, decisions trained per batch (self-play: both seats') and decisions/s.
The card's name and power limit are read in the same run; the network is randomly initialised (seed 0) and keeps training
through the timed batches."""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

from azul_deep_reinforcement_learning_b200.train import SelfPlayTrainer  # noqa: E402
from bench_opponent import card  # noqa: E402


def bench(games, reps, self_play):
    tr = SelfPlayTrainer(games, seed=0, self_play=self_play)
    for _ in range(2):
        tr.step()
    tr.enable_step_graph(warmup=0)
    tr.step()                                                # the first replay
    torch.cuda.synchronize()
    ms, decisions = [], []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        tr.step(defer_stats=True)
        b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b))
        decisions.append(tr.fetch_stats()["transitions"])
    t = sum(ms) / len(ms)
    d = sum(decisions) / len(decisions)
    return {"ms": t, "ms_min": min(ms), "ms_max": max(ms), "episodes_per_s": games / (t * 1e-3), "decisions": d,
            "decisions_per_s": d / (t * 1e-3)}


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--games", type=int, default=16384)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args(argv)
    if not torch.cuda.is_available():
        raise SystemExit("bench_train_selfplay: no CUDA device")
    out = {"card": card(), "games": args.games, "vs_random": bench(args.games, args.reps, False),
           "self_play": bench(args.games, args.reps, True)}
    out["self_play_over_vs_random"] = out["self_play"]["ms"] / out["vs_random"]["ms"]
    s = json.dumps(out, indent=1)
    print(s)
    if args.out:
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
