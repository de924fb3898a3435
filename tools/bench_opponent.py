"""Whole-episode rollouts against the random opponent, a frozen policy opponent and the greedy agent, and two-seat self-play,
timed with CUDA events.

    python tools/bench_opponent.py [--games 16384 131072] [--reps 5] [--out FILE]

Per batch size: (a) the persistent runner-mode rollout vs the random opponent, (b) the persistent rollout vs a policy
opponent (azb_policy_rollout_vs_policy), (c) the eager run_episodes vs the same policy opponent (one policy launch per
agent decision, one or more opponent launches each followed by a host read, one reward launch), (d) the persistent rollout
vs the greedy agent (azb_policy_rollout_vs_greedy), (e) the eager run_episodes vs the greedy agent (one policy launch and
one azb_opponent_greedy launch per agent decision, a host read every 8 decisions), (f) the persistent two-seat self-play
(azb_policy_rollout_selfplay: the agent's network plays both seats, and both seats' decisions are recorded).  A timed batch
is a whole PersistentEpisodes.run / SelfPlayEpisodes.run (episode start, the rollout, discounted returns) or a whole
run_episodes, after one warm-up batch.
Reported: ms per batch, episodes/s, recorded decisions/s (row f: both seats'), and the opponent passes per agent decision -- the most any CTA
needed in one decision (the kernel's counter) and, from a separate counting run of the eager path, the mean and maximum
over decisions of the launches in which some game of the batch moved.  The card's name and power limit are read in the
same run.  Both networks are randomly initialised (seed 0 / 1); the agent samples (mode 0)."""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

from azul_deep_reinforcement_learning_b200.azulnet.model import ActorCritic  # noqa: E402
from azul_deep_reinforcement_learning_b200.engine import PackedPolicy, policy_step  # noqa: E402
from azul_deep_reinforcement_learning_b200.selfplay import (BatchedGameRunner, PersistentEpisodes,  # noqa: E402
                                                            SelfPlayEpisodes, run_episodes)


def card():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        info["power_limit_and_max_sm_clock"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"
    except (OSError, subprocess.SubprocessError, IndexError):
        info["power_limit_and_max_sm_clock"] = "unknown"
    return info


def timed(fn, reps):
    fn()                                                     # warm-up: module loads, allocations
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = fn()
        b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b))
    return ms, out


def count_eager_passes(runner, packed):
    """Launches per agent decision in which some game of the batch took an opponent move (eager path, counting run)."""
    per_decision = []
    orig = runner._opponent_policy_moves

    def counting(max_rounds=64, check_every=1):
        k = 0
        for _ in range(max_rounds):
            out = policy_step(runner.engine, runner.opponent, mode=runner.opponent_mode, apply_step=True, want_mask=False,
                              act_filter=1)
            if not bool((out["action"] != 255).any()):
                break
            k += 1
        per_decision.append(k)

    runner._opponent_policy_moves = counting
    run_episodes(runner, packed, max_decisions=160, record_obs=False)
    runner._opponent_policy_moves = orig
    return per_decision[1:]                                  # [0] belongs to the episode start


def bench(n, reps):
    torch.manual_seed(0)
    net = ActorCritic(136, 180).cuda()
    torch.manual_seed(1)
    opp = ActorCritic(136, 180).cuda()
    res = {"games": n}

    ra = BatchedGameRunner(n, seed=11)
    ea = PersistentEpisodes(ra, PackedPolicy(ra.engine, net))
    ms, r = timed(lambda: ea.run(), reps)
    res["a_persistent_vs_random"] = _rates(n, ms, int(r.meta[0]))

    rb = BatchedGameRunner(n, seed=11)
    rb.opponent = PackedPolicy(rb.engine, opp)
    eb = PersistentEpisodes(rb, PackedPolicy(rb.engine, net))
    ms, r = timed(lambda: eb.run(), reps)
    res["b_persistent_vs_policy"] = _rates(n, ms, int(r.meta[0]))
    res["b_persistent_vs_policy"]["max_opponent_passes_per_decision_per_cta"] = int(eb.opp_passes[0])

    rc = BatchedGameRunner(n, seed=11, opponent=PackedPolicy(rb.engine, opp))
    pc = PackedPolicy(rc.engine, net)
    ms, batch = timed(lambda: run_episodes(rc, pc, max_decisions=160, record_obs=False), max(2, reps // 2))
    res["c_eager_vs_policy"] = _rates(n, ms, int(batch["active"].sum()))
    passes = count_eager_passes(rc, pc)
    res["c_eager_vs_policy"]["opponent_passes_per_decision_batch_mean"] = sum(passes) / max(len(passes), 1)
    res["c_eager_vs_policy"]["opponent_passes_per_decision_batch_max"] = max(passes) if passes else 0

    rd = BatchedGameRunner(n, seed=11, opponent="greedy")
    ed = PersistentEpisodes(rd, PackedPolicy(rd.engine, net))
    ms, r = timed(lambda: ed.run(), reps)
    res["d_persistent_vs_greedy"] = _rates(n, ms, int(r.meta[0]))

    re_ = BatchedGameRunner(n, seed=11, opponent="greedy")
    pe = PackedPolicy(re_.engine, net)
    ms, batch = timed(lambda: run_episodes(re_, pe, max_decisions=160, record_obs=False), max(2, reps // 2))
    res["e_eager_vs_greedy"] = _rates(n, ms, int(batch["active"].sum()))

    rf = BatchedGameRunner(n, seed=11)
    ef = SelfPlayEpisodes(rf.engine, PackedPolicy(rf.engine, net))
    ms, r = timed(lambda: ef.run(), reps)
    res["f_persistent_selfplay"] = _rates(n, ms, int(r.meta[0]))
    res["f_persistent_selfplay"]["unfinished"] = n - int(ef.out["done"].sum())
    res["b_over_a"] = res["b_persistent_vs_policy"]["ms"] / res["a_persistent_vs_random"]["ms"]
    res["d_over_a"] = res["d_persistent_vs_greedy"]["ms"] / res["a_persistent_vs_random"]["ms"]
    res["e_over_d"] = res["e_eager_vs_greedy"]["ms"] / res["d_persistent_vs_greedy"]["ms"]
    res["c_over_b"] = res["c_eager_vs_policy"]["ms"] / res["b_persistent_vs_policy"]["ms"]
    res["f_over_a"] = res["f_persistent_selfplay"]["ms"] / res["a_persistent_vs_random"]["ms"]
    res["f_over_b"] = res["f_persistent_selfplay"]["ms"] / res["b_persistent_vs_policy"]["ms"]
    return res


def _rates(n, ms, decisions):
    t = sum(ms) / len(ms)
    return {"ms": t, "ms_min": min(ms), "ms_max": max(ms), "episodes_per_s": n / (t * 1e-3),
            "decisions": decisions, "decisions_per_s": decisions / (t * 1e-3)}


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--games", type=int, nargs="+", default=[16384, 131072])
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args(argv)
    if not torch.cuda.is_available():
        raise SystemExit("bench_opponent: no CUDA device")
    out = {"card": card(), "results": [bench(n, args.reps) for n in args.games]}
    s = json.dumps(out, indent=1)
    print(s)
    if args.out:
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
