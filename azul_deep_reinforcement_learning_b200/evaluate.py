"""Measure a saved network against an opponent over many games -- the ``scripts/run_batch.py`` / ``NNRunner.run_batch``
equivalent (reference scripts/run_batch.py, nn_runner.py:49-51).

    python -m azul_deep_reinforcement_learning_b200.evaluate NET [--opponent FILE|random] [--games N]
                                                             [--mode sample|argmax] [--seed S]

``NET`` plays seat 1 and ``--opponent`` seat 2 (a frozen network, or ``random``: ``RandomAgent``).  The ``--games``
episodes are played in parallel, one per game slot, whole in ONE launch of the persistent policy kernel; with a network
opponent both seats select their moves the same way (``--mode``).  Printed and returned: the ``GameStatistics`` means
per game (what ``SelfPlayTrainer`` logs), the games not finished within the decision bound and the agent decisions played.
"""
import argparse
import json

import torch

from .engine import PackedPolicy
from .selfplay import BatchedGameRunner, PersistentEpisodes, load_network
from .train import STAT_FIELDS, summarize_stats

MODES = {"sample": 0, "argmax": 1}
REPORT_KEYS = ("games", "player_score", "opponent_score", "win_percent", "rounds", "percent_first_player", "floor_penalty",
               "max_combo", "completed_rows", "completed_columns", "completed_colors", "reward", "unfinished", "decisions")


def evaluate(net, opponent="random", games=2048, mode=0, seed=0, device=0, rules=None, max_decisions=160):
    """Play ``games`` episodes of ``net`` (seat 1) against ``opponent`` ("random", or anything ``selfplay.load_network``
    takes); ``mode`` 0 samples, 1 takes the argmax.  Returns a dict of per-game means (``REPORT_KEYS``) plus
    ``max_opponent_passes`` (network opponent: the most opponent moves one agent decision had to wait for)."""
    dev = torch.device("cuda", device)
    runner = BatchedGameRunner(games, rules=rules, seed=seed, device=device)
    packed = PackedPolicy(runner.engine, load_network(net, dev))
    if not (isinstance(opponent, str) and opponent == "random"):
        runner.opponent, runner.opponent_mode = PackedPolicy(runner.engine, load_network(opponent, dev)), int(mode)
    # the statistics come from the final states (azb_stats): the decision records are not needed beyond their count
    episodes = PersistentEpisodes(runner, packed, max_decisions=max_decisions, capacity=128)
    with torch.no_grad():
        records = episodes.run(mode=int(mode))
        e = runner.engine
        per_game = e.stats().long()                                           # [G, 10], azb_stats order
        ended = e.export_records()[:, _end_of_game_column()] != 0
        sums = [float(records.meta[0]), 0.0, 0.0, 0.0, float(records.reward_sum), float(games)]
        sums += [float(x) for x in per_game.sum(0).tolist()]
        sums += [float((per_game[:, 0] > per_game[:, 1]).sum()), float((~ended).sum())]
    assert len(sums) == STAT_FIELDS
    st = summarize_stats(sums)
    out = {k: st[k] for k in REPORT_KEYS if k in st}
    out["decisions"] = int(records.meta[0])
    out["max_opponent_passes"] = int(episodes.opp_passes[0]) if runner.opponent is not None else 0
    return out


def _end_of_game_column():
    from .layout import UnpackedLayout
    return UnpackedLayout(2).end_of_game


def parse_args(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("net", help="the network in seat 1: any file Agent(base_net_file=...) accepts")
    ap.add_argument("--opponent", default="random", metavar="FILE|random",
                    help="seat 2: a saved network, or 'random' (RandomAgent; default)")
    ap.add_argument("--games", type=int, default=2048, help="episodes, played in parallel (default 2048)")
    ap.add_argument("--mode", default="sample", choices=sorted(MODES), help="move selection of both networks")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--max-decisions", type=int, default=160, help="agent decisions after which a game counts as unfinished")
    args = ap.parse_args(argv)
    if args.games < 1:
        ap.error("--games must be >= 1")
    return args


def main(argv=None):
    args = parse_args(argv)
    out = evaluate(args.net, args.opponent, games=args.games, mode=MODES[args.mode], seed=args.seed,
                   max_decisions=args.max_decisions)
    print(json.dumps(out))
    return out


if __name__ == "__main__":
    main()
