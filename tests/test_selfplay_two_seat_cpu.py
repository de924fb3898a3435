"""Two-seat self-play without a GPU: the command line and the trainer's argument checks, and the per-seat discounted
returns of the host restatement against the recurrence azb_discounted_returns runs (one running return per seat, picked by
flags bit 2)."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")


def test_cli_self_play_and_eval_every():
    from azul_deep_reinforcement_learning_b200.train import parse_args
    a = parse_args(["256", "run1", "--self-play", "--eval-every", "5", "--eval-games", "512"])
    assert a.self_play and a.eval_every == 5 and a.eval_games == 512 and a.opponent is None
    b = parse_args([])
    assert not b.self_play and b.eval_every == 0
    for bad in (["--self-play", "--opponent", "old.pt"], ["--self-play", "--opponent", "greedy"],
                ["--self-play", "--opponent-refresh", "3"], ["--eval-every", "-1"], ["--self-play", "--eval-every", "-2"],
                ["--eval-games", "0"]):
        with pytest.raises(SystemExit):
            parse_args(bad)


def test_trainer_rejects_self_play_with_an_opponent():
    from azul_deep_reinforcement_learning_b200.train import SelfPlayTrainer
    for kw in ({"opponent": "greedy"}, {"opponent": "old.pt"}, {"opponent_refresh": 2}):
        with pytest.raises(ValueError):
            SelfPlayTrainer(64, self_play=True, **kw)


def _bit2_recurrence(reward, flags, gamma):
    """The kernel's walk: backwards over the iterations, one running return per seat chosen by bit 2."""
    T, G = reward.shape
    q = np.zeros((T, G))
    run = np.zeros((2, G))
    for t in reversed(range(T)):
        on = (flags[t] & 1) == 1
        s = (flags[t] >> 2) & 1
        for seat in (0, 1):
            sel = on & (s == seat)
            run[seat] = np.where(sel, reward[t] + gamma * run[seat], run[seat])
        q[t] = np.where(on, np.where(s == 1, run[1], run[0]), 0.0)
    return q


def _per_game_lists(reward, flags, gamma):
    """nn_runner.py:72-75 on each seat's own list of decisions, game by game."""
    T, G = reward.shape
    q = np.zeros((T, G))
    for g in range(G):
        for seat in (0, 1):
            ts = [t for t in range(T) if flags[t, g] & 1 and (flags[t, g] >> 2) & 1 == seat]
            run = 0.0
            for t in reversed(ts):
                run = reward[t, g] + gamma * run
                q[t, g] = run
    return q


@pytest.mark.parametrize("T,G,p_on,p_seat2", [(1, 7, 1.0, 0.5), (37, 64, 0.6, 0.5), (120, 40, 0.9, 0.0), (64, 33, 0.5, 1.0)])
def test_two_seat_returns_restatement_agrees_with_bit2_recurrence(T, G, p_on, p_seat2):
    from azul_deep_reinforcement_learning_b200.selfplay import discounted_returns_two_seat
    rng = np.random.default_rng(T * 1000 + G)
    gamma = 0.99
    on = rng.random((T, G)) < p_on
    seat2 = rng.random((T, G)) < p_seat2
    over = rng.random((T, G)) < 0.1
    flags = (on.astype(np.uint8) | (over & on).astype(np.uint8) << 1 | (seat2 & on).astype(np.uint8) << 2)
    flags[rng.random((T, G)) < 0.05] |= 4                        # bit 2 without bit 0: not a decision
    flags[(flags & 1) == 0] &= 4
    reward = rng.integers(-40, 41, (T, G)).astype(np.float64)
    want = _per_game_lists(reward, flags, gamma)
    rec = _bit2_recurrence(reward, flags, gamma)
    assert np.allclose(rec, want, rtol=1e-12, atol=1e-12)
    got = discounted_returns_two_seat(torch.from_numpy(reward), torch.from_numpy(flags), gamma).numpy()
    assert np.allclose(got, want, rtol=1e-12, atol=1e-12)
    # seat 1 only (bit 2 never set): the one recurrence of the runner modes
    only1 = flags & 3
    assert np.allclose(_bit2_recurrence(reward, only1, gamma),
                       discounted_returns_two_seat(torch.from_numpy(reward), torch.from_numpy(only1), gamma).numpy())
