"""The greedy agent without a GPU: the naive restatement (tests/harness/greedy_oracle.c) against a brute force built from
the oracle's primitives, the header's greedy_action / opponent_greedy (csrc/azb_rules.cuh through the g++ harness) against
the restatement, and the command lines that select the greedy opponent."""
import numpy as np
import pytest

from azul_deep_reinforcement_learning_b200.layout import UnpackedLayout
from oracle import oracle as O
from tests.harness import greedy as GH
from tests.helpers import FUZZ_CONFIGS, TRACE_CONFIGS, fuzz_key, load_fuzz, load_kat, load_trace

WORDS = [0, 0xFFFFFFFF, 0x80000000, 0x12345678, 0x9E3779B9, 0xDEADBEEF]
OFFSET = 1000                   # raises the mover's score so that count_score's clamp at zero never applies


def _states(players, pool):
    """Reachable states of the golden traces, kat.npz and fuzz.npz, plus random-agent playouts (finished games among them)
    of this configuration: int32 records [N, U]."""
    U = O.lib().ao_record_size(players)
    out = []
    for p, rules in TRACE_CONFIGS:
        tr = load_trace(p, rules)
        if p == players:
            out += [tr["full_states"], tr["initial_states"], tr["final_states"]]
    if players == 2:
        kat = load_kat()
        out += [kat["fixture_records"], kat["kat_records"]]
    fz = load_fuzz()
    for p, fpool in FUZZ_CONFIGS:
        if p == players:
            k = fuzz_key(p, fpool)
            out += [fz[k + "_before"], fz[k + "_scored"], fz[k + "_stepped"]]
    rng = np.random.default_rng(100 * players + pool)
    for k in (0, 3, 11, 29, 57, 140):
        recs = O.fresh_records(64, players, pool, 0, seed=7 + k, gid0=1000 * k)
        O.rollout_random(recs, players, pool, 0, 7 + k, 1000 * k, int(k + rng.integers(0, 5)))
        out.append(recs)
    states = np.concatenate([np.asarray(s, np.int32).reshape(-1, U) for s in out])
    return np.ascontiguousarray(states)


def _brute_force(rec, players, pool, word):
    """ao_move on a copy and ao_score_preview with the mover's score raised by OFFSET, for every legal action."""
    L = UnpackedLayout(players)
    g = O.Game(players, pool, record=rec)
    cur = int(rec[L.scalars])
    s = cur - 1 if cur > 0 else players - 1
    best, T = None, []
    for a in range(180):
        d, c, p = a % 6, (a // 6) % 5, a // 30
        if not g.is_legal_move(d, c, p):
            continue
        h = g.copy()
        h.move(d, c, p)
        h.rec[L.score + s] += OFFSET
        v = int(h.score_preview()[s]) - OFFSET
        if best is None or v > best:
            best, T = v, []
        if v == best:
            T.append(a)
    if not T:
        return -1, 0
    return T[(int(word) * len(T)) >> 32], len(T)


@pytest.mark.parametrize("players,pool", FUZZ_CONFIGS)
def test_oracle_greedy_equals_brute_force(players, pool):
    states = _states(players, pool)
    words = WORDS + [int(w) for w in np.random.default_rng(players + 10 * pool).integers(0, 2 ** 32, 4)]
    tied = 0
    for i, rec in enumerate(states[::3]):
        for w in words:
            want, n_best = _brute_force(rec, players, pool, w)
            assert GH.ao_greedy_action(rec, players, pool, w) == want, (i, w)
        assert GH.ao_greedy_ties(rec, players, pool) == n_best
        tied += n_best >= 2
    assert tied >= 20, tied                                            # tie-breaks were exercised


def _packable(rec, players):
    return GH.host_lib().hh_greedy_action(np.ascontiguousarray(rec, np.int32).ctypes.data, players, 0, 0) >= 0


@pytest.mark.parametrize("players,pool", FUZZ_CONFIGS)
def test_header_greedy_action_equals_oracle(players, pool):
    states = _states(players, pool)
    words = WORDS + [int(w) for w in np.random.default_rng(7 * players + pool).integers(0, 2 ** 32, 6)]
    checked = tied = 0
    for i, rec in enumerate(states):
        if not _packable(rec, players):
            continue
        ties = GH.ao_greedy_ties(rec, players, pool)
        tied += ties >= 2
        for w in words:
            want = GH.ao_greedy_action(rec, players, pool, w)
            assert GH.hh_greedy_action(rec, players, pool, w) == (180 if want < 0 else want), (i, w)
        checked += 1
    assert checked >= 0.9 * len(states) and tied >= 20, (checked, len(states), tied)


@pytest.mark.parametrize("require_two", [1, 0])
@pytest.mark.parametrize("players,pool", FUZZ_CONFIGS)
def test_header_opponent_greedy_equals_oracle(players, pool, require_two):
    """Seeded playouts: the agent (seat 1) plays the random agent's move, then the greedy opponent loop; state, reward
    difference, mask and status after every hand-back."""
    L = UnpackedLayout(players)
    seed = 3 + players + 10 * pool
    recs = O.fresh_records(48, players, pool, 0, seed)
    for gid in range(recs.shape[0]):
        a, b = recs[gid].copy(), recs[gid].copy()
        for t in range(120):
            da, ma = GH.ao_opponent_greedy(a, players, pool, seed, gid, require_two)
            db, mb = GH.hh_opponent_greedy(b, players, pool, seed, gid, require_two)
            assert (da, ma.tolist()) == (db, mb.tolist()) and np.array_equal(a, b), (gid, t)
            if a[L.scalars + 3] or int(ma.astype(np.int64).sum()) == 0:
                break
            w = O.philox4x32_10([gid, t, 7, 0], [seed, 0])[0]          # the agent's move: any legal action
            act = O.random_action(ma, w)
            for r in (a, b):
                g = O.Game(players, pool, record=r)
                assert g.step(act, seed=seed, gid=gid) == 0
                r[:] = g.rec


def test_training_and_evaluate_cli_accept_greedy():
    from azul_deep_reinforcement_learning_b200.evaluate import parse_args as eval_args
    from azul_deep_reinforcement_learning_b200.train import parse_args as train_args
    a = train_args(["256", "run1", "--opponent", "greedy"])
    assert (a.opponent, a.opponent_refresh) == ("greedy", 0)
    assert eval_args(["net.pt", "--opponent", "greedy"]).opponent == "greedy"
    with pytest.raises(SystemExit):
        train_args(["256", "--opponent", "greedy", "--opponent-refresh", "5"])


def test_greedy_opponent_never_loads_a_network(monkeypatch):
    """The keyword selects the agent: nothing tries to read a file called 'greedy' (a checkpoint of that name is
    passed as ./greedy)."""
    from azul_deep_reinforcement_learning_b200 import selfplay

    def refuse(*a, **k):
        raise AssertionError("load_network called")

    monkeypatch.setattr(selfplay, "load_network", refuse)
    assert selfplay.resolve_opponent(None, "greedy") == "greedy"
    assert selfplay.resolve_opponent(None, None) is None
    with pytest.raises(AssertionError):
        selfplay.resolve_opponent(None, "./greedy")
    with pytest.raises(ValueError):
        selfplay.BatchedGameRunner(16, opponent="greedy!")
