"""The packed bit-plane rules (csrc/azb_rules.cuh, the header the CUDA kernels are built from)
compiled for the host and checked against the golden vectors and the oracle.  CPU-only; this
is the pre-GPU gate for the rules arithmetic -- the -m gpu tests repeat it through the C-ABI."""
import numpy as np
import pytest

from azul_deep_reinforcement_learning_b200.layout import UnpackedLayout
from oracle import oracle as O
from tests import harness as H
from tests.helpers import TRACE_CONFIGS, TraceGame, load_kat, load_trace, stream_digest


@pytest.mark.parametrize("players,rules", TRACE_CONFIGS)
def test_packed_rules_replay_golden(players, rules):
    tr = load_trace(players, rules)
    pool = int(tr["tile_pool"])
    L = UnpackedLayout(players)
    for i in range(len(tr["first_player"])):
        tg = TraceGame(tr, i)
        rec = np.zeros(L.size, np.int32)
        rec[L.n_players] = players
        rec[L.next_first_player] = tg.first_player
        if pool:
            rec[L.box:L.box + 5] = 20
        rc, _, _ = H.op(rec, players, pool, H.OP_NEW_ROUND, draws=tg.draws[0])
        assert rc == 0 and np.array_equal(rec, tg.initial)
        rnd, masks, states = 1, [], []
        for t, a in enumerate(tg.actions):
            _, m, _ = H.op(rec, players, pool, H.OP_ROUNDTRIP, want_mask=True)
            turn = rec[L.turn_counter]
            draws = tg.draws[rnd] if rnd < len(tg.draws) else np.full(20, -1, np.int8)
            rc, _, _ = H.op(rec, players, pool, H.OP_STEP, a=int(a), draws=draws)
            assert rc == 0
            rnd += int(rec[L.turn_counter] != turn)
            masks.append(m); states.append(rec.copy())
            if tg.full:
                assert np.array_equal(m, tg.masks[t]), (i, t)
                assert np.array_equal(rec, tg.states[t + 1]), (i, t, np.nonzero(rec != tg.states[t + 1]))
        assert np.array_equal(rec, tg.final)
        assert stream_digest(masks, states) == tg.sha
        assert H.op(rec, players, pool, H.OP_STEP, a=0, draws=np.full(20, -1, np.int8))[0] == -2


def test_packed_rules_known_answers():
    kat = load_kat()
    L = UnpackedLayout(2)
    for s in range(len(kat["kat_names"])):
        pool = int(kat["kat_pool"][s])
        rec = kat["fixture_records"][int(kat["kat_fixture"][s])].astype(np.int32).copy()
        if pool == 1:
            rec[L.box:L.box + 5] = 20
        for k in range(int(kat["kat_op_offsets"][s]), int(kat["kat_op_offsets"][s + 1])):
            code, a, b, c = [int(x) for x in kat["kat_ops"][k]]
            expect_ret = int(kat["kat_returns"][k])
            if code == 0:
                rc = H.op(rec, 2, pool, H.OP_MOVE, a=a + 6 * b + 30 * c)[0]
            elif code == 1:
                d = kat["kat_draws"][k]
                rc = H.op(rec, 2, pool, H.OP_STEP, a=a + 6 * b + 30 * c, draws=d if d[0] >= 0 else np.full(20, -1, np.int8))[0]
            elif code == 2:
                rc = H.op(rec, 2, pool, H.OP_NEXT)[0]
            elif code == 3:
                rc = H.op(rec, 2, pool, H.OP_SCORE)[0]
            elif code == 4:
                _, m, _ = H.op(rec, 2, pool, H.OP_ROUNDTRIP, want_mask=True)
                rc = int(m[c] >> (a + 6 * b) & 1)
            assert rc == expect_ret, (kat["kat_names"][s], k)
            assert np.array_equal(rec, kat["kat_records"][k].astype(np.int32)), (kat["kat_names"][s], k)


def test_packed_fixture_masks_and_roundtrip():
    kat = load_kat()
    for name, rec, mask in zip(kat["fixture_names"], kat["fixture_records"], kat["fixture_masks"]):
        r = rec.astype(np.int32).copy()
        rc, m, _ = H.op(r, 2, 0, H.OP_ROUNDTRIP, want_mask=True)
        assert rc == 0 and np.array_equal(r, rec.astype(np.int32)), name
        assert np.array_equal(m, mask), name


@pytest.mark.parametrize("players", [2, 3, 4])
@pytest.mark.parametrize("pool", [0, 1])
@pytest.mark.parametrize("first_rule", [0, 1])
def test_packed_rollout_matches_oracle(players, pool, first_rule):
    """Seeded Philox rollouts with auto-reset: identical records and counters."""
    seed, gid0, n, k = 0x5EED + players, 1000, 48, 150
    a = O.fresh_records(n, players, pool, first_rule, seed, gid0)
    b = a.copy()
    for i in range(n):   # packed reset must agree with the oracle reset too
        r = np.zeros_like(b[i]); r[UnpackedLayout(players).n_players] = players
        assert H.op(r, players, pool, H.OP_RESET, seed=seed, gid=gid0 + i, first_rule=first_rule)[0] == 0
        assert np.array_equal(r, a[i])
    ca = O.rollout_random(a, players, pool, first_rule, seed, gid0, k)
    cb = H.rollout(b, players, pool, first_rule, seed, gid0, k)
    assert np.array_equal(a, b), np.nonzero((a != b).any(axis=1))
    assert np.array_equal(ca, cb), (ca, cb)
    assert ca[0] == n * k and ca[1] > 0
    # continuing in two halves gives the same result as one call (RNG position lives in the state)
    c = O.fresh_records(n, players, pool, first_rule, seed, gid0)
    H.rollout(c, players, pool, first_rule, seed, gid0, 77)
    H.rollout(c, players, pool, first_rule, seed, gid0, k - 77)
    assert np.array_equal(c, b)


def test_packed_random_action_matches_oracle():
    rng = np.random.default_rng(1)
    for _ in range(3000):
        m = rng.integers(0, 2 ** 30, size=6, dtype=np.uint64).astype(np.uint32)
        m &= rng.integers(0, 2 ** 30, size=6, dtype=np.uint64).astype(np.uint32)
        if rng.random() < 0.3:
            m[rng.integers(0, 6)] = 0
        w = int(rng.integers(0, 2 ** 32, dtype=np.uint64))
        a, b = O.random_action(m, w), H.random_action(m, w)
        assert (a == b) or (a == -1 and b == 180)


def test_packed_score_preview_and_predicates():
    kat = load_kat()
    names = list(kat["fixture_names"])
    for name in ("game_end_of_round_1", "game_end_of_round_2", "game_sample_1"):
        rec = kat["fixture_records"][names.index(name)].astype(np.int32).copy()
        g = O.Game(2, 0, record=rec.copy())
        before = rec.copy()
        _, _, prev = H.op(rec, 2, 0, H.OP_PREVIEW, want_preview=True)
        assert np.array_equal(prev, g.score_preview()) and np.array_equal(rec, before)
        assert H.op(rec, 2, 0, H.OP_EOR)[0] == int(g.is_end_of_round())
        assert H.op(rec, 2, 0, H.OP_EOG)[0] == int(g.is_end_of_game())


def test_box_beyond_127_tiles_is_flagged():
    """The Lid refill keeps the cumulative box counts in 7-bit fields (a game has 100 tiles): a box that no game can
    produce is flagged with the bad-import status bit instead of drawing from corrupted thresholds."""
    from azul_deep_reinforcement_learning_b200.layout import STATUS_BAD_IMPORT
    players, pool, seed, gid0 = 2, 1, 77, 5
    L = UnpackedLayout(players)
    recs = O.fresh_records(4, players, pool, 0, seed, gid0)
    ok = recs.copy()
    recs[:, L.box:L.box + 5] = 40                  # 200 tiles in the bag
    H.rollout(recs, players, pool, 0, seed, gid0, 40)
    H.rollout(ok, players, pool, 0, seed, gid0, 40)
    assert (recs[:, L.status] & STATUS_BAD_IMPORT).all()
    assert not (ok[:, L.status] & STATUS_BAD_IMPORT).any()


def test_import_rejects_unrepresentable():
    L = UnpackedLayout(2)
    rec = np.zeros(L.size, np.int32); rec[L.n_players] = 2
    rec[L.pattern_lines + 5 * 2 + 0] = 1
    rec[L.pattern_lines + 5 * 2 + 3] = 1          # two colours in one pattern row
    assert H.op(rec, 2, 0, H.OP_ROUNDTRIP)[0] == -16


@pytest.mark.parametrize("pool", [0, 1])
def test_packed_opponent_loop_matches_oracle(pool):
    """GameRunner.step's opponent loop + reward preview (game_runner.py:46-52): packed rules vs oracle."""
    seed, n = 99 + pool, 64
    recs = O.fresh_records(n, 2, pool, 0, seed, 0)
    rng = np.random.default_rng(3)
    for it in range(70):
        for i in range(n):
            a, b = recs[i].copy(), recs[i].copy()
            da, ma = O.opponent_random(a, 2, pool, seed, i, require_two=(it > 0))
            db, mb = H.opponent(b, 2, pool, seed, i, require_two=(it > 0))
            assert da == db and np.array_equal(ma, mb) and np.array_equal(a, b)
            L = UnpackedLayout(2)
            if not a[L.end_of_game] and ma.any():
                assert a[L.current_player] == 1
                g = O.Game(2, pool, record=a)
                act = O.random_action(ma, int(rng.integers(0, 2 ** 32)))
                assert g.step(act, None, seed, i) == 0          # the agent's own move, then the opponent again
                recs[i] = g.rec
            else:
                recs[i] = O.fresh_records(1, 2, pool, 0, seed + it + 1, i)[0]


def test_packed_rules_random_boards():
    from tests.helpers import FUZZ_CONFIGS, fuzz_key, load_fuzz
    fz = load_fuzz()
    for players, pool in FUZZ_CONFIGS:
        k = fuzz_key(players, pool)
        for i in range(len(fz[k + "_action"])):
            rec = fz[k + "_before"][i].astype(np.int32).copy()
            rc, m, _ = H.op(rec, players, pool, H.OP_ROUNDTRIP, want_mask=True)
            assert rc == 0 and np.array_equal(m, fz[k + "_mask"][i]), (k, i)
            # the single-action legality test of the step kernel agrees with the mask for all 256 action bytes
            assert H.op(rec.copy(), players, pool, H.OP_LEGAL_SINGLE)[0] == 0, (k, i)
            sc = rec.copy()
            assert H.op(sc, players, pool, H.OP_SCORE)[0] == 0
            assert np.array_equal(sc, fz[k + "_scored"][i].astype(np.int32)), (k, i)
            a = int(fz[k + "_action"][i])
            if a != 255:
                assert H.op(rec, players, pool, H.OP_STEP, a=a, draws=fz[k + "_draws"][i])[0] == 0
                assert np.array_equal(rec, fz[k + "_stepped"][i].astype(np.int32)), (k, i)
