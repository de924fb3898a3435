"""The C oracle against the reference's ``GameRunner`` goldens (tests/golden/runner_*.npz, recorded from the live
reference by oracle/record_golden_runner.py): every env step of every episode (agent's and opponent's), the ``while``
test of ``GameRunner.step`` / ``reset`` (game_runner.py:46,84) at every state, and reward / done / player_score /
observation / legal mask / record at every hand-back to the agent.  CPU only."""
import numpy as np
import pytest

from azul_deep_reinforcement_learning_b200.layout import UnpackedLayout
from oracle import oracle as O
from tests.helpers import RUNNER_RULES, RunnerEpisode, load_model_golden, load_runner


@pytest.mark.parametrize("rules", RUNNER_RULES)
def test_oracle_replays_reference_game_runner(rules):
    tr = load_runner(rules)
    pool = int(tr["tile_pool"])
    L = UnpackedLayout(2)
    n_forced = 0
    for e in range(len(tr["seeds"])):
        ep = RunnerEpisode(tr, e)
        # Azul(rules) + new_round() of GameRunner.reset (game_runner.py:79-80)
        g = O.Game(2, pool, first_player=ep.first_player)
        g.new_round(ep.init_draws)
        assert np.array_equal(g.rec, ep.init_record)
        player_score, hb = 0, 0
        in_reset = True
        for s in range(ep.n_steps + 1):
            # the loop test on the current state decides who moves next
            cont = O.runner_continues(g.rec, 2, require_two=not in_reset)
            handback = not cont
            assert handback == (hb < ep.n_hb and ep.hb_step[hb] == s), (e, s)
            if handback:
                # game_runner.py:48-55 (and :81 after reset): reward from a count_score on a copy
                sc = g.score_preview()
                new_score = int(sc[0]) - int(sc[1])
                if in_reset:
                    new_score_ref, reward = 0, 0
                    in_reset = False
                    player_score = 0                          # game_runner.py:81
                else:
                    reward = new_score - player_score
                    player_score = new_score
                assert reward == int(ep.hb_reward[hb]), (e, s)
                assert player_score == int(ep.hb_player_score[hb])
                assert bool(g.is_end_of_game()) == bool(ep.hb_done[hb])
                assert np.array_equal(g.rec[:L.total_steps], ep.hb_records[hb][:L.total_steps])
                assert np.array_equal(O.observe(g.rec, 2, 0), ep.hb_obs[hb])
                assert np.array_equal(g.legal_mask(), ep.hb_mask[hb])
                assert ep.hb_move_counter[hb] == s
                hb += 1
            if s == ep.n_steps:
                break
            seat = int(g.rec[L.current_player])
            assert seat == int(ep.step_seat[s])
            if seat == 1 and not handback:
                n_forced += 1                                 # seat 1's forced move played by the opponent (:46)
            assert g.step(int(ep.step_action[s]), ep.step_draws(s)) == 0
        assert hb == ep.n_hb and bool(ep.hb_done[-1])
        assert np.array_equal(g.rec[:L.total_steps], ep.final_record[:L.total_steps])
        # Azul.get_statistics (azul.py:314-315)
        st = O.statistics(g.rec, 2)
        want = dict(zip(ep.stat_keys, ep.stats))
        assert st[0] == want["player_score"] and st[1] == want["opponent_score"] and st[2] == want["rounds"]
        assert abs(100.0 * st[3] / st[4] - want["percent_first_player"]) < 1e-9
        assert st[5] == want["floor_penalty"] and st[6] == want["max_combo"]
        assert st[7] == want["completed_rows"] and st[8] == want["completed_columns"] and st[9] == want["completed_colors"]
        assert float(st[0] > st[1]) == want["win_percent"]
    assert n_forced > 20          # the ":46" rule (opponent plays seat 1 when it has < 2 legal moves) is exercised


def test_oracle_observation_matches_reference_get_state():
    """``get_state(perspective=current_player-1)`` as the opponent sees it (game_runner.py:38) and from seat 1:
    the 4,096 decision states of model.npz."""
    z = load_model_golden()
    recs, obs = z["records"].astype(np.int32), z["obs"].astype(np.int32)
    for i in range(recs.shape[0]):
        assert np.array_equal(O.observe(recs[i], 2, -1), obs[i]), i
        m = O.Game(2, 0, record=recs[i]).legal_mask()
        assert np.array_equal(m, z["mask"][i])
