"""Whole episodes against a frozen policy opponent in one persistent launch (azb_policy_rollout_vs_policy), the sync-free
episode start, training against a frozen or lagged network and the evaluation entry point -- against the eager
GameRunner(opponent=Agent) path of selfplay.BatchedGameRunner."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

from azul_deep_reinforcement_learning_b200.layout import UnpackedLayout  # noqa: E402

pytestmark = pytest.mark.gpu

N_RAGGED = 148 * 128 + 333                 # two tiles on some CTAs: several parts in the runner block
RULES = {1: {"first_player": "Random", "tile_pool": "Lid"}, 0: {"first_player": "Random", "tile_pool": "Random"}}


def _eager_runner(n, pool, seed, opp_net, mode):
    """BatchedGameRunner(opponent=PackedPolicy) whose agent decides with ``mode`` too (run_episodes samples)."""
    from azul_deep_reinforcement_learning_b200.engine import BatchedAzul, PackedPolicy
    from azul_deep_reinforcement_learning_b200.selfplay import BatchedGameRunner

    class Runner(BatchedGameRunner):
        def step_policy(self, packed, mode=0):
            return super().step_policy(packed, mode=self.opponent_mode)

    helper = BatchedAzul(n, 2, pool, 0, seed=seed, reset=False)
    return Runner(n, rules=RULES[pool], seed=seed, opponent=PackedPolicy(helper, opp_net) if opp_net is not None else None,
                  opponent_mode=mode)


def _nets(seed):
    from azul_deep_reinforcement_learning_b200.azulnet.model import ActorCritic
    torch.manual_seed(seed)
    return ActorCritic(136, 180), ActorCritic(136, 180)


@pytest.mark.parametrize("n", [700, N_RAGGED])
@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("pool", [1, 0])
def test_persistent_rollout_vs_policy_equals_eager_loop(pool, mode, n):
    """PersistentEpisodes against a PackedPolicy opponent == run_episodes on BatchedGameRunner(opponent=PackedPolicy):
    per game the same actions, rewards, logp / value records, recorded states (observation and mask), done flags, final
    state and player_score; discounted returns within the runner-mode tolerance."""
    _check_against_eager(pool, mode, n, same_image=False, seed=40 + 2 * pool + mode)


def test_persistent_rollout_vs_own_image():
    """The opponent's image may be the agent's own buffer (self-play against the current network)."""
    _check_against_eager(1, 0, 1500, same_image=True, seed=9)


def _check_against_eager(pool, mode, n, same_image, seed):
    from azul_deep_reinforcement_learning_b200.engine import PackedPolicy, mask_to_bool
    from azul_deep_reinforcement_learning_b200.selfplay import PersistentEpisodes, discounted_returns, run_episodes
    net, opp = _nets(seed)
    a = _eager_runner(n, pool, 31 + seed, net if same_image else opp, mode)
    b = _eager_runner(n, pool, 31 + seed, net if same_image else opp, mode)
    pa, pb = PackedPolicy(a.engine, net), PackedPolicy(b.engine, net)
    if same_image:
        a.opponent, b.opponent = pa, pb
    assert torch.equal(a.engine.state, b.engine.state)
    pers = PersistentEpisodes(b, pb, max_decisions=160, want_logp_value=True)

    # the sync-free start equals GameRunner.reset with the Agent opponent and leaves seat 1 to move with >= 2 actions
    a.reset()
    pers.start(mode)
    torch.cuda.synchronize()
    assert torch.equal(a.engine.state, b.engine.state) and torch.equal(a.mask, b.mask)
    assert int(b.player_score.abs().sum()) == 0
    rec = b.engine.export_records().cpu().numpy()
    L = UnpackedLayout(2)
    assert (rec[:, L.current_player] == 1).all() and bool((mask_to_bool(b.mask).sum(dim=1) >= 2).all())

    eager = run_episodes(a, pa, max_decisions=160, record_obs=True)
    r = pers.run(gamma=0.99, mode=mode)
    torch.cuda.synchronize()
    assert 1 <= int(pers.opp_passes[0]) <= 64
    assert torch.equal(a.engine.state, b.engine.state) and torch.equal(a.player_score, b.player_score)
    act = eager["active"]                                         # [T, G]
    T = act.shape[0]
    n_dec, used = int(r.meta[0]), int(r.meta[1])
    assert n_dec == int(act.sum()) and used <= 160 and n_dec <= r.cap
    flags = r.flags_rec[:T]
    assert torch.equal((flags & 1).bool(), act) and int(r.flags_rec[T:].sum()) == 0
    slots = r.slot_rec[:T][act].long()
    assert int(slots.min()) >= 0 and len(torch.unique(slots)) == n_dec
    assert torch.equal(r.action_rec[slots].long(), eager["action"][act])
    assert torch.equal(r.reward_rec[:T][act].float(), eager["reward"][act])
    assert torch.equal(r.logp_rec[slots], eager["logp"][act]) and torch.equal(r.value_rec[slots], eager["value"][act])
    assert torch.equal(r.view.observe_bf16(-1)[slots], eager["obs"][act])
    assert torch.equal(r.view.legal_mask()[:, slots], eager["mask"].permute(1, 0, 2)[:, act])
    # done flag: on the last decision of every finished game
    done_t = ((flags >> 1) & 1).bool()
    assert int(done_t.sum()) == n - eager["unfinished"] and bool((done_t <= act).all())
    if mode == 0:
        assert eager["unfinished"] == 0
    # azb_discounted_returns accumulates in double: so does the reference here (argmax games can run all 160 decisions, and
    # a float32 recurrence drifts past the tolerance over that many steps)
    q = discounted_returns(eager["reward"].double(), act, 0.99).float()
    assert torch.allclose(r.qval[slots], q[act], rtol=1e-6, atol=1e-5)


def test_entry_point_rejects_bad_arguments():
    """A null opponent image, a 3-player handle and an unknown mode are refused before any launch; so is a persistent
    rollout whose agent mode differs from the opponent's."""
    import ctypes
    from azul_deep_reinforcement_learning_b200.engine import BatchedAzul, EpisodeRecords, PackedPolicy, _ptr
    from azul_deep_reinforcement_learning_b200.selfplay import PersistentEpisodes
    net, opp = _nets(1)
    for players, mode, null_opp in ((2, 0, True), (3, 0, False), (2, 2, False)):
        e = BatchedAzul(256, players, 1, 0, seed=1)
        helper = e if players == 2 else BatchedAzul(256, 2, 1, 0, seed=1)
        p, q = PackedPolicy(helper, net), PackedPolicy(helper, opp)
        r = EpisodeRecords(helper, 4)
        ps = torch.zeros(256, dtype=torch.int16, device="cuda")
        rc = e.lib.azb_policy_rollout_vs_policy(
            e._h, _ptr(e.state), _ptr(p.buf), None if null_opp else _ptr(q.buf), mode, 4, _ptr(ps), _ptr(r.meta), r.cap,
            _ptr(r.state_rec), _ptr(r.action_rec), None, None, _ptr(r.slot_rec), _ptr(r.reward_rec), _ptr(r.flags_rec),
            ctypes.c_void_p(r.meta.data_ptr() + 4), None, None, None, None, e._stream())
        assert rc == -1, (players, mode, null_opp)                     # AZB_E_INVALID
    b = _eager_runner(256, 1, 3, opp, 1)
    pers = PersistentEpisodes(b, PackedPolicy(b.engine, net))
    with pytest.raises(ValueError):
        pers.run(mode=0)


def test_trainer_against_frozen_network_and_lagged_copy():
    """SelfPlayTrainer(opponent=...) trains through the captured batch graph; without refresh the opponent image never
    changes, with opponent_refresh = 1 it equals a fresh pack of the network after every batch."""
    from azul_deep_reinforcement_learning_b200.engine import PackedPolicy
    from azul_deep_reinforcement_learning_b200.train import SelfPlayTrainer
    _, frozen = _nets(5)
    tr = SelfPlayTrainer(512, seed=2, opponent=frozen)
    image = tr.opponent.buf.clone()
    hist = tr.train(batches=3, log=None)                               # batch 3 is the replay of the captured graph
    assert tr._graph is not None
    assert len(hist) == 3 and all(np.isfinite(h["ac_loss"]) for h in hist)
    assert all(h["games"] == 512 and h["unfinished"] == 0 for h in hist)
    assert all(25 * 512 < h["transitions"] < 80 * 512 for h in hist)
    assert torch.equal(tr.opponent.buf, image)
    assert torch.equal(image, PackedPolicy(tr.runner.engine, frozen.to(tr.device)).buf)

    lag = SelfPlayTrainer(512, seed=3, opponent_refresh=1)
    first = lag.opponent.buf.clone()
    lag.enable_step_graph(warmup=1)
    for _ in range(2):
        lag.step()
        torch.cuda.synchronize()
        assert torch.equal(lag.opponent.buf, PackedPolicy(lag.runner.engine, lag.net).buf)
    assert not torch.equal(lag.opponent.buf, first)


def _expected(per_game, ended):
    games = per_game.shape[0]
    s = per_game.sum(0).double() / games
    return {"player_score": float(s[0]), "opponent_score": float(s[1]), "rounds": float(s[2]),
            "win_percent": float((per_game[:, 0] > per_game[:, 1]).sum()) / games, "unfinished": int((~ended).sum())}


def test_evaluate_matches_eager_and_runner_mode(tmp_path):
    """evaluate() against a saved network in argmax mode reports the statistics azb_stats gives on the eager path's final
    states; against the random opponent those of the existing runner mode."""
    from azul_deep_reinforcement_learning_b200.engine import PackedPolicy
    from azul_deep_reinforcement_learning_b200.evaluate import evaluate
    from azul_deep_reinforcement_learning_b200.selfplay import BatchedGameRunner, PersistentEpisodes, run_episodes
    net, opp = _nets(8)
    torch.save(opp.state_dict(), str(tmp_path / "opp.pt"))
    n, seed = 2048, 17
    L = UnpackedLayout(2)
    for opponent in ("file", "random"):
        got = evaluate(net, str(tmp_path / "opp.pt") if opponent == "file" else "random", games=n, mode=1, seed=seed)
        ref = BatchedGameRunner(n, seed=seed)                          # the same construction as evaluate()
        packed = PackedPolicy(ref.engine, net.cuda())
        if opponent == "file":
            ref.opponent, ref.opponent_mode = PackedPolicy(ref.engine, opp.cuda()), 1
            ref.step_policy = lambda p, mode=0, _f=ref.step_policy: _f(p, mode=1)
            batch = run_episodes(ref, packed, max_decisions=160, record_obs=False)
            decisions = int(batch["active"].sum())
            assert 1 <= got["max_opponent_passes"] <= 64
        else:
            r = PersistentEpisodes(ref, packed, max_decisions=160).run(mode=1)
            decisions = int(r.meta[0])
        torch.cuda.synchronize()
        per_game = ref.engine.stats().long().cpu()
        ended = torch.from_numpy(ref.engine.export_records().cpu().numpy()[:, L.end_of_game] != 0)
        want = _expected(per_game, ended)
        for k, v in want.items():
            assert got[k] == v, (opponent, k, got[k], v)
        assert got["games"] == n and got["decisions"] == decisions
        for k in ("percent_first_player", "floor_penalty", "max_combo", "completed_rows", "completed_columns",
                  "completed_colors"):
            assert np.isfinite(got[k]), k
