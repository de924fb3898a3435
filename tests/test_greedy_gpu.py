"""The greedy agent on the GPU: azb_greedy_action and azb_opponent_greedy against the CPU restatement
(tests/harness/greedy_oracle.c) game by game, whole episodes against it in one persistent launch
(azb_policy_rollout_vs_greedy) against the eager BatchedGameRunner(opponent="greedy") loop, training and evaluation
against it, and that it plays sensibly."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

from azul_deep_reinforcement_learning_b200.layout import UnpackedLayout  # noqa: E402
from tests.harness import greedy as GH  # noqa: E402

pytestmark = pytest.mark.gpu

CONFIGS = [(p, pool) for p in (2, 3, 4) for pool in (0, 1)]
N_RAGGED = 148 * 128 + 333                 # two tiles on some CTAs: several parts in the runner block
RULES = {1: {"first_player": "Random", "tile_pool": "Lid"}, 0: {"first_player": "Random", "tile_pool": "Random"}}
M32 = 0xFFFFFFFF


def _philox_words(seed, gid, block):
    """Philox4x32-10(ctr = (gid, block, ACTION = 0, 0), key = seed) for arrays of gid / block (uint64 arithmetic)."""
    c0, c1 = gid.astype(np.uint64), block.astype(np.uint64)
    c2, c3 = np.zeros_like(c0), np.zeros_like(c0)
    k0, k1 = np.uint64(seed & M32), np.uint64((seed >> 32) & M32)
    m = np.uint64(M32)
    for _ in range(10):
        p0, p1 = np.uint64(0xD2511F53) * c0, np.uint64(0xCD9E8D57) * c2
        c0, c1, c2, c3 = ((p1 >> np.uint64(32)) ^ c1 ^ k0) & m, p1 & m, ((p0 >> np.uint64(32)) ^ c3 ^ k1) & m, p0 & m
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & m, (k1 + np.uint64(0xBB67AE85)) & m
    return np.stack([c0, c1, c2, c3], axis=1)


def _action_words(seed, gid0, recs, players):
    L = UnpackedLayout(players)
    steps = recs[:, L.total_steps].astype(np.int64) & M32
    gid = gid0 + np.arange(recs.shape[0], dtype=np.int64)
    w = _philox_words(seed, gid, steps >> 2)
    return w[np.arange(recs.shape[0]), steps & 3]


def _snapshots(players, pool, seed, n, ks):
    """n games of a random-agent rollout, exported after each of the step counts in ks: records [len(ks) * n, U]."""
    from azul_deep_reinforcement_learning_b200.engine import BatchedAzul
    e = BatchedAzul(n, players, pool, 0, seed=seed)
    out, done = [], 0
    for k in ks:
        e.rollout_random(k - done)
        done = k
        out.append(e.export_records().cpu().numpy())
    return e, np.concatenate(out)


def _finished_games(players, pool, seed, n):
    """n finished games: every seat played by the greedy agent until the end (azb_greedy_action + azb_step)."""
    from azul_deep_reinforcement_learning_b200.engine import BatchedAzul
    e = BatchedAzul(n, players, pool, 0, seed=seed)
    for _ in range(400):
        st = e.step(e.greedy_action(), want_mask=False)
        if bool(((st["done"] != 0) | ((st["status"] & 4) != 0)).all()):
            break
    return e.export_records().cpu().numpy()


@pytest.mark.parametrize("players,pool", CONFIGS)
def test_greedy_action_equals_oracle(players, pool):
    """azb_greedy_action == ao_greedy_action (with the game's own Philox word) on 65,536 reachable states from rollout
    snapshots, plus finished games; the state is untouched."""
    from azul_deep_reinforcement_learning_b200.engine import BatchedAzul
    seed = 1000 + 10 * players + pool
    _, snaps = _snapshots(players, pool, seed, 16384, (0, 9, 31, 77))
    fin = _finished_games(players, pool, seed + 1, 2048)
    L = UnpackedLayout(players)
    assert int((fin[:, L.end_of_game] != 0).sum()) >= 1900
    recs = np.ascontiguousarray(np.concatenate([snaps, fin]), dtype=np.int32)
    e = BatchedAzul(recs.shape[0], players, pool, 0, seed=seed, game_id_base=77, reset=False)
    assert bool((e.import_records(recs) != 0).all())
    before = e.state.clone()
    got = e.greedy_action().cpu().numpy()
    assert torch.equal(e.state, before)
    words = _action_words(seed, 77, recs, players)
    want = np.array([GH.ao_greedy_action(r, players, pool, int(w)) for r, w in zip(recs, words)])
    ended = recs[:, L.end_of_game] != 0
    want = np.where(ended | (want < 0), 255, want)
    bad = np.nonzero(got != want)[0]
    assert bad.size == 0, (bad[:10], got[bad[:10]], want[bad[:10]])
    assert (got[ended] == 255).all() and (got[~ended] < 180).mean() > 0.99


@pytest.mark.parametrize("require_two", [1, 0])
@pytest.mark.parametrize("players,pool", CONFIGS)
def test_opponent_greedy_equals_oracle(players, pool, require_two):
    """azb_opponent_greedy == ao_opponent_greedy game by game: record, reward, mask, done and status; the observation
    output equals azb_observe_bf16 of the resulting state."""
    from azul_deep_reinforcement_learning_b200.engine import BatchedAzul
    seed = 2000 + 10 * players + pool
    _, recs = _snapshots(players, pool, seed, 2048, (0, 13, 40))
    n = recs.shape[0]
    e = BatchedAzul(n, players, pool, 0, seed=seed, game_id_base=5, reset=False)
    e.import_records(recs)
    score = torch.randint(-20, 20, (n,), dtype=torch.int16, device=e.device)
    score0 = score.cpu().numpy().astype(np.int32)
    out = e.opponent_greedy(score, require_two=bool(require_two), want_mask=True, want_obs=True)
    torch.cuda.synchronize()
    got = e.export_records().cpu().numpy()
    mask = out["mask"].cpu().numpy().astype(np.uint32)
    reward, done, status = (out[k].cpu().numpy() for k in ("reward", "done", "status"))
    L = UnpackedLayout(players)
    for g in range(n):
        r = np.ascontiguousarray(recs[g].copy())
        diff, m = GH.ao_opponent_greedy(r, players, pool, seed, 5 + g, require_two)
        assert np.array_equal(got[g], r), g
        assert np.array_equal(mask[:, g], m), g
        assert int(reward[g]) == diff - score0[g] and int(score[g]) == diff, g
        assert int(done[g]) == int(r[L.end_of_game] != 0) and int(status[g]) == int(r[L.status]), g
    assert torch.equal(out["obs"], e.observe_bf16(0))


def _runner(n, pool, seed, agent_mode):
    """BatchedGameRunner(opponent="greedy") whose agent decides with ``agent_mode`` (run_episodes samples)."""
    from azul_deep_reinforcement_learning_b200.selfplay import BatchedGameRunner

    class Runner(BatchedGameRunner):
        def step_policy(self, packed, mode=0):
            return super().step_policy(packed, mode=agent_mode)

    return Runner(n, rules=RULES[pool], seed=seed, opponent="greedy")


@pytest.mark.parametrize("n", [700, N_RAGGED])
@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("pool", [1, 0])
def test_persistent_rollout_vs_greedy_equals_eager_loop(pool, mode, n):
    """PersistentEpisodes on BatchedGameRunner(opponent="greedy") == run_episodes on the same runner: per game the same
    actions, rewards, logp / value records, recorded states (observation and mask), done flags, final state and
    player_score; discounted returns within the runner-mode tolerance."""
    from azul_deep_reinforcement_learning_b200.azulnet.model import ActorCritic
    from azul_deep_reinforcement_learning_b200.engine import PackedPolicy, mask_to_bool
    from azul_deep_reinforcement_learning_b200.selfplay import PersistentEpisodes, discounted_returns, run_episodes
    seed = 60 + 2 * pool + mode
    torch.manual_seed(seed)
    net = ActorCritic(136, 180)
    a, b = _runner(n, pool, 31 + seed, mode), _runner(n, pool, 31 + seed, mode)
    pa, pb = PackedPolicy(a.engine, net), PackedPolicy(b.engine, net)
    pers = PersistentEpisodes(b, pb, max_decisions=160, want_logp_value=True)
    a.reset()
    pers.start(mode)
    torch.cuda.synchronize()
    assert torch.equal(a.engine.state, b.engine.state) and torch.equal(a.mask, b.mask)
    rec = b.engine.export_records().cpu().numpy()
    L = UnpackedLayout(2)
    assert (rec[:, L.current_player] == 1).all() and bool((mask_to_bool(b.mask).sum(dim=1) >= 2).all())

    eager = run_episodes(a, pa, max_decisions=160, record_obs=True)
    r = pers.run(gamma=0.99, mode=mode)
    torch.cuda.synchronize()
    assert torch.equal(a.engine.state, b.engine.state) and torch.equal(a.player_score, b.player_score)
    act = eager["active"]
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
    done_t = ((flags >> 1) & 1).bool()
    assert int(done_t.sum()) == n - eager["unfinished"] and bool((done_t <= act).all())
    assert eager["unfinished"] == 0 or mode == 1
    q = discounted_returns(eager["reward"].double(), act, 0.99).float()
    assert torch.allclose(r.qval[slots], q[act], rtol=1e-6, atol=1e-5)


def test_vs_greedy_rejects_bad_arguments():
    """A 3-player handle and an unknown mode are refused before any launch; so is an unknown opponent keyword."""
    import ctypes
    from azul_deep_reinforcement_learning_b200.azulnet.model import ActorCritic
    from azul_deep_reinforcement_learning_b200.engine import BatchedAzul, EpisodeRecords, PackedPolicy, _ptr
    from azul_deep_reinforcement_learning_b200.selfplay import BatchedGameRunner
    net = ActorCritic(136, 180)
    for players, mode in ((3, 0), (2, 2), (4, 1)):
        e = BatchedAzul(256, players, 1, 0, seed=1)
        helper = e if players == 2 else BatchedAzul(256, 2, 1, 0, seed=1)
        p = PackedPolicy(helper, net)
        r = EpisodeRecords(helper, 4)
        ps = torch.zeros(256, dtype=torch.int16, device="cuda")
        rc = e.lib.azb_policy_rollout_vs_greedy(
            e._h, _ptr(e.state), _ptr(p.buf), mode, 4, _ptr(ps), _ptr(r.meta), r.cap, _ptr(r.state_rec), _ptr(r.action_rec),
            None, None, _ptr(r.slot_rec), _ptr(r.reward_rec), _ptr(r.flags_rec), ctypes.c_void_p(r.meta.data_ptr() + 4),
            None, None, None, None, None, None, e._stream())
        assert rc == -1, (players, mode)                               # AZB_E_INVALID
    with pytest.raises(ValueError):
        BatchedGameRunner(256, opponent="grredy")


def test_trainer_against_greedy():
    """SelfPlayTrainer(opponent="greedy") trains through the captured batch graph (batch 3 is its replay)."""
    from azul_deep_reinforcement_learning_b200.train import SelfPlayTrainer
    tr = SelfPlayTrainer(512, seed=4, opponent="greedy")
    assert tr.runner.opponent == "greedy" and tr.opponent is None
    hist = tr.train(batches=3, log=None)
    assert tr._graph is not None
    assert len(hist) == 3 and all(np.isfinite(h["ac_loss"]) for h in hist)
    assert all(h["games"] == 512 and h["unfinished"] == 0 for h in hist)
    with pytest.raises(ValueError):
        SelfPlayTrainer(64, opponent="greedy", opponent_refresh=2)


def test_evaluate_against_greedy_matches_eager():
    """evaluate(net, "greedy", mode=1) reports the statistics azb_stats gives on the eager path's final states."""
    from azul_deep_reinforcement_learning_b200.azulnet.model import ActorCritic
    from azul_deep_reinforcement_learning_b200.engine import PackedPolicy
    from azul_deep_reinforcement_learning_b200.evaluate import evaluate
    from azul_deep_reinforcement_learning_b200.selfplay import BatchedGameRunner, run_episodes
    torch.manual_seed(8)
    net = ActorCritic(136, 180)
    n, seed = 2048, 17
    got = evaluate(net, "greedy", games=n, mode=1, seed=seed)
    ref = BatchedGameRunner(n, seed=seed, opponent="greedy")             # the same construction as evaluate()
    ref.step_policy = lambda p, mode=0, _f=ref.step_policy: _f(p, mode=1)
    batch = run_episodes(ref, PackedPolicy(ref.engine, net.cuda()), max_decisions=160, record_obs=False)
    torch.cuda.synchronize()
    L = UnpackedLayout(2)
    per_game = ref.engine.stats().long().cpu()
    ended = torch.from_numpy(ref.engine.export_records().cpu().numpy()[:, L.end_of_game] != 0)
    s = per_game.sum(0).double() / n
    want = {"player_score": float(s[0]), "opponent_score": float(s[1]), "rounds": float(s[2]),
            "win_percent": float((per_game[:, 0] > per_game[:, 1]).sum()) / n, "unfinished": int((~ended).sum())}
    for k, v in want.items():
        assert got[k] == v, (k, got[k], v)
    assert got["games"] == n and got["decisions"] == int(batch["active"].sum()) and got["max_opponent_passes"] == 0


def test_greedy_agent_is_sensible():
    """Greedy in seat 1 beats the random opponent in more than 60 % of 4,096 games, and an untrained network scores less
    against the greedy agent than against the random one."""
    from azul_deep_reinforcement_learning_b200.azulnet.model import ActorCritic
    from azul_deep_reinforcement_learning_b200.evaluate import evaluate
    from azul_deep_reinforcement_learning_b200.selfplay import BatchedGameRunner
    n = 4096
    runner = BatchedGameRunner(n, seed=21)
    done = torch.zeros(n, dtype=torch.bool, device=runner.device)
    for _ in range(200):
        out = runner.step(runner.engine.greedy_action())
        done |= (out["done"] != 0) | ((out["status"] & 4) != 0)
        if bool(done.all()):
            break
    st = runner.engine.stats().long()
    win = float((st[:, 0] > st[:, 1]).double().mean())
    assert bool(done.all()) and win > 0.6, win
    torch.manual_seed(3)
    net = ActorCritic(136, 180)
    vs_greedy = evaluate(net, "greedy", games=n, seed=5)
    vs_random = evaluate(net, "random", games=n, seed=5)
    print("greedy vs random: seat-1 wins %.4f, score %.2f vs %.2f; untrained net player_score vs greedy %.2f, vs random %.2f"
          % (win, float(st[:, 0].double().mean()), float(st[:, 1].double().mean()), vs_greedy["player_score"],
             vs_random["player_score"]))
    assert vs_greedy["player_score"] < vs_random["player_score"], (vs_greedy, vs_random)
