"""Batched GameRunner semantics and the self-play training loop on the GPU."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

from azul_deep_reinforcement_learning_b200.layout import UnpackedLayout  # noqa: E402
from oracle import oracle as O  # noqa: E402

pytestmark = pytest.mark.gpu


def test_batched_game_runner_matches_oracle_runner():
    """GameRunner.reset / step (game_runner.py:43-55,76-85) for 512 games against the C oracle's statement of
    the same loop: agent actions are fed in, opponent moves come from the shared Philox schedule."""
    from azul_deep_reinforcement_learning_b200.selfplay import BatchedGameRunner
    n, seed = 512, 77
    gr = BatchedGameRunner(n, seed=seed)
    recs = O.fresh_records(n, 2, 1, 0, seed, 0)
    pscore = np.zeros(n, np.int64)
    masks = np.zeros((n, 6), np.uint32)
    for i in range(n):
        _, masks[i] = O.opponent_random(recs[i], 2, 1, seed, i, require_two=False)
    assert np.array_equal(gr.engine.export_records().cpu().numpy(), recs)
    assert np.array_equal(gr.mask.cpu().numpy().astype(np.uint32).T, masks)
    L = UnpackedLayout(2)
    rng = np.random.default_rng(0)
    for t in range(45):
        act = np.full(n, 255, np.uint8)
        want_reward = np.zeros(n, np.int64)
        want_done = np.zeros(n, np.uint8)
        for i in range(n):
            g = O.Game(2, 1, record=recs[i])
            if not g.rec[L.end_of_game] and masks[i].any():
                a = O.random_action(masks[i], int(rng.integers(0, 2 ** 32)))
                act[i] = a
                assert g.step(a, None, seed, i) == 0
            recs[i] = g.rec
            d, masks[i] = O.opponent_random(recs[i], 2, 1, seed, i, require_two=True)
            want_reward[i] = d - pscore[i]
            pscore[i] = d
            want_done[i] = recs[i][L.end_of_game]
        out = gr.step(torch.from_numpy(act))
        assert np.array_equal(gr.engine.export_records().cpu().numpy(), recs), t
        assert np.array_equal(out["reward"].cpu().numpy().astype(np.int64), want_reward), t
        assert np.array_equal(out["done"].cpu().numpy(), want_done), t
        assert np.array_equal(out["mask"].cpu().numpy().astype(np.uint32).T, masks), t
        assert np.array_equal(gr.player_score.cpu().numpy().astype(np.int64), pscore)
    assert want_done.sum() > 0
    # GameRunner invariant after step: seat 1 to move with >= 2 legal actions, or the game is over
    cur = recs[:, L.current_player]
    nvalid = np.array([sum(bin(int(w)).count("1") for w in m) for m in masks])
    assert (((cur == 1) & (nvalid >= 2)) | (recs[:, L.end_of_game] == 1) | (recs[:, L.status] & 4 != 0)).all()


def test_reward_kat_from_reference_fixture():
    """tests/test_game_runner.py:52-62: from game_end_of_round_3 with player_score 49-32, stepping (0,3,0)
    yields reward -6 (deterministic: the move ends the round, seat 1 starts the next with 72 legal moves)."""
    from azul_deep_reinforcement_learning_b200.selfplay import BatchedGameRunner
    from tests.helpers import load_kat
    kat = load_kat()
    rec = kat["fixture_records"][list(kat["fixture_names"]).index("game_end_of_round_3")].astype(np.int32)[None, :].copy()
    L = UnpackedLayout(2)
    rec[0, L.box:L.box + 5] = 20
    gr = BatchedGameRunner(1, seed=3)
    assert bool(gr.engine.import_records(rec).all())
    gr.player_score.fill_(49 - 32)
    out = gr.step(torch.tensor([0 + 6 * 3 + 30 * 0], dtype=torch.uint8))
    assert int(out["reward"][0]) == -6 and int(out["done"][0]) == 0
    r = gr.engine.export_records().cpu().numpy()[0]
    assert int(gr.player_score[0]) == r[L.score] - r[L.score + 1] and r[L.current_player] == 1


def test_selfplay_training_runs_and_learns_something():
    from azul_deep_reinforcement_learning_b200.train import SelfPlayTrainer
    tr = SelfPlayTrainer(games_per_rank=512, seed=1)
    before = [p.detach().clone() for p in tr.net.parameters()]
    hist = tr.train(batches=3, log=None)
    assert len(hist) == 3 and all(np.isfinite(h["ac_loss"]) for h in hist)
    assert all(h["games"] == 512 and h["unfinished"] == 0 for h in hist)
    assert all(25 * 512 < h["transitions"] < 80 * 512 for h in hist)            # SURVEY §3.3: ~30-36 decisions per game
    assert any(not torch.equal(a, b) for a, b in zip(before, tr.net.parameters()))
    assert 0 <= hist[0]["win_percent"] <= 1 and 3 <= hist[0]["rounds"] <= 12


def test_agent_opponent_in_batched_runner():
    """GameRunner(opponent=Agent) (scripts/run_batch.py:6-8): the frozen policy plays seat 2 and seat 1's forced moves."""
    from azul_deep_reinforcement_learning_b200.azulnet.model import ActorCritic
    from azul_deep_reinforcement_learning_b200.engine import BatchedAzul, PackedPolicy, mask_to_bool
    from azul_deep_reinforcement_learning_b200.selfplay import BatchedGameRunner, run_episodes
    torch.manual_seed(3)
    net, opp = ActorCritic(136, 180), ActorCritic(136, 180)
    n = 1024
    helper = BatchedAzul(n, 2, 1, 0, seed=5, reset=False)
    gr = BatchedGameRunner(n, seed=5, opponent=PackedPolicy(helper, opp))
    packed = PackedPolicy(gr.engine, net)
    L = UnpackedLayout(2)
    for t in range(30):
        rec = gr.engine.export_records().cpu().numpy()
        nvalid = mask_to_bool(gr.mask).sum(dim=1).cpu().numpy()
        live = rec[:, L.end_of_game] == 0
        assert ((rec[live, L.current_player] == 1) & (nvalid[live] >= 2)).all(), t      # invariant of GameRunner.step
        before_steps = rec[:, L.total_steps].copy()
        out = gr.step_policy(packed)
        after = gr.engine.export_records().cpu().numpy()
        moved = after[:, L.total_steps] - before_steps
        assert (moved[live] >= 1).all() and (moved[~live] == 0).all()
        assert int((out["status"] & 1).max()) == 0
    # a whole batch of episodes against the Agent opponent terminates and produces rewards
    batch = run_episodes(gr, packed, max_decisions=200)
    assert batch["unfinished"] < n // 20 and float(batch["reward"].abs().sum()) > 0


def test_fused_a2c_loss_gradient_matches_autograd():
    """azb_a2c_loss_grad (one kernel: masked log-softmax, the three terms of Agent.update, their gradient) against PyTorch
    autograd of train.a2c_loss_terms -- the formula test_train_cpu pins to the reference's Agent.update -- on recorded
    decisions of a real rollout.  fp32 both sides; tolerance 2e-5 of the gradient scale."""
    from azul_deep_reinforcement_learning_b200.azulnet.model import ActorCritic
    from azul_deep_reinforcement_learning_b200.engine import PackedPolicy, mask_rows_to_bool
    from azul_deep_reinforcement_learning_b200.selfplay import BatchedGameRunner, discounted_returns, run_episodes
    from azul_deep_reinforcement_learning_b200.train import ACTOR_COEFF, CRITIC_COEFF, ENTROPY_COEFF, a2c_loss_terms
    torch.manual_seed(3)
    net = ActorCritic(136, 180).cuda()
    with torch.no_grad():
        for p in net.parameters():
            p.mul_(2.5)
    gr = BatchedGameRunner(300, seed=8)
    batch = run_episodes(gr, PackedPolicy(gr.engine, net))
    act = batch["active"]
    T, G = act.shape
    sel = act.reshape(-1).nonzero(as_tuple=True)[0]
    obs = batch["obs"].reshape(T * G, -1)[sel].float()
    assert obs.dtype == torch.float32 and batch["obs"].dtype == torch.bfloat16
    rows = batch["mask"].permute(0, 2, 1).reshape(T * G, 6)[sel].contiguous()
    action = batch["action"].reshape(-1)[sel]
    qval = discounted_returns(batch["reward"], act, 0.99).reshape(-1)[sel]
    n = int(sel.numel())
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        # reference: autograd through the torch formula
        a, c, e = a2c_loss_terms(net, obs, mask_rows_to_bool(rows), action, qval)
        ((ACTOR_COEFF * a + CRITIC_COEFF * c + ENTROPY_COEFF * e) / n).backward()
        want = [p.grad.clone() for p in net.parameters()]
        net.zero_grad()
        # fused kernel at the network outputs, autograd through the layers
        logits = net.actor_linear2(torch.relu(net.actor_linear1(obs)))
        value = net.forward_critic(obs).squeeze(1)
        sums = torch.zeros(3, dtype=torch.float64, device="cuda")
        dl, dv = gr.engine.a2c_loss_grad(logits.detach(), value.detach().contiguous(), rows, action, qval, 1.0 / n,
                                         (ACTOR_COEFF, CRITIC_COEFF, ENTROPY_COEFF), sums)
        torch.autograd.backward([logits, value], [dl, dv])
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev
    legal = mask_rows_to_bool(rows)
    assert float(dl[~legal].abs().max()) == 0.0                      # no gradient into illegal actions
    for p, w in zip(net.parameters(), want):
        assert float((p.grad - w).abs().max()) <= 2e-5 * max(1.0, float(w.abs().max())), p.shape
    ref = torch.stack([a, c, e]).double()
    assert float(((sums - ref).abs() / ref.abs().clamp_min(1.0)).max()) < 1e-5


def _a2c_reference(logits, value, legal, action, qval, scale, coeffs):
    """float64 statement of azb_a2c_loss_grad: (dlogits, dvalue, sums); rows whose action is not legal contribute nothing."""
    ca, cc, ce = coeffs
    ok = (action >= 0) & (action < 180) & legal.gather(1, action.clamp(0, 179)[:, None]).squeeze(1)
    l, m = logits.double()[ok], legal[ok]
    masked = l.masked_fill(~m, float("-inf"))
    lse = torch.logsumexp(masked, 1)
    log_prob = l.gather(1, action[ok][:, None]).squeeze(1) - lse
    k = m.sum(1).double()
    entropy = -((l * m).sum(1) / k - lse)
    adv = qval.double()[ok] - value.double()[ok]
    p = torch.exp(masked - lse[:, None])
    onehot = torch.nn.functional.one_hot(action[ok], 180).double()
    dl = torch.zeros(logits.shape, dtype=torch.float64, device=logits.device)
    dv = torch.zeros(value.shape, dtype=torch.float64, device=logits.device)
    dl[ok] = scale * torch.where(m, ca * (-adv)[:, None] * (onehot - p) + ce * (p - 1.0 / k[:, None]), 0.0)
    dv[ok] = scale * (ca * log_prob - 2.0 * cc * adv)
    return dl, dv, torch.stack([(-log_prob * adv).sum(), (adv * adv).sum(), entropy.sum()]), ok


@pytest.mark.parametrize("kind", ["one_legal", "all_legal", "only_150_179", "logits_1e4", "no_legal", "action_-1",
                                  "action_180", "illegal_action"])
def test_fused_a2c_loss_grad_edge_rows(kind):
    """azb_a2c_loss_grad against a float64 reference on synthetic masks: every other row of 128 is of the given kind.
    A single legal action has log-prob and entropy 0 (its gradient row is exactly zero); all 180 legal and only 150..179
    legal reach the lanes that hold columns past 180; logits of size 1e4 need the max subtraction; rows whose action
    is not legal (no legal action, action -1 or 180, an action outside the mask) get zero gradients and stay out of
    the sums."""
    from azul_deep_reinforcement_learning_b200.engine import BatchedAzul
    gen = torch.Generator(device="cuda").manual_seed(5)
    n, edge = 128, torch.arange(0, 128, 2, device="cuda")
    logits = torch.randn(n, 180, generator=gen, device="cuda") * 3.0
    value = torch.randn(n, generator=gen, device="cuda") * 10.0
    qval = torch.rand(n, generator=gen, device="cuda") * 80.0 - 40.0
    u = torch.rand(n, 180, generator=gen, device="cuda")
    legal = u < 0.3
    legal[:, 7] = True
    if kind == "one_legal":
        legal[edge] = False
        legal[edge, (u[edge, 0] * 180).long()] = True
    elif kind == "all_legal":
        legal[edge] = True
    elif kind == "only_150_179":
        legal[edge] = False
        legal[edge, 150:] = True
    elif kind == "logits_1e4":
        logits[edge] *= 1e4 / 3.0
    elif kind == "no_legal":
        legal[edge] = False
    action = torch.where(legal, u, -1.0).argmax(1)
    if kind.startswith("action_"):
        action[edge] = int(kind[len("action_"):])
    elif kind == "illegal_action":
        action[edge] = torch.where(legal, -1.0, u).argmax(1)[edge]
    words = (legal.view(n, 6, 30).long() << torch.arange(30, device="cuda")).sum(2).to(torch.int32).contiguous()
    eng = BatchedAzul(1, 2, 0, 0, seed=1)
    coeffs, scale = (1.0, 0.5, 0.1), 0.5
    sums = torch.zeros(3, dtype=torch.float64, device="cuda")
    dl, dv = eng.a2c_loss_grad(logits, value, words, action, qval, scale, coeffs, sums)
    want_dl, want_dv, want_sums, ok = _a2c_reference(logits, value, legal, action, qval, scale, coeffs)
    assert int(ok.sum()) == (n if kind in ("one_legal", "all_legal", "only_150_179", "logits_1e4") else n // 2)
    assert int(torch.count_nonzero(dl[~ok])) == 0 and int(torch.count_nonzero(dv[~ok])) == 0
    if kind == "one_legal":
        assert int(torch.count_nonzero(dl[edge])) == 0
    assert float((dl.double() - want_dl).abs().max()) <= 1e-5 * float(want_dl.abs().max())
    assert float((dv.double() - want_dv).abs().max()) <= 1e-5 * float(want_dv.abs().max())
    assert float(((sums - want_sums).abs() / want_sums.abs().clamp_min(1.0)).max()) <= 1e-5, (sums, want_sums)


@pytest.mark.parametrize("n", [1000, 256 * 148 + 3])
def test_train_stats_match_per_game_statistics(n):
    """azb_train_stats decodes the 2-player packed words itself: its 18 outputs equal the sums of azb_stats and of the
    exported records, exactly, with some games ended; the decision count is clamped to the record capacity (+1e9 on the
    unfinished count when it overflowed); the loss and reward sums pass through.  Other player counts are rejected."""
    from types import SimpleNamespace
    from azul_deep_reinforcement_learning_b200.engine import BatchedAzul, _ptr, train_stats
    eng = BatchedAzul(n, 2, 1, 0, seed=n)
    eng.rollout_random(45)
    eng.state[3, torch.arange(n, device="cuda") % 7 == 3] |= 1 << 12            # MISC bit 12: end_of_game
    per_game = eng.stats().long().sum(0).tolist()
    rec = eng.export_records().cpu().numpy()
    L = UnpackedLayout(2)
    wins = int((rec[:, L.score] > rec[:, L.score + 1]).sum())
    unfinished = int((rec[:, L.end_of_game] == 0).sum())
    assert 0 < unfinished < n and 0 < wins < n
    loss = torch.tensor([1.5, -2.25, 3.0], dtype=torch.float64, device="cuda")
    for n_dec, cap in ((500, 700), (700, 700), (701, 700)):
        recs = SimpleNamespace(meta=torch.tensor([n_dec, 0], dtype=torch.int32, device="cuda"), cap=cap,
                               reward_sum=torch.tensor([-17.0], dtype=torch.float64, device="cuda"))
        out = torch.full((18,), 123.0, dtype=torch.float64, device="cuda")
        train_stats(eng, recs, loss, out)
        want = [min(n_dec, cap), 1.5, -2.25, 3.0, -17.0, n] + per_game + [wins, unfinished + (1e9 if n_dec > cap else 0)]
        assert out.tolist() == want, (n_dec, cap)
    for players in (3, 4):
        other = BatchedAzul(64, players, 0, 0, seed=1)
        assert other.lib.azb_train_stats(other._h, _ptr(other.state), _ptr(recs.meta), 700, _ptr(loss), _ptr(recs.reward_sum),
                                         _ptr(out), other._stream()) == -1                # AZB_E_INVALID


@pytest.mark.parametrize("k", [1, 3, 4, 5, 161])
def test_discounted_returns_on_synthetic_records(k):
    """azb_discounted_returns against a float64 loop of nn_runner.py:72-75 cast to float32 (1 ulp: r + gamma * q may be
    fused) on synthetic records: gaps in the decision flags, decisions without a slot, a walk bounded by the iterations
    the rollout ran.  Slots never named keep their contents; the reward sum is the exact sum of the walked rewards."""
    from azul_deep_reinforcement_learning_b200.engine import BatchedAzul, EpisodeRecords, discounted_returns_records
    n, gamma = 1000, 0.99
    rng = np.random.default_rng(k)
    eng = BatchedAzul(n, 2, 0, 0, seed=k, reset=False)
    recs = EpisodeRecords(eng, k, capacity=k * n)
    flags = (rng.random((k, n)) < 0.7).astype(np.uint8) | (rng.integers(0, 2, (k, n)) << 1).astype(np.uint8)
    reward = rng.integers(-40, 41, (k, n)).astype(np.int16)
    slot = rng.permutation(k * n).reshape(k, n).astype(np.int32)
    slot[rng.random((k, n)) < 0.1] = -1
    used = k - k // 3
    recs.flags_rec.copy_(torch.from_numpy(flags))
    recs.reward_rec.copy_(torch.from_numpy(reward))
    recs.slot_rec.copy_(torch.from_numpy(slot))
    recs.qval.fill_(float("nan"))
    recs.meta[1] = used
    discounted_returns_records(eng, recs, gamma)
    want = np.full(k * n, np.nan, np.float32)
    q, total = np.zeros(n), 0
    for t in reversed(range(used)):
        on = (flags[t] & 1) == 1
        q = np.where(on, reward[t] + gamma * q, q)
        total += int(reward[t][on].sum())
        w = on & (slot[t] >= 0)
        want[slot[t][w]] = q[w].astype(np.float32)
    got = recs.qval.cpu().numpy()
    named = ~np.isnan(want)
    assert named.sum() > 0 and bool(np.isnan(got[~named]).all())
    assert bool((np.abs(got[named] - want[named]) <= np.spacing(np.abs(want[named]))).all())
    assert float(recs.reward_sum) == total


def test_training_cli_csv_checkpoint_resume_and_reload(tmp_path):
    """scripts/training.py equivalent (train.py main): writes <net>.csv (one row per batch) and <net>.pt; --resume continues
    the batch numbering, appends to the CSV, restores parameters + Adam state; the checkpoint loads as an opponent Agent."""
    import csv
    from azul_deep_reinforcement_learning_b200 import train
    from azul_deep_reinforcement_learning_b200.azulnet.agent import Agent
    name = str(tmp_path / "run1")
    train.main(["128", name, "--batches", "2", "--seed", "3"])
    rows = list(csv.DictReader(open(name + ".csv")))
    assert [int(r["batch"]) for r in rows] == [1, 2]
    for k in ("reward", "actor_loss", "critic_loss", "entropy_loss", "ac_loss", "player_score", "opponent_score", "rounds",
              "percent_first_player", "floor_penalty", "max_combo", "completed_rows", "completed_columns", "completed_colors",
              "win_percent"):                                        # agent.py:12 + game_runner.py:12 statistic names
        assert k in rows[0] and np.isfinite(float(rows[0][k])), k
    ck = torch.load(name + ".pt", map_location="cpu", weights_only=False)
    assert ck["batch"] == 2 and ck["optimizer"]["state"][0]["step"] == 2
    # resume: two more batches
    train.main(["128", name, "--batches", "4", "--seed", "3", "--resume", name + ".pt"])
    rows = list(csv.DictReader(open(name + ".csv")))
    assert [int(r["batch"]) for r in rows] == [1, 2, 3, 4]
    ck2 = torch.load(name + ".pt", map_location="cpu", weights_only=False)
    assert ck2["batch"] == 4 and ck2["optimizer"]["state"][0]["step"] == 4
    assert not torch.equal(ck["ac_net"]["actor_linear1.weight"], ck2["ac_net"]["actor_linear1.weight"])
    # a resumed trainer starts from exactly the saved parameters
    tr = train.SelfPlayTrainer(64, seed=3)
    assert tr.load_checkpoint(name + ".pt") == 4
    for k, v in tr.net.state_dict().items():
        assert torch.equal(v.cpu(), ck2["ac_net"][k])
    # ... and the checkpoint is a valid base_net / opponent (scripts/run_batch.py:6-8)
    a = Agent(base_net_file=name)
    assert torch.equal(a.ac_net.actor_linear2.bias, ck2["ac_net"]["actor_linear2.bias"])


def test_opponent_random_observation_for_3_and_4_players():
    """azb_opponent_random with the observation output for P = 3, 4 (shared-memory staging sized per player count)."""
    from azul_deep_reinforcement_learning_b200.engine import BatchedAzul
    for players in (3, 4):
        eng = BatchedAzul(1000, players, 1, 0, seed=players)
        eng.rollout_random(7)
        ps = torch.zeros(1000, dtype=torch.int16, device="cuda")
        out = eng.opponent_random(ps, require_two=True, want_obs=True)
        torch.cuda.synchronize()
        assert torch.equal(out["obs"].float(), eng.observe(0))
        rec = eng.export_records().cpu().numpy()
        L = UnpackedLayout(players)
        for i in range(0, 1000, 37):
            assert np.array_equal(O.observe(rec[i], players, 0), out["obs"][i].float().cpu().numpy().astype(np.int32))


def test_persistent_selfplay_rollout_equals_stepwise():
    """azb_policy_rollout (self-play, K decisions in one launch, state resident) == K launches of azb_policy_step with
    auto-reset: identical states and counters, for both pools and a ragged batch with several tiles per CTA."""
    from azul_deep_reinforcement_learning_b200.azulnet.model import ActorCritic
    from azul_deep_reinforcement_learning_b200.engine import BatchedAzul, PackedPolicy, policy_step
    torch.manual_seed(4)
    net = ActorCritic(136, 180)
    for pool, n in ((1, 148 * 128 * 2 + 77), (0, 1000)):
        a = BatchedAzul(n, 2, pool, 0, seed=13)
        b = BatchedAzul(n, 2, pool, 0, seed=13)
        pa, pb = PackedPolicy(a, net), PackedPolicy(b, net)
        K = 70                                                    # longer than a game: resets happen
        for _ in range(K):
            last = policy_step(a, pa, mode=0, apply_step=True, auto_reset=True, want_mask=False)
        got = b.policy_rollout(pb, K, want_last=True)
        torch.cuda.synchronize()
        assert torch.equal(a.state, b.state)
        assert torch.equal(a.counters, b.counters) and int(a.counters[1]) > 0
        assert torch.equal(last["action"], got["action"]) and torch.equal(last["logp"], got["logp"])


@pytest.mark.parametrize("n", [700, 148 * 128 + 333])
def test_persistent_runner_rollout_equals_episode_loop(n):
    """azb_policy_rollout (runner mode: agent decision + opponent loop + reward + record, whole episodes in one launch)
    reproduces run_episodes (one policy launch + one opponent launch per decision): per game the same actions, rewards,
    decision states and final state; discounted returns equal nn_runner.py:72-75 on those rewards.  The in-kernel opponent
    loop votes across the warp (one count_score + refill pass per warp), the step-wise launches run one game per thread:
    a ragged batch of one tile per CTA, and one with two tiles on some CTAs (two parts in the runner phase)."""
    from azul_deep_reinforcement_learning_b200.azulnet.model import ActorCritic
    from azul_deep_reinforcement_learning_b200.engine import PackedPolicy
    from azul_deep_reinforcement_learning_b200.selfplay import (BatchedGameRunner, PersistentEpisodes, discounted_returns,
                                                                 run_episodes)
    torch.manual_seed(6)
    net = ActorCritic(136, 180)
    a, b = BatchedGameRunner(n, seed=31), BatchedGameRunner(n, seed=31)
    pa, pb = PackedPolicy(a.engine, net), PackedPolicy(b.engine, net)
    eager = run_episodes(a, pa, max_decisions=160, record_obs=True)
    pers = PersistentEpisodes(b, pb, max_decisions=160, want_logp_value=True)
    r = pers.run(gamma=0.99)
    torch.cuda.synchronize()
    assert eager["unfinished"] == 0
    assert torch.equal(a.engine.state, b.engine.state) and torch.equal(a.player_score, b.player_score)
    act = eager["active"]                                         # [T, G]
    T = act.shape[0]
    n_dec, used = int(r.meta[0]), int(r.meta[1])
    assert n_dec == int(act.sum()) and used <= 160 and n_dec <= r.cap
    flags = r.flags_rec[:T]
    assert torch.equal((flags & 1).bool(), act) and int(r.flags_rec[T:].sum()) == 0
    slots = r.slot_rec[:T][act].long()
    assert int(slots.min()) >= 0 and len(torch.unique(slots)) == n_dec      # every decision owns one slot
    assert torch.equal(r.action_rec[slots].long(), eager["action"][act])
    assert torch.equal(r.reward_rec[:T][act].float(), eager["reward"][act])
    assert torch.equal(r.logp_rec[slots], eager["logp"][act]) and torch.equal(r.value_rec[slots], eager["value"][act])
    # the recorded states reproduce the recorded observations and masks
    obs = r.view.observe_bf16(-1)
    assert torch.equal(obs[slots], eager["obs"][act])
    mask = r.view.legal_mask()                                    # [6, cap]
    assert torch.equal(mask[:, slots], eager["mask"].permute(1, 0, 2)[:, act])
    # done flag: the last decision of every game
    done_t = ((flags >> 1) & 1).bool()
    assert int(done_t.sum()) == n and bool((done_t <= act).all())
    q = discounted_returns(eager["reward"], act, 0.99)
    assert torch.allclose(r.qval[slots], q[act], rtol=1e-6, atol=1e-5)
    assert abs(float(r.reward_sum) - float(eager["reward"][act].sum())) < 1e-6


def _autograd_reference(net, recs, n, coeffs):
    """fp32 torch autograd of train.a2c_loss_terms (pinned to the reference's Agent.update by tests/test_update_golden_cpu.py)
    on the first n decision records: gradient SUMS per parameter name, loss sums, logits, value."""
    from azul_deep_reinforcement_learning_b200.engine import mask_rows_to_bool
    from azul_deep_reinforcement_learning_b200.train import a2c_loss_terms
    obs = recs.view.observe(-1)[:n]
    rows = recs.view.legal_mask().t()[:n].contiguous()
    action, qval = recs.action_rec[:n].long(), recs.qval[:n]
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        net.zero_grad()
        a, c, e = a2c_loss_terms(net, obs, mask_rows_to_bool(rows), action, qval)
        (coeffs[0] * a + coeffs[1] * c + coeffs[2] * e).backward()
        with torch.no_grad():
            logits = net.actor_linear2(torch.relu(net.actor_linear1(obs)))
            value = net.forward_critic(obs).squeeze(1)
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev
    return {k: p.grad.clone() for k, p in net.named_parameters()}, torch.stack([a, c, e]).double().detach(), logits, value


@pytest.mark.parametrize("games,scale", [(300, 1.0), (1500, 2.5)])
def test_tensor_core_update_gradients_match_autograd(games, scale):
    """azb_a2c_update_gradients (forward recomputation, loss and the whole backward pass as tcgen05 GEMMs, fp16 operands /
    fp32 accumulation) against fp32 autograd of the reference's loss on the decision records of a real rollout:
    recomputed logits / value, the three loss sums and all eight parameter gradients; decision count read on the device."""
    from azul_deep_reinforcement_learning_b200.azulnet.model import ActorCritic
    from azul_deep_reinforcement_learning_b200.engine import PARAM_ORDER, PackedPolicy, UpdateGradients
    from azul_deep_reinforcement_learning_b200.selfplay import BatchedGameRunner, PersistentEpisodes
    torch.manual_seed(3)
    net = ActorCritic(136, 180).cuda()
    with torch.no_grad():
        for p in net.parameters():
            p.mul_(scale)
    gr = BatchedGameRunner(games, seed=8)
    packed = PackedPolicy(gr.engine, net)
    recs = PersistentEpisodes(gr, packed, max_decisions=160).run(gamma=0.99)
    n = int(recs.meta[0])
    assert 20 * games < n <= recs.cap
    coeffs = (1.0, 0.5, 0.1)
    want, want_sums, want_logits, want_value = _autograd_reference(net, recs, n, coeffs)
    upd = UpdateGradients(gr.engine, recs.cap)
    logits, value = upd.run(packed, recs.state_rec, recs.action_rec, recs.qval, n_dec=recs.meta[:1], coeffs=coeffs, want_outputs=True)
    torch.cuda.synchronize()
    # forward recomputation: same bound as the policy kernel (per element, floor = the row's largest |logit|)
    floor = want_logits.abs().max(dim=1, keepdim=True).values
    assert bool(((logits - want_logits).abs() <= 1e-3 * torch.maximum(want_logits.abs(), floor)).all())
    assert bool(((value - want_value).abs() <= 1e-3 * torch.maximum(want_value.abs(), want_value.abs().max())).all())
    assert float(((upd.sums - want_sums).abs() / want_sums.abs().clamp_min(1.0)).max()) < 2e-3
    # gradients: the critic and the actor's second layer to ~1e-3 of the tensor's largest entry; the actor's first layer
    # additionally sees hidden units whose pre-activation lies within the forward rounding error of zero switch their ReLU
    # derivative (each switch moves an entry by a whole term of the sum): a few per cent at 10^4 decisions, less with more
    for name in PARAM_ORDER:
        g, w = upd.grads[name].double(), want[name].double()
        err = float((g - w).abs().max())
        tol = 6e-2 if name.startswith("actor_linear1") else 1e-2
        assert err <= tol * float(w.abs().max()), (name, err, float(w.abs().max()))
        assert float((g * w).sum() / (g.norm() * w.norm())) > 0.9998, name
    # a second call without zeroing accumulates; n_fixed (host count) gives the same result as the device counter
    flat1 = upd.flat.clone()
    upd.run(packed, recs.state_rec, recs.action_rec, recs.qval, n_fixed=n, coeffs=coeffs, zero=False)
    torch.cuda.synchronize()
    assert float((upd.flat - 2 * flat1).abs().max()) <= 2e-3 * float(flat1.abs().max())


def test_tensor_core_update_in_chunks_equals_one_pass():
    """azb_a2c_update_gradients works through the records in workspace-sized chunks: 1,024-decision chunks give the same
    gradient sums (up to the order of the fp32 atomic additions) as one pass."""
    from azul_deep_reinforcement_learning_b200 import _lib
    from azul_deep_reinforcement_learning_b200.azulnet.model import ActorCritic
    from azul_deep_reinforcement_learning_b200.engine import PackedPolicy, UpdateGradients
    from azul_deep_reinforcement_learning_b200.selfplay import BatchedGameRunner, PersistentEpisodes
    torch.manual_seed(9)
    net = ActorCritic(136, 180).cuda()
    gr = BatchedGameRunner(300, seed=12)
    packed = PackedPolicy(gr.engine, net)
    recs = PersistentEpisodes(gr, packed, max_decisions=160).run(gamma=0.99)
    n = int(recs.meta[0])
    one = UpdateGradients(gr.engine, recs.cap)
    one.run(packed, recs.state_rec, recs.action_rec, recs.qval, n_dec=recs.meta[:1])
    lib = _lib.load()
    try:
        _lib.check(lib.azb_update_set_chunk_rows(1024))
        many = UpdateGradients(gr.engine, recs.cap)
        assert many.workspace.numel() < one.workspace.numel() // 8
        many.run(packed, recs.state_rec, recs.action_rec, recs.qval, n_dec=recs.meta[:1])
        fixed = UpdateGradients(gr.engine, recs.cap)
        fixed.run(packed, recs.state_rec, recs.action_rec, recs.qval, n_fixed=n)
        torch.cuda.synchronize()
    finally:
        _lib.check(lib.azb_update_set_chunk_rows(1 << 20))
    scale = float(one.flat.abs().max())
    assert n > 5 * 1024 and float((many.flat - one.flat).abs().max()) <= 1e-4 * scale
    assert float((fixed.flat - one.flat).abs().max()) <= 1e-4 * scale
    assert float(((many.sums - one.sums).abs() / one.sums.abs().clamp_min(1.0)).max()) < 1e-9
