"""Two-seat self-play in one persistent launch (azb_policy_rollout_selfplay, SelfPlayEpisodes): the persistent rollout against
a step-wise loop built from existing entry points, the zero-sum rewards, the argument checks, the tensor-core update on
both seats' decisions and the trainer with --self-play."""
import ctypes

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from azul_deep_reinforcement_learning_b200.layout import UnpackedLayout  # noqa: E402

pytestmark = pytest.mark.gpu

N_RAGGED = 148 * 128 * 2 + 333             # three tiles on some CTAs: several parts in the closing block
RULES = {1: {"first_player": "Random", "tile_pool": "Lid"}, 0: {"first_player": "Random", "tile_pool": "Random"}}


def _engine(n, pool, seed):
    from azul_deep_reinforcement_learning_b200.engine import BatchedAzul, rules_to_ints
    p, first = rules_to_ints(2, RULES[pool])
    return BatchedAzul(n, 2, p, first, seed=seed, reset=False)


def _popcount(mask):
    m = mask.to(torch.int64) & 0xFFFFFFFF
    return ((m.unsqueeze(-1) >> torch.arange(32, device=m.device)) & 1).sum(dim=(0, 2))


def _stepwise(eng, packed, mode, K):
    """The two-seat semantics, one policy_step(apply_step = 1, act_filter = 0) per iteration, with the seat and pending
    bookkeeping in torch: returns the per-(iteration, game) records, the recorded states' observation and mask (in record
    order: iteration, then game), the games that got stuck and the iterations run."""
    from azul_deep_reinforcement_learning_b200.engine import policy_step
    L = UnpackedLayout(2)
    n, dev = eng.n_games, eng.device
    eng.reset()
    score = torch.zeros((2, n), dtype=torch.int64, device=dev)
    pending = torch.full((2, n), -1, dtype=torch.int64, device=dev)
    flags = torch.zeros((K, n), dtype=torch.uint8, device=dev)
    reward = torch.zeros((K, n), dtype=torch.int64, device=dev)
    action = torch.full((K, n), 255, dtype=torch.int64, device=dev)
    logp = torch.zeros((K, n), dtype=torch.float32, device=dev)
    value = torch.zeros((K, n), dtype=torch.float32, device=dev)
    stuck = torch.zeros(n, dtype=torch.bool, device=dev)
    obs, masks = [], []
    cols = torch.arange(n, device=dev)
    used = 0
    for t in range(K):
        rec = eng.export_records()
        alive = (rec[:, L.end_of_game] == 0) & ~stuck
        if not bool(alive.any()):
            break
        used = t + 1
        mask = eng.legal_mask()
        seat2 = rec[:, L.current_player] != 1
        decides = (_popcount(mask) >= 2) & alive
        obs.append(eng.observe_bf16(-1)[decides])
        masks.append(mask[:, decides])
        out = policy_step(eng, packed, mode=mode, apply_step=True, want_mask=False, act_filter=0)
        flags[t] = decides.to(torch.uint8) | ((decides & seat2).to(torch.uint8) << 2)
        action[t] = torch.where(decides, out["action"].long(), action[t])
        logp[t] = torch.where(decides, out["logp"], logp[t])
        value[t] = torch.where(decides, out["value"], value[t])
        for s in (0, 1):
            sel = decides & (seat2 == bool(s))
            pending[s] = torch.where(sel, t, pending[s])
        # closing: after the move and the round's end
        rec = eng.export_records()
        over = rec[:, L.end_of_game] != 0
        nv = _popcount(eng.legal_mask())
        stuck |= ~over & (nv == 0)
        every = over | stuck
        prev = eng.score_preview().long()
        d1 = prev[0] - prev[1]
        mover2 = rec[:, L.current_player] != 1
        for s in (0, 1):
            d = d1 if s == 0 else -d1
            close = (every | ((mover2 == bool(s)) & (nv >= 2))) & (pending[s] >= 0)
            tt, gg = pending[s][close], cols[close]
            reward[tt, gg] = d[close] - score[s][close]
            flags[tt, gg] |= (over[close].to(torch.uint8) << 1)
            score[s] = torch.where(close, d, score[s])
            pending[s] = torch.where(close, -1, pending[s])
    return {"flags": flags, "reward": reward, "action": action, "logp": logp, "value": value, "score": score,
            "obs": torch.cat(obs), "mask": torch.cat(masks, dim=1), "stuck": stuck, "used": used}


@pytest.mark.parametrize("n", [700, N_RAGGED])
@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("pool", [1, 0])
def test_selfplay_rollout_equals_stepwise(pool, mode, n):
    """SelfPlayEpisodes == the step-wise loop, per game: actions, seats, rewards, logp / value records, recorded states
    (observation and mask), flags, final state and player_score bit for bit; the returns within the runner-mode tolerance
    of the host per-seat returns."""
    from azul_deep_reinforcement_learning_b200.azulnet.model import ActorCritic
    from azul_deep_reinforcement_learning_b200.engine import PackedPolicy
    from azul_deep_reinforcement_learning_b200.selfplay import SelfPlayEpisodes, discounted_returns_two_seat
    seed = 80 + 2 * pool + mode
    torch.manual_seed(seed)
    net = ActorCritic(136, 180)
    a, b = _engine(n, pool, 41 + seed), _engine(n, pool, 41 + seed)
    pa, pb = PackedPolicy(a, net), PackedPolicy(b, net)
    K = 320
    ref = _stepwise(a, pa, mode, K)
    sp = SelfPlayEpisodes(b, pb, max_decisions=K, want_logp_value=True)
    r = sp.run(gamma=0.99, mode=mode)
    torch.cuda.synchronize()
    # the kernel marks a stuck game in its state (AZB_ST_STUCK); the step-wise loop cannot, so those games compare without it
    state = b.state.clone()
    st = ref["stuck"]
    assert bool(((state[3, st] >> 13) & 1).all())
    state[3, st] = a.state[3, st]
    assert torch.equal(state, a.state)
    assert torch.equal(sp.player_score.long(), ref["score"])
    n_dec, used = int(r.meta[0]), int(r.meta[1])
    assert used == ref["used"] and n_dec <= r.cap
    T = used
    flags = ref["flags"][:T]
    act = (flags & 1).bool()
    assert n_dec == int(act.sum())
    assert torch.equal(r.flags_rec[:T], flags) and int(r.flags_rec[T:].sum()) == 0
    assert bool(((flags >> 2) & 1).bool().any()) and bool((((flags >> 2) & 1) == 0)[act].any())
    assert torch.equal(r.reward_rec[:T][act].long(), ref["reward"][:T][act])
    slots = r.slot_rec[:T][act].long()
    assert int(slots.min()) >= 0 and len(torch.unique(slots)) == n_dec
    assert torch.equal(r.action_rec[slots].long(), ref["action"][:T][act])
    assert torch.equal(r.logp_rec[slots], ref["logp"][:T][act]) and torch.equal(r.value_rec[slots], ref["value"][:T][act])
    # records in the reference's order (iteration, then game) = the boolean index order of act
    assert torch.equal(r.view.observe_bf16(-1)[slots], ref["obs"])
    assert torch.equal(r.view.legal_mask()[:, slots], ref["mask"])
    unfinished = int((a.export_records()[:, UnpackedLayout(2).end_of_game] == 0).sum())
    assert unfinished == 0 or mode == 1
    q = discounted_returns_two_seat(ref["reward"][:T].double(), flags, 0.99).float()
    assert torch.allclose(r.qval[slots], q[act], rtol=1e-6, atol=1e-5)


def test_selfplay_rewards_are_zero_sum():
    """At a size where CTAs own two or more tiles: per finished episode seat s's rewards sum to d_s of the final state (its
    score preview minus the other seat's), the two sums negate each other, and reward_sum is 0 when nothing is unfinished."""
    from azul_deep_reinforcement_learning_b200.azulnet.model import ActorCritic
    from azul_deep_reinforcement_learning_b200.engine import PackedPolicy
    from azul_deep_reinforcement_learning_b200.selfplay import SelfPlayEpisodes
    n = 148 * 128 * 3 + 77
    torch.manual_seed(5)
    eng = _engine(n, 1, 9)
    sp = SelfPlayEpisodes(eng, PackedPolicy(eng, ActorCritic(136, 180)))
    r = sp.run(gamma=0.99, mode=0)
    torch.cuda.synchronize()
    T = int(r.meta[1])
    f = r.flags_rec[:T]
    rw = r.reward_rec[:T].long() * (f & 1).long()
    seat2 = ((f >> 2) & 1).bool()
    s1, s2 = (rw * ~seat2).sum(0), (rw * seat2).sum(0)
    prev = eng.score_preview().long()
    d1 = prev[0] - prev[1]
    ended = eng.export_records()[:, UnpackedLayout(2).end_of_game] != 0
    assert int(ended.sum()) == n
    assert torch.equal(s1, d1) and torch.equal(s2, -d1) and torch.equal(s1, -s2)
    assert torch.equal(sp.player_score[0].long(), d1) and torch.equal(sp.player_score[1].long(), -d1)
    assert float(r.reward_sum[0]) == 0.0
    # the last decision of every finished episode carries the game-over bit, for both seats
    last = (f & 2).bool()
    assert bool((last.sum(0) == 2).all())
    per_game = int(r.meta[0]) / n
    assert 30 < per_game < 200, per_game


def test_selfplay_rejects_bad_arguments():
    """A 3-player handle, mode 2, k_decisions 0 and null record buffers are each refused before any launch."""
    from azul_deep_reinforcement_learning_b200.azulnet.model import ActorCritic
    from azul_deep_reinforcement_learning_b200.engine import BatchedAzul, EpisodeRecords, PackedPolicy, _ptr
    net = ActorCritic(136, 180)
    helper = BatchedAzul(256, 2, 1, 0, seed=1)
    p = PackedPolicy(helper, net)
    r = EpisodeRecords(helper, 4)
    ps = torch.zeros((2, 256), dtype=torch.int16, device="cuda")
    pend = torch.zeros((2, 256), dtype=torch.int32, device="cuda")
    three = BatchedAzul(256, 3, 1, 0, seed=1)

    def call(e, mode=0, k=4, state_rec=True, flags_rec=True, pending=True):
        return e.lib.azb_policy_rollout_selfplay(
            e._h, _ptr(e.state), _ptr(p.buf), mode, k, _ptr(ps), _ptr(pend) if pending else None, _ptr(r.meta), r.cap,
            _ptr(r.state_rec) if state_rec else None, _ptr(r.action_rec), None, None, _ptr(r.slot_rec), _ptr(r.reward_rec),
            _ptr(r.flags_rec) if flags_rec else None, ctypes.c_void_p(r.meta.data_ptr() + 4), None, None, None,
            e._stream())

    before = helper.state.clone()
    for rc in (call(three), call(helper, mode=2), call(helper, k=0), call(helper, state_rec=False),
               call(helper, flags_rec=False), call(helper, pending=False)):
        assert rc == -1                                                   # AZB_E_INVALID
    torch.cuda.synchronize()
    assert torch.equal(helper.state, before) and int(r.meta[0]) == 0


def test_tensor_core_update_on_two_seat_records():
    """azb_a2c_update_gradients on a two-seat batch (seat 2's decisions included) against fp32 autograd of the reference's
    loss on observations rebuilt from the records, from the mover's perspective."""
    from azul_deep_reinforcement_learning_b200.azulnet.model import ActorCritic
    from azul_deep_reinforcement_learning_b200.engine import PARAM_ORDER, PackedPolicy, UpdateGradients, mask_rows_to_bool
    from azul_deep_reinforcement_learning_b200.selfplay import SelfPlayEpisodes
    from azul_deep_reinforcement_learning_b200.train import a2c_loss_terms
    torch.manual_seed(6)
    net = ActorCritic(136, 180).cuda()
    eng = _engine(600, 1, 13)
    packed = PackedPolicy(eng, net)
    r = SelfPlayEpisodes(eng, packed).run(gamma=0.99)
    n = int(r.meta[0])
    T = int(r.meta[1])
    assert int(((r.flags_rec[:T] & 5) == 5).sum()) > 10 * 600          # plenty of seat-2 decisions
    coeffs = (1.0, 0.5, 0.1)
    obs = r.view.observe_bf16(-1)[:n].float()
    rows = r.view.legal_mask()[:, :n].t().contiguous()
    action, qval = r.action_rec[:n].long(), r.qval[:n]
    net.zero_grad()
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        a, c, e = a2c_loss_terms(net, obs, mask_rows_to_bool(rows), action, qval)
        (coeffs[0] * a + coeffs[1] * c + coeffs[2] * e).backward()
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev
    want = {k: p.grad.clone() for k, p in net.named_parameters()}
    upd = UpdateGradients(eng, r.cap)
    upd.run(packed, r.state_rec, r.action_rec, r.qval, n_dec=r.meta[:1], coeffs=coeffs)
    torch.cuda.synchronize()
    want_sums = torch.stack([a, c, e]).double().detach()
    assert float(((upd.sums - want_sums).abs() / want_sums.abs().clamp_min(1.0)).max()) < 2e-3
    for name in PARAM_ORDER:
        g, w = upd.grads[name].double(), want[name].double()
        assert float((g * w).sum() / (g.norm() * w.norm())) > 0.999, name


def test_trainer_self_play():
    """SelfPlayTrainer(self_play=True) trains through the captured batch graph (batch 3 is its replay); with eval_every=2
    the evaluation columns are filled on the evaluated rows and blank elsewhere."""
    from azul_deep_reinforcement_learning_b200.selfplay import SelfPlayEpisodes
    from azul_deep_reinforcement_learning_b200.train import EVAL_FIELDS, SelfPlayTrainer
    tr = SelfPlayTrainer(512, seed=4, self_play=True)
    assert isinstance(tr.episodes, SelfPlayEpisodes) and tr.runner.opponent is None
    hist = tr.train(batches=3, log=None, eval_every=2, eval_games=256)
    assert tr._graph is not None
    assert len(hist) == 3 and all(np.isfinite(h["ac_loss"]) for h in hist)
    assert all(h["games"] == 512 and h["unfinished"] == 0 and h["reward"] == 0.0 for h in hist)
    assert all(h["transitions"] > 512 * 30 for h in hist)
    for h in hist:
        filled = h["batch"] % 2 == 0
        for k in EVAL_FIELDS:
            assert (h[k] is not None) == filled, (h["batch"], k)
    ev = hist[1]
    assert 0.0 <= ev["eval_win_percent"] <= 1.0 and ev["eval_opponent_score"] > 0
