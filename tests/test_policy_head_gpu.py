"""The output head of the fused policy kernel -- masked softmax, inverse-CDF sampling with one Philox word, argmax, log pi,
entropy and the move it plays -- against a float64 reference of the same operations, at designed logits.

The actor's second layer has weight 0 and bias v, so every game gets the logits v (as fp16 hi + lo bias inputs) whatever its
state; the legal masks come from real states (random rollouts, both tile pools, a ragged batch).  The reference is fed the
logits the kernel reports, so this isolates the head from the MLP, whose rounding tests/test_policy_gpu.py covers.  The
draw of a game is reproduced from its Philox word: counter (game_id_base + g, steps >> 2, PURPOSE_POLICY = 4, 0), key
(seed_lo, seed_hi), word steps & 3, u = (word >> 8) / 2^24, where steps is the record's total_steps (packed word 6, which
is what k_policy reads as gm.steps)."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

pytestmark = pytest.mark.gpu

N = 65536 + 77                      # ragged: the last tile holds 77 games
SEED = 0x1234_5678_9ABC
LOG2E = 1.4426950408889634
EPS = 2.0 ** -24                    # fp32 unit roundoff


# ---- the states, the network with designed logits and one launch -------------------------------------------------------
def _engine(pool, depth, seed=SEED):
    from azul_deep_reinforcement_learning_b200.engine import BatchedAzul
    eng = BatchedAzul(N, 2, pool, 0, seed=seed, game_id_base=1000 * depth)
    eng.rollout_random(depth)       # auto-reset: games at every stage of a round and of a game
    return eng


def _net(bias):
    from azul_deep_reinforcement_learning_b200.azulnet.model import ActorCritic
    torch.manual_seed(0)
    net = ActorCritic(136, 180)
    with torch.no_grad():
        net.actor_linear2.weight.zero_()
        net.actor_linear2.bias.copy_(torch.as_tensor(np.asarray(bias, dtype=np.float32)))
    return net


def _launch(eng, net, mode, apply_step=False):
    from azul_deep_reinforcement_learning_b200.engine import PackedPolicy, mask_to_bool, policy_step
    with torch.no_grad():
        out = policy_step(eng, PackedPolicy(eng, net), mode=mode, apply_step=apply_step, want_logits=True)
        torch.cuda.synchronize()
    r = {k: out[k].cpu().numpy() for k in ("action", "logp", "entropy", "status")}
    r["mask"] = mask_to_bool(out["mask"]).cpu().numpy()
    r["logits"] = out["logits"].cpu().numpy()
    r["action"] = r["action"].astype(np.int64)
    return r


# ---- Philox4x32-10 (oracle/azul_oracle.c ao_philox4x32_10), vectorised over games -------------------------------------
def _philox(c0, c1, c2, c3, k0, k1):
    M32 = np.uint64(0xFFFFFFFF)
    c = [np.asarray(x, dtype=np.uint64) & M32 for x in (c0, c1, c2, c3)]
    k0, k1 = np.uint64(k0), np.uint64(k1)
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c[0]
        p1 = np.uint64(0xCD9E8D57) * c[2]
        c = [((p1 >> np.uint64(32)) ^ c[1] ^ k0) & M32, p1 & M32, ((p0 >> np.uint64(32)) ^ c[3] ^ k1) & M32, p0 & M32]
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & M32, (k1 + np.uint64(0xBB67AE85)) & M32
    return np.stack(c, axis=1)


def _sampling_words(eng):
    """Each game's sampling word for the engine's current states; the game's step count is read from its record."""
    from azul_deep_reinforcement_learning_b200.layout import UnpackedLayout
    steps = eng.export_records()[:, UnpackedLayout(2).total_steps].cpu().numpy().astype(np.uint64)
    assert np.array_equal(steps, eng.state[6].cpu().numpy().astype(np.uint32).astype(np.uint64))   # packed word 6 = STEPS
    gid = np.arange(eng.n_games, dtype=np.uint64) + np.uint64(eng.game_id_base)
    w = _philox(gid, steps >> np.uint64(2), np.full_like(gid, 4), np.zeros_like(gid), eng.seed & 0xFFFFFFFF, eng.seed >> 32)
    return w[np.arange(eng.n_games), (steps & np.uint64(3)).astype(np.int64)].astype(np.uint32)


def test_philox_matches_oracle():
    from oracle import oracle as O
    rng = np.random.default_rng(3)
    ctr = rng.integers(0, 2 ** 32, size=(16, 4), dtype=np.uint64)
    key = rng.integers(0, 2 ** 32, size=2, dtype=np.uint64)
    got = _philox(ctr[:, 0], ctr[:, 1], ctr[:, 2], ctr[:, 3], int(key[0]), int(key[1]))
    for i in range(16):
        assert np.array_equal(got[i].astype(np.uint32), O.philox4x32_10(ctr[i].astype(np.uint32), key.astype(np.uint32)))


# ---- the float64 reference of the head ----------------------------------------------------------------------------------
def _reference(logits, mask, words):
    """float64: masked log_softmax, entropy -mean(logp over legal), argmax (lowest legal index among the maxima), the
    inverse-CDF draw of u = (word >> 8) / 2^24 (the first action whose cumulative probability exceeds u) and the distance of
    u to the nearest CDF boundary."""
    l = np.where(mask, logits.astype(np.float64), -np.inf)
    n = mask.sum(axis=1)
    has = n > 0
    mx = np.where(has, l.max(axis=1), 0.0)
    with np.errstate(invalid="ignore", divide="ignore"):
        lse = mx + np.log(np.exp(l - mx[:, None]).sum(axis=1))
        logp = l - lse[:, None]
        p = np.where(mask, np.exp(logp), 0.0)
    ent = -np.where(mask, logp, 0.0).sum(axis=1) / np.maximum(n, 1)
    cdf = np.cumsum(p, axis=1)
    cdf /= np.where(has, cdf[:, -1], 1.0)[:, None]
    u = (words >> 8).astype(np.float64) / 2.0 ** 24
    sample = (cdf <= u[:, None]).sum(axis=1)                 # = first index with cdf > u (illegal columns repeat a value)
    dist = np.where(mask, np.abs(cdf - u[:, None]), np.inf).min(axis=1)
    spread = np.where(mask, mx[:, None] - l, 0.0).max(axis=1)
    return {"logp": logp, "p": p, "entropy": ent, "argmax": np.argmax(l, axis=1), "sample": sample, "dist": dist,
            "n": n, "max": np.where(has, np.abs(l).max(axis=1, where=mask, initial=0.0), 0.0), "spread": spread}


def _band(ref):
    """Half-width of the band around a CDF boundary inside which the kernel's fp32 draw may differ from the float64 one.

    The kernel forms each legal weight as 2^x with x = fma(l, log2e, -fl(m log2e)) for the running maximum m of its 16-column
    chunk, and rescales chunk sums and part sums by 2^((m' - m) log2e) with exact differences of two maxima.  Per weight, x is
    off by the residual of fl(m log2e) (<= M log2e 2^-24 for M = max |legal logit|; weights of different chunks carry
    different residuals, so at most twice that between two weights), and by the roundings of the fma, of the rescale
    arguments and of fp32 log2e itself (<= S log2e 2^-24 each for S = the row's logit spread, four of them); ex2.approx adds
    2 ulp per exponential (two on any path).  As 2^x has relative error ln2 dx, and ln2 log2e = 1, a weight is off by at most
    (2 M + 4 S + 8) 2^-24 relative, and a normalised CDF value by twice that.  The fp32 sums along the three-level scan (part
    prefix, chunk, 16 columns: <= 24 additions) and the product u gse add <= 26 2^-24.  The band takes that sum,
    (4 M + 8 S + 42) 2^-24, times 2 as margin.  Spreads beyond 104 nats do not matter: those weights are below 2^-150 of the
    largest and flush to 0 in fp32 whatever their error."""
    return 2.0 * EPS * (4.0 * ref["max"] + 8.0 * np.minimum(ref["spread"], 104.0) + 42.0)


def _random_logits(rng, scale=10.0, clip=30.0):
    """|v| <= 30 with illegal-heavy and empty parts: part 2 holds the largest logits, one chunk of part 1 sits far below."""
    v = np.clip(rng.normal(0.0, scale, 180), -clip, clip).astype(np.float32)
    v[96:144] = np.clip(v[96:144] + 15.0, -clip, clip)
    v[64:80] -= 25.0
    return np.clip(v, -clip, clip).astype(np.float32)


@pytest.fixture(scope="module")
def sampled():
    """Sampling mode: four logit vectors, each over the states of one (pool, depth)."""
    rng = np.random.default_rng(11)
    runs = []
    for pool, depth in ((0, 3), (1, 17), (0, 41), (1, 90)):
        eng = _engine(pool, depth)
        words = _sampling_words(eng)
        v = _random_logits(rng)
        out = _launch(eng, _net(v), mode=0)
        runs.append((out, words, _reference(out["logits"], out["mask"], words)))
    return runs


def _check_draws(out, ref, label, max_share=0.01):
    """The kernel's draw is the reference draw for every game with u outside the band; returns the games inside."""
    has = ref["n"] > 0
    band = _band(ref)
    inside = has & (ref["dist"] <= band)
    bad = has & ~inside & (out["action"] != ref["sample"])
    assert not bad.any(), (label, np.flatnonzero(bad)[:8], out["action"][bad][:8], ref["sample"][bad][:8],
                           (ref["dist"] / band)[bad][:8])
    assert inside.sum() <= max_share * has.sum(), (label, int(inside.sum()), int(has.sum()))
    assert (out["action"][~has] == 255).all()
    return inside


def test_sampled_draw_logp_entropy(sampled):
    for i, (out, words, ref) in enumerate(sampled):
        has = ref["n"] > 0
        assert has.mean() > 0.9
        # the logits are v in every game (fp16 hi + lo of the bias: within 2^-20 relative)
        assert np.allclose(out["logits"], out["logits"][0], rtol=0, atol=0)
        _check_draws(out, ref, i)
        a = out["action"][has]
        assert out["mask"][has, a].all() and (ref["p"][has, a] > 0).all()
        want = ref["logp"][has, a]
        tol = 2e-6 * (8.0 + ref["max"][has] + ref["spread"][has])
        assert (np.abs(out["logp"][has] - want) <= tol).all(), np.abs(out["logp"][has] - want).max()
        assert (np.abs(out["entropy"][has] - ref["entropy"][has]) <= tol).all()
        assert (out["status"] & 1 == 0).all()


def test_single_legal_action(sampled):
    """One legal action: it is drawn, and log pi and entropy are 0 within the rounding of logit -> weight -> log."""
    seen = 0
    for out, words, ref in sampled:
        one = ref["n"] == 1
        seen += int(one.sum())
        only = np.argmax(out["mask"][one], axis=1)
        assert np.array_equal(out["action"][one], only)
        tol = 8.0 * EPS * (16.0 + ref["max"][one])
        assert (np.abs(out["logp"][one]) <= tol).all(), np.abs(out["logp"][one]).max()
        assert (np.abs(out["entropy"][one]) <= tol).all(), np.abs(out["entropy"][one]).max()
    assert seen >= 100, seen


TIES = [(15, 16), (47, 48), (95, 96), (143, 144), (40, 150), (15, 16, 47, 48, 95, 96, 143, 144)]


@pytest.mark.parametrize("pool", [0, 1])
def test_argmax_ties_pick_lowest_legal_index(pool):
    """Equal maximal logits across chunk (15 / 16) and part (47 / 48, 95 / 96, 143 / 144) boundaries and across parts: argmax
    mode plays the lowest legal index among them (np.argmax, azulnet/agent.py); log pi and entropy as the reference."""
    rng = np.random.default_rng(5 + pool)
    eng = _engine(pool, 23 if pool else 7)
    for tie in TIES:
        v = rng.uniform(-6.0, 2.0, 180).astype(np.float32)
        v[list(tie)] = 5.0                                     # exact in fp16: hi = 5, lo = 0, the same fp32 logit
        out = _launch(eng, _net(v), mode=1)
        ref = _reference(out["logits"], out["mask"], np.zeros(N, np.uint32))
        has = ref["n"] > 0
        assert (out["logits"][:, list(tie)] == 5.0).all()
        assert np.array_equal(out["action"][has], ref["argmax"][has]), tie
        legal = out["mask"][:, list(tie)]
        # non-vacuous: games where the lower index of a tie is legal and where only a higher one is
        assert (legal[:, 0] & legal[:, 1:].any(axis=1)).sum() >= 20, tie
        assert (~legal[:, 0] & legal[:, 1:].any(axis=1)).sum() >= 20, tie
        a = out["action"][has]
        assert (np.abs(out["logp"][has] - ref["logp"][has, a]) <= 5e-5).all()
        assert (np.abs(out["entropy"][has] - ref["entropy"][has]) <= 5e-5).all()


# ---- extreme spreads and offsets -----------------------------------------------------------------------------------------
def _spread_logits(rng, offset):
    """Chunk 0 of every part within 3 nats of ``offset``; the part's two other chunks 100..120 nats below it."""
    v = np.empty(192, np.float64)
    for q in range(4):
        v[48 * q:48 * q + 16] = offset + rng.uniform(0.0, 3.0, 16)
        v[48 * q + 16:48 * q + 48] = offset - 100.0 - rng.uniform(0.0, 20.0, 32)
    return v[:180].astype(np.float32)


def _ex2(x):
    """ex2.approx.ftz on the host: 2^x rounded to fp32, results below 2^-126 flushed to 0."""
    with np.errstate(over="ignore", invalid="ignore"):
        y = np.exp2(x.astype(np.float64)).astype(np.float32)
    return np.where(np.abs(y) < np.float32(2.0 ** -126), np.float32(0.0), y)


def _fma(a, b, c):
    """fmaf for fp32 operands (the product is exact in float64; the sum is rounded twice, which may differ in the last bit)"""
    return (np.asarray(a, np.float64) * np.asarray(b, np.float64) + np.asarray(c, np.float64)).astype(np.float32)


def former_sampling(logits, mask, words):
    """The sampling step as k_policy did it before part and chunk weights were formed alike (azb_policy.cu, epilogues 2a and
    2b), restated in fp32: the part weights wq from exact differences of maxima, the chunk weights from
    fma(chunk max, log2e, -fl(gmx log2e)).  Their sums disagree by up to ~1e-4 of a part's weight at |gmx| ~ 1e4, and at
    gmx < -88.7 a chunk before the part's first legal action got weight 0 * inf = NaN.  A target in such a gap fell back
    to the part's last LEGAL chunk; when that chunk's weights had all underflowed, no action was chosen and the move was
    action 0.  Returns the action that arithmetic picks per game (-1: none, i.e. action 0 was played)."""
    f32 = np.float32
    L2E = f32(LOG2E)
    n = len(words)
    lg = np.full((n, 192), -np.inf, f32)
    lg[:, :180] = np.where(mask, logits, -np.inf)
    lg = lg.reshape(n, 4, 3, 16)
    bits = np.zeros((n, 192), bool)
    bits[:, :180] = mask
    bits = bits.reshape(n, 4, 3, 16)
    with np.errstate(all="ignore"):
        mx = np.full((n, 4), -np.inf, f32)
        se = np.zeros((n, 4), f32)
        cs = np.zeros((n, 4, 3), f32)
        cms = np.zeros((n, 4, 3), f32)
        vs = np.zeros((n, 4, 3, 16), f32)
        for c in range(3):
            nm = np.maximum(mx, lg[:, :, c].max(axis=-1))
            ms = np.where(nm == -np.inf, f32(0), nm).astype(f32)
            ms2 = (ms * L2E).astype(f32)
            vs[:, :, c] = _ex2(_fma(lg[:, :, c], L2E, -ms2[..., None]))
            s = np.zeros((n, 4), f32)
            for i in range(16):
                s = (s + vs[:, :, c, i]).astype(f32)
            se = ((se * _ex2(_fma(mx, L2E, -ms2))).astype(f32) + s).astype(f32)
            cs[:, :, c], cms[:, :, c] = s, ms
            mx = nm
        npart = bits.reshape(n, 4, 48).sum(axis=-1)
        gmx = np.where(npart > 0, mx, -np.inf).max(axis=1).astype(f32)
        wq = np.where(npart > 0, (se * _ex2(((mx - gmx[:, None]).astype(f32) * L2E).astype(f32))).astype(f32), f32(0))
        gse = np.zeros(n, f32)
        run = np.zeros((n, 4), f32)
        for q in range(4):
            gse = (gse + wq[:, q]).astype(f32)
            run[:, q] = gse
        target = (((words >> 8).astype(f32) * f32(1.0 / 16777216.0)).astype(f32) * gse).astype(f32)
        hit = target[:, None] < run
        last = 3 - np.argmax((npart > 0)[:, ::-1], axis=1)
        owner = np.where(hit.any(axis=1), np.argmax(hit, axis=1), last)
        rows = np.arange(n)
        prefix = np.where(owner > 0, run[rows, np.maximum(owner - 1, 0)], f32(0)).astype(f32)
        gm2 = (gmx * L2E).astype(f32)
        sc = _ex2(_fma(cms[rows, owner], L2E, -gm2[:, None]))
        wc = (cs[rows, owner] * sc).astype(f32)
        k = np.full(n, -1)
        acc = prefix.copy()
        base = prefix.copy()
        for c in range(3):
            nacc = (acc + wc[:, c]).astype(f32)
            h = (k < 0) & (target < nacc)
            base = np.where(h, acc, base)
            k = np.where(h, c, k)
            acc = nacc
        ob = bits[rows, owner]
        fall = k < 0
        kf = np.where(ob[:, 2].any(axis=-1), 2, np.where(ob[:, 1].any(axis=-1), 1, 0))
        fb = (((prefix + np.where(kf > 0, wc[:, 0], f32(0))).astype(f32) + np.where(kf > 1, wc[:, 1], f32(0)))).astype(f32)
        base = np.where(fall, fb, base)
        k = np.where(fall, kf, k)
        sk = sc[rows, k]
        v = vs[rows, owner, k]
        cum = base
        chosen = np.full(n, -1)
        for i in range(16):
            upd = (v[:, i] > 0) & (cum <= target)
            chosen = np.where(upd, i, chosen)
            cum = _fma(v[:, i], sk, cum)
    return np.where(chosen >= 0, 48 * owner + 16 * k + chosen, -1)


OFFSETS = [0.0, 50.0, 1000.0, 10000.0, -1000.0]
FRACTIONS = np.linspace(0.0, 1.0, 6, endpoint=False)


@pytest.mark.parametrize("pool", [0, 1])
def test_extreme_spread_and_offset(pool):
    """Chunk 0 of each part >= 100 nats above the part's other chunks, at offsets 0, 50, 1e3, 1e4 and -1e3 (with fractional
    offsets): every played action is legal and has float64 probability > 1e-30, no status reports an illegal move, log pi
    matches float64 within a tolerance that grows with the offset, and the fused step equals azb_step on the reported
    actions.  The batch is not vacuous: the former fp32 arithmetic of the sampling step (``former_sampling``) chooses no
    action -- and so played action 0 -- in some of its games."""
    from azul_deep_reinforcement_learning_b200.engine import BatchedAzul
    rng = np.random.default_rng(17 + pool)
    eng = _engine(pool, 29)
    s0 = eng.state.clone()
    twin = BatchedAzul(N, 2, pool, 0, seed=eng.seed, game_id_base=eng.game_id_base, reset=False)
    words = _sampling_words(eng)
    former_none = 0
    for off in OFFSETS:
        for frac in FRACTIONS:
            v = _spread_logits(rng, off + frac)
            eng.state.copy_(s0)
            out = _launch(eng, _net(v), mode=0, apply_step=True)
            ref = _reference(out["logits"], out["mask"], words)
            has = ref["n"] > 0
            a = out["action"]
            label = (off, float(frac))
            assert out["mask"][has, a[has]].all(), (label, np.flatnonzero(has & ~out["mask"][np.arange(N), np.minimum(a, 179)])[:8])
            assert (ref["p"][has, a[has]] > 1e-30).all(), (label, ref["p"][has, a[has]].min())
            assert (out["status"] & 1 == 0).all(), label
            tol = 1e-3 + 8.0 * EPS * abs(off)
            err = np.abs(out["logp"][has] - ref["logp"][has, a[has]])
            assert (err <= tol).all(), (label, err.max(), tol)
            # (the band is wide here, 5e-3 at 1e4, and the few heavy actions of chunk 0 share it: the share is not bounded)
            _check_draws(out, ref, label, max_share=1.0)
            twin.state.copy_(s0)
            st = twin.step(torch.as_tensor(a.astype(np.uint8)), None, want_mask=False)
            assert int((st["status"] & 1).sum()) == 0, label
            assert torch.equal(twin.state, eng.state), label
            old = former_sampling(out["logits"], out["mask"], words)
            none = has & (old < 0)
            former_none += int(none.sum())
    assert former_none >= 5, former_none


@pytest.mark.parametrize("c", [64.0, 1024.0, -1024.0])
def test_offset_invariance(c):
    """v and v + c draw the same actions outside the band of v + c (log-softmax is shift invariant)."""
    rng = np.random.default_rng(23)
    eng = _engine(1, 17)
    words = _sampling_words(eng)
    v = _random_logits(rng)
    base = _launch(eng, _net(v), mode=0)
    shifted = _launch(eng, _net(v + np.float32(c)), mode=0)
    ref = _reference(shifted["logits"], shifted["mask"], words)
    inside = _check_draws(shifted, ref, c, max_share=0.05)
    ref0 = _reference(base["logits"], base["mask"], words)
    inside |= ref0["dist"] <= _band(ref0)
    has = ref["n"] > 0
    assert np.array_equal(base["action"][has & ~inside], shifted["action"][has & ~inside])


# ---- parameters beyond the fp16 range --------------------------------------------------------------------------------------
def test_parameters_beyond_fp16_follow_the_rounding_spec():
    """Biases at +-7e4 and +-1e6 (b2a, b1a, b1c), weights at +-7e4 (W2a, W1a) and a hidden unit driven into saturation by its
    bias alone (W1a row 0): logits and value equal torch_forward(emulate_f16=True) -- weights clamp to +-65504, a bias enters
    as fp16 hi = half(clamp(b)) plus lo = half(clamp(b - hi)), the actor's hidden units saturate at 65504."""
    from azul_deep_reinforcement_learning_b200.azulnet.model import ActorCritic
    from tests.helpers import torch_forward
    torch.manual_seed(2)
    net = ActorCritic(136, 180)
    big = torch.tensor([7e4, -7e4, 1e6, -1e6])
    with torch.no_grad():
        net.actor_linear2.bias[[0, 50, 100, 170]] = big
        net.actor_linear1.bias[[1, 2, 3, 4]] = big
        net.critic_linear1.bias[[5, 6, 7, 8]] = big
        net.actor_linear2.weight[10, 20] = 7e4
        net.actor_linear2.weight[11, 21] = -7e4
        net.actor_linear1.weight[20, 3] = 7e4
        net.actor_linear1.weight[21, 40] = -7e4
        net.actor_linear1.weight[0].zero_()
        net.actor_linear1.bias[0] = 7e4
    eng = _engine(1, 31)
    out = _launch(eng, net, mode=1)
    ref = torch_forward(net, eng.observe(-1), emulate_f16=True)
    assert float(ref["ha"][:, 0].min()) == 65504.0                              # unit 0 saturated in every game
    assert float(ref["ha"][:, 1].min()) == 65504.0 and float(ref["ha"][:, 3].min()) == 65504.0
    # per element: fp32 accumulation of the products and the hi / lo bias terms (<= 2^-16 of their absolute sum), plus one
    # fp16 rounding step of a hidden unit whose fp32 pre-activation sits on a rounding boundary
    absl = ref["ha"].abs() @ ref["w2a"].abs().T + ref["b2a"].abs()
    err = (torch.as_tensor(out["logits"], device=absl.device).double() - ref["logits"]).abs()
    assert bool((err <= 2e-4 * absl + 1e-3).all()), float((err / (absl + 1)).max())
    absv = torch.relu(ref["hc_pre"]).abs() @ ref["w2c"].abs() + ref["b2c"].abs()
    absv = absv + (ref["x"].abs() @ ref["w1c"].abs().T + ref["b1c"].abs()) @ ref["w2c"].abs()
    with torch.no_grad():
        from azul_deep_reinforcement_learning_b200.engine import PackedPolicy, policy_step
        val = policy_step(eng, PackedPolicy(eng, net), mode=1, apply_step=False)["value"].double()
    assert bool(((val - ref["value"]).abs() <= 1e-5 * absv + 1e-3).all()), float((val - ref["value"]).abs().max())


# ---- the persistent launches share the head ----------------------------------------------------------------------------------
def _check_records(recs, label):
    from azul_deep_reinforcement_learning_b200.engine import mask_to_bool
    nd = min(int(recs.meta[0]), recs.cap)
    assert nd > 0, label
    legal = mask_to_bool(recs.view.legal_mask())[:nd]
    act = recs.action_rec[:nd].long()
    assert bool((act < 180).all()), label
    ok = legal.gather(1, act[:, None]).squeeze(1)
    assert bool(ok.all()), (label, int((~ok).sum()), nd)


def test_persistent_rollouts_play_legal_actions_at_extreme_logits():
    """The extreme network of test_extreme_spread_and_offset (offset 1e4) in one PersistentEpisodes run (random opponent)
    and one SelfPlayEpisodes run: every recorded action is legal in its recorded state."""
    from azul_deep_reinforcement_learning_b200.engine import BatchedAzul, PackedPolicy
    from azul_deep_reinforcement_learning_b200.selfplay import BatchedGameRunner, PersistentEpisodes, SelfPlayEpisodes
    net = _net(_spread_logits(np.random.default_rng(31), 10000.37))
    gr = BatchedGameRunner(8192 + 45, seed=77)
    _check_records(PersistentEpisodes(gr, PackedPolicy(gr.engine, net), max_decisions=160).run(), "runner")
    eng = BatchedAzul(8192 + 45, 2, 1, 0, seed=78, reset=False)
    _check_records(SelfPlayEpisodes(eng, PackedPolicy(eng, net), max_decisions=320).run(), "selfplay")
    torch.cuda.synchronize()
