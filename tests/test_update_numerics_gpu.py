"""azb_a2c_update_gradients (csrc/azb_update.cu) against a float64 reference that rounds where the kernel rounds.

The kernel's operands are fp16 and its sums fp32, so against the fp32 network (test_selfplay_gpu.py) it can only be held
to a few per cent.  Here the reference takes the same fp16 operands (tests/helpers.torch_forward: observation, W1a, W1c,
W2a, the actor's hidden activations, the biases as fp16 hi + lo) and, like the kernel, rounds the logit gradient dL and
the hidden-layer gradients dHa / dHc to fp16 before the weight-gradient products; the ReLU derivatives come from the
pre-activations.  Everything else is float64.  What remains is fp32 accumulation order, __expf / __logf, and the rare
fp16 rounding where the kernel's fp32 value and the float64 one straddle a rounding boundary.

Bounds, each about 2 to 10 times the largest error measured over these cases (B200, 1,000 W power limit): logits
within 2e-4 of the row's largest |logit| (measured 1.4e-4: the fp16 rounding of a hidden activation whose fp32 and float64 values straddle a
rounding boundary moves it by an fp16 ulp), value within 1e-6 of max(1, largest |value|) (1.7e-7); each gradient tensor
within a fraction of its largest entry, and exactly zero where the reference is: 2e-4 for the actor's layers (largest:
actor_linear1.weight 1.1e-4, the same straddles in dL and dHa), 1e-4 for actor_linear2.bias (1.2e-5) and
critic_linear1 (1.4e-5), 5e-6 for critic_linear2.weight (6.6e-7); critic_linear2.bias, a single sum over the decisions
that can cancel to a small fraction of its terms, within 1e-6 of the sum of their magnitudes (1.5e-7); loss sums
within 5e-5 relative (7.8e-6).

The records are states of random rollouts of both tile pools (seat 1 or seat 2 to move), with legal actions drawn
uniformly and returns uniform in [-40, 40], plus states with exactly one legal action and rows the kernel must ignore:
no legal action, action 255 (no decision) and an in-range action that is illegal in its state."""
import pytest

torch = pytest.importorskip("torch")

from tests.helpers import f16, torch_forward  # noqa: E402

pytestmark = pytest.mark.gpu

COEFFS = (1.0, 0.5, 0.1)
TOL = {"logits": 2e-4, "value": 1e-6, "actor_linear1.weight": 2e-4, "actor_linear1.bias": 2e-4, "actor_linear2.weight": 2e-4,
       "actor_linear2.bias": 1e-4, "critic_linear1.weight": 1e-4, "critic_linear1.bias": 1e-4, "critic_linear2.weight": 5e-6,
       "critic_linear2.bias": 1e-6, "sums": 5e-5}
N_BAD = 16                      # rows of each unusable kind


class Records:
    """Packed states [17, N] with the decision taken on each (uint8) and its return (float32); observation (mover's
    perspective) and legal mask rebuilt from the states by the engine.  Without ``action`` an action is drawn uniformly
    among the legal ones (``legal`` False: among the illegal ones) and a return uniformly in [-40, 40]."""

    def __init__(self, state, action=None, qval=None, gen=None, legal=True):
        from azul_deep_reinforcement_learning_b200.engine import BatchedAzul, mask_to_bool
        self.state = state.contiguous()
        self.view = BatchedAzul(state.shape[1], 2, 0, 0, reset=False)
        self.view.state.copy_(self.state)
        self.obs = self.view.observe(-1)
        self.mask = mask_to_bool(self.view.legal_mask())
        if action is None:
            u = torch.rand(self.mask.shape, generator=gen, device="cuda")
            action = torch.where(self.mask if legal else ~self.mask, u, -1.0).argmax(1).to(torch.uint8)
            qval = torch.rand(state.shape[1], generator=gen, device="cuda") * 80.0 - 40.0
        self.action, self.qval = action.contiguous(), qval.contiguous()

    def cat(self, other, at=None):
        """``other``'s rows inserted before the rows ``at`` (default: appended)."""
        n, m = self.state.shape[1], other.state.shape[1]
        pos = torch.arange(n, device="cuda")
        if at is not None:
            pos = pos + torch.searchsorted(at, pos, right=True)
            ins = at + torch.arange(m, device="cuda")
        else:
            ins = n + torch.arange(m, device="cuda")
        order = torch.empty(n + m, dtype=torch.long, device="cuda")
        order[pos] = torch.arange(n, device="cuda")
        order[ins] = n + torch.arange(m, device="cuda")
        return Records(torch.cat([self.state, other.state], 1)[:, order], torch.cat([self.action, other.action])[order],
                       torch.cat([self.qval, other.qval])[order])


def _random_states(n, pool, k, seed):
    from azul_deep_reinforcement_learning_b200.engine import BatchedAzul
    eng = BatchedAzul(n, 2, pool, 0, seed=seed)
    eng.rollout_random(k)
    return eng.state.clone()


@pytest.fixture(scope="module")
def data():
    from azul_deep_reinforcement_learning_b200.azulnet.model import ActorCritic
    from azul_deep_reinforcement_learning_b200.engine import BatchedAzul, mask_to_bool
    gen = torch.Generator(device="cuda").manual_seed(11)
    state = torch.cat([_random_states(3000, pool, k, 100 + 10 * pool + k) for pool in (0, 1) for k in (0, 9, 26, 55)], 1)
    # states with exactly one legal action (one source / colour pair left that only the floor line takes: a few per cent
    # of mid-round states), searched for in a larger pool
    single = []
    for pool in (0, 1):
        for k in (14, 33, 61):
            eng = BatchedAzul(1 << 13, 2, pool, 0, seed=7 + 3 * pool + k)
            eng.rollout_random(k)
            single.append(eng.state[:, mask_to_bool(eng.legal_mask()).sum(1) == 1])
    single = torch.cat(single, 1)[:, :24]
    assert single.shape[1] > 0
    base, one = Records(state, gen=gen), Records(single, gen=gen)
    assert bool((one.mask.sum(1) == 1).all())
    clean = base.cat(one, at=torch.arange(one.state.shape[1], device="cuda") * 97 + 1)
    # unusable rows, built from clean states: no legal action (factories, centre and first-player token cleared), no
    # decision (action 255), an in-range action that is illegal in the state
    src = slice(5000, 5000 + N_BAD)
    empty = clean.state[:, src].clone()
    empty[0:3] = 0
    empty[3] &= ~31
    bad = [Records(empty, clean.action[src], clean.qval[src]),
           Records(clean.state[:, src], torch.full((N_BAD,), 255, dtype=torch.uint8, device="cuda"), clean.qval[src]),
           Records(clean.state[:, src], gen=gen, legal=False)]
    assert int(bad[0].mask.sum()) == 0 and not bool(bad[2].mask.gather(1, bad[2].action.long()[:, None]).any())
    bad = bad[0].cat(bad[1]).cat(bad[2])
    mixed = clean.cat(bad, at=torch.arange(bad.state.shape[1], device="cuda") * 41 + 3)
    nets = {}
    for scale in (1.0, 3.0):
        torch.manual_seed(0)
        net = ActorCritic(136, 180)
        with torch.no_grad():
            for p in net.parameters():
                p.mul_(scale)
        nets[scale] = net
    return {"clean": clean, "bad": bad, "mixed": mixed, "nets": nets}


def _reference(net, r, n, coeffs):
    """Gradient sums, loss sums, logits and value of the first n records, emulating the kernel's roundings."""
    o = torch_forward(net, r.obs[:n], emulate_f16=True)
    ca, cc, ce = coeffs
    mask, act = r.mask[:n], r.action[:n].long()
    ok = (act < 180) & mask.gather(1, act.clamp(max=179)[:, None]).squeeze(1)
    m, a, q = mask[ok], act[ok], r.qval[:n][ok].double()
    logits, value = o["logits"][ok], o["value"][ok]
    masked = logits.masked_fill(~m, float("-inf"))
    lse = torch.logsumexp(masked, 1)
    log_prob = logits.gather(1, a[:, None]).squeeze(1) - lse
    k = m.sum(1).double()
    entropy = -((logits * m).sum(1) / k - lse)
    adv = q - value
    p = torch.exp(masked - lse[:, None])
    onehot = torch.nn.functional.one_hot(a, 180).double()
    dl = torch.where(m, ca * (-adv)[:, None] * (onehot - p) + ce * (p - 1.0 / k[:, None]), 0.0)
    dl = f16(dl.float()).double()
    dv = ca * log_prob - 2.0 * cc * adv
    ha_on, hc_on = o["ha_pre"][ok] > 0, o["hc_pre"][ok] > 0
    dha = f16(((dl @ o["w2a"]) * ha_on).float()).double()
    dhc = f16((dv[:, None] * o["w2c"][None, :] * hc_on).float()).double()
    x = o["x"][ok]
    grads = {"actor_linear1.weight": dha.T @ x, "actor_linear1.bias": dha.sum(0),
             "actor_linear2.weight": dl.T @ o["ha"][ok], "actor_linear2.bias": dl.sum(0),
             "critic_linear1.weight": dhc.T @ x, "critic_linear1.bias": dhc.sum(0),
             "critic_linear2.weight": (dv[:, None] * torch.relu(o["hc_pre"][ok])).sum(0)[None, :],
             "critic_linear2.bias": dv.sum()[None]}
    sums = torch.stack([(-log_prob * adv).sum(), (adv * adv).sum(), entropy.sum()])
    # grad b2c is one sum over all decisions, which can cancel far below its summands: it is measured against those
    scales = {name: float(g.abs().max()) for name, g in grads.items()}
    scales["critic_linear2.bias"] = float(dv.abs().sum())
    return {"grads": grads, "scales": scales, "sums": sums, "logits": o["logits"], "value": o["value"], "ok": ok}


def _kernel(r, packed, cap, coeffs=COEFFS, n_fixed=0, n_dec=None):
    from azul_deep_reinforcement_learning_b200.engine import UpdateGradients
    upd = UpdateGradients(r.view, cap)
    nd = None if n_dec is None else torch.tensor([n_dec], dtype=torch.int32, device="cuda")
    logits, value = upd.run(packed, r.state[:, :cap].contiguous(), r.action[:cap].contiguous(), r.qval[:cap].contiguous(),
                            n_dec=nd, n_fixed=n_fixed, coeffs=coeffs, want_outputs=True)
    torch.cuda.synchronize()
    return upd, logits, value


def _compare(upd, logits, value, ref):
    """Asserts the bounds of the module docstring; returns each quantity's error over its scale."""
    from azul_deep_reinforcement_learning_b200.engine import PARAM_ORDER
    ok, ref_l, ref_v = ref["ok"], ref["logits"], ref["value"]
    n = ref_l.shape[0]
    err = {}
    row_scale = ref_l.abs().max(1).values
    err["logits"] = float(((logits[:n].double() - ref_l).abs().max(1).values / row_scale).max())
    if bool(ok.any()):
        err["value"] = float((value[:n][ok].double() - ref_v[ok]).abs().max()) / max(1.0, float(ref_v[ok].abs().max()))
    for name in PARAM_ORDER:
        g, w = upd.grads[name].double(), ref["grads"][name]
        d, scale = float((g - w).abs().max()), ref["scales"][name]
        assert scale > 0 or d == 0.0, (name, d)
        err[name] = d / scale if scale > 0 else 0.0
    err["sums"] = float(((upd.sums - ref["sums"]).abs() / ref["sums"].abs().clamp_min(1.0)).max())
    for k, e in err.items():
        assert e <= TOL[k], (k, e, err)
    return err


def _packed(d, scale):
    from azul_deep_reinforcement_learning_b200.engine import PackedPolicy
    return PackedPolicy(d["mixed"].view, d["nets"][scale])


@pytest.mark.parametrize("n", [1, 63, 64, 65, 127, 128, 129, 1000, 148 * 128 + 1])
def test_update_matches_rounded_reference_at_ragged_counts(data, n):
    """Host-side counts that end inside, on and just past a 64-decision half tile and a 128-decision tile, and one tile
    more than a B200 has SMs (a CTA works on a second tile while the next one's states are prefetched)."""
    r = data["mixed"]
    net = data["nets"][1.0]
    ref = _reference(net, r, n, COEFFS)
    assert int(ref["ok"].sum()) >= 1
    _compare(*_kernel(r, _packed(data, 1.0), n + 5, n_fixed=n), ref)


def test_update_device_side_count(data):
    """The count read on the device: below the capacity, above it (clamped: the result of a run over the whole
    capacity), and zero (nothing is added)."""
    r, net, packed = data["mixed"], data["nets"][1.0], _packed(data, 1.0)
    n, cap = 1000, 1300
    _compare(*_kernel(r, packed, cap, n_dec=n), _reference(net, r, n, COEFFS))
    over, logits, value = _kernel(r, packed, cap, n_dec=cap + 1000)
    _compare(over, logits[:cap], value[:cap], _reference(net, r, cap, COEFFS))
    at_cap = _kernel(r, packed, cap, n_fixed=cap)[0]
    assert float((over.flat - at_cap.flat).abs().max()) <= 1e-6 * float(at_cap.flat.abs().max())
    assert float((over.sums - at_cap.sums).abs().max()) <= 1e-9 * float(at_cap.sums.abs().max())
    zero = _kernel(r, packed, cap, n_dec=0)[0]
    assert int(torch.count_nonzero(zero.flat)) == 0 and int(torch.count_nonzero(zero.sums)) == 0


@pytest.mark.parametrize("chunk_rows", [128, 256])
def test_update_in_small_chunks_matches_reference(data, chunk_rows):
    """Workspace-sized chunks whose boundaries fall inside the batch."""
    from azul_deep_reinforcement_learning_b200 import _lib
    r, n = data["mixed"], 3 * 256 + 5
    lib = _lib.load()
    try:
        _lib.check(lib.azb_update_set_chunk_rows(chunk_rows))
        got = _kernel(r, _packed(data, 1.0), n, n_fixed=n)
    finally:
        _lib.check(lib.azb_update_set_chunk_rows(1 << 20))
    assert got[0].workspace.numel() == lib.azb_update_workspace_bytes(chunk_rows)       # sized for one chunk
    _compare(*got, _reference(data["nets"][1.0], r, n, COEFFS))


@pytest.mark.parametrize("scale", [1.0, 3.0])
@pytest.mark.parametrize("coeffs", [(1.0, 0.5, 0.1), (1.0, 0.0, 0.0), (0.0, 1.0, 0.0), (0.0, 0.0, 1.0)])
def test_update_coefficients_and_weight_scales(data, coeffs, scale):
    """Each loss term on its own, at the default initialisation and at three times it (peaked softmaxes).  A term that is
    switched off leaves its gradients exactly zero: no actor or entropy term, no actor gradient; no actor or critic term,
    no gradient at the value, so no critic gradient."""
    r, n = data["mixed"], 3000
    upd, logits, value = _kernel(r, _packed(data, scale), n, coeffs=coeffs, n_fixed=n)
    _compare(upd, logits, value, _reference(data["nets"][scale], r, n, coeffs))
    actor = [k for k in upd.grads if k.startswith("actor")]
    critic = [k for k in upd.grads if k.startswith("critic")]
    if coeffs[0] == 0.0 and coeffs[2] == 0.0:
        assert all(int(torch.count_nonzero(upd.grads[k])) == 0 for k in actor)
    if coeffs[0] == 0.0 and coeffs[1] == 0.0:
        assert all(int(torch.count_nonzero(upd.grads[k])) == 0 for k in critic)


def test_update_ignores_unusable_rows(data):
    """Rows without a legal action, with action 255 or with an illegal action, appended to a batch, change nothing."""
    clean, n = data["clean"], 2000
    head = Records(clean.state[:, :n], clean.action[:n], clean.qval[:n])
    both = head.cat(data["bad"])
    packed = _packed(data, 1.0)
    ref = _reference(data["nets"][1.0], head, n, COEFFS)
    a = _kernel(head, packed, n, n_fixed=n)
    b = _kernel(both, packed, both.state.shape[1], n_fixed=both.state.shape[1])
    _compare(*a, ref)
    _compare(b[0], b[1][:n], b[2][:n], ref)
    assert float((a[0].flat - b[0].flat).abs().max()) <= 1e-6 * float(a[0].flat.abs().max())
    assert float(((a[0].sums - b[0].sums).abs() / a[0].sums.abs()).max()) <= 1e-9
