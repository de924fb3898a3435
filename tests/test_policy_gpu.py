"""K4 parity: the fused policy kernel (tcgen05 MLP + masked softmax + sampling + step) against plain
PyTorch fp32 evaluations of the same ActorCritic (reference azulnet/model.py:12-41) on the same states.

Tolerances (north star: logits within 1e-3 relative at reduced precision): the kernel rounds observation,
weights and the hidden activations to fp16 (11-bit significand; the tensor cores take fp16 and bf16 at the same
rate) and accumulates in fp32, so it is compared (a) tightly, 2e-4 of the logit scale, with a float64 torch
evaluation of the SAME fp16-rounded operands, and (b) at the north star's 1e-3 of the logit scale with the
untouched fp32 model."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

pytestmark = pytest.mark.gpu


def _setup(n=4096, pool=1, seed=7, k=23):
    from azul_deep_reinforcement_learning_b200.azulnet.model import ActorCritic
    from azul_deep_reinforcement_learning_b200.engine import BatchedAzul, PackedPolicy
    torch.manual_seed(0)
    net = ActorCritic(136, 180)
    # a wider spread than the default init so that masks / argmax are meaningful
    with torch.no_grad():
        for p in net.parameters():
            p.mul_(3.0)
    eng = BatchedAzul(n, 2, pool, 0, seed=seed)
    eng.rollout_random(k)                       # mid-game states with varied walls / scores
    packed = PackedPolicy(eng, net)
    return net, eng, packed


def test_policy_logits_and_value_match_torch():
    from azul_deep_reinforcement_learning_b200.engine import policy_step
    from tests.helpers import torch_forward
    with torch.no_grad():
        for pool in (0, 1):
            net, eng, packed = _setup(pool=pool)
            obs = eng.observe(-1)
            out = policy_step(eng, packed, mode=1, apply_step=False, want_logits=True)
            torch.cuda.synchronize()
            ref = torch_forward(net, obs, emulate_f16=True)
            ref_l, ref_v = ref["logits"].float(), ref["value"].float()
            scale = float(ref_l.abs().max())
            err = float((out["logits"] - ref_l).abs().max())
            assert err <= 2e-4 * scale, (err, scale)
            assert float((out["value"] - ref_v).abs().max()) <= 2e-4 * max(1.0, float(ref_v.abs().max()))
            full = torch_forward(net, obs, emulate_f16=False)
            full_l, full_v = full["logits"].float(), full["value"].float()
            assert float((out["logits"] - full_l).abs().max()) <= 1e-3 * float(full_l.abs().max())
            assert float((out["value"] - full_v).abs().max()) <= 1e-3 * max(1.0, float(full_v.abs().max()))


def test_policy_softmax_argmax_entropy_and_mask():
    from azul_deep_reinforcement_learning_b200.engine import mask_to_bool, policy_step
    with torch.no_grad():
        net, eng, packed = _setup()
        ref_mask = mask_to_bool(eng.legal_mask())
        out = policy_step(eng, packed, mode=1, apply_step=False, want_logits=True)
        assert torch.equal(mask_to_bool(out["mask"]), ref_mask)
        logits = out["logits"].masked_fill(~ref_mask, float("-inf"))
        logp_all = torch.log_softmax(logits, dim=1)                              # model.py:40
        act = out["action"].long()
        assert bool(ref_mask.gather(1, act[:, None]).all())                      # only legal actions
        best = logits.max(dim=1).values
        chosen = logits.gather(1, act[:, None]).squeeze(1)
        assert float((best - chosen).abs().max()) <= 1e-4                         # argmax (up to exact ties)
        assert float((out["logp"] - logp_all.gather(1, act[:, None]).squeeze(1)).abs().max()) <= 2e-3
        ent = -(logp_all.masked_fill(~ref_mask, 0.0).sum(dim=1) / ref_mask.sum(dim=1))   # nn_runner.py:36-40
        assert float((out["entropy"] - ent).abs().max()) <= 2e-3 * max(1.0, float(ent.abs().max()))
        assert int(out["status"].max()) == 0 and int(out["done"].max()) == 0


def test_policy_sampling_distribution_and_step_parity():
    """Many copies of one state (different game ids -> different Philox words): the sampled actions follow
    softmax(masked logits); with apply_step the resulting states equal azb_step on the sampled actions."""
    from azul_deep_reinforcement_learning_b200.azulnet.model import ActorCritic
    from azul_deep_reinforcement_learning_b200.engine import BatchedAzul, PackedPolicy, mask_to_bool, policy_step
    with torch.no_grad():
        torch.manual_seed(1)
        net = ActorCritic(136, 180)
        n = 1 << 16
        src = BatchedAzul(1, 2, 1, 0, seed=5)
        src.rollout_random(9)
        rec = src.export_records().cpu().numpy()
        eng = BatchedAzul(n, 2, 1, 0, seed=11, reset=False)
        assert bool(eng.import_records(np.repeat(rec, n, axis=0)).all())
        packed = PackedPolicy(eng, net)
        before = eng.state.clone()
        out = policy_step(eng, packed, mode=0, apply_step=False, want_logits=True)
        assert torch.equal(before, eng.state)
        mask = mask_to_bool(out["mask"])[0]
        p = torch.softmax(out["logits"][0].masked_fill(~mask, float("-inf")), dim=0).double().cpu().numpy()
        counts = np.bincount(out["action"].cpu().numpy(), minlength=180).astype(np.float64)
        assert counts[~mask.cpu().numpy()].sum() == 0
        sel = p > 0
        chi2 = float((((counts[sel] - n * p[sel]) ** 2) / (n * p[sel])).sum())
        dof = int(sel.sum()) - 1
        assert chi2 < dof + 6 * np.sqrt(2 * dof) + 10, (chi2, dof)
        # fused step == separate step with the same actions (both use the Philox refill schedule)
        twin = BatchedAzul(n, 2, 1, 0, seed=11, reset=False)
        twin.state.copy_(eng.state)
        out2 = policy_step(eng, packed, mode=0, apply_step=True)
        assert torch.equal(out2["action"], out["action"])
        twin.step(out["action"], None)
        assert torch.equal(twin.state, eng.state)


def test_policy_selfplay_runs_to_game_end_and_ragged_batch():
    from azul_deep_reinforcement_learning_b200.engine import policy_step
    with torch.no_grad():
        net, eng, packed = _setup(n=1000, k=0)      # ragged: 1000 is not a multiple of the 128-game tile
        done_any = torch.zeros(1000, dtype=torch.bool, device=eng.device)
        for _ in range(300):
            out = policy_step(eng, packed, mode=0, apply_step=True)
            done_any |= out["done"].bool()
            assert int((out["status"] & 1).max()) == 0          # never an illegal action
        assert float(done_any.float().mean()) > 0.9               # (a random-init policy plays long games)
        before = eng.state.clone()
        out = policy_step(eng, packed, mode=0, apply_step=True)
        ended = out["done"].bool() & done_any
        assert bool(((out["status"][ended] & 2) != 0).all())      # ended games: flagged GameEnded ...
        assert torch.equal(before[:, ended], eng.state[:, ended])  # ... and left untouched
        assert bool((out["action"][ended] == 255).all())


def test_policy_selfplay_auto_reset_counters():
    """apply_step = 2: finished games are tallied and replaced; counters stay consistent with the states."""
    from azul_deep_reinforcement_learning_b200.engine import policy_step
    with torch.no_grad():
        net, eng, packed = _setup(n=2048, k=0)
        steps = 260
        n_done = 0
        for _ in range(steps):
            out = policy_step(eng, packed, mode=0, apply_step=True, auto_reset=True, want_mask=False)
            n_done += int(out["done"].sum())
            assert int(out["status"].max()) == 0
        c = eng.read_counters()
        assert c["steps"] == 2048 * steps and c["games"] == n_done > 0 and c["stuck"] == 0
        rec = eng.export_records().cpu().numpy()
        from azul_deep_reinforcement_learning_b200.layout import UnpackedLayout
        L = UnpackedLayout(2)
        assert (rec[:, L.end_of_game] == 0).all() and (rec[:, 0:30].sum(axis=1) > 0).all()
        # every new_round after the initial azb_reset is counted once: finished games' rounds + running games' rounds
        assert c["rounds"] == c["turns"] + int(rec[:, L.turn_counter].sum()) - 2048


def test_policy_finishing_phase_many_tiles_per_cta():
    """More than 96 tiles per CTA with EVERY game flagged (a whole batch of ended games asking for fresh ones): the
    finishing phase at the end of the policy kernel works through its dense list in groups; every slot ends up with a
    fresh, playable game and the next step runs normally."""
    from azul_deep_reinforcement_learning_b200.engine import BatchedAzul, PackedPolicy, policy_step
    from azul_deep_reinforcement_learning_b200.azulnet.model import ActorCritic
    from azul_deep_reinforcement_learning_b200.layout import UnpackedLayout
    with torch.no_grad():
        n = 148 * 128 * 100 + 77                                  # 100+ tiles for every CTA of a 148-SM GPU, ragged tail
        torch.manual_seed(0)
        eng = BatchedAzul(n, 2, 1, 0, seed=3)
        packed = PackedPolicy(eng, ActorCritic(136, 180))
        eng.state[3] |= 1 << 12                                   # MISC bit 12: end_of_game in every slot
        out = policy_step(eng, packed, mode=0, apply_step=True, auto_reset=True, want_mask=False)
        assert bool((out["done"] == 1).all())                     # (the boards still hold tiles, so an action is reported; it is not played)
        misc = eng.state[3]
        assert int(((misc >> 12) & 1).sum()) == 0 and int((misc >> 28).sum()) == 0      # nobody ended, no transient flag left
        L = UnpackedLayout(2)
        for lo in (0, n // 2, n - 512):
            sub = BatchedAzul(512, 2, 1, 0, seed=3, game_id_base=lo, reset=False)
            sub.state.copy_(eng.state[:, lo:lo + 512])
            rec = sub.export_records().cpu().numpy()
            assert (rec[:, 0:30].sum(axis=1) == 20).all() and (rec[:, L.score:L.score + 2] == 0).all()   # 20 tiles on the factories
        out = policy_step(eng, packed, mode=0, apply_step=True, auto_reset=True, want_mask=False)
        assert bool((out["action"] < 180).all()) and int(out["status"].max()) == 0
        assert eng.read_counters()["rounds"] == n and eng.read_counters()["steps"] == n
