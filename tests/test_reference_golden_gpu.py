"""The CUDA path (through the C ABI) against goldens recorded from the LIVE reference above the bare rules engine
(tests/golden/runner_*.npz, model.npz, update.npz; oracle/record_golden_runner.py):

* ``GameRunner.reset`` / ``step`` (game_runner.py:43-55,76-85): every env step of 2 x 64 reference episodes through
  ``azb_step`` with the recorded actions and draws, the opponent-loop stop rule of ``azb_opponent_random`` at EVERY state
  of the trace, reward / done / legal mask / observation / record at every hand-back, ``azb_stats`` at the end;
* ``ActorCritic.forward_actor / forward_critic`` (model.py:23-41) on 4,096 reachable decision states through the fused
  policy kernel: logits, value, log pi, entropy term, argmax;
* ``Agent.update`` (agent.py:39-62) through the trainer's update: loss terms, gradients, parameters after two Adam steps.

Tolerances (DESIGN.md §0): integer outputs bit-exact.  Logits / value (fp16 tensor-core operands, fp32 accumulation)
per element |got - ref| <= 1e-3 * max(|ref|, floor) with floor = the largest |logit| of that decision's row (the largest
|value| of the batch for the value head); log-probabilities and the entropy term 2e-3 + 1e-3 * floor absolute (they are differences of logits and a
log-sum-exp).  Gradients of the update: see test_trainer_decision_updates_match_reference_agent_update."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

from azul_deep_reinforcement_learning_b200.layout import UnpackedLayout  # noqa: E402
from tests.helpers import (PARAM_NAMES, RUNNER_RULES, RunnerEpisode, load_model_golden, load_runner,  # noqa: E402
                           load_update_golden, mask_words_to_bool, net_from_golden)

pytestmark = pytest.mark.gpu

LOGIT_RTOL = 1e-3
LOGP_ATOL = 2e-3


@pytest.mark.parametrize("rules", RUNNER_RULES)
def test_game_runner_traces_on_gpu(rules):
    from azul_deep_reinforcement_learning_b200.engine import BatchedAzul
    tr = load_runner(rules)
    pool = int(tr["tile_pool"])
    E = len(tr["seeds"])
    eps = [RunnerEpisode(tr, e) for e in range(E)]
    L = UnpackedLayout(2)
    eng = BatchedAzul(E, 2, pool, 1, seed=1, reset=False)
    twin = BatchedAzul(E, 2, pool, 1, seed=1, reset=False)
    assert bool(eng.import_records(np.stack([ep.init_record for ep in eps])).all())
    pos = np.zeros(E, np.int64)               # env steps of the episode executed so far
    hb = np.zeros(E, np.int64)                # hand-backs seen so far
    pscore = torch.zeros(E, dtype=torch.int16, device="cuda")
    n_forced = n_hb = 0
    for tick in range(max(ep.n_steps for ep in eps) + 1):
        # ---- the stop rule on the current state of every game, both loop variants (game_runner.py:46 / :84) ----
        steps_before = eng.state[6].clone()
        outs = {}
        for require_two in (False, True):
            twin.state.copy_(eng.state)
            ps = pscore.clone()
            o = twin.opponent_random(ps, require_two=require_two, want_obs=True)
            o["stopped"] = (twin.state[6] == steps_before).cpu().numpy()
            o["ps"] = ps
            outs[require_two] = {k: ((v.float() if v.dtype == torch.bfloat16 else v).cpu().numpy() if torch.is_tensor(v) else v) for k, v in o.items()}
        rec = eng.export_records().cpu().numpy()
        obs0 = eng.observe(0).cpu().numpy()
        new_ps = pscore.cpu().numpy().copy()
        for e, ep in enumerate(eps):
            if pos[e] > ep.n_steps:
                continue
            in_reset = hb[e] == 0
            o = outs[not in_reset]
            want_hb = hb[e] < ep.n_hb and ep.hb_step[hb[e]] == pos[e]
            assert bool(o["stopped"][e]) == bool(want_hb), (rules, e, int(pos[e]))
            if want_hb:
                h = int(hb[e])
                if in_reset:
                    new_ps[e] = 0                                             # game_runner.py:81
                else:
                    assert int(o["reward"][e]) == int(ep.hb_reward[h]), (e, h)
                    new_ps[e] = o["ps"][e]
                assert int(new_ps[e]) == int(ep.hb_player_score[h])
                assert int(o["done"][e]) == int(ep.hb_done[h])
                assert np.array_equal(o["mask"][:, e].astype(np.uint32), ep.hb_mask[h])
                assert np.array_equal(rec[e][:L.total_steps], ep.hb_records[h][:L.total_steps])
                assert np.array_equal(obs0[e].astype(np.int32), ep.hb_obs[h])
                assert np.array_equal(o["obs"][e].astype(np.float32).astype(np.int32), ep.hb_obs[h])     # the bf16 record of training
                hb[e] += 1
                n_hb += 1
        pscore.copy_(torch.from_numpy(new_ps))
        # ---- the next recorded env step of every unfinished episode (agent's or opponent's) through azb_step ----
        act = np.full(E, 255, np.uint8)
        draws = np.full((E, 20), -1, np.int8)
        for e, ep in enumerate(eps):
            s = int(pos[e])
            if s < ep.n_steps:
                assert int(rec[e][L.current_player]) == int(ep.step_seat[s])
                if ep.step_seat[s] == 1 and s >= ep.n_reset_steps and not (hb[e] > 0 and ep.hb_step[hb[e] - 1] == s):
                    n_forced += 1
                act[e] = ep.step_action[s]
                d = ep.step_draws(s)
                if d is not None:
                    draws[e] = d
            pos[e] += 1
        if (act != 255).any():
            out = eng.step(torch.from_numpy(act), torch.from_numpy(draws))
            st = out["status"].cpu().numpy()
            assert ((st & 3) == 0).all()
    assert n_hb == int(tr["hb_offsets"][-1]) and n_forced > 20
    rec = eng.export_records().cpu().numpy()
    stats = eng.stats().cpu().numpy()
    for e, ep in enumerate(eps):
        assert np.array_equal(rec[e][:L.total_steps], ep.final_record[:L.total_steps])
        want = dict(zip(ep.stat_keys, ep.stats))                              # Azul.get_statistics, azul.py:314-315
        st = stats[e]
        assert st[0] == want["player_score"] and st[1] == want["opponent_score"] and st[2] == want["rounds"]
        assert abs(100.0 * st[3] / st[4] - want["percent_first_player"]) < 1e-9
        assert [st[5], st[6], st[7], st[8], st[9]] == [want[k] for k in ("floor_penalty", "max_combo", "completed_rows", "completed_columns", "completed_colors")]


def _policy_on_golden_states(z, scale, mode):
    from azul_deep_reinforcement_learning_b200.engine import BatchedAzul, PackedPolicy, policy_step
    n = z["records"].shape[0]
    eng = BatchedAzul(n, 2, 1, 1, seed=9, reset=False)
    assert bool(eng.import_records(z["records"].astype(np.int32)).all())
    net = net_from_golden(z, "param_", scale)
    packed = PackedPolicy(eng, net)
    out = policy_step(eng, packed, mode=mode, apply_step=False, want_logits=True)
    torch.cuda.synchronize()
    return eng, {k: v.cpu().numpy() for k, v in out.items()}


@pytest.mark.parametrize("tag,scale", [("s1", 1.0), ("s3", 3.0)])
def test_policy_kernel_matches_reference_actor_critic(tag, scale):
    z = load_model_golden()
    n, nf = z["records"].shape[0], z[tag + "_logits_full"].shape[0]
    eng, out = _policy_on_golden_states(z, scale, mode=1)
    valid = mask_words_to_bool(z["mask"])
    # the kernel's own observation and mask equal the reference's get_state / check_all_valid for these states
    assert np.array_equal(eng.observe(-1).cpu().numpy().astype(np.int32), z["obs"].astype(np.int32))
    assert np.array_equal(out["mask"].T.astype(np.uint32), z["mask"])
    # logits: per element against the reference rows (full rows for the first nf states, 4 entries per state for all)
    floor = z[tag + "_logits_absmax"].astype(np.float64)
    ref_full = z[tag + "_logits_full"].astype(np.float64)
    err = np.abs(out["logits"][:nf] - ref_full)
    bound = LOGIT_RTOL * np.maximum(np.abs(ref_full), floor[:nf, None])
    assert (err <= bound).all(), float((err / bound).max())
    sel = z["sel_actions"].astype(np.int64)
    got_sel = np.take_along_axis(out["logits"], sel, axis=1)
    ref_sel = z[tag + "_logits_sel"].astype(np.float64)
    assert (np.abs(got_sel - ref_sel) <= LOGIT_RTOL * np.maximum(np.abs(ref_sel), floor[:, None])).all()
    # value (critic head)
    ref_v = z[tag + "_value"].astype(np.float64)
    assert (np.abs(out["value"] - ref_v) <= LOGIT_RTOL * np.maximum(np.abs(ref_v), np.abs(ref_v).max())).all()
    # entropy term -mean(log pi over legal) (nn_runner.py:36-40)
    assert (np.abs(out["entropy"] - z[tag + "_entropy"]) <= LOGP_ATOL + LOGIT_RTOL * floor).all()
    # "Max" action selection (agent.py:70-71): the reference's argmax, or an action whose probability ties it
    same = out["action"] == z[tag + "_argmax"]
    p_chosen = np.exp(out["logp"].astype(np.float64))
    assert (same | (np.abs(p_chosen - z[tag + "_pmax"]) <= 2e-3 * z[tag + "_pmax"])).all()
    assert same.mean() > 0.995
    assert np.abs(p_chosen - z[tag + "_pmax"]).max() <= 3e-3 * float(z[tag + "_pmax"].max())
    assert valid[np.arange(n), out["action"]].all()


@pytest.mark.parametrize("tag,scale", [("s1", 1.0), ("s3", 3.0)])
def test_policy_kernel_sampled_logp_matches_reference(tag, scale):
    """Sampling mode: log pi(action) of whatever action the kernel drew equals the reference's log_softmax entry."""
    z = load_model_golden()
    nf = z[tag + "_logits_full"].shape[0]
    _, out = _policy_on_golden_states(z, scale, mode=0)
    valid = mask_words_to_bool(z["mask"])[:nf]
    act = out["action"][:nf].astype(np.int64)
    assert valid[np.arange(nf), act].all()
    ref = torch.from_numpy(z[tag + "_logits_full"].astype(np.float64)).masked_fill(~torch.from_numpy(valid), float("-inf"))
    ref_logp = torch.log_softmax(ref, dim=1).numpy()                          # model.py:40 on the reference's own logits
    floor = z[tag + "_logits_absmax"][:nf].astype(np.float64)
    assert (np.abs(out["logp"][:nf] - ref_logp[np.arange(nf), act]) <= LOGP_ATOL + LOGIT_RTOL * floor).all()
    assert len(np.unique(act)) > 20


@pytest.mark.parametrize("path,grad_tol,flip_frac", [("autograd-fp32", 2e-4, 2e-3), ("autograd-tf32", 6e-2, 0.06), ("tensor", 6e-2, 0.06)])
def test_trainer_decision_updates_match_reference_agent_update(path, grad_tol, flip_frac):
    """Two ``Agent.update`` calls of the live reference (update.npz) through the trainer: the loss terms, the gradient of the
    first update and the parameters after both Adam steps -- for the fp32 autograd path, the TF32 autograd path and the
    hand-written tensor-core path (azb_a2c_update_gradients on packed decision states).  Gradient tolerance per tensor,
    relative to its largest entry: fp32 2e-4; reduced-precision operands (10/11-bit significands) 6e-2 at these ~350
    decisions -- hidden units whose pre-activation lies within the forward rounding error of zero switch their ReLU
    derivative, each such switch moves an entry by a whole term of the sum (cosine with the fp32 gradient > 0.999)."""
    from azul_deep_reinforcement_learning_b200.engine import BatchedAzul
    from azul_deep_reinforcement_learning_b200.train import SelfPlayTrainer
    z = load_update_golden()
    tr = SelfPlayTrainer(64, learning_rate=float(z["learning_rate"]), gamma=float(z["gamma"]), seed=0, device=0,
                         tf32_update=(path != "autograd-fp32"))
    tr.load_parameters({n: torch.from_numpy(z["param0_" + n]) for n in PARAM_NAMES})
    named = dict(tr.net.named_parameters())
    for b in (0, 1):
        idx = np.nonzero(z["batch"] == b)[0]
        action = torch.from_numpy(z["action"][idx].astype(np.int64)).cuda()
        qval = torch.from_numpy(z["qvals"][idx].astype(np.float32)).cuda()
        if path == "tensor":
            view = BatchedAzul(len(idx), 2, 1, 0, seed=0, reset=False)
            assert bool(view.import_records(z["records"][idx].astype(np.int32)).all())
            st = tr.update_states(view.state, action.to(torch.uint8), qval)
        else:
            obs = torch.from_numpy(z["obs"][idx].astype(np.float32)).cuda().to(torch.bfloat16)
            rows = torch.from_numpy(z["mask"][idx].astype(np.int64)).to(torch.int32).cuda().contiguous()
            st = tr.update_decisions(obs, rows, action, qval)
        losses = z["losses"][b]                                                  # reward, actor, critic, entropy, ac
        for k, want in (("actor_loss", losses[1]), ("critic_loss", losses[2]), ("entropy_loss", losses[3]), ("ac_loss", losses[4])):
            assert abs(st[k] - want) <= 2e-3 * abs(want), (b, k, st[k], want)
        if b == 0:
            for name in PARAM_NAMES:
                want = torch.from_numpy(z["grad1_" + name]).cuda()
                got = tr.last_grads[name]
                err = float((got - want).abs().max())
                assert err <= grad_tol * float(want.abs().max()), (name, err, float(want.abs().max()))
                cos = float((got.double() * want.double()).sum() / (got.double().norm() * want.double().norm()))
                assert cos > 0.999, (name, cos)
        for name in PARAM_NAMES:
            want = torch.from_numpy(z["param%d_" % (b + 1) + name]).cuda()
            diff = (named[name].detach() - want).abs()
            # Adam's first steps are ~lr * sign(g): only entries whose gradient is at rounding level may land elsewhere
            assert float(diff.max()) <= 2.1 * float(z["learning_rate"]) * (b + 1), name
            assert float((diff > 2e-5).float().mean()) < flip_frac, (name, float((diff > 2e-5).float().mean()))
