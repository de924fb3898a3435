"""Host-side model / update code against goldens recorded from the LIVE reference (tests/golden/model.npz,
update.npz; oracle/record_golden_runner.py): ``ActorCritic.forward_*`` (model.py:23-41), the discounted returns of
``NNRunner.train`` (nn_runner.py:72-75) and one full ``Agent.update`` (agent.py:39-62: loss terms, gradients, Adam
step).  CPU only; the GPU kernels are checked against the same files in tests/test_reference_golden_gpu.py."""
import numpy as np
import torch

from tests.helpers import PARAM_NAMES, load_model_golden, load_update_golden, mask_words_to_bool, net_from_golden


def test_facade_actor_critic_matches_reference_forward():
    z = load_model_golden()
    obs = torch.from_numpy(z["obs"].astype(np.float32))
    valid = torch.from_numpy(mask_words_to_bool(z["mask"]))
    sel = torch.from_numpy(z["sel_actions"].astype(np.int64))
    for tag, scale in (("s1", 1.0), ("s3", 3.0)):
        net = net_from_golden(z, "param_", scale)
        with torch.no_grad():
            value = net.forward_critic(obs).squeeze(1)
            dist, logp = net.forward_actor(obs, valid)
        # same torch CPU ops as the reference on the same parameters: identical up to summation order
        assert torch.allclose(value, torch.from_numpy(z[tag + "_value"]), rtol=1e-5, atol=1e-5)
        assert torch.allclose(logp.gather(1, sel), torch.from_numpy(z[tag + "_logp_sel"]), rtol=1e-5, atol=1e-5)
        ent = -(logp.masked_fill(~valid, 0.0).sum(1) / valid.sum(1))
        assert torch.allclose(ent, torch.from_numpy(z[tag + "_entropy"]), rtol=1e-5, atol=1e-5)
        assert torch.equal(dist.argmax(1).to(torch.uint8), torch.from_numpy(z[tag + "_argmax"]))


def test_discounted_returns_match_nn_runner_train():
    """nn_runner.py:72-75 on the recorded episodes, through the batched [T, G] routine of the step-wise episode loop."""
    from azul_deep_reinforcement_learning_b200.selfplay import discounted_returns
    z = load_update_golden()
    reward, done, qref = z["reward"].astype(np.float64), z["done"], z["qvals"]
    ends = np.nonzero(done)[0]
    starts = np.concatenate([[0], ends[:-1] + 1])
    T, G = int((ends - starts + 1).max()), len(ends)
    r = torch.zeros(T, G, dtype=torch.float64)
    act = torch.zeros(T, G, dtype=torch.bool)
    for g, (a, b) in enumerate(zip(starts, ends)):
        r[: b - a + 1, g] = torch.from_numpy(reward[a:b + 1])
        act[: b - a + 1, g] = True
    q = discounted_returns(r, act, float(z["gamma"]))
    for g, (a, b) in enumerate(zip(starts, ends)):
        assert np.allclose(q[: b - a + 1, g].numpy(), qref[a:b + 1], rtol=1e-12, atol=1e-9)
    assert np.allclose(z["episode_rewards"], [reward[a:b + 1].sum() for a, b in zip(starts, ends)])


def test_a2c_loss_terms_and_adam_step_match_reference_agent_update():
    """The trainer's loss (train.a2c_loss_terms: sums over decisions) / N, its autograd gradient and the Adam step
    equal what the reference's Agent.update produced on the same decisions: losses, p.grad, parameters after 1 and 2 steps."""
    from azul_deep_reinforcement_learning_b200.train import ACTOR_COEFF, CRITIC_COEFF, ENTROPY_COEFF, a2c_loss_terms
    z = load_update_golden()
    net = net_from_golden(z, "param0_", 1.0)
    opt = torch.optim.Adam(net.parameters(), lr=float(z["learning_rate"]))      # agent.py:37
    named = dict(net.named_parameters())
    for b in (0, 1):
        idx = np.nonzero(z["batch"] == b)[0]
        obs = torch.from_numpy(z["obs"][idx].astype(np.float32))
        valid = torch.from_numpy(mask_words_to_bool(z["mask"][idx]))
        action = torch.from_numpy(z["action"][idx].astype(np.int64))
        qval = torch.from_numpy(z["qvals"][idx].astype(np.float32))             # agent.py:41 FloatTensor
        if b == 0:
            # what the rollout recorded with these parameters: value, log pi(action), entropy term (nn_runner.py:32-40)
            with torch.no_grad():
                _, logp = net.forward_actor(obs, valid)
                assert torch.allclose(net.forward_critic(obs).squeeze(1), torch.from_numpy(z["value"][idx]), rtol=1e-5, atol=1e-5)
                assert torch.allclose(logp.gather(1, action[:, None]).squeeze(1), torch.from_numpy(z["logp"][idx]), rtol=1e-5, atol=1e-5)
        a, c, e = a2c_loss_terms(net, obs, valid, action, qval)
        n = float(len(idx))
        losses = z["losses"][b]                                                  # reward, actor, critic, entropy, ac
        assert abs(float(a) / n - losses[1]) <= 1e-5 * abs(losses[1])
        assert abs(float(c) / n - losses[2]) <= 1e-5 * abs(losses[2])
        assert abs(float(e) / n - losses[3]) <= 1e-5 * abs(losses[3])
        loss = (ACTOR_COEFF * a + CRITIC_COEFF * c + ENTROPY_COEFF * e) / n
        assert abs(float(loss) - losses[4]) <= 1e-5 * abs(losses[4])
        opt.zero_grad()
        loss.backward()
        if b == 0:
            for name in PARAM_NAMES:
                g, want = named[name].grad, torch.from_numpy(z["grad1_" + name])
                assert torch.allclose(g, want, rtol=1e-4, atol=1e-6 * float(want.abs().max())), name
        opt.step()
        for name in PARAM_NAMES:
            want = torch.from_numpy(z["param%d_" % (b + 1) + name])
            # an Adam step moves every parameter by ~lr * sign(g) (first step) -- entries whose gradient is at rounding
            # level may differ by up to that; everything else agrees to float precision
            diff = (named[name].detach() - want).abs()
            assert float(diff.max()) <= 2.1 * float(z["learning_rate"]) * (b + 1), name
            assert float((diff > 1e-6).float().mean()) < 2e-3, (name, float((diff > 1e-6).float().mean()))
