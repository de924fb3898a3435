"""Host-side training logic on CPU: the batched A2C loss equals ``Agent.update``'s (agent.py:39-62) on the same
transitions, discounted returns follow nn_runner.py:72-75, and the 2-rank gradient all-reduce (gloo)
reproduces the single-process global-batch gradient."""
import os
import sys

import numpy as np
import torch
import torch.multiprocessing as mp

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _fake_batch(n, seed):
    g = torch.Generator().manual_seed(seed)
    obs = torch.randint(0, 5, (n, 136), generator=g).float()
    mask = torch.rand(n, 180, generator=g) < 0.15
    mask[:, 0] = True
    action = torch.multinomial(mask.float(), 1, generator=g).squeeze(1)
    qval = torch.randn(n, generator=g) * 3
    return obs, mask, action, qval


def test_batched_loss_equals_agent_update_formula():
    from azul_deep_reinforcement_learning_b200.azulnet.model import ActorCritic
    from azul_deep_reinforcement_learning_b200.train import ACTOR_COEFF, CRITIC_COEFF, ENTROPY_COEFF, a2c_loss_terms
    torch.manual_seed(0)
    net = ActorCritic(136, 180)
    obs, mask, action, qval = _fake_batch(57, 1)
    a, c, e = a2c_loss_terms(net, obs, mask, action, qval)
    loss = (ACTOR_COEFF * a + CRITIC_COEFF * c + ENTROPY_COEFF * e) / 57
    grads = torch.autograd.grad(loss, list(net.parameters()))
    # the reference formulation: per-decision lists, then Agent.update's means (agent.py:39-57)
    values, log_probs, entropy = [], [], []
    for i in range(57):
        s = obs[i:i + 1]
        values.append(net.forward_critic(s))
        _, logp = net.forward_actor(s, mask[i:i + 1])
        log_probs.append(logp.squeeze(0)[action[i]])
        entropy.append(-logp.masked_select(mask[i:i + 1]).mean())
    v = torch.stack(values).squeeze(2)
    adv = qval.reshape(-1, 1) - v
    ref = (-torch.stack(log_probs) * adv.squeeze(1)).mean() + 0.5 * adv.pow(2).mean() + 0.1 * torch.stack(entropy).mean()
    ref_grads = torch.autograd.grad(ref, list(net.parameters()))
    assert abs(float(loss) - float(ref)) < 1e-4 * max(1.0, abs(float(ref)))
    for g1, g2 in zip(grads, ref_grads):
        assert torch.allclose(g1, g2, rtol=1e-4, atol=1e-5)


def test_alive_chain_equals_the_sequential_bookkeeping():
    """The vectorised `active` / `alive` flags of a chunk of decisions equal the per-decision recurrence
    acted = alive & ok; alive = acted & ~done (what NNRunner.run_episode's while-loop does per game)."""
    from azul_deep_reinforcement_learning_b200.selfplay import _alive_chain
    g = torch.Generator().manual_seed(4)
    C, G = 13, 257
    status = (torch.rand(C, G, generator=g) < 0.08).to(torch.uint8) * 2 + (torch.rand(C, G, generator=g) < 0.05).to(torch.uint8) * 4
    done = (torch.rand(C, G, generator=g) < 0.1).to(torch.uint8)
    alive0 = torch.rand(G, generator=g) < 0.8
    active, alive = _alive_chain(status, done, alive0)
    a = alive0.clone()
    for t in range(C):
        acted = a & ((status[t] & 6) == 0)
        assert torch.equal(active[t], acted), t
        a = acted & ~done[t].bool()
    assert torch.equal(alive, a)


def test_network_outputs_match_the_module():
    """train.network_outputs (custom Linear with a GEMM bias gradient) == the nn.Module forward, values and gradients."""
    from azul_deep_reinforcement_learning_b200.azulnet.model import ActorCritic
    from azul_deep_reinforcement_learning_b200.train import network_outputs
    torch.manual_seed(5)
    net = ActorCritic(136, 180)
    x = torch.randn(37, 136)
    gl, gv = torch.randn(37, 180), torch.randn(37)
    logits = net.actor_linear2(torch.relu(net.actor_linear1(x)))
    value = net.forward_critic(x).squeeze(1)
    torch.autograd.backward([logits, value], [gl, gv])
    want = [p.grad.clone() for p in net.parameters()]
    net.zero_grad()
    l2, v2 = network_outputs(net, x)
    assert torch.allclose(l2, logits, atol=1e-6) and torch.allclose(v2, value, atol=1e-6)
    torch.autograd.backward([l2, v2], [gl, gv])
    for p, w in zip(net.parameters(), want):
        assert torch.allclose(p.grad, w, rtol=1e-5, atol=1e-6), p.shape


def test_discounted_returns():
    from azul_deep_reinforcement_learning_b200.selfplay import discounted_returns
    r = torch.tensor([[1.0, 2.0], [0.0, -1.0], [3.0, 5.0]])
    act = torch.tensor([[True, True], [True, True], [True, False]])
    q = discounted_returns(r, act, 0.99)
    assert torch.allclose(q[:, 0], torch.tensor([1 + 0.99 * (0 + 0.99 * 3), 0 + 0.99 * 3, 3.0]))
    assert torch.allclose(q[:2, 1], torch.tensor([2 + 0.99 * -1.0, -1.0]))


def _worker(rank, world, port, out_dir):
    sys.path.insert(0, REPO)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    from azul_deep_reinforcement_learning_b200 import parallel
    from azul_deep_reinforcement_learning_b200.azulnet.model import ActorCritic
    from azul_deep_reinforcement_learning_b200.engine import PARAM_ORDER
    from azul_deep_reinforcement_learning_b200.train import a2c_loss_terms, allreduce_flat_and_stats
    parallel.init("gloo")
    torch.manual_seed(0)
    net = ActorCritic(136, 180)
    n = 40 + 25 * rank                                      # ranks hold different numbers of transitions
    obs, mask, action, qval = _fake_batch(n, 10 + rank)
    # the trainer's form: unscaled gradient sums in ONE flat fp32 buffer (PARAM_ORDER) + the count in the statistics
    # vector, both all-reduced, then divided by the global count
    a, c, e = a2c_loss_terms(net, obs, mask, action, qval)
    (a + 0.5 * c + 0.1 * e).backward()
    named = dict(net.named_parameters())
    flat = torch.cat([named[name].grad.reshape(-1) for name in PARAM_ORDER]).float()
    stats = torch.tensor([float(n), 7.0 + rank], dtype=torch.float64)
    allreduce_flat_and_stats(flat, stats)
    assert stats.tolist() == [105.0, 15.0]
    flat /= stats[0].float()
    grads, off = {}, 0
    for name in PARAM_ORDER:
        k = named[name].numel()
        grads[name] = flat[off:off + k].view_as(named[name])
        off += k
    torch.save([grads[name] for name, _ in net.named_parameters()], os.path.join(out_dir, "grads%d.pt" % rank))
    torch.distributed.destroy_process_group()


def test_two_rank_flat_gradient_allreduce_matches_global_batch(tmp_path):
    from azul_deep_reinforcement_learning_b200.azulnet.model import ActorCritic
    from azul_deep_reinforcement_learning_b200.train import a2c_loss_terms
    from tests.helpers import free_port
    mp.spawn(_worker, args=(2, free_port(), str(tmp_path)), nprocs=2, join=True)
    torch.manual_seed(0)
    net = ActorCritic(136, 180)
    parts = [_fake_batch(40, 10), _fake_batch(65, 11)]
    obs, mask, action, qval = [torch.cat([p[i] for p in parts]) for i in range(4)]
    a, c, e = a2c_loss_terms(net, obs, mask, action, qval)
    ref = torch.autograd.grad((a + 0.5 * c + 0.1 * e) / 105, list(net.parameters()))
    for r in range(2):
        got = torch.load(tmp_path / ("grads%d.pt" % r))
        for g1, g2 in zip(got, ref):
            assert torch.allclose(g1, g2, rtol=1e-4, atol=1e-6), r


def _flat_worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    sys.path.insert(0, REPO)
    import torch.distributed as dist
    from azul_deep_reinforcement_learning_b200.train import allreduce_flat_and_stats
    dist.init_process_group("gloo")
    g = torch.Generator().manual_seed(100 + rank)
    flat = torch.randn(82081, generator=g)
    stats = torch.tensor([10.0 + rank, 1.5 * (rank + 1)], dtype=torch.float64)
    allreduce_flat_and_stats(flat, stats)
    if rank == 0:
        # by value: a torch tensor in a multiprocessing queue travels as a handle into the SENDER's shared memory, which
        # is gone if this process exits before the parent has rebuilt it
        out.put((flat.numpy().copy(), str(flat.dtype), stats.tolist()))
    dist.destroy_process_group()


def test_flat_gradient_and_stats_allreduce_two_ranks_gloo():
    """The trainer's collectives (one flat fp32 gradient all-reduce + one float64 statistics all-reduce) on two gloo ranks."""
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    from tests.helpers import free_port
    port = free_port()
    procs = [ctx.Process(target=_flat_worker, args=(r, 2, port, out)) for r in range(2)]
    for p in procs:
        p.start()
    flat, flat_dtype, stats = out.get(timeout=120)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    want = sum(torch.randn(82081, generator=torch.Generator().manual_seed(100 + r)) for r in range(2))
    assert torch.allclose(torch.from_numpy(flat), want) and flat_dtype == "torch.float32"
    assert stats == [21.0, 4.5]


def test_saved_networks_load_back_through_agent(tmp_path):
    """Every format the package (or the reference, nn_runner.py:83-84 / agent.py:36) writes loads back through
    ``Agent(base_net_file=...)``: pickled module (.mx), bare state_dict (.pt), trainer checkpoint dict (.pt)."""
    from azul_deep_reinforcement_learning_b200.azulnet.agent import Agent
    from azul_deep_reinforcement_learning_b200.azulnet.model import ActorCritic
    torch.manual_seed(11)
    net = ActorCritic(136, 180)
    want = {k: v.clone() for k, v in net.state_dict().items()}
    torch.save(net, str(tmp_path / "module.mx"))
    torch.save(net.state_dict(), str(tmp_path / "bare.pt"))
    torch.save({"ac_net": net.state_dict(), "optimizer": torch.optim.Adam(net.parameters()).state_dict(), "batch": 7},
               str(tmp_path / "ckpt.pt"))
    for name in ("module.mx", "module", "bare.pt", "bare", "ckpt.pt", "ckpt"):
        a = Agent(base_net_file=str(tmp_path / name))
        got = a.ac_net.state_dict()
        assert set(got) == set(want) and all(torch.equal(got[k], want[k]) for k in want), name
        assert len(a.ac_optimizer.param_groups[0]["params"]) == 8
