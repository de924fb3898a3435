"""Batched counterparts of ``GameRunner`` / ``NNRunner`` (reference game_runner.py:9-85, nn_runner.py:13-84).

``BatchedGameRunner`` is G copies of the reference's 2-player env wrapper advancing in lock-step on one
GPU: seat 1 is the learning agent, seat 2 a random agent (``RandomAgent``, game_runner.py:87-97, drawing
from the Philox schedule), the greedy agent (``azb_greedy_action``: the best one-move score) or a frozen network.
``PersistentEpisodes`` plays whole episodes in one launch of the fused policy kernel; that is how the trainer plays.  ``run_episodes`` is the step-wise loop the persistent
kernel is checked against: one agent decision costs up to three launches, the observation
(``azb_observe_bf16``, only when the caller records it), the fused policy kernel (``azb_policy_step``: MLP on
tcgen05 + masked softmax + sampling + the agent's ``Azul.step``) and the opponent loop + reward
(``azb_opponent_random`` / ``azb_opponent_greedy``).
"""
import os

import torch

from .engine import (BatchedAzul, EpisodeRecords, PackedPolicy, discounted_returns_records, mask_to_bool, policy_step,
                     rules_to_ints, runner_rollout)

DEFAULT_RULES = {"first_player": "Random", "tile_pool": "Lid"}      # game_runner.py:23
GREEDY = "greedy"                   # the opponent keyword of the greedy agent


class BatchedGameRunner:
    def __init__(self, n_games, rules=None, seed=0, device=0, game_id_base=0, opponent=None, opponent_mode=0):
        """``opponent``: None = RandomAgent (game_runner.py:29-30), ``"greedy"`` = the greedy agent, or a ``PackedPolicy`` =
        a frozen ``Agent`` (scripts/run_batch.py:6-8) whose moves come from the fused policy kernel."""
        if isinstance(opponent, str) and opponent != GREEDY:
            raise ValueError("unknown opponent %r: None (random), %r or a PackedPolicy" % (opponent, GREEDY))
        self.opponent, self.opponent_mode = opponent, opponent_mode
        rules = DEFAULT_RULES if rules is None else rules
        pool, first = rules_to_ints(2, rules)
        self.engine = BatchedAzul(n_games, 2, pool, first, seed=seed, device=device, game_id_base=game_id_base, reset=False)
        self.n_games, self.device = n_games, self.engine.device
        self.player_score = torch.zeros(n_games, dtype=torch.int16, device=self.device)
        self.mask = None
        self.reset()

    def reset(self):
        """``GameRunner.reset`` (game_runner.py:76-85): fresh games, the opponent plays until seat 1 is to move."""
        self.engine.reset()
        self.player_score.zero_()
        out = self._opponent_moves(require_two=False)
        self.player_score.zero_()                     # game_runner.py:81: the score baseline restarts at 0
        self.mask = out["mask"]
        return out

    def get_state(self):
        """``GameRunner.get_state()`` for every game: float32 [G, 136] from seat 1's perspective."""
        return self.engine.observe(0)

    def get_valid_moves(self):
        return mask_to_bool(self.mask)

    def _opponent_policy_moves(self, max_rounds=64, check_every=1):
        """``while (current_player != 1 or #valid < 2) and not end: opponent_move()`` (game_runner.py:46-47) with an
        Agent opponent: each launch lets every game that is still in the opponent's hands take one policy decision
        (``act_filter = 1``); typically one or two launches per agent decision.  The loop runs until no game acted
        (checked on the host every ``check_every`` launches: a launch in which nobody acts changes nothing); a round
        is at most 20 takes long, so ``max_rounds`` launches can only be exceeded by a bug -- that raises."""
        for i in range(max_rounds):
            out = policy_step(self.engine, self.opponent, mode=self.opponent_mode, apply_step=True, want_mask=False,
                              act_filter=1)
            if (i + 1) % check_every == 0 and not bool((out["action"] != 255).any()):
                return
        if bool((out["action"] != 255).any()):
            raise RuntimeError("opponent loop did not hand the move back to seat 1 within %d policy launches" % max_rounds)

    def _opponent_moves(self, require_two):
        """The opponent loop + reward (game_runner.py:46-52; :84-85 without ``require_two``)."""
        if self.opponent == GREEDY:
            return self.engine.opponent_greedy(self.player_score, require_two=require_two)
        if self.opponent is not None:                 # a fresh board always offers seat 1 >= 2 actions, so the
            self._opponent_policy_moves()             # ":46" and ":84" loop conditions coincide in reset
        return self.engine.opponent_random(self.player_score, require_two=require_two)

    def _after_agent_move(self):
        out = self._opponent_moves(require_two=True)
        self.mask = out["mask"]
        return out

    def step(self, actions):
        """``GameRunner.step`` (game_runner.py:43-55) with one action per game (uint8, 255 = skip that game).
        Returns dict(reward int16, done uint8, status uint8 [step status | opponent status], mask)."""
        st = self.engine.step(actions, None, want_mask=False)
        out = self._after_agent_move()
        out["status"] = out["status"] | st["status"]
        return out

    def step_policy(self, packed, mode=0):
        """Agent decision by the fused policy kernel + its env step, then the opponent loop and the reward."""
        pol = policy_step(self.engine, packed, mode=mode, apply_step=True, want_mask=False)
        out = self._after_agent_move()
        out.update(action=pol["action"], logp=pol["logp"], value=pol["value"], entropy=pol["entropy"],
                   policy_status=pol["status"])
        return out


RAW_KEYS = ("obs", "mask", "reward", "value", "logp", "entropy", "action", "status", "done")


def _one_decision(runner, packed, rec, record_obs):
    """One agent decision for every game; appends the raw outputs of the kernels (what ``NNRunner.run_episode``
    records, nn_runner.py:27-45) without any per-decision bookkeeping -- see :func:`_alive_chain`."""
    if record_obs:
        rec["obs"].append(runner.engine.observe_bf16(0))
    rec["mask"].append(runner.mask)          # every opponent_random call returns a new tensor: no copy needed
    out = runner.step_policy(packed)
    rec["reward"].append(out["reward"])
    rec["value"].append(out["value"])
    rec["logp"].append(out["logp"])
    rec["entropy"].append(out["entropy"])
    rec["action"].append(out["action"])
    rec["status"].append(out["policy_status"])
    rec["done"].append(out["done"])


def _alive_chain(status, done, alive0):
    """``active[t]`` = the game was still running when decision t was taken and a decision was taken
    (policy status without ENDED / STUCK); a game stays alive while it acts and is not done.  Vectorised over the
    decisions of a chunk: status, done uint8 [C, G]; alive0 bool [G].  Returns (active bool [C, G], alive bool [G])."""
    ok = (status & 6) == 0
    live = (ok & (done == 0)).to(torch.uint8)
    chain = torch.cummin(live, dim=0).values.bool()                       # alive after decision t (given alive0)
    before = torch.cat([torch.ones_like(chain[:1]), chain[:-1]])
    return before & ok & alive0, chain[-1] & alive0


def _finish_batch(chunks, alive):
    out = {k: torch.cat([c[k] for c in chunks]) for k in chunks[0]}
    out["reward"] = out["reward"].to(torch.float32)
    out["action"] = out["action"].to(torch.int64)
    del out["status"], out["done"]
    out["unfinished"] = int(alive.sum())
    return out


def _stack_chunk(rec, alive):
    chunk = {k: torch.stack(v) for k, v in rec.items() if v}
    chunk["active"], alive = _alive_chain(chunk["status"], chunk["done"], alive)
    return chunk, alive


def run_episodes(runner, packed, max_decisions=160, check_every=8, record_obs=True):
    """``NNRunner.run_episode`` for every game of ``runner`` at once (nn_runner.py:17-47).

    Returns a dict of [T, G] tensors: reward (float32), value, logp, entropy (from the kernel), action
    (int64), active (bool: the game was still running when the decision was taken), mask (int32
    [T, 6, G] legal-mask words) and, when ``record_obs``, obs (bfloat16 [T, G, 136]) for the autograd
    recomputation."""
    G, dev = runner.n_games, runner.device
    runner.reset()
    alive = torch.ones(G, dtype=torch.bool, device=dev)
    chunks, t = [], 0
    while t < max_decisions:
        rec = {k: [] for k in RAW_KEYS}
        for _ in range(min(check_every, max_decisions - t)):
            _one_decision(runner, packed, rec, record_obs)
        t += check_every
        chunk, alive = _stack_chunk(rec, alive)
        chunks.append(chunk)
        if not bool(alive.any()):
            break
    return _finish_batch(chunks, alive)


class PersistentEpisodes:
    """``NNRunner.run_episode`` for every game slot with the whole episode loop on the device: ``GameRunner.reset`` (a few
    launches), then ONE persistent launch of the fused policy kernel that takes every agent decision, plays the opponent's
    moves, takes the rewards and writes the decision records, then the discounted returns (one launch).  The recorded
    decisions are those of :func:`run_episodes` (same Philox schedule); only their storage differs (compact slots in
    arbitrary order instead of [T, G]).

    The opponent is the runner's: the random agent (``runner.opponent`` None), the greedy agent (``"greedy"``) or a frozen
    network (a ``PackedPolicy``, ``GameRunner(opponent=Agent(...))``), which then plays with the same selection mode as the
    agent.  Nothing in :meth:`run` waits for the GPU, so a whole batch can be captured in a CUDA graph."""

    def __init__(self, runner, packed, max_decisions=160, capacity=None, want_logp_value=False):
        self.runner, self.packed = runner, packed
        n = runner.n_games
        if capacity is None:                       # ~30 decisions per episode on average; small batches get the full K x G
            capacity = max_decisions * n if n <= 4096 else 56 * n
        self.records = EpisodeRecords(runner.engine, max_decisions, capacity, want_logp_value)
        self.out = {"mask": torch.zeros((6, n), dtype=torch.int32, device=runner.device),
                    "done": torch.zeros(n, dtype=torch.uint8, device=runner.device),
                    "status": torch.zeros(n, dtype=torch.uint8, device=runner.device)}
        # policy opponent: the most opponent passes one decision of the last run needed
        self.opp_passes = torch.zeros(1, dtype=torch.int32, device=runner.device)

    def start(self, mode=0):
        """``GameRunner.reset`` (game_runner.py:76-85) for every slot.  Against a policy opponent without the host reads of
        ``BatchedGameRunner.reset``: on a fresh board the opponent moves at most once before seat 1 is to move with >= 2
        legal actions, so ONE opponent launch replaces its loop; the resulting state is the same."""
        runner = self.runner
        if not isinstance(runner.opponent, PackedPolicy):        # the random or the greedy agent: no host reads
            return runner.reset()
        e = runner.engine
        e.reset()
        runner.player_score.zero_()
        policy_step(e, runner.opponent, mode=mode, apply_step=True, want_mask=False, act_filter=1)
        out = e.opponent_random(runner.player_score, require_two=False)
        runner.player_score.zero_()                  # game_runner.py:81: the score baseline restarts at 0
        runner.mask = out["mask"]
        return out

    def run(self, gamma=0.99, mode=0):
        opponent = self.runner.opponent
        policy = isinstance(opponent, PackedPolicy)
        if policy and self.runner.opponent_mode != mode:
            raise ValueError("the persistent rollout plays both seats with one selection mode: agent mode %d, opponent mode %d"
                             % (mode, self.runner.opponent_mode))
        r = self.records
        self.start(mode)
        r.clear()
        if policy:
            self.opp_passes.zero_()
        runner_rollout(self.runner.engine, self.packed, r, self.runner.player_score, mode=mode, out=self.out,
                       opponent=opponent, opp_passes=self.opp_passes if policy else None)
        discounted_returns_records(self.runner.engine, r, gamma)
        self.runner.mask = self.out["mask"]
        return r


def load_network(net, device=None):
    """An ``ActorCritic`` from a module, a ``state_dict``, a trainer checkpoint dict (``{"ac_net": ...}``) or a file path (every
    format ``Agent(base_net_file=...)`` accepts, through ``azulnet.agent.load_ac_net``)."""
    from .azulnet.agent import load_ac_net
    from .azulnet.model import ActorCritic
    if isinstance(net, (str, os.PathLike)):
        net = load_ac_net(os.fspath(net))
    elif isinstance(net, dict):
        sd = net["ac_net"] if "ac_net" in net else net
        net = ActorCritic(136, 180)
        net.load_state_dict(sd)
    elif not isinstance(net, torch.nn.Module):
        raise TypeError("expected an ActorCritic, a state_dict or a file path, got %r" % type(net).__name__)
    return net.to(device) if device is not None else net


def resolve_opponent(engine, opponent, device=None):
    """The runner's opponent for an opponent choice: None (the random agent) stays None, ``"greedy"`` selects the greedy
    agent (a checkpoint file of that name is passed as ``./greedy``), anything else is a network (``load_network``) packed
    for the policy kernel of ``engine``."""
    if opponent is None or (isinstance(opponent, str) and opponent == GREEDY):
        return opponent
    return PackedPolicy(engine, load_network(opponent, device))


def discounted_returns(reward, active, gamma):
    """q_t = r_t + gamma * q_{t+1} per episode (nn_runner.py:72-75), [T, G]; inactive slots contribute 0."""
    T = reward.shape[0]
    q = torch.zeros_like(reward)
    run = torch.zeros_like(reward[0])
    r = reward * active
    for t in range(T - 1, -1, -1):
        run = r[t] + gamma * run
        q[t] = run
    return q
