"""Self-play A2C training on the GPU rollout engine -- the ``scripts/training.py`` / ``NNRunner.train``
equivalent (reference scripts/training.py:8-22, nn_runner.py:53-84, agent.py:39-62).

    python -m azul_deep_reinforcement_learning_b200.train [batch_size] [net_name] [--batches N]
                                                      [--opponent FILE|greedy] [--opponent-refresh N]
                                                      [--self-play] [--eval-every N] [--eval-games E]
    torchrun --nproc-per-node 8 -m azul_deep_reinforcement_learning_b200.train 1024 run1

``batch_size`` episodes are played IN PARALLEL per rank (one game slot each) instead of one after the
other; everything else follows the reference: discounted returns with gamma = 0.99, the loss of
``Agent.update`` (advantage not detached in the actor term, "entropy" = -mean(log pi over legal moves)
added with +0.1), Adam(lr 3e-4).  Rollouts are one launch of the persistent fused tensor-core policy kernel per batch
(fp16 operands, fp32 accumulation); the update recomputes the forward pass and runs the whole backward pass on the
recorded decision states with hand-written tcgen05 kernels (azb_a2c_update_gradients).  With several ranks each one plays
its own shard of the global game-id range and the only collectives are one flat fp32 gradient all-reduce per update (C1,
82,081 values) and the statistics reduction (C2, 18 float64).
"""
import argparse
import csv
import os
import time

import torch
import torch.distributed as dist

from . import parallel
from .azulnet.model import ActorCritic
from .engine import PackedPolicy, UpdateGradients, train_stats
from .selfplay import GREEDY, BatchedGameRunner, PersistentEpisodes, SelfPlayEpisodes, resolve_opponent

ACTOR_COEFF, CRITIC_COEFF, ENTROPY_COEFF = 1.0, 0.5, 0.1          # agent.py:47-49


def a2c_loss_terms(net, obs, mask, action, qval):
    """Sums (not means) of the three loss terms of ``Agent.update`` over N transitions (agent.py:45-56).

    obs [N,136] float32, mask [N,180] bool, action [N] int64, qval [N] float32.  Returned as sums so that
    several ranks can divide by the GLOBAL transition count and all-reduce exact global-batch gradients."""
    value = net.forward_critic(obs).squeeze(1)
    logits = net.actor_linear2(torch.relu(net.actor_linear1(obs))).masked_fill(~mask, float("-inf"))
    logp_all = torch.log_softmax(logits, dim=1)
    log_prob = logp_all.gather(1, action[:, None]).squeeze(1)                     # nn_runner.py:32
    entropy = -(logp_all.masked_fill(~mask, 0.0).sum(dim=1) / mask.sum(dim=1))    # nn_runner.py:36-40
    advantage = qval - value                                                      # agent.py:45 (not detached)
    return (-log_prob * advantage).sum(), advantage.pow(2).sum(), entropy.sum()


class _Linear(torch.autograd.Function):
    """``x @ w.T + b`` whose bias gradient is a GEMM with a row of ones (tensor cores) instead of autograd's column
    reduction over the [N, out] gradient -- a fifth of the update's GPU time at 5*10^5 decisions."""

    @staticmethod
    def forward(ctx, x, w, b):
        ctx.save_for_backward(x, w)
        return torch.addmm(b, x, w.t())

    @staticmethod
    def backward(ctx, dy):
        x, w = ctx.saved_tensors
        dx = dy @ w if ctx.needs_input_grad[0] else None
        dw = dy.t() @ x
        db = (torch.ones(1, dy.shape[0], dtype=dy.dtype, device=dy.device) @ dy).squeeze(0)
        return dx, dw, db


def network_outputs(net, x):
    """(logits [N,180] raw, value [N]) of ``ActorCritic`` (model.py:23-41 before the mask) through :class:`_Linear`."""
    lin = _Linear.apply
    logits = lin(torch.relu(lin(x, net.actor_linear1.weight, net.actor_linear1.bias)), net.actor_linear2.weight, net.actor_linear2.bias)
    value = lin(torch.relu(lin(x, net.critic_linear1.weight, net.critic_linear1.bias)), net.critic_linear2.weight, net.critic_linear2.bias)
    return logits, value.squeeze(1)


def allreduce_flat_and_stats(flat, stats):
    """What the trainer does per update, in place: C1 = ONE fp32 all-reduce of the flat gradient buffer (82,081 sums), C2 =
    one float64 all-reduce of the statistics vector.  No-op for a single process."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(flat, op=dist.ReduceOp.SUM)
        dist.all_reduce(stats, op=dist.ReduceOp.SUM)
    return flat, stats


STAT_FIELDS = 18        # n_decisions, 3 loss sums, reward sum, games, 10 game statistics sums, wins, unfinished


def summarize_stats(s, update_sync_s=None):
    """The STAT_FIELDS sums (``azb_train_stats`` order) -> the per-batch numbers: mean losses per decision, and per game the
    reward and the ``GameStatistics`` fields (agent.py:12, game_runner.py:10-22)."""
    n_global, games = max(s[0], 1.0), s[5]
    out = {"transitions": s[0], "games": games, "actor_loss": s[1] / n_global, "critic_loss": s[2] / n_global,
           "entropy_loss": s[3] / n_global, "reward": s[4] / games}
    if update_sync_s is not None:
        out["update_sync_s"] = update_sync_s
    out["ac_loss"] = ACTOR_COEFF * out["actor_loss"] + CRITIC_COEFF * out["critic_loss"] + ENTROPY_COEFF * out["entropy_loss"]
    g = [x / games for x in s[6:16]]
    out.update(player_score=g[0], opponent_score=g[1], rounds=g[2],
               percent_first_player=100.0 * s[9] / max(s[10], 1.0), floor_penalty=g[5], max_combo=g[6],
               completed_rows=g[7], completed_columns=g[8], completed_colors=g[9])
    out["win_percent"] = s[16] / games
    out["unfinished"] = int(s[17])
    return out


EVAL_FIELDS = ("eval_win_percent", "eval_player_score", "eval_opponent_score")     # train(eval_every=N) columns


class SelfPlayTrainer:
    """``NNRunner.train`` (nn_runner.py:53-84) with ``games_per_rank`` episodes played in parallel per rank.

    :meth:`rollout` plays the whole batch in one launch of the persistent fused policy kernel (``PersistentEpisodes``) and
    returns its compact decision records; :meth:`update` runs ``Agent.update`` on them with ``azb_a2c_update_gradients``
    (hand-written tcgen05 forward / backward).  :meth:`enable_step_graph` captures both as one CUDA graph.
    :meth:`update_decisions` (PyTorch autograd over cuBLAS GEMMs, TF32 or -- ``tf32_update=False`` -- fp32) and
    :meth:`update_states` (the tensor-core kernels) run one ``Agent.update`` on explicitly given decisions: the entry points
    the tests hold against the reference.

    ``opponent``: None plays the random agent (``RandomAgent``); ``"greedy"`` the greedy agent (the best one-move score, a
    fixed-strength yardstick); an ``ActorCritic``, a ``state_dict`` or a file path (anything ``Agent(base_net_file=...)``
    loads) plays a frozen network in seat 2 (``GameRunner(opponent=Agent(...))``), sampling like the agent.  ``opponent_refresh`` = N > 0: the opponent's weights are replaced by the current network's
    after every N batches -- self-play against a lagged copy of itself.

    ``self_play=True``: the network plays BOTH seats (``SelfPlayEpisodes``, one persistent launch per batch) and learns from
    every decision with a choice, seat 2's included; it takes no ``opponent`` or ``opponent_refresh``.  ``max_decisions``
    then bounds the moves of both seats together (default 320; 160 agent decisions otherwise).  The batch statistics keep
    their meaning -- seat 1 against seat 2, decisions of both seats -- so ``reward`` is 0 when every episode finished (the
    two seats' rewards cancel) and the scores and ``win_percent`` are symmetric up to noise: ``train(eval_every=N)``
    measures progress against the greedy agent instead."""

    def __init__(self, games_per_rank=1024, learning_rate=3e-4, gamma=0.99, seed=0, device=0, rank=0, world=1,
                 rules=None, max_decisions=None, tf32_update=True, opponent=None, opponent_refresh=0, self_play=False):
        if self_play and (opponent is not None or opponent_refresh):
            raise ValueError("self_play plays both seats with the network: it takes no opponent or opponent_refresh")
        self.rank, self.world, self.gamma = rank, world, gamma
        self.rules, self.self_play = rules, bool(self_play)
        self.tf32_update = tf32_update
        self.device = torch.device("cuda", device)
        torch.manual_seed(seed)                              # identical initial weights on every rank
        self.net = ActorCritic(136, 180).to(self.device)
        self.params = list(self.net.parameters())
        self.opt = torch.optim.Adam(self.params, lr=learning_rate, fused=True, capturable=True)   # agent.py:37 (one fused kernel; graph-capturable)
        self.runner = BatchedGameRunner(games_per_rank, rules=rules, seed=seed, device=device,
                                        game_id_base=parallel.shard(rank, games_per_rank))
        self.packed = PackedPolicy(self.runner.engine, self.net)
        self.opponent, self.opponent_refresh, self.batches_done = None, int(opponent_refresh), 0
        is_greedy = isinstance(opponent, str) and opponent == GREEDY
        if opponent_refresh and is_greedy:
            raise ValueError("opponent_refresh replaces a network opponent: the greedy agent has no weights")
        if opponent_refresh and opponent is None:
            opponent = self.net                              # a lagged copy of the network itself
        # a network is packed once into its own fixed buffer: a captured batch reads it there, a refresh re-packs it in place
        self.runner.opponent, self.runner.opponent_mode = resolve_opponent(self.runner.engine, opponent, self.device), 0
        if isinstance(self.runner.opponent, PackedPolicy):
            self.opponent = self.runner.opponent
        if self.self_play:
            self.episodes = SelfPlayEpisodes(self.runner.engine, self.packed, max_decisions=max_decisions or 320)
        else:
            self.episodes = PersistentEpisodes(self.runner, self.packed, max_decisions=max_decisions or 160)
        # every parameter gradient is a view into ONE flat fp32 buffer (PARAM_ORDER): the tensor-core kernels add into
        # it, autograd accumulates into the views in place, and the gradient all-reduce is a single collective on it
        self.tc = UpdateGradients(self.runner.engine, self.episodes.records.cap)
        for name, p in self.net.named_parameters():
            p.grad = self.tc.grads[name]
        self._host_stats = torch.zeros((2, STAT_FIELDS), dtype=torch.float64).pin_memory()
        self._pending = []                                   # (slot, event) of statistics on their way to the host
        self._slot = 0
        self._graph = None
        self.history = []

    # ---- rollout ---------------------------------------------------------------------------
    def rollout(self):
        """Every game slot plays one episode; returns the ``EpisodeRecords`` of the agent's decisions (self-play: both
        seats') with their discounted returns."""
        with torch.no_grad():
            self.packed.update(self.net)
            return self.episodes.run(self.gamma)

    def load_parameters(self, state_dict):
        """Replace the network parameters (e.g. a checkpoint or a reference ``ac_net.state_dict()``); Adam restarts."""
        self.net.load_state_dict({k: v.to(self.device) for k, v in state_dict.items()})
        self.opt = torch.optim.Adam(self.params, lr=self.opt.param_groups[0]["lr"], fused=True, capturable=True)
        self._graph = None

    # ---- gradients -------------------------------------------------------------------------
    def accumulate_gradients(self, obs, masks, action, qval, chunk=1 << 18):
        """The "autograd" path: forward recomputation + the loss of ``Agent.update`` (agent.py:45-56) + back-propagation
        for N recorded decisions: obs bfloat16 / float32 [N,136], masks int32 [N,6] (legal-mask words), action int64 [N],
        qval float32 [N].  Leaves the SUMS over the decisions (not yet divided by a count) in ``p.grad`` and returns the
        float64 [3] sums of the actor / critic / entropy terms.  The dense layers run through cuBLAS (TF32 or fp32);
        everything between the network outputs and the loss is one kernel (azb_a2c_loss_grad)."""
        self.tc.flat.zero_()
        sums = torch.zeros(3, dtype=torch.float64, device=self.device)
        tf32 = torch.backends.cuda.matmul.allow_tf32
        torch.backends.cuda.matmul.allow_tf32 = self.tf32_update
        try:
            for lo in range(0, int(obs.shape[0]), chunk):
                x = obs[lo:lo + chunk].float()
                logits, value = network_outputs(self.net, x)
                dlogits, dvalue = self.runner.engine.a2c_loss_grad(
                    logits.detach(), value.detach().contiguous(), masks[lo:lo + chunk].contiguous(), action[lo:lo + chunk],
                    qval[lo:lo + chunk], 1.0, (ACTOR_COEFF, CRITIC_COEFF, ENTROPY_COEFF), sums)
                torch.autograd.backward([logits, value], [dlogits, dvalue])
        finally:
            torch.backends.cuda.matmul.allow_tf32 = tf32
        return sums

    def _step(self, n, sums):
        for p in self.params:
            p.grad.mul_(1.0 / n)
        self.last_grads = {name: p.grad.clone() for name, p in self.net.named_parameters()}
        self.opt.step()
        a, c, e = (sums / n).cpu().tolist()
        return {"actor_loss": a, "critic_loss": c, "entropy_loss": e,
                "ac_loss": ACTOR_COEFF * a + CRITIC_COEFF * c + ENTROPY_COEFF * e}

    def update_decisions(self, obs, masks, action, qval):
        """One single-process ``Agent.update`` (agent.py:39-62) on N explicitly given decisions through the autograd path:
        means over the N decisions, Adam step.  Returns the loss statistics of agent.py:58-59; ``self.last_grads`` holds
        the mean gradients."""
        return self._step(int(obs.shape[0]), self.accumulate_gradients(obs, masks, action, qval))

    def update_states(self, state_rec, action, qval):
        """:meth:`update_decisions` through the tensor-core path: state_rec int32 [17, N] (packed states the decisions
        were taken on), action uint8 [N], qval float32 [N]."""
        n = int(state_rec.shape[1])
        tc = self.tc if self.tc.cap == n else UpdateGradients(self.runner.engine, n)
        self.packed.update(self.net)
        tc.run(self.packed, state_rec.contiguous(), action, qval, n_fixed=n, coeffs=(ACTOR_COEFF, CRITIC_COEFF, ENTROPY_COEFF))
        if tc is not self.tc:
            self.tc.flat.copy_(tc.flat)
        return self._step(n, tc.sums)

    # ---- update ----------------------------------------------------------------------------
    def update(self, batch, defer_stats=False):
        """``Agent.update`` (agent.py:39-62) on the decision records of :meth:`rollout` (see :meth:`_update_device`);
        then the statistics start their way to the host."""
        self._push_stats(self._update_device(batch))
        return None if defer_stats else self.fetch_stats()

    def _push_stats(self, stats):
        slot = self._slot
        self._slot ^= 1
        self._host_stats[slot].copy_(stats, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
        self._pending.append((slot, ev))

    # ---- the whole batch as one CUDA graph ----------------------------------------------------
    def enable_step_graph(self, warmup=2):
        """Capture rollout + update (every launch of a batch, collectives and the fused Adam step included) in ONE CUDA
        graph: a batch is then a single graph launch (the ~60 small launches of a batch otherwise leave the GPU idle for a
        fifth of the step).  Nothing in a batch waits for the host."""
        for _ in range(warmup):
            self.update(self.rollout())
            self._batch_done()
        torch.cuda.synchronize(self.device)
        self._graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self._graph):
            self._graph_stats = self._update_device(self.rollout())
        return self

    def step(self, defer_stats=False):
        """One training batch: rollout + update (one graph launch when :meth:`enable_step_graph` was called)."""
        if self._graph is not None:
            self._graph.replay()
            self._push_stats(self._graph_stats)
            self._batch_done()
            return None if defer_stats else self.fetch_stats()
        out = self.update(self.rollout(), defer_stats)
        self._batch_done()
        return out

    def _batch_done(self):
        """Every ``opponent_refresh`` batches the opponent's image is re-packed from the current network: one launch of its
        own, outside a captured batch, into the buffer that batch reads -- the next replay plays against the new weights."""
        self.batches_done += 1
        if self.opponent is not None and self.opponent_refresh > 0 and self.batches_done % self.opponent_refresh == 0:
            with torch.no_grad():
                self.opponent.update(self.net)

    def _update_device(self, recs):
        """``Agent.update`` (agent.py:39-62) on the ``EpisodeRecords`` of a rollout; returns the device statistics.

        Gradients are accumulated as SUMS over the local decisions in the flat fp32 buffer; one fp32 all-reduce carries
        them and a tiny float64 one the decision count and the batch statistics; every rank then divides by the global
        count (the means of agent.py:47-56 over the global batch) and takes the same Adam step.  Nothing here waits for
        the GPU: the statistics travel to pinned host memory asynchronously and are read by :meth:`fetch_stats`
        (``defer_stats=True``: later -- the training loop reads them one batch late -- otherwise right away)."""
        self.tc.run(self.packed, recs.state_rec, recs.action_rec, recs.qval, n_dec=recs.meta[:1],
                    coeffs=(ACTOR_COEFF, CRITIC_COEFF, ENTROPY_COEFF))
        stats = train_stats(self.runner.engine, recs, self.tc.sums,
                            torch.empty(STAT_FIELDS, dtype=torch.float64, device=self.device))
        allreduce_flat_and_stats(self.tc.flat, stats)                    # C1: 82,081 fp32 gradient sums, C2: 18 float64 counters
        self.tc.flat.mul_((1.0 / stats[0].clamp_min(1.0)).float())
        self.opt.step()
        return stats

    def fetch_stats(self):
        """Statistics of the oldest update whose numbers have not been read yet (waits for that copy only)."""
        slot, ev = self._pending.pop(0)
        t0 = time.perf_counter()
        ev.synchronize()
        s = self._host_stats[slot].tolist()
        if s[17] >= 1e9:
            raise RuntimeError("decision records overflowed their capacity (raise max_decisions / capacity)")
        return summarize_stats(s, update_sync_s=time.perf_counter() - t0)

    def save_checkpoint(self, path, batch):
        """``<net_name>.pt``: network ``state_dict`` (parameter names of model.py:17-21, loadable by
        ``Agent(base_net_file=...)``), optimiser state and the number of batches done (nn_runner.py:83-84 saves the
        pickled module instead)."""
        torch.save({"ac_net": {k: v.detach().cpu() for k, v in self.net.state_dict().items()},
                    "optimizer": self.opt.state_dict(), "batch": int(batch)}, path)

    def load_checkpoint(self, path):
        """Resume from :meth:`save_checkpoint` output (or from any file ``Agent(base_net_file=...)`` accepts: then Adam
        restarts).  Returns the number of batches already done."""
        from .azulnet.agent import load_ac_net
        obj = torch.load(path, map_location="cpu", weights_only=False)
        if isinstance(obj, dict) and "ac_net" in obj:
            self.net.load_state_dict({k: v.to(self.device) for k, v in obj["ac_net"].items()})
            if "optimizer" in obj:
                self.opt.load_state_dict(obj["optimizer"])
            self._graph = None                               # a captured batch refers to the old optimiser state
            return int(obj.get("batch", 0))
        self.load_parameters(load_ac_net(path).state_dict())
        return 0

    def evaluate_greedy(self, games=2048):
        """The current network (seat 1, argmax) against the greedy agent over ``games`` episodes: the ``EVAL_FIELDS``."""
        from .evaluate import evaluate
        ev = evaluate(self.net, "greedy", games=games, mode=1, seed=self.rank, device=self.device.index, rules=self.rules)
        return {"eval_win_percent": ev["win_percent"], "eval_player_score": ev["player_score"],
                "eval_opponent_score": ev["opponent_score"]}

    def train(self, batches=1000, net_name=None, log=print, start_batch=0, checkpoint_every=1000, graph=True, eval_every=0,
              eval_games=2048):
        """Batches ``start_batch + 1 .. batches``.  With ``net_name``: one CSV row per batch in ``<net_name>.csv``
        (appended to when resuming) and ``<net_name>.pt`` every ``checkpoint_every`` batches and at the end.  The host
        never waits for the batch it just launched: a batch's statistics are read (and logged) while the next one runs.

        ``eval_every`` = N > 0: after every N-th batch rank 0 plays :meth:`evaluate_greedy` (``eval_games`` episodes) with
        the network that batch produced; every row then has the ``EVAL_FIELDS`` columns, blank between evaluations.  An
        evaluation waits for the GPU, and its time counts towards the evaluated batch's ``batch_s``."""
        if eval_every < 0:
            raise ValueError("eval_every must be >= 0")
        writer = fh = None
        marks = []                                           # (batch number, host time at launch, evaluation or None)

        def finish(b, t_launch, ev):
            nonlocal writer, fh
            st = self.fetch_stats()
            now = time.perf_counter()
            st.update(batch=b, batch_s=now - t_launch, games_per_sec=st["games"] / max(now - t_launch, 1e-9))
            if eval_every > 0:
                st.update(ev or dict.fromkeys(EVAL_FIELDS))
            self.history.append(st)
            if self.rank != 0:
                return
            if net_name is not None:
                if writer is None:
                    resume = start_batch > 0 and os.path.exists(net_name + ".csv")
                    fh = open(net_name + ".csv", "a" if resume else "w", newline="")
                    writer = csv.DictWriter(fh, fieldnames=list(st.keys()))
                    if not resume:
                        writer.writeheader()
                writer.writerow(st)
                fh.flush()
            if log:
                log("batch %d: %.0f games/s  reward %.2f  score %.1f vs %.1f  win %.1f%%  loss %.3f" % (
                    b, st["games_per_sec"], st["reward"], st["player_score"], st["opponent_score"],
                    100 * st["win_percent"], st["ac_loss"]))
                if ev:
                    log("batch %d: vs greedy (argmax) win %.1f%%  score %.1f vs %.1f" % (
                        b, 100 * ev["eval_win_percent"], ev["eval_player_score"], ev["eval_opponent_score"]))

        for b in range(start_batch, batches):
            if graph and self._graph is None and b >= start_batch + 2:
                self.enable_step_graph(warmup=0)             # the first two batches ran launch by launch (lazy initialisation)
            t0 = time.perf_counter()
            self.step(defer_stats=True)
            # the evaluation is queued behind this batch's update on the stream: it plays the network that batch produced
            ev = self.evaluate_greedy(eval_games) if eval_every > 0 and self.rank == 0 and (b + 1) % eval_every == 0 else None
            marks.append((b + 1, t0, ev))
            if len(marks) > 1:                               # the previous batch's numbers are on the host by now
                finish(*marks.pop(0))
            if self.rank == 0 and net_name is not None and ((b + 1) % checkpoint_every == 0 or b + 1 == batches):
                self.save_checkpoint(net_name + ".pt", b + 1)                  # nn_runner.py:83-84, as a state_dict
        while marks:
            finish(*marks.pop(0))
        if fh:
            fh.close()
        return self.history


def parse_args(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("batch_size", nargs="?", type=int, default=10, help="episodes per batch and rank (scripts/training.py:8-11)")
    ap.add_argument("net_name", nargs="?", default=None, help="write <net_name>.csv / .pt (scripts/training.py:12-15)")
    ap.add_argument("--batches", type=int, default=1000)
    ap.add_argument("--lr", type=float, default=3e-4)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--resume", default=None, metavar="FILE",
                    help="continue from a checkpoint written by this script (<net_name>.pt) or start from any saved "
                         "network Agent(base_net_file=...) accepts")
    ap.add_argument("--checkpoint-every", type=int, default=1000)
    ap.add_argument("--opponent", default=None, metavar="FILE|greedy",
                    help="play seat 2 with this frozen network (any file Agent(base_net_file=...) accepts), or with the "
                         "greedy agent ('greedy': the move with the best one-move score), instead of the random agent; "
                         "pass a network file named greedy as ./greedy")
    ap.add_argument("--opponent-refresh", type=int, default=0, metavar="N",
                    help="replace the opponent by the current network after every N batches (self-play against a lagged "
                         "copy; without --opponent it starts as the initial network)")
    ap.add_argument("--self-play", action="store_true",
                    help="the network plays both seats and learns from both seats' decisions (no --opponent, no "
                         "--opponent-refresh; the logged reward is then 0)")
    ap.add_argument("--eval-every", type=int, default=0, metavar="N",
                    help="after every N batches play the network (argmax) against the greedy agent and log "
                         "eval_win_percent / eval_player_score / eval_opponent_score (default 0: never)")
    ap.add_argument("--eval-games", type=int, default=2048, metavar="E", help="episodes per evaluation (default 2048)")
    args = ap.parse_args(argv)
    if args.opponent_refresh < 0:
        ap.error("--opponent-refresh must be >= 0")
    if args.self_play and (args.opponent is not None or args.opponent_refresh):
        ap.error("--self-play plays both seats with the network: it cannot be combined with --opponent or --opponent-refresh")
    if args.eval_every < 0:
        ap.error("--eval-every must be >= 0")
    if args.eval_games < 1:
        ap.error("--eval-games must be >= 1")
    if args.opponent == GREEDY and args.opponent_refresh:
        ap.error("--opponent-refresh replaces a network opponent: it does not apply to --opponent greedy")
    return args


def main(argv=None):
    args = parse_args(argv)
    rank, world, local = parallel.world()
    if world > 1:
        parallel.init("nccl", local)
    torch.cuda.set_device(local)
    tr = SelfPlayTrainer(args.batch_size, learning_rate=args.lr, seed=args.seed, device=local, rank=rank, world=world,
                         opponent=args.opponent, opponent_refresh=args.opponent_refresh, self_play=args.self_play)
    start = tr.load_checkpoint(args.resume) if args.resume else 0
    tr.train(batches=args.batches, net_name=args.net_name, start_batch=start, checkpoint_every=args.checkpoint_every,
             eval_every=args.eval_every, eval_games=args.eval_games)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
