#!/usr/bin/env python
"""Generate the goldens ABOVE the bare rules engine by driving the UNMODIFIED reference (build container only).

TEST INFRASTRUCTURE ONLY.  Run as ``python -m oracle.record_golden_runner`` from the repo root; needs
/root/reference.  Nothing here is imported by the product package.  ``oracle/record_golden.py`` records
the ``Azul`` traces; this module records what sits on top of them (SURVEY.md §8 rows a13-a19):

* ``runner_{rules}.npz`` -- ``N_EPISODES`` episodes of the reference ``GameRunner`` (game_runner.py:9-85)
  per rule set: ``reset()`` and every ``step()`` with every env step inside them (the agent's and the
  opponent's: seat, action, the 20 draws of a ``new_round`` it triggered), and at every hand-back to the
  agent: reward, done, ``player_score``, ``move_counter``, ``get_state()``, ``get_valid_moves()`` and the
  full post-step record; at the end ``Azul.get_statistics()``.
* ``model.npz`` -- ``ActorCritic(136,180)`` (model.py:12-41) under ``torch.manual_seed(0)`` (what
  ``Agent()`` builds, agent.py:31-34) evaluated by the reference's own ``forward_actor`` /
  ``forward_critic`` on ``N_MODEL`` reachable states (records, reference ``get_state`` observation from
  the mover's perspective, legal mask): value, entropy term, log-probabilities of sampled legal
  actions, argmax, and the full logit rows of the first ``N_MODEL_FULL`` states; for the default
  initialisation and for the same parameters scaled by 3 (peaked policies; those outputs in ``model_s3.npz``).
* ``update.npz`` -- ``NNRunner.train(batch_size=B, batches=2)`` (nn_runner.py:53-84) on the reference
  ``Agent`` (agent.py:39-62): every decision of both batches (record, observation, mask, sampled
  action, reward), the discounted returns the reference fed to ``Agent.update``, the four loss
  statistics of each update, the gradients left in ``p.grad`` by the first update and the parameters
  after each Adam step (those in ``update_steps.npz``).

Hooks are attribute swaps in the reference's module namespaces (the ``random`` module object seen by
``azulnet.azul``, the ``Azul`` name seen by ``azulnet.game_runner``, bound methods of live objects);
the reference sources are untouched.
"""
import os
import random as _random
import sys

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

from azul_deep_reinforcement_learning_b200.layout import unpacked_size  # noqa: E402
from oracle.record_golden import RecordingRandom, mask_words, ref_to_record  # noqa: E402
from oracle.ref_loader import load_reference  # noqa: E402

N_EPISODES = 64
N_MODEL = 4096
N_MODEL_FULL = 512
UPDATE_EPISODES = 12
RULESETS = {"default": {}, "lid": {"first_player": "Random", "tile_pool": "Lid"}}
PARAM_NAMES = ["actor_linear1.weight", "actor_linear1.bias", "actor_linear2.weight", "actor_linear2.bias",
               "critic_linear1.weight", "critic_linear1.bias", "critic_linear2.weight", "critic_linear2.bias"]


class Tracer:
    """Log of every ``Azul.step`` / ``Azul.new_round`` executed by the games a GameRunner creates."""

    def __init__(self, ref, proxy):
        self.proxy, self.events = proxy, []
        tracer = self

        class TracedAzul(ref.Azul):
            def new_round(self):
                n0 = len(tracer.proxy.draws)
                super().new_round()
                self._last_draws = list(tracer.proxy.draws[n0:])

            def step(self, display, color, pattern):
                seat = int(self.current_player)
                self._last_draws = None
                self._steps = getattr(self, "_steps", 0)
                super().step(display, color, pattern)          # raises before mutation (azul.py:298-302)
                self._steps += 1
                tracer.events.append(dict(seat=seat, action=display + 6 * color + 30 * pattern,
                                          draws=self._last_draws, record=ref_to_record(self, self._steps)))

        self.cls = TracedAzul


def record_runner(ref, rules_name, out_dir, model_pool):
    """GameRunner episodes; also feeds ``model_pool`` with (record, obs, mask) of every decision point."""
    import torch
    azul_mod, gr_mod = sys.modules["azulnet.azul"], sys.modules["azulnet.game_runner"]
    rules = RULESETS[rules_name]
    U = unpacked_size(2)
    eps = []
    seed = 0
    while len(eps) < N_EPISODES:
        seed += 1
        proxy = RecordingRandom()
        tracer = Tracer(ref, proxy)
        azul_mod.random, gr_mod.Azul = proxy, tracer.cls
        try:
            _random.seed(70000 + seed)
            rng = np.random.default_rng(seed)
            agent_rand = ref.RandomAgent()

            class Opp:                                         # RandomAgent (game_runner.py:87-97) + a log of what it saw
                def get_a_output(self, state, valid_moves):
                    g = gr.game
                    model_pool.append((ref_to_record(g, getattr(g, "_steps", 0)), np.asarray(state, dtype=np.int64),
                                       mask_words(valid_moves.numpy()[0])))
                    return agent_rand.get_a_output(state, valid_moves)

            gr = ref.GameRunner(opponent=Opp(), rules=dict(rules))
            try:
                gr.reset()                                     # game_runner.py:76-85
                game = gr.game
                init_first = proxy.first[-1] if rules.get("first_player") == "Random" else 1
                # the record right after Azul(rules) + new_round(): rebuilt from the reset game's first draws
                n_reset_steps = len(tracer.events)
                hbs = []

                def handback(reward, done):
                    g = gr.game
                    valid = ref.check_all_valid(g)
                    hbs.append(dict(step=len(tracer.events), reward=int(reward), done=int(bool(done)),
                                    player_score=int(gr.player_score), move_counter=int(gr.move_counter),
                                    obs=np.asarray(gr.get_state(), dtype=np.int64), mask=mask_words(valid),
                                    record=ref_to_record(g, getattr(g, "_steps", 0))))
                    return valid

                valid = handback(0, False)
                done = False
                while not done:
                    model_pool.append((hbs[-1]["record"], hbs[-1]["obs"], hbs[-1]["mask"]))
                    if rng.random() < 0.3:                     # some uniform choices: more straight-to-floor moves
                        a = int(rng.choice(np.nonzero(valid)[0]))
                    else:
                        a = int(agent_rand.get_a_output(None, torch.from_numpy(valid.reshape(1, 180))))
                    reward, done = gr.step(a)                  # game_runner.py:43-55
                    valid = handback(reward, done)
            except (ValueError, IndexError):                   # stuck round: the reference crashes (SURVEY §5); skip the seed
                continue
            assert gr.game is game
            stats = game.get_statistics()
            # every new_round of the reset game: the first 20 draws after the constructor game's 20
            draws_rows, step_draw_idx = [], []
            # draws consumed by the reset game's initial new_round (the GameRunner ctor's own game drew 20 before it)
            all_draws = np.asarray(proxy.draws, dtype=np.int8).reshape(-1, 20)
            init_draws = all_draws[1]
            init = ref.Azul(rules=dict(rules))                 # rebuild the initial record on the reference itself
            init.next_first_player = init_first
            azul_mod.random = _ReplayRandom(init_draws)
            init.new_round()
            azul_mod.random = proxy
            for ev in tracer.events:
                if ev["draws"]:
                    step_draw_idx.append(len(draws_rows))
                    draws_rows.append(np.asarray(ev["draws"], dtype=np.int8))
                else:
                    step_draw_idx.append(-1)
            assert 2 + len(draws_rows) == all_draws.shape[0]
            eps.append(dict(seed=seed, first=init_first, init_draws=init_draws, init_record=ref_to_record(init, 0),
                            events=tracer.events, hbs=hbs, draws=draws_rows, step_draw_idx=step_draw_idx,
                            n_reset_steps=n_reset_steps,
                            stats=np.asarray([stats[k] for k in STAT_KEYS], dtype=np.float64)))
        finally:
            azul_mod.random, gr_mod.Azul = _random, ref.Azul

    step_off = np.cumsum([0] + [len(e["events"]) for e in eps]).astype(np.int64)
    hb_off = np.cumsum([0] + [len(e["hbs"]) for e in eps]).astype(np.int64)
    draw_off = np.cumsum([0] + [len(e["draws"]) for e in eps]).astype(np.int64)
    out = dict(
        tile_pool=np.int32(1 if rules.get("tile_pool") == "Lid" else 0),
        first_player_rule=np.int32(0 if rules.get("first_player") == "Random" else 1),
        seeds=np.asarray([e["seed"] for e in eps], dtype=np.int32),
        first_player=np.asarray([e["first"] for e in eps], dtype=np.int8),
        init_draws=np.stack([e["init_draws"] for e in eps]),
        init_records=np.stack([e["init_record"] for e in eps]).astype(np.int16),
        n_reset_steps=np.asarray([e["n_reset_steps"] for e in eps], dtype=np.int32),
        step_offsets=step_off, hb_offsets=hb_off, draw_offsets=draw_off,
        step_seat=np.concatenate([[ev["seat"] for ev in e["events"]] for e in eps]).astype(np.int8),
        step_action=np.concatenate([[ev["action"] for ev in e["events"]] for e in eps]).astype(np.uint8),
        step_draw_idx=np.concatenate([e["step_draw_idx"] for e in eps]).astype(np.int32),   # row inside the episode's draws, -1 none
        draws=np.concatenate([np.stack(e["draws"]) if e["draws"] else np.zeros((0, 20), np.int8) for e in eps]),
        final_records=np.stack([e["events"][-1]["record"] for e in eps]).astype(np.int16),
        hb_step=np.concatenate([[h["step"] for h in e["hbs"]] for e in eps]).astype(np.int32),   # env steps of the episode done before it
        hb_reward=np.concatenate([[h["reward"] for h in e["hbs"]] for e in eps]).astype(np.int16),
        hb_done=np.concatenate([[h["done"] for h in e["hbs"]] for e in eps]).astype(np.uint8),
        hb_player_score=np.concatenate([[h["player_score"] for h in e["hbs"]] for e in eps]).astype(np.int16),
        hb_move_counter=np.concatenate([[h["move_counter"] for h in e["hbs"]] for e in eps]).astype(np.int32),
        hb_obs=np.concatenate([np.stack([h["obs"] for h in e["hbs"]]) for e in eps]).astype(np.int16),
        hb_mask=np.concatenate([np.stack([h["mask"] for h in e["hbs"]]) for e in eps]).astype(np.uint32),
        hb_records=np.concatenate([np.stack([h["record"] for h in e["hbs"]]) for e in eps]).astype(np.int16),
        stat_keys=np.asarray(STAT_KEYS), stats=np.stack([e["stats"] for e in eps]),
    )
    assert out["hb_records"].shape[1] == U and out["hb_obs"].shape[1] == 136
    path = os.path.join(out_dir, "runner_%s.npz" % rules_name)
    np.savez_compressed(path, **out)
    forced = sum(1 for e in eps for i, ev in enumerate(e["events"]) if ev["seat"] == 1 and i >= e["n_reset_steps"]) - \
        sum(len(e["hbs"]) - 1 for e in eps)
    print("%s: %d episodes, %d env steps, %d hand-backs, %d seat-1 moves played by the opponent (game_runner.py:46), %.1f KiB" % (
        os.path.basename(path), len(eps), int(step_off[-1]), int(hb_off[-1]), forced, os.path.getsize(path) / 1024))


STAT_KEYS = ["player_score", "opponent_score", "rounds", "percent_first_player", "floor_penalty", "max_combo",
             "completed_rows", "completed_columns", "completed_colors", "win_percent"]


class _ReplayRandom:
    """``random`` stand-in that replays 20 recorded colours (both pool kinds draw one colour per call)."""

    def __init__(self, draws):
        self.it = iter(int(d) for d in draws)

    def randrange(self, *a):
        return next(self.it)

    def choices(self, population, weights=None, **kw):
        return [next(self.it)]


def get_params(net):
    sd = net.state_dict()
    return {n: sd[n].detach().cpu().numpy().astype(np.float32).copy() for n in PARAM_NAMES}


def record_model(ref, out_dir, model_pool):
    import torch
    rng = np.random.default_rng(4096)
    # distinct decision states with at least one legal action, game not over
    seen, pool = set(), []
    for rec, obs, mask in model_pool:
        key = rec.tobytes() + obs.tobytes()
        if key in seen or not mask.any():
            continue
        seen.add(key)
        pool.append((rec, obs, mask))
    idx = rng.permutation(len(pool))[:N_MODEL]
    assert len(idx) == N_MODEL, "only %d distinct decision states" % len(pool)
    recs = np.stack([pool[i][0] for i in idx]).astype(np.int16)
    obs = np.stack([pool[i][1] for i in idx]).astype(np.int16)
    masks = np.stack([pool[i][2] for i in idx]).astype(np.uint32)
    valid = ((masks[:, :, None] >> np.arange(30, dtype=np.uint32)) & 1).astype(bool).reshape(N_MODEL, 180)
    sel = np.stack([rng.choice(np.nonzero(v)[0], size=4) for v in valid]).astype(np.uint8)

    torch.manual_seed(0)
    agent = ref.Agent()                                        # agent.py:31-34: ActorCritic(136, 180)
    net = agent.ac_net
    # the parameters are not stored here: they equal update.npz's param0_* (the same Agent() under torch.manual_seed(0))
    out = dict(records=recs, obs=obs, mask=masks, sel_actions=sel)
    x = torch.from_numpy(obs.astype(np.float32))
    m = torch.from_numpy(valid)
    for tag, scale in (("s1", 1.0), ("s3", 3.0)):
        if scale != 1.0:
            with torch.no_grad():
                for p in net.parameters():
                    p.mul_(scale)
        with torch.no_grad():
            value = net.forward_critic(x)                                          # model.py:23-27
            dist, logp = net.forward_actor(x, m)                                   # model.py:28-41
            logits = net.actor_linear2(torch.relu(net.actor_linear1(x)))           # the rows before model.py:37
        logp_np = logp.numpy()
        out[tag + "_value"] = value.numpy().reshape(-1).astype(np.float32)
        out[tag + "_entropy"] = np.asarray([-logp_np[i][valid[i]].mean() for i in range(N_MODEL)], dtype=np.float32)   # nn_runner.py:36-40
        out[tag + "_logp_sel"] = np.take_along_axis(logp_np, sel.astype(np.int64), axis=1).astype(np.float32)
        out[tag + "_argmax"] = dist.numpy().argmax(axis=1).astype(np.uint8)         # agent.py:71 "Max"
        out[tag + "_pmax"] = dist.numpy().max(axis=1).astype(np.float32)
        out[tag + "_logits_full"] = logits.numpy()[:N_MODEL_FULL].astype(np.float32)
        out[tag + "_logits_absmax"] = np.abs(logits.numpy()).max(axis=1).astype(np.float32)
        out[tag + "_logits_sel"] = np.take_along_axis(logits.numpy(), sel.astype(np.int64), axis=1).astype(np.float32)
    out["scales"] = np.asarray([1.0, 3.0], dtype=np.float32)
    path = os.path.join(out_dir, "model.npz")
    np.savez_compressed(os.path.join(out_dir, "model_s3.npz"), **{k: out.pop(k) for k in list(out) if k.startswith("s3_")})
    np.savez_compressed(path, **out)
    print("model.npz: %d states (%d with full logit rows), %.1f KiB" % (N_MODEL, N_MODEL_FULL, os.path.getsize(path) / 1024))


def record_update(ref, out_dir):
    """Two batches of ``NNRunner.train`` on the live reference with every input of ``Agent.update`` captured."""
    import torch
    azul_mod, gr_mod = sys.modules["azulnet.azul"], sys.modules["azulnet.game_runner"]
    proxy = RecordingRandom()
    azul_mod.random = proxy
    try:
        _random.seed(424242)
        sys.modules["azulnet.game_runner"].random.seed(424242)
        np.random.seed(2024)
        torch.manual_seed(0)
        agent = ref.Agent(learning_rate=3e-4)                  # scripts/training.py:19
        gr = ref.GameRunner()                                  # scripts/training.py:20: default rules, RandomAgent opponent
        runner = ref.NNRunner(agent, gr)
        params0 = get_params(agent.ac_net)
        decisions, updates = [], []
        orig_get, orig_update, orig_step = agent.get_ac_output, agent.update, gr.step
        pending = {}

        def get_ac_output(state, valid_moves, action_selection="Distribution"):
            r = orig_get(state, valid_moves, action_selection)
            g = gr.game
            pending.update(record=ref_to_record(g), obs=np.asarray(state, dtype=np.int64),
                           mask=mask_words(valid_moves.numpy()[0]), action=int(r[0]), value=float(r[3]),
                           logp=float(r[2].squeeze(0)[r[0]]))
            return r

        def step(i):
            reward, done = orig_step(i)
            assert pending["action"] == int(i)
            decisions.append(dict(pending, reward=int(reward), done=int(bool(done)), batch=len(updates)))
            return reward, done

        def update(qvals, rewards, values, log_probs, entropy):
            orig_update(qvals, rewards, values, log_probs, entropy)               # agent.py:39-62
            buf = agent.agent_statistics.statisticsBuffer
            updates.append(dict(
                qvals=np.asarray(qvals, dtype=np.float64).reshape(-1), episode_rewards=np.asarray(rewards, dtype=np.float64),
                entropy=np.asarray([float(e) for e in entropy], dtype=np.float32),
                losses=np.asarray([buf[k][-1] for k in ("reward", "actor_loss", "critic_loss", "entropy_loss", "ac_loss")], dtype=np.float64),
                grads={n: p.grad.detach().numpy().astype(np.float32).copy() for n, p in agent.ac_net.named_parameters()},
                params=get_params(agent.ac_net)))

        agent.get_ac_output, agent.update, gr.step = get_ac_output, update, step
        runner.train(net_name=None, batch_size=UPDATE_EPISODES, batches=2)        # nn_runner.py:53-84
    finally:
        azul_mod.random = _random
    assert len(updates) == 2
    D = len(decisions)
    out = dict(
        records=np.stack([d["record"] for d in decisions]).astype(np.int16),
        obs=np.stack([d["obs"] for d in decisions]).astype(np.int16),
        mask=np.stack([d["mask"] for d in decisions]).astype(np.uint32),
        action=np.asarray([d["action"] for d in decisions], dtype=np.uint8),
        reward=np.asarray([d["reward"] for d in decisions], dtype=np.int16),
        done=np.asarray([d["done"] for d in decisions], dtype=np.uint8),
        batch=np.asarray([d["batch"] for d in decisions], dtype=np.uint8),
        value=np.asarray([d["value"] for d in decisions], dtype=np.float32),       # critic output when the decision was taken
        logp=np.asarray([d["logp"] for d in decisions], dtype=np.float32),
        qvals=np.concatenate([u["qvals"] for u in updates]),                      # nn_runner.py:72-75, in decision order
        entropy=np.concatenate([u["entropy"] for u in updates]),
        gamma=np.float64(agent.gamma), learning_rate=np.float64(agent.learning_rate),
        losses=np.stack([u["losses"] for u in updates]),                          # reward, actor, critic, entropy, ac
        episode_rewards=np.concatenate([u["episode_rewards"] for u in updates]),
    )
    assert out["qvals"].shape[0] == D
    for n in PARAM_NAMES:
        out["param0_" + n] = params0[n]
        out["grad1_" + n] = updates[0]["grads"][n]
        out["param1_" + n] = updates[0]["params"][n]
        out["param2_" + n] = updates[1]["params"][n]
    path = os.path.join(out_dir, "update.npz")
    np.savez_compressed(os.path.join(out_dir, "update_steps.npz"),
                        **{k: out.pop(k) for k in list(out) if k.startswith(("param1_", "param2_"))})
    np.savez_compressed(path, **out)
    print("update.npz: %d decisions in 2 batches of %d episodes, losses %s, %.1f KiB" % (
        D, UPDATE_EPISODES, np.array2string(out["losses"], precision=4), os.path.getsize(path) / 1024))


def main():
    ref = load_reference()
    out_dir = os.path.join(REPO, "tests", "golden")
    os.makedirs(out_dir, exist_ok=True)
    model_pool = []
    for rules_name in RULESETS:
        record_runner(ref, rules_name, out_dir, model_pool)
    record_model(ref, out_dir, model_pool)
    record_update(ref, out_dir)


if __name__ == "__main__":
    main()
