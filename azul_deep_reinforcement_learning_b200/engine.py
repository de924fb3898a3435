"""Host side of the batched engine: a thin owner of device buffers around the C ABI.

PyTorch is used for device memory and streams only; every operation on the game state is a
hand-written sm_100a kernel reached through ``include/azb.h``.
"""
import ctypes

import numpy as np
import torch

from . import _lib
from .layout import (FIRST_PLAYER_RANDOM, MASK_WORDS, N_ACTIONS, TILE_POOL_LID, TILE_POOL_RANDOM, state_words,
                     unpacked_size)

N_COUNTERS = 16
COUNTER_NAMES = [
    "steps", "games", "rounds", "score_seat0", "score_seat1", "wins_seat0", "stuck", "bag_empty", "turns",
    "floor_penalty_seat0", "max_combo_seat0", "rows_seat0", "columns_seat0", "colours_seat0",
    "first_player_seat0", "score_all",
]
ACTION_SKIP = 255


def rules_to_ints(players, rules):
    """Reference ``rules`` dict (azul.py:35-56) -> (tile_pool, first_player) integers."""
    from .azulnet.azul import IllegalRule
    first = 1
    if "first_player" in rules:
        fp = rules["first_player"]
        if fp == "Random":
            first = FIRST_PLAYER_RANDOM
        elif type(fp) == int and 1 <= fp <= players:
            first = fp
        else:
            raise IllegalRule
    pool = TILE_POOL_RANDOM
    if "tile_pool" in rules:
        tp = rules["tile_pool"]
        if tp == "Random":
            pool = TILE_POOL_RANDOM
        elif tp == "Lid":
            pool = TILE_POOL_LID
        else:
            raise IllegalRule
    return pool, first


def _ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


class BatchedAzul:
    """``n_games`` independent Azul games on one GPU.

    Reference counterpart: ``n_games`` ``azulnet.Azul`` objects (azul.py:17) plus the mask / random
    agent / reward helpers of ``azulnet.game_runner``.  State lives in ``self.state``
    (uint32 ``[W, n_games]`` as an int32 tensor, packed structure-of-arrays).
    """

    def __init__(self, n_games, players=2, tile_pool=TILE_POOL_RANDOM, first_player=1, seed=0, device=0,
                 game_id_base=0, reset=True):
        if not torch.cuda.is_available():
            raise _lib.AzbError("no CUDA device: the engine has no CPU path")
        self.lib = _lib.load()
        self.n_games, self.players, self.tile_pool, self.first_player = int(n_games), players, tile_pool, first_player
        self.seed, self.game_id_base = int(seed), int(game_id_base)
        self.device = torch.device("cuda", device)
        h = ctypes.c_void_p()
        _lib.check(self.lib.azb_create(ctypes.byref(h), device, self.n_games, players, tile_pool, first_player,
                                      self.seed & (2 ** 64 - 1), self.game_id_base))
        self._h = h
        self.W = state_words(players)
        self.U = unpacked_size(players)
        self.state = torch.zeros((self.W, self.n_games), dtype=torch.int32, device=self.device)
        self.counters = torch.zeros(N_COUNTERS, dtype=torch.int64, device=self.device)
        if reset:
            self.reset()

    def __del__(self):
        h = getattr(self, "_h", None)
        if h:
            self.lib.azb_destroy(h)
            self._h = None

    # -- helpers ---------------------------------------------------------------------------
    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _new(self, shape, dtype):
        return torch.empty(shape, dtype=dtype, device=self.device)

    def set_block_threads(self, threads):
        _lib.check(self.lib.azb_set_block_threads(self._h, threads))

    def set_rollout_defer(self, games):
        _lib.check(self.lib.azb_set_rollout_defer(self._h, games))

    # -- K6 ----------------------------------------------------------------------------------
    def reset(self, which=None):
        """Fresh game (``Azul(rules)`` + ``new_round()``) in all slots or where ``which`` is non-zero."""
        if which is not None:
            which = which.to(device=self.device, dtype=torch.uint8).contiguous()
        _lib.check(self.lib.azb_reset(self._h, _ptr(self.state), _ptr(which), self._stream()))

    # -- K2 ----------------------------------------------------------------------------------
    def legal_mask(self, out=None):
        """uint32 ``[6, n_games]`` (int32 tensor); word p bit (d + 6c) <=> action d + 6c + 30p."""
        out = self._new((MASK_WORDS, self.n_games), torch.int32) if out is None else out
        _lib.check(self.lib.azb_legal_mask(self._h, _ptr(self.state), _ptr(out), self._stream()))
        return out

    # -- K1 ----------------------------------------------------------------------------------
    def step(self, action, draws=None, want_mask=True, want_preview=False):
        """One ``Azul.step`` per game.  Returns dict(done, status[, mask][, preview])."""
        action = action.to(device=self.device, dtype=torch.uint8).contiguous()
        assert action.numel() == self.n_games
        if draws is not None:
            draws = draws.to(device=self.device, dtype=torch.int8).contiguous()
            assert draws.numel() == 20 * self.n_games
        mask = self._new((MASK_WORDS, self.n_games), torch.int32) if want_mask else None
        preview = self._new((self.players, self.n_games), torch.int16) if want_preview else None
        done = self._new((self.n_games,), torch.uint8)
        status = self._new((self.n_games,), torch.uint8)
        _lib.check(self.lib.azb_step(self._h, _ptr(self.state), _ptr(action), _ptr(draws), _ptr(mask), _ptr(preview),
                                    _ptr(done), _ptr(status), self._stream()))
        out = {"done": done, "status": status}
        if want_mask:
            out["mask"] = mask
        if want_preview:
            out["preview"] = preview
        return out

    # -- K1+K2+K3+K6 fused -------------------------------------------------------------------
    def rollout_random(self, k_steps, mask_out=None):
        """``k_steps`` random-agent env steps per game with auto-reset; counters accumulate on device."""
        _lib.check(self.lib.azb_rollout_random(self._h, _ptr(self.state), int(k_steps), _ptr(mask_out),
                                              _ptr(self.counters), self._stream()))

    def rollout_random_host(self, host_state, k_steps, host_mask=None, host_counters=None):
        """End-to-end form of :meth:`rollout_random` on HOST buffers (pinned for async copies).

        ``host_state`` (int32 ``[W, n_games]``) is copied to the device, rolled out for ``k_steps`` and
        copied back in place; the final legal mask and the accumulated counters are copied to
        ``host_mask`` / ``host_counters`` when given.  Returns after the results are on the host.
        """
        self.state.copy_(host_state, non_blocking=True)
        mask = None
        if host_mask is not None:
            if getattr(self, "_mask_buf", None) is None:
                self._mask_buf = self._new((MASK_WORDS, self.n_games), torch.int32)
            mask = self._mask_buf
        self.rollout_random(k_steps, mask)
        host_state.copy_(self.state, non_blocking=True)
        if host_mask is not None:
            host_mask.copy_(mask, non_blocking=True)
        if host_counters is not None:
            host_counters.copy_(self.counters, non_blocking=True)
        torch.cuda.current_stream(self.device).synchronize()

    def read_counters(self):
        c = self.counters.cpu().numpy()
        return dict(zip(COUNTER_NAMES, (int(x) for x in c)))

    # -- K5 ----------------------------------------------------------------------------------
    def score_preview(self):
        out = self._new((self.players, self.n_games), torch.int16)
        _lib.check(self.lib.azb_score_preview(self._h, _ptr(self.state), _ptr(out), self._stream()))
        return out

    # -- K7 ----------------------------------------------------------------------------------
    def import_records(self, records):
        """int32 ``[n_games, U]`` unpacked records -> packed state; returns the per-game ok flags."""
        rec = torch.as_tensor(np.ascontiguousarray(records, dtype=np.int32)).to(self.device)
        assert rec.shape == (self.n_games, self.U), rec.shape
        ok = self._new((self.n_games,), torch.uint8)
        _lib.check(self.lib.azb_import_state(self._h, _ptr(rec), _ptr(self.state), _ptr(ok), self._stream()))
        return ok

    def export_records(self):
        rec = self._new((self.n_games, self.U), torch.int32)
        _lib.check(self.lib.azb_export_state(self._h, _ptr(self.state), _ptr(rec), self._stream()))
        return rec

    def observe(self, perspective=-1):
        """``GameRunner.get_state`` for every game: float32 ``[n_games, 32 + 52P]``."""
        obs = self._new((self.n_games, 32 + 52 * self.players), torch.float32)
        _lib.check(self.lib.azb_observe(self._h, _ptr(self.state), int(perspective), _ptr(obs), self._stream()))
        return obs

    def observe_bf16(self, perspective=-1):
        """:meth:`observe` in bfloat16 (what the policy kernel feeds its first layer; what training records)."""
        obs = self._new((self.n_games, 32 + 52 * self.players), torch.bfloat16)
        _lib.check(self.lib.azb_observe_bf16(self._h, _ptr(self.state), int(perspective), _ptr(obs), self._stream()))
        return obs

    def a2c_loss_grad(self, logits, value, mask_rows, action, qval, scale, coeffs, sums=None):
        """The loss of ``Agent.update`` (agent.py:45-56) at the network outputs, and its gradient, in one kernel.

        logits float32 [N,180] (raw), value float32 [N], mask_rows int32 [N,6], action int64 [N], qval float32 [N];
        ``coeffs`` = (actor, critic, entropy).  Returns (dlogits [N,180], dvalue [N]); ``sums`` (float64 [3], optional)
        accumulates the unscaled sums of the three loss terms."""
        n = logits.shape[0]
        for t, dt in ((logits, torch.float32), (value, torch.float32), (mask_rows, torch.int32), (action, torch.int64), (qval, torch.float32)):
            assert t.dtype == dt and t.is_contiguous() and t.device == self.device and t.shape[0] == n, (t.dtype, t.shape)
        assert logits.shape == (n, N_ACTIONS) and mask_rows.shape == (n, MASK_WORDS)
        dlogits, dvalue = torch.empty_like(logits), torch.empty_like(value)
        _lib.check(self.lib.azb_a2c_loss_grad(self._h, n, _ptr(logits), _ptr(value), _ptr(mask_rows), _ptr(action), _ptr(qval),
                                              float(scale), float(coeffs[0]), float(coeffs[1]), float(coeffs[2]),
                                              _ptr(dlogits), _ptr(dvalue), _ptr(sums), self._stream()))
        return dlogits, dvalue

    def stats(self):
        out = self._new((self.n_games, 10), torch.int32)
        _lib.check(self.lib.azb_stats(self._h, _ptr(self.state), _ptr(out), self._stream()))
        return out

    # -- per-function entry points of the reference (façade) ------------------------------
    def move(self, action):
        action = action.to(device=self.device, dtype=torch.uint8).contiguous()
        _lib.check(self.lib.azb_move(self._h, _ptr(self.state), _ptr(action), self._stream()))

    def next_player(self):
        _lib.check(self.lib.azb_next_player(self._h, _ptr(self.state), self._stream()))

    def count_score(self):
        _lib.check(self.lib.azb_count_score(self._h, _ptr(self.state), self._stream()))

    def new_round(self, draws=None):
        if draws is not None:
            draws = draws.to(device=self.device, dtype=torch.int8).contiguous()
            assert draws.numel() == 20 * self.n_games
        _lib.check(self.lib.azb_new_round(self._h, _ptr(self.state), _ptr(draws), self._stream()))

    def opponent_random(self, player_score, require_two=True, want_mask=True, want_obs=False):
        """``GameRunner.step``'s opponent loop + reward for every game (K a14).  ``player_score`` (int16 [G]) is
        updated in place; returns dict(reward int16, done, status uint8[, mask][, obs bfloat16 [G, 32 + 52P]: the
        observation of the resulting state from seat 1's perspective])."""
        return self._opponent(self.lib.azb_opponent_random, player_score, require_two, want_mask, want_obs)

    def opponent_greedy(self, player_score, require_two=True, want_mask=True, want_obs=False):
        """:meth:`opponent_random` with the greedy agent (``azb_greedy_action``) as the opponent."""
        return self._opponent(self.lib.azb_opponent_greedy, player_score, require_two, want_mask, want_obs)

    def _opponent(self, fn, player_score, require_two, want_mask, want_obs):
        n = self.n_games
        reward, done, status = self._new((n,), torch.int16), self._new((n,), torch.uint8), self._new((n,), torch.uint8)
        mask = self._new((MASK_WORDS, n), torch.int32) if want_mask else None
        obs = self._new((n, 32 + 52 * self.players), torch.bfloat16) if want_obs else None
        _lib.check(fn(self._h, _ptr(self.state), int(bool(require_two)), _ptr(player_score), _ptr(reward), _ptr(done),
                      _ptr(status), _ptr(mask), _ptr(obs), self._stream()))
        out = {"reward": reward, "done": done, "status": status}
        if want_mask:
            out["mask"] = mask
        if want_obs:
            out["obs"] = obs
        return out

    def greedy_action(self):
        """The greedy agent's action for the seat to move in every game: uint8 [G] (``ACTION_SKIP`` when the game is over
        or no action is legal).  The state is not touched."""
        out = self._new((self.n_games,), torch.uint8)
        _lib.check(self.lib.azb_greedy_action(self._h, _ptr(self.state), _ptr(out), self._stream()))
        return out

    # -- K4, persistent form ------------------------------------------------------------------
    def policy_rollout(self, packed, k_decisions, mode=0, want_last=False):
        """Self-play (BASELINE.json configs[3]): ``k_decisions`` env steps per game in ONE launch, every seat's move sampled
        from the policy (``mode`` 1: argmax), finished games tallied in ``self.counters`` and replaced; the packed state
        stays on the device between decisions.  ``want_last``: returns the last decision's action / logp / value."""
        out = None
        if want_last:
            if getattr(self, "_last_out", None) is None:
                self._last_out = {"action": self._new((self.n_games,), torch.uint8), "logp": self._new((self.n_games,), torch.float32),
                                  "value": self._new((self.n_games,), torch.float32)}
            out = self._last_out
        _lib.check(self.lib.azb_policy_rollout(
            self._h, _ptr(self.state), _ptr(packed.buf), int(mode), int(k_decisions), 0, None, None, 0, None, None, None, None,
            None, None, None, None, _ptr(out["action"]) if out else None, _ptr(out["logp"]) if out else None,
            _ptr(out["value"]) if out else None, None, None, None, _ptr(self.counters), self._stream()))
        return out

    def policy_rollout_host(self, packed, host_state, k_decisions, host_last=None, host_counters=None, mode=0):
        """End-to-end form of :meth:`policy_rollout` on HOST buffers (pinned): state in, ``k_decisions`` decisions per game,
        state + the last decision's action / logp / value + the counters out.  Returns after the results are on the host."""
        self.state.copy_(host_state, non_blocking=True)
        out = self.policy_rollout(packed, k_decisions, mode, want_last=host_last is not None)
        host_state.copy_(self.state, non_blocking=True)
        if host_last is not None:
            for k, v in host_last.items():
                v.copy_(out[k], non_blocking=True)
        if host_counters is not None:
            host_counters.copy_(self.counters, non_blocking=True)
        torch.cuda.current_stream(self.device).synchronize()

    def round_flags(self):
        out = self._new((self.n_games,), torch.uint8)
        _lib.check(self.lib.azb_round_flags(self._h, _ptr(self.state), _ptr(out), self._stream()))
        return out


class BatchedAzulByPlayers:
    """``n_games`` games under the opt-in rule "factory count by player count" (SURVEY §8f rank 4, the reference's
    azul.py:72 TODO): ``factories`` = 2 * players + 1 displays (7 / 9 for 3 / 4 players; ``factories=5`` runs the reference's
    rule through the same kernels), 30 * (factories + 1) actions, legal mask = int64 ``[6, n_games]`` (word p bit
    d + S*c, S = factories + 1), actions uint16 (0xFFFF = skip).  The default engine (:class:`BatchedAzul`) is untouched."""

    def __init__(self, n_games, players, tile_pool=TILE_POOL_RANDOM, first_player=1, seed=0, device=0, game_id_base=0,
                 factories=None, reset=True):
        if not torch.cuda.is_available():
            raise _lib.AzbError("no CUDA device: the engine has no CPU path")
        self.lib = _lib.load()
        self.factories = int(2 * players + 1 if factories is None else factories)
        self.n_games, self.players, self.tile_pool, self.first_player = int(n_games), players, tile_pool, first_player
        self.seed, self.game_id_base = int(seed), int(game_id_base)
        self.device = torch.device("cuda", device)
        self.W = _lib.check(self.lib.azb_v_state_words(players, self.factories))
        self.U = _lib.check(self.lib.azb_v_record_size(players, self.factories))
        self.n_actions = self.lib.azb_v_n_actions(self.factories)
        h = ctypes.c_void_p()
        _lib.check(self.lib.azb_create(ctypes.byref(h), device, self.n_games, players, tile_pool, first_player,
                                      self.seed & (2 ** 64 - 1), self.game_id_base))
        self._h = h
        self.state = torch.zeros((self.W, self.n_games), dtype=torch.int32, device=self.device)
        self.counters = torch.zeros(N_COUNTERS, dtype=torch.int64, device=self.device)
        if reset:
            self.reset()

    def __del__(self):
        h = getattr(self, "_h", None)
        if h:
            self.lib.azb_destroy(h)
            self._h = None

    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def reset(self, which=None):
        if which is not None:
            which = which.to(device=self.device, dtype=torch.uint8).contiguous()
        _lib.check(self.lib.azb_v_reset(self._h, self.factories, _ptr(self.state), _ptr(which), self._stream()))

    def legal_mask(self):
        out = torch.empty((MASK_WORDS, self.n_games), dtype=torch.int64, device=self.device)
        _lib.check(self.lib.azb_v_legal_mask(self._h, self.factories, _ptr(self.state), _ptr(out), self._stream()))
        return out

    def step(self, action, draws=None):
        """One ``Azul.step`` per game (action int16 / uint16 tensor, 0xFFFF = skip).  Returns dict(mask, done, status)."""
        action = action.to(device=self.device).to(torch.int32).to(torch.uint16 if hasattr(torch, "uint16") else torch.int16).contiguous()
        if draws is not None:
            draws = draws.to(device=self.device, dtype=torch.int8).contiguous()
            assert draws.numel() == 4 * self.factories * self.n_games
        mask = torch.empty((MASK_WORDS, self.n_games), dtype=torch.int64, device=self.device)
        done = torch.empty(self.n_games, dtype=torch.uint8, device=self.device)
        status = torch.empty(self.n_games, dtype=torch.uint8, device=self.device)
        _lib.check(self.lib.azb_v_step(self._h, self.factories, _ptr(self.state), _ptr(action), _ptr(draws), _ptr(mask),
                                      _ptr(done), _ptr(status), self._stream()))
        return {"mask": mask, "done": done, "status": status}

    def rollout_random(self, k_steps):
        _lib.check(self.lib.azb_v_rollout_random(self._h, self.factories, _ptr(self.state), int(k_steps), _ptr(self.counters),
                                                self._stream()))

    def import_records(self, records):
        rec = torch.as_tensor(np.ascontiguousarray(records, dtype=np.int32)).to(self.device)
        assert rec.shape == (self.n_games, self.U), rec.shape
        ok = torch.empty(self.n_games, dtype=torch.uint8, device=self.device)
        _lib.check(self.lib.azb_v_import_state(self._h, self.factories, _ptr(rec), _ptr(self.state), _ptr(ok), self._stream()))
        return ok

    def export_records(self):
        rec = torch.empty((self.n_games, self.U), dtype=torch.int32, device=self.device)
        _lib.check(self.lib.azb_v_export_state(self._h, self.factories, _ptr(self.state), _ptr(rec), self._stream()))
        return rec

    def read_counters(self):
        return dict(zip(COUNTER_NAMES, (int(x) for x in self.counters.cpu().numpy())))


class PackedPolicy:
    """The ``ActorCritic`` parameters (model.py:17-21) in the fp16 shared-memory image of the policy kernel."""

    def __init__(self, engine, ac_net):
        self.engine = engine
        lib = engine.lib
        self.buf = torch.empty(lib.azb_policy_packed_bytes(), dtype=torch.uint8, device=engine.device)
        self.update(ac_net)

    def update(self, ac_net):
        """Re-pack after an optimiser step (weights are read from the module's current parameters)."""
        e = self.engine
        t = [ac_net.actor_linear1.weight, ac_net.actor_linear1.bias, ac_net.actor_linear2.weight, ac_net.actor_linear2.bias,
             ac_net.critic_linear1.weight, ac_net.critic_linear1.bias, ac_net.critic_linear2.weight, ac_net.critic_linear2.bias]
        assert tuple(t[0].shape) == (180, 136) and tuple(t[2].shape) == (180, 180) and tuple(t[6].shape) == (1, 180)
        t = [x.detach().to(device=e.device, dtype=torch.float32).contiguous() for x in t]
        _lib.check(e.lib.azb_policy_pack_weights(e._h, *[_ptr(x) for x in t], _ptr(self.buf), e._stream()))
        self._keep = t          # keep the staging tensors alive until the pack kernel ran


def policy_step(engine, packed, mode=0, apply_step=True, want_logits=False, want_mask=True, auto_reset=False,
                act_filter=0):
    """K4 in one launch: observation -> MLP (tcgen05) -> masked softmax -> sample / argmax -> [Azul.step].

    Returns dict(action uint8, logp, value, entropy float32, done, status uint8[, mask int32 [6,G]][, logits [G,180]])."""
    n, dev = engine.n_games, engine.device
    out = {
        "action": torch.empty(n, dtype=torch.uint8, device=dev), "logp": torch.empty(n, dtype=torch.float32, device=dev),
        "value": torch.empty(n, dtype=torch.float32, device=dev), "entropy": torch.empty(n, dtype=torch.float32, device=dev),
        "done": torch.empty(n, dtype=torch.uint8, device=dev), "status": torch.empty(n, dtype=torch.uint8, device=dev),
    }
    mask = torch.empty((MASK_WORDS, n), dtype=torch.int32, device=dev) if want_mask else None
    logits = torch.empty((n, N_ACTIONS), dtype=torch.float32, device=dev) if want_logits else None
    _lib.check(engine.lib.azb_policy_step(
        engine._h, _ptr(engine.state), _ptr(packed.buf), int(mode), (2 if auto_reset else 1) if apply_step else 0, _ptr(out["action"]),
        _ptr(out["logp"]), _ptr(out["value"]), _ptr(out["entropy"]), _ptr(mask), _ptr(out["done"]), _ptr(out["status"]),
        _ptr(logits), _ptr(engine.counters) if auto_reset else None, int(act_filter), engine._stream()))
    if want_mask:
        out["mask"] = mask
    if want_logits:
        out["logits"] = logits
    return out


class EpisodeRecords:
    """Device buffers for the decision records of ``azb_policy_rollout``'s runner mode (one episode per game slot, at most
    ``max_decisions`` agent decisions each, ``capacity`` decisions in total) -- what ``NNRunner.run_episode`` /
    ``NNRunner.train`` collect in Python lists (nn_runner.py:17-47,58-75)."""

    def __init__(self, engine, max_decisions, capacity=None, want_logp_value=False):
        n, dev = engine.n_games, engine.device
        self.engine, self.k, self.cap = engine, int(max_decisions), int(capacity or max_decisions * n)
        # a sibling handle over the compact state records: observation / legal mask of a recorded decision are functions
        # of the packed state it was taken on
        self.view = BatchedAzul(self.cap, 2, engine.tile_pool, engine.first_player, seed=engine.seed, device=dev.index, reset=False)
        self.state_rec = self.view.state
        self.action_rec = torch.zeros(self.cap, dtype=torch.uint8, device=dev)
        self.qval = torch.zeros(self.cap, dtype=torch.float32, device=dev)
        self.logp_rec = torch.zeros(self.cap, dtype=torch.float32, device=dev) if want_logp_value else None
        self.value_rec = torch.zeros(self.cap, dtype=torch.float32, device=dev) if want_logp_value else None
        self.slot_rec = torch.full((self.k, n), -1, dtype=torch.int32, device=dev)
        self.reward_rec = torch.zeros((self.k, n), dtype=torch.int16, device=dev)
        self.flags_rec = torch.zeros((self.k, n), dtype=torch.uint8, device=dev)
        self.meta = torch.zeros(2, dtype=torch.int32, device=dev)           # [0] n_dec, [1] decision iterations run
        self.reward_sum = torch.zeros(1, dtype=torch.float64, device=dev)

    def clear(self):
        self.meta.zero_()
        self.flags_rec.zero_()
        self.reward_sum.zero_()


def runner_rollout(engine, packed, records, player_score, mode=0, out=None, opponent=None, opp_passes=None):
    """``NNRunner.run_episode`` for every game slot in ONE launch (``azb_policy_rollout``, runner mode): agent decisions by the
    fused policy kernel, opponent loop + reward after each, decision records into ``records``.  The episodes must have
    been started (``BatchedGameRunner.reset``, or :meth:`selfplay.PersistentEpisodes.start` against a policy opponent).

    ``opponent``: None plays the random opponent; ``"greedy"`` the greedy agent (``azb_policy_rollout_vs_greedy``); a
    :class:`PackedPolicy` plays a frozen network with the same ``mode`` (``azb_policy_rollout_vs_policy``).  ``opp_passes``
    (uint32 / int32 [1], optional, zeroed by the caller) then receives the most opponent passes one decision needed."""
    r = records
    mask, done, status = (_ptr(out["mask"]), _ptr(out["done"]), _ptr(out["status"])) if out else (None, None, None)
    if isinstance(opponent, str):
        assert opponent == "greedy", opponent
        _lib.check(engine.lib.azb_policy_rollout_vs_greedy(
            engine._h, _ptr(engine.state), _ptr(packed.buf), int(mode), r.k, _ptr(player_score), _ptr(r.meta), r.cap,
            _ptr(r.state_rec), _ptr(r.action_rec), _ptr(r.logp_rec), _ptr(r.value_rec), _ptr(r.slot_rec), _ptr(r.reward_rec),
            _ptr(r.flags_rec), ctypes.c_void_p(r.meta.data_ptr() + 4), None, None, None, mask, done, status, engine._stream()))
        return
    if opponent is not None:
        _lib.check(engine.lib.azb_policy_rollout_vs_policy(
            engine._h, _ptr(engine.state), _ptr(packed.buf), _ptr(opponent.buf), int(mode), r.k, _ptr(player_score),
            _ptr(r.meta), r.cap, _ptr(r.state_rec), _ptr(r.action_rec), _ptr(r.logp_rec), _ptr(r.value_rec), _ptr(r.slot_rec),
            _ptr(r.reward_rec), _ptr(r.flags_rec), ctypes.c_void_p(r.meta.data_ptr() + 4), _ptr(opp_passes),
            mask, done, status, engine._stream()))
        return
    _lib.check(engine.lib.azb_policy_rollout(
        engine._h, _ptr(engine.state), _ptr(packed.buf), int(mode), r.k, 1, _ptr(player_score), _ptr(r.meta), r.cap,
        _ptr(r.state_rec), _ptr(r.action_rec), _ptr(r.logp_rec), _ptr(r.value_rec), _ptr(r.slot_rec), _ptr(r.reward_rec),
        _ptr(r.flags_rec), ctypes.c_void_p(r.meta.data_ptr() + 4), None, None, None, mask, done, status,
        None, engine._stream()))


def selfplay_rollout(engine, packed, records, player_score, pending, mode=0, out=None):
    """Two-seat self-play for every game slot in ONE launch (``azb_policy_rollout_selfplay``): the network plays both seats,
    every decision with >= 2 legal actions is recorded into ``records`` (flags bit 2 marks seat 2's), and each seat's reward
    is its score-preview lead gained since its previous decision.  ``player_score``: int16 [2, G], zeroed when the episodes
    start (``azb_reset``, no opening moves); ``pending``: int32 [2, G] scratch.  ``out``: optional dict of mask / done /
    status buffers that receive the final state's."""
    r = records
    mask, done, status = (_ptr(out["mask"]), _ptr(out["done"]), _ptr(out["status"])) if out else (None, None, None)
    assert player_score.dtype == torch.int16 and player_score.shape == (2, engine.n_games) and player_score.is_contiguous()
    assert pending.dtype == torch.int32 and pending.shape == (2, engine.n_games) and pending.is_contiguous()
    _lib.check(engine.lib.azb_policy_rollout_selfplay(
        engine._h, _ptr(engine.state), _ptr(packed.buf), int(mode), r.k, _ptr(player_score), _ptr(pending), _ptr(r.meta),
        r.cap, _ptr(r.state_rec), _ptr(r.action_rec), _ptr(r.logp_rec), _ptr(r.value_rec), _ptr(r.slot_rec),
        _ptr(r.reward_rec), _ptr(r.flags_rec), ctypes.c_void_p(r.meta.data_ptr() + 4), mask, done, status,
        engine._stream()))


def train_stats(engine, records, loss_sums, out):
    """The 18 batch statistics (``azb_train_stats``) into ``out`` (float64 [18]) in one launch."""
    _lib.check(engine.lib.azb_train_stats(engine._h, _ptr(engine.state), _ptr(records.meta), records.cap, _ptr(loss_sums),
                                         _ptr(records.reward_sum), _ptr(out), engine._stream()))
    return out


def discounted_returns_records(engine, records, gamma):
    """nn_runner.py:72-75 on the decision records: fills ``records.qval`` (compact) and ``records.reward_sum``."""
    r = records
    _lib.check(engine.lib.azb_discounted_returns(engine._h, r.k, float(gamma), _ptr(r.reward_rec), _ptr(r.flags_rec),
                                                _ptr(r.slot_rec), _ptr(r.qval), _ptr(r.reward_sum),
                                                ctypes.c_void_p(r.meta.data_ptr() + 4), engine._stream()))


PARAM_ORDER = ["actor_linear1.weight", "actor_linear1.bias", "actor_linear2.weight", "actor_linear2.bias",
               "critic_linear1.weight", "critic_linear1.bias", "critic_linear2.weight", "critic_linear2.bias"]
PARAM_SHAPES = [(180, 136), (180,), (180, 180), (180,), (180, 136), (180,), (1, 180), (1,)]


class UpdateGradients:
    """``Agent.update``'s gradient (agent.py:39-62) on the tensor cores (``azb_a2c_update_gradients``): a flat fp32 buffer
    holding the eight parameter gradients (``self.grads[name]`` are views into it, in PARAM_ORDER), the float64 [3] loss
    sums and the kernels' workspace for ``capacity`` decisions."""

    def __init__(self, engine, capacity):
        self.engine, self.cap = engine, int(capacity)
        dev = engine.device
        sizes = [int(np.prod(sh)) for sh in PARAM_SHAPES]
        self.flat = torch.zeros(sum(sizes), dtype=torch.float32, device=dev)
        self.grads, off = {}, 0
        for name, sh, n in zip(PARAM_ORDER, PARAM_SHAPES, sizes):
            self.grads[name] = self.flat[off:off + n].view(sh)
            off += n
        self.sums = torch.zeros(3, dtype=torch.float64, device=dev)
        self.workspace = torch.empty(engine.lib.azb_update_workspace_bytes(self.cap), dtype=torch.uint8, device=dev)

    def run(self, packed, state_rec, action, qval, n_dec=None, n_fixed=0, coeffs=(1.0, 0.5, 0.1), want_outputs=False, zero=True):
        """Gradient SUMS over the decisions into ``self.flat`` (zeroed first unless ``zero`` is False); ``n_dec``: device
        uint32 / int32 [1] tensor with the decision count (no host sync), else ``n_fixed``."""
        e = self.engine
        assert state_rec.dtype == torch.int32 and state_rec.shape == (17, self.cap) and state_rec.is_contiguous()
        assert action.dtype == torch.uint8 and qval.dtype == torch.float32 and action.numel() >= self.cap and qval.numel() >= self.cap
        if zero:
            self.flat.zero_()
            self.sums.zero_()
        logits = value = None
        if want_outputs:
            n = int(n_dec) if n_dec is not None else int(n_fixed)
            logits = torch.zeros((n, N_ACTIONS), dtype=torch.float32, device=e.device)
            value = torch.zeros(n, dtype=torch.float32, device=e.device)
        g = self.grads
        _lib.check(e.lib.azb_a2c_update_gradients(
            e._h, _ptr(state_rec), self.cap, _ptr(action), _ptr(qval), _ptr(n_dec), int(n_fixed), _ptr(packed.buf),
            float(coeffs[0]), float(coeffs[1]), float(coeffs[2]), _ptr(self.workspace),
            *[_ptr(g[name]) for name in PARAM_ORDER], _ptr(self.sums), _ptr(logits), _ptr(value), e._stream()))
        return logits, value


def mask_to_bool(mask6):
    """uint32 ``[6, G]`` mask words -> bool ``[G, 180]`` in the reference's action order."""
    m = mask6.to(torch.int64) & 0xFFFFFFFF
    bits = (m.unsqueeze(-1) >> torch.arange(30, device=m.device)) & 1      # [6, G, 30]
    return bits.permute(1, 0, 2).reshape(m.shape[1], N_ACTIONS).bool()


def mask_rows_to_bool(rows):
    """int32 ``[N, 6]`` mask words (one row per decision) -> bool ``[N, 180]``; 32-bit arithmetic only (the 30 mask
    bits never reach the sign bit)."""
    shifts = torch.arange(30, device=rows.device, dtype=torch.int32)
    return ((rows.unsqueeze(-1) >> shifts) & 1).reshape(rows.shape[0], N_ACTIONS).bool()
