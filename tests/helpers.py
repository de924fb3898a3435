"""Shared helpers for the parity tests (golden-trace access, the emulated-precision network forward; no game logic)."""
import hashlib
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
TRACE_CONFIGS = [(p, r) for p in (2, 3, 4) for r in ("default", "lid")]


def load_trace(players, rules):
    z = np.load(os.path.join(GOLDEN, "trace_p%d_%s.npz" % (players, rules)))
    return {k: z[k] for k in z.files}


def load_kat():
    z = np.load(os.path.join(GOLDEN, "kat.npz"))
    return {k: z[k] for k in z.files}


class TraceGame:
    """View of game ``i`` inside a loaded trace."""

    def __init__(self, tr, i):
        s0, s1 = int(tr["step_offsets"][i]), int(tr["step_offsets"][i + 1])
        r0, r1 = int(tr["round_offsets"][i]), int(tr["round_offsets"][i + 1])
        self.actions = tr["actions"][s0:s1]
        self.draws = tr["draws"][r0:r1]                # [rounds, 20], round 0 = the initial new_round
        self.first_player = int(tr["first_player"][i])
        self.initial = tr["initial_states"][i].astype(np.int32)
        self.final = tr["final_states"][i].astype(np.int32)
        self.sha = bytes(tr["stream_sha256"][i].tobytes())
        self.full = i < int(tr["n_full"])
        if self.full:
            # full_states rows: game j contributes T_j + 1 rows
            off = s0 + i
            self.states = tr["full_states"][off:off + (s1 - s0) + 1].astype(np.int32)
            self.masks = tr["full_masks"][s0:s1]


def stream_digest(masks, states):
    h = hashlib.sha256()
    for m, s in zip(masks, states):
        h.update(np.asarray(m, dtype="<u4").tobytes())
        h.update(np.asarray(s, dtype="<i4").tobytes())
    return h.digest()


def load_fuzz():
    z = np.load(os.path.join(GOLDEN, "fuzz.npz"))
    return {k: z[k] for k in z.files}


FUZZ_CONFIGS = [(p, pool) for p in (2, 3, 4) for pool in (0, 1)]


def fuzz_key(players, pool):
    return "p%d_%s" % (players, "lid" if pool else "default")


# ---- GameRunner goldens (oracle/record_golden_runner.py) -------------------------------------
RUNNER_RULES = ["default", "lid"]


def load_runner(rules):
    z = np.load(os.path.join(GOLDEN, "runner_%s.npz" % rules))
    return {k: z[k] for k in z.files}


class RunnerEpisode:
    """View of episode ``e`` of a runner golden: the env steps since ``GameRunner.reset`` and the hand-backs."""

    def __init__(self, tr, e):
        s0, s1 = int(tr["step_offsets"][e]), int(tr["step_offsets"][e + 1])
        h0, h1 = int(tr["hb_offsets"][e]), int(tr["hb_offsets"][e + 1])
        d0, d1 = int(tr["draw_offsets"][e]), int(tr["draw_offsets"][e + 1])
        self.n_steps, self.n_hb = s1 - s0, h1 - h0
        self.first_player = int(tr["first_player"][e])
        self.init_draws = tr["init_draws"][e]
        self.init_record = tr["init_records"][e].astype(np.int32)
        self.final_record = tr["final_records"][e].astype(np.int32)
        self.n_reset_steps = int(tr["n_reset_steps"][e])
        self.step_seat, self.step_action = tr["step_seat"][s0:s1], tr["step_action"][s0:s1]
        self.step_draw_idx = tr["step_draw_idx"][s0:s1]
        self.draws = tr["draws"][d0:d1]
        self.hb_step, self.hb_reward, self.hb_done = tr["hb_step"][h0:h1], tr["hb_reward"][h0:h1], tr["hb_done"][h0:h1]
        self.hb_player_score, self.hb_move_counter = tr["hb_player_score"][h0:h1], tr["hb_move_counter"][h0:h1]
        self.hb_obs, self.hb_mask = tr["hb_obs"][h0:h1].astype(np.int32), tr["hb_mask"][h0:h1]
        self.hb_records = tr["hb_records"][h0:h1].astype(np.int32)
        self.stat_keys, self.stats = [str(k) for k in tr["stat_keys"]], tr["stats"][e]

    def step_draws(self, s):
        """the 20 colours of the ``new_round`` env step ``s`` triggered, or None"""
        i = int(self.step_draw_idx[s])
        return None if i < 0 else self.draws[i]


# ---- model / update goldens (oracle/record_golden_runner.py) ----------------------------------
PARAM_NAMES = ["actor_linear1.weight", "actor_linear1.bias", "actor_linear2.weight", "actor_linear2.bias",
               "critic_linear1.weight", "critic_linear1.bias", "critic_linear2.weight", "critic_linear2.bias"]


def _load_golden(*names):
    out = {}
    for name in names:
        z = np.load(os.path.join(GOLDEN, name))
        out.update({k: z[k] for k in z.files})
    return out


def load_model_golden():
    """model.npz: the decision states and the outputs at the default parameters (s1_*); model_s3.npz: the outputs at the
    parameters scaled by 3.  The parameters (param_*) are update.npz's param0_*: both goldens record ``Agent()`` under
    ``torch.manual_seed(0)``, so they are stored once."""
    z = _load_golden("model.npz", "model_s3.npz")
    u = np.load(os.path.join(GOLDEN, "update.npz"))
    z.update({"param_" + n: u["param0_" + n] for n in PARAM_NAMES})
    return z


def load_update_golden():
    """update.npz: the decisions, losses, initial parameters and first gradient; update_steps.npz: the parameters after
    each of the two Adam steps (param1_*, param2_*)."""
    return _load_golden("update.npz", "update_steps.npz")


def mask_words_to_bool(words):
    """uint32 [N, 6] -> bool [N, 180] in the reference's action order (game_runner.py:102-103)."""
    w = np.asarray(words, dtype=np.uint32)
    return (((w[:, :, None] >> np.arange(30, dtype=np.uint32)) & 1) != 0).reshape(w.shape[0], 180)


def net_from_golden(z, prefix, scale=1.0, device="cpu"):
    """The package's ``ActorCritic`` loaded with the recorded reference parameters (times ``scale``)."""
    import torch
    from azul_deep_reinforcement_learning_b200.azulnet.model import ActorCritic
    net = ActorCritic(136, 180)
    net.load_state_dict({n: torch.from_numpy(z[prefix + n] * np.float32(scale)) for n in PARAM_NAMES})
    return net.to(device)


def free_port():
    """A TCP port nobody listens on right now (rendezvous of the world_size-2 gloo tests on 127.0.0.1)."""
    import socket
    with socket.socket(socket.AF_INET, socket.SOCK_STREAM) as sk:
        sk.bind(("127.0.0.1", 0))
        return sk.getsockname()[1]


# ---- the network as the tensor-core kernels evaluate it (azb_policy.cu k_pack_weights, azb_tc.cuh) --------------------
def f16(x):
    """Round to fp16 and back (float32)."""
    import torch
    return x.to(torch.float16).to(torch.float32)


def torch_forward(net, obs, emulate_f16):
    """ActorCritic on ``obs`` [N, 136] in float64 on the GPU.  With ``emulate_f16`` the operands are rounded where the
    tensor-core kernels round them: the observation, W1a / W1c / W2a (clamped to +-65504) and the actor's hidden
    activations to fp16; the biases b1a / b1c / b2a enter as fp16 hi + lo (hi = half(b), lo = half(b - hi)); w2c, b2c and
    the critic's hidden activations stay unrounded.  Returns a dict of float64 tensors: x, the weights as used (w1a, b1a,
    w2a, b2a, w1c, b1c, w2c [180], b2c), ha_pre / hc_pre (pre-activations), ha (relu'd, rounded as layer 2 reads it),
    logits [N, 180] and value [N]."""
    import torch
    p = {k: v.detach().cuda().float() for k, v in net.state_dict().items()}
    w1a, b1a = p["actor_linear1.weight"], p["actor_linear1.bias"]
    w2a, b2a = p["actor_linear2.weight"], p["actor_linear2.bias"]
    w1c, b1c = p["critic_linear1.weight"], p["critic_linear1.bias"]
    x = obs.cuda().float()
    if emulate_f16:
        def w16(w):
            return f16(w.clamp(-65504.0, 65504.0))

        def b16(b):
            hi = w16(b)
            return hi.double() + w16(b - hi).double()
        x, w1a, w2a, w1c = f16(x), w16(w1a), w16(w2a), w16(w1c)
        b1a, b2a, b1c = b16(b1a), b16(b2a), b16(b1c)
    o = {"x": x.double(), "w1a": w1a.double(), "b1a": b1a.double(), "w2a": w2a.double(), "b2a": b2a.double(),
         "w1c": w1c.double(), "b1c": b1c.double(), "w2c": p["critic_linear2.weight"].double().reshape(-1),
         "b2c": p["critic_linear2.bias"].double().reshape(())}
    o["ha_pre"] = o["x"] @ o["w1a"].T + o["b1a"]
    o["hc_pre"] = o["x"] @ o["w1c"].T + o["b1c"]
    ha = torch.relu(o["ha_pre"])
    o["ha"] = f16(ha.clamp_max(65504.0).float()).double() if emulate_f16 else ha
    o["logits"] = o["ha"] @ o["w2a"].T + o["b2a"]
    o["value"] = torch.relu(o["hc_pre"]) @ o["w2c"] + o["b2c"]
    return o
