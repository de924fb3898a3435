"""ctypes binding of include/azb.h.  There is no CPU fallback: a missing library or device is an error."""
import ctypes
import os

from .build import LIB_PATH

_lib = None

ABI_VERSION = 1
SYMBOLS = [
    "azb_abi_version", "azb_state_words", "azb_record_size", "azb_obs_size", "azb_last_error",
    "azb_create", "azb_destroy", "azb_set_block_threads", "azb_set_rollout_defer", "azb_reset", "azb_legal_mask", "azb_step",
    "azb_rollout_random", "azb_score_preview", "azb_import_state", "azb_export_state", "azb_observe",
    "azb_stats", "azb_move", "azb_next_player", "azb_count_score", "azb_new_round", "azb_round_flags",
    "azb_opponent_random", "azb_policy_packed_bytes", "azb_policy_pack_weights", "azb_policy_step",
    "azb_observe_bf16", "azb_a2c_loss_grad", "azb_policy_rollout", "azb_policy_rollout_vs_policy", "azb_discounted_returns",
    "azb_greedy_action", "azb_opponent_greedy", "azb_policy_rollout_vs_greedy",
    "azb_update_workspace_bytes", "azb_a2c_update_gradients", "azb_update_set_chunk_rows", "azb_train_stats",
    "azb_v_state_words", "azb_v_record_size", "azb_v_n_actions", "azb_v_reset", "azb_v_legal_mask", "azb_v_step",
    "azb_v_rollout_random", "azb_v_import_state", "azb_v_export_state",
]


class AzbError(RuntimeError):
    """A C-ABI call returned a negative code."""


def load():
    """Load libazb.so (built in-tree by build.py / __graft_entry__.build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise AzbError(
            "CUDA library %s is missing: run `python -m azul_deep_reinforcement_learning_b200.build` "
            "(or __graft_entry__.build()).  There is no CPU fallback." % LIB_PATH)
    L = ctypes.CDLL(LIB_PATH)
    vp, i32, i64, u64 = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_uint64
    L.azb_abi_version.restype = i32
    L.azb_last_error.restype = ctypes.c_char_p
    for name in ("azb_state_words", "azb_record_size", "azb_obs_size"):
        getattr(L, name).argtypes = [i32]
    L.azb_create.argtypes = [ctypes.POINTER(vp), i32, i64, i32, i32, i32, u64, u64]
    L.azb_destroy.argtypes = [vp]
    L.azb_set_block_threads.argtypes = [vp, i32]
    L.azb_set_rollout_defer.argtypes = [vp, i32]
    L.azb_reset.argtypes = [vp, vp, vp, vp]
    L.azb_legal_mask.argtypes = [vp, vp, vp, vp]
    L.azb_step.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp]
    L.azb_rollout_random.argtypes = [vp, vp, i32, vp, vp, vp]
    L.azb_score_preview.argtypes = [vp, vp, vp, vp]
    L.azb_import_state.argtypes = [vp, vp, vp, vp, vp]
    L.azb_export_state.argtypes = [vp, vp, vp, vp]
    L.azb_observe.argtypes = [vp, vp, i32, vp, vp]
    L.azb_observe_bf16.argtypes = [vp, vp, i32, vp, vp]
    L.azb_stats.argtypes = [vp, vp, vp, vp]
    L.azb_move.argtypes = [vp, vp, vp, vp]
    L.azb_next_player.argtypes = [vp, vp, vp]
    L.azb_count_score.argtypes = [vp, vp, vp]
    L.azb_new_round.argtypes = [vp, vp, vp, vp]
    L.azb_round_flags.argtypes = [vp, vp, vp, vp]
    L.azb_opponent_random.argtypes = [vp, vp, i32, vp, vp, vp, vp, vp, vp, vp]
    L.azb_opponent_greedy.argtypes = [vp, vp, i32, vp, vp, vp, vp, vp, vp, vp]
    L.azb_greedy_action.argtypes = [vp, vp, vp, vp]
    L.azb_policy_pack_weights.argtypes = [vp] * 11
    L.azb_policy_step.argtypes = [vp, vp, vp, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, vp]
    f32 = ctypes.c_float
    L.azb_a2c_loss_grad.argtypes = [vp, i64, vp, vp, vp, vp, vp, f32, f32, f32, f32, vp, vp, vp, vp]
    L.azb_policy_rollout.argtypes = [vp, vp, vp, i32, i32, i32, vp, vp, i64] + [vp] * 16
    L.azb_policy_rollout_vs_policy.argtypes = [vp, vp, vp, vp, i32, i32, vp, vp, i64] + [vp] * 13
    L.azb_policy_rollout_vs_greedy.argtypes = [vp, vp, vp, i32, i32, vp, vp, i64] + [vp] * 15
    L.azb_discounted_returns.argtypes = [vp, i32, ctypes.c_double, vp, vp, vp, vp, vp, vp, vp]
    L.azb_update_set_chunk_rows.argtypes = [i64]
    L.azb_train_stats.argtypes = [vp, vp, vp, i64, vp, vp, vp, vp]
    L.azb_update_workspace_bytes.argtypes = [i64]
    L.azb_update_workspace_bytes.restype = i64
    L.azb_a2c_update_gradients.argtypes = [vp, vp, i64, vp, vp, vp, i64, vp, f32, f32, f32] + [vp] * 13
    L.azb_v_state_words.argtypes = [i32, i32]
    L.azb_v_record_size.argtypes = [i32, i32]
    L.azb_v_n_actions.argtypes = [i32]
    L.azb_v_reset.argtypes = [vp, i32, vp, vp, vp]
    L.azb_v_legal_mask.argtypes = [vp, i32, vp, vp, vp]
    L.azb_v_step.argtypes = [vp, i32, vp, vp, vp, vp, vp, vp, vp]
    L.azb_v_rollout_random.argtypes = [vp, i32, vp, i32, vp, vp]
    L.azb_v_import_state.argtypes = [vp, i32, vp, vp, vp, vp]
    L.azb_v_export_state.argtypes = [vp, i32, vp, vp, vp]
    if L.azb_abi_version() != ABI_VERSION:
        raise AzbError("libazb.so ABI %d != binding ABI %d: rebuild" % (L.azb_abi_version(), ABI_VERSION))
    _lib = L
    return L


def check(rc):
    if rc < 0:
        raise AzbError("azb call failed (%d): %s" % (rc, load().azb_last_error().decode()))
    return rc
