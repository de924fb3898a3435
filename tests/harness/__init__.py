"""TEST HARNESS ONLY: g++ build of csrc/azb_rules.cuh (the header the CUDA kernels include) so the
packed-state rules can be checked against the oracle on a machine without a GPU.  The product
package never imports or loads this."""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "_build", "librules_host.so")
_HDR = os.path.join(os.path.dirname(os.path.dirname(_HERE)), "azul_deep_reinforcement_learning_b200", "csrc",
                    "azb_rules.cuh")
_lib = None


def lib():
    global _lib
    if _lib is None:
        src = os.path.join(_HERE, "rules_host.cpp")
        newest = max(os.path.getmtime(src), os.path.getmtime(_HDR))
        if not os.path.exists(_SO) or os.path.getmtime(_SO) < newest:
            os.makedirs(os.path.dirname(_SO), exist_ok=True)
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wno-unknown-pragmas",
                                   "-o", _SO, src])
        L = ctypes.CDLL(_SO)
        L.hh_op.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p,
                            ctypes.c_uint64, ctypes.c_uint32, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]
        L.hh_rollout.argtypes = [ctypes.c_void_p, ctypes.c_int64, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                 ctypes.c_uint64, ctypes.c_uint32, ctypes.c_int, ctypes.c_void_p]
        L.hh_opponent.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_uint64, ctypes.c_uint32, ctypes.c_int,
                                  ctypes.c_void_p, ctypes.c_void_p]
        L.hh_random_action.argtypes = [ctypes.c_void_p, ctypes.c_uint32]
        _lib = L
    return _lib


OP_MOVE, OP_STEP, OP_NEXT, OP_SCORE, OP_NEW_ROUND, OP_RESET, OP_PREVIEW, OP_EOR, OP_EOG, OP_ROUNDTRIP = \
    0, 1, 2, 3, 5, 6, 7, 8, 9, 100
OP_LEGAL_SINGLE = 10          # returns the number of action bytes where move_is_legal != mask bit


def op(rec, players, pool, code, a=0, draws=None, seed=0, gid=0, first_rule=1, want_mask=False, want_preview=False):
    assert rec.dtype == np.int32 and rec.flags.c_contiguous
    d = None if draws is None else np.ascontiguousarray(draws, dtype=np.int8)
    mask = np.zeros(6, np.uint32) if want_mask else None
    prev = np.zeros(players, np.int32) if want_preview else None
    rc = lib().hh_op(rec.ctypes.data, players, pool, code, int(a), None if d is None else d.ctypes.data, seed, gid,
                     first_rule, None if mask is None else mask.ctypes.data, None if prev is None else prev.ctypes.data)
    return rc, mask, prev


def rollout(recs, players, pool, first_rule, seed, gid0, k):
    cnt = np.zeros(16, np.int64)
    rc = lib().hh_rollout(recs.ctypes.data, recs.shape[0], players, pool, first_rule, seed, gid0, k, cnt.ctypes.data)
    assert rc == 0
    return cnt


def random_action(mask6, word):
    m = np.ascontiguousarray(mask6, dtype=np.uint32)
    return lib().hh_random_action(m.ctypes.data, int(word) & 0xFFFFFFFF)


def opponent(rec, players, pool, seed, gid, require_two=True):
    mask = np.zeros(6, np.uint32)
    diff = np.zeros(1, np.int32)
    rc = lib().hh_opponent(rec.ctypes.data, players, pool, seed, gid, int(require_two), mask.ctypes.data, diff.ctypes.data)
    assert rc == 0
    return int(diff[0]), mask


# ---- the "factory count by player count" variant (csrc/azb_variant.cuh) ------------------------------------------
_VSO = os.path.join(_HERE, "_build", "libvariant_host.so")
_VHDR = os.path.join(os.path.dirname(_HDR), "azb_variant.cuh")
_vlib = None


def vlib():
    global _vlib
    if _vlib is None:
        src = os.path.join(_HERE, "variant_host.cpp")
        newest = max(os.path.getmtime(src), os.path.getmtime(_HDR), os.path.getmtime(_VHDR))
        if not os.path.exists(_VSO) or os.path.getmtime(_VSO) < newest:
            os.makedirs(os.path.dirname(_VSO), exist_ok=True)
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wno-unknown-pragmas", "-o", _VSO, src])
        L = ctypes.CDLL(_VSO)
        L.vh_op.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p,
                            ctypes.c_uint64, ctypes.c_uint32, ctypes.c_int, ctypes.c_void_p]
        L.vh_rollout.argtypes = [ctypes.c_void_p, ctypes.c_int64, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                 ctypes.c_uint64, ctypes.c_uint32, ctypes.c_int, ctypes.c_void_p]
        L.vh_random_action.argtypes = [ctypes.c_void_p, ctypes.c_uint32, ctypes.c_int]
        _vlib = L
    return _vlib


V_OP_MASK, V_OP_STEP, V_OP_RESET, V_OP_ROUNDTRIP = 0, 1, 6, 100


def v_op(rec, players, factories, pool, code, a=0, draws=None, seed=0, gid=0, first_rule=1):
    assert rec.dtype == np.int32 and rec.flags.c_contiguous
    d = None if draws is None else np.ascontiguousarray(draws, dtype=np.int8)
    mask = np.zeros(6, np.uint64)
    rc = vlib().vh_op(rec.ctypes.data, players, factories, pool, code, int(a), None if d is None else d.ctypes.data, seed, gid,
                      first_rule, mask.ctypes.data)
    return rc, mask


def v_rollout(recs, players, factories, pool, first_rule, seed, gid0, k):
    cnt = np.zeros(16, np.int64)
    assert vlib().vh_rollout(recs.ctypes.data, recs.shape[0], players, factories, pool, first_rule, seed, gid0, k, cnt.ctypes.data) == 0
    return cnt
