"""TEST HARNESS ONLY: the greedy agent on the CPU, twice -- the naive restatement (greedy_oracle.c, built with the oracle's
rule functions) and the g++ build of csrc/azb_rules.cuh's greedy_action / opponent_greedy (greedy_host.cpp).  The product
package never imports or loads this."""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(os.path.dirname(_HERE))
_HDR = os.path.join(_ROOT, "azul_deep_reinforcement_learning_b200", "csrc", "azb_rules.cuh")
_ORACLE_C = os.path.join(_ROOT, "oracle", "azul_oracle.c")
_libs = {}


def _build(name, src, deps, cmd):
    if name not in _libs:
        so = os.path.join(_HERE, "_build", name)
        newest = max(os.path.getmtime(p) for p in [src] + deps)
        if not os.path.exists(so) or os.path.getmtime(so) < newest:
            os.makedirs(os.path.dirname(so), exist_ok=True)
            subprocess.check_call(cmd + ["-o", so, src])
        _libs[name] = ctypes.CDLL(so)
    return _libs[name]


def oracle_lib():
    L = _build("libgreedy_oracle.so", os.path.join(_HERE, "greedy_oracle.c"), [_ORACLE_C],
               ["gcc", "-O2", "-fPIC", "-std=c11", "-shared", "-lpthread"])
    vp, I, U32, U64 = ctypes.c_void_p, ctypes.c_int, ctypes.c_uint32, ctypes.c_uint64
    L.ao_greedy_action.argtypes = [vp, I, I, U32]
    L.ao_greedy_ties.argtypes = [vp, I, I]
    L.ao_opponent_greedy.argtypes = [vp, I, I, U64, U32, I, vp]
    return L


def host_lib():
    L = _build("libgreedy_host.so", os.path.join(_HERE, "greedy_host.cpp"), [_HDR],
               ["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wno-unknown-pragmas"])
    vp, I, U32, U64 = ctypes.c_void_p, ctypes.c_int, ctypes.c_uint32, ctypes.c_uint64
    L.hh_greedy_action.argtypes = [vp, I, I, U32]
    L.hh_opponent_greedy.argtypes = [vp, I, I, U64, U32, I, vp, vp]
    return L


def _rec(rec):
    r = np.ascontiguousarray(rec, dtype=np.int32)
    return r, r.ctypes.data


def ao_greedy_action(rec, players, pool, word):
    """The naive greedy pick on one record: the action index, -1 when no action is legal."""
    r, p = _rec(rec)
    return oracle_lib().ao_greedy_action(p, players, pool, int(word) & 0xFFFFFFFF)


def ao_greedy_ties(rec, players, pool):
    """How many legal actions share the best value (0 when none is legal)."""
    r, p = _rec(rec)
    return oracle_lib().ao_greedy_ties(p, players, pool)


def ao_opponent_greedy(rec, players, pool, seed, gid, require_two=True):
    """In place on one int32 record; returns (score difference seat 1 - seat 2 after a count_score on a copy, mask)."""
    assert rec.dtype == np.int32 and rec.flags.c_contiguous
    m = np.zeros(6, np.uint32)
    d = oracle_lib().ao_opponent_greedy(rec.ctypes.data, players, pool, seed, gid, int(require_two), m.ctypes.data)
    return int(d), m


def hh_greedy_action(rec, players, pool, word):
    """azb_rules.cuh's greedy_action on one record: the action index, 180 when no action is legal."""
    r, p = _rec(rec)
    rc = host_lib().hh_greedy_action(p, players, pool, int(word) & 0xFFFFFFFF)
    assert rc >= 0, rc
    return rc


def hh_opponent_greedy(rec, players, pool, seed, gid, require_two=True):
    assert rec.dtype == np.int32 and rec.flags.c_contiguous
    m = np.zeros(6, np.uint32)
    diff = np.zeros(1, np.int32)
    assert host_lib().hh_opponent_greedy(rec.ctypes.data, players, pool, seed, gid, int(require_two), m.ctypes.data,
                                         diff.ctypes.data) == 0
    return int(diff[0]), m
