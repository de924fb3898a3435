"""CPU-side checks of the drop-in boundary: the C-ABI library builds, loads and exports every symbol
include/azb.h declares; without a GPU it refuses to run instead of falling back to anything."""
import ctypes
import os
import re

import pytest

from azul_deep_reinforcement_learning_b200 import _lib, build, layout

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    build.build()
    return _lib.load()


def test_header_symbols_exported(lib):
    hdr = open(os.path.join(REPO, "include", "azb.h")).read()
    declared = set(re.findall(r"^\s*(?:const char\*|int64_t|int)\s+(azb_\w+)\s*\(", hdr, flags=re.M))
    assert declared == set(_lib.SYMBOLS), declared ^ set(_lib.SYMBOLS)
    for name in declared:
        assert hasattr(lib, name), name


def test_every_entry_point_is_documented_for_the_binding():
    """INTEGRATION.md names every entry point of include/azb.h (the reference function it replaces, or what it answers)."""
    hdr = open(os.path.join(REPO, "include", "azb.h")).read()
    doc = open(os.path.join(REPO, "INTEGRATION.md")).read()
    declared = set(re.findall(r"^\s*(?:const char\*|int64_t|int)\s+(azb_\w+)\s*\(", hdr, flags=re.M))
    missing = sorted(n for n in declared if n not in doc)
    assert not missing, missing


def test_sizes(lib):
    assert lib.azb_abi_version() == 1
    for p in (2, 3, 4):
        assert lib.azb_state_words(p) == layout.state_words(p) == 7 + 5 * p
        assert lib.azb_record_size(p) == layout.unpacked_size(p)
        assert lib.azb_obs_size(p) == 32 + 52 * p
    assert lib.azb_obs_size(2) == 136                       # agent.py:29
    assert lib.azb_state_words(5) < 0
    assert [layout.algorithmic_bytes_per_step(p) for p in (2, 3, 4)] == [161, 201, 241]   # BASELINE.md §4


def test_create_rejects_bad_rules_and_missing_device(lib):
    import torch
    h = ctypes.c_void_p()
    assert lib.azb_create(ctypes.byref(h), 0, 16, 5, 0, 1, 0, 0) == -1          # players
    assert lib.azb_create(ctypes.byref(h), 0, 16, 2, 2, 1, 0, 0) == -1          # tile_pool
    assert lib.azb_create(ctypes.byref(h), 0, 16, 2, 0, 3, 0, 0) == -1          # IllegalRule, tests/test_azul.py:48
    if not torch.cuda.is_available():
        assert lib.azb_create(ctypes.byref(h), 0, 16, 2, 0, 1, 0, 0) == -3      # no device -> loud failure
        assert b"no CPU path" in lib.azb_last_error()
        from azul_deep_reinforcement_learning_b200.engine import BatchedAzul
        with pytest.raises(_lib.AzbError):
            BatchedAzul(16)


def test_native_source_has_no_compile_time_switches():
    """The shipped CUDA sources compile one way: preprocessor conditionals only tell the device pass from the host pass
    and C from C++ (and guard the public header), so no -D flag builds a library that computes something else."""
    allowed = {"__CUDACC__", "__CUDA_ARCH__", "__cplusplus", "AZB_H"}
    csrc = os.path.join(REPO, "azul_deep_reinforcement_learning_b200", "csrc")
    paths = [os.path.join(csrc, f) for f in sorted(os.listdir(csrc))] + [os.path.join(REPO, "include", "azb.h")]
    found = []
    for path in paths:
        if not os.path.isfile(path):
            continue
        for no, line in enumerate(open(path), 1):
            m = re.match(r"\s*#\s*(?:if|ifdef|ifndef|elif)\b(.*)", line)
            if m:
                names = set(re.findall(r"[A-Za-z_]\w*", m.group(1).split("//")[0])) - {"defined"}
                if not names or not names <= allowed:           # `#if 0` switches code off just as well
                    found.append("%s:%d: %s" % (os.path.relpath(path, REPO), no, line.strip()))
    assert not found, found


def test_product_never_imports_oracle():
    pkg = os.path.join(REPO, "azul_deep_reinforcement_learning_b200")
    for root, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(root, f)).read()
                assert "import oracle" not in src and "from oracle" not in src and "azul_oracle" not in src, f
                assert "tests.harness" not in src and "rules_host" not in src, f
