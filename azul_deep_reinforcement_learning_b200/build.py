"""In-tree build of the CUDA library (``libazb.so``) for sm_100a.

``nvcc`` cross-compiles without a GPU, so this runs in the build container; the resulting ``.so``
is git-ignored but travels to the GPU box with the repo snapshot.
"""
import os
import shutil
import subprocess

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, "csrc")
LIB_PATH = os.path.join(PKG_DIR, "libazb.so")
SOURCES = [os.path.join(CSRC, "azb.cu"), os.path.join(CSRC, "azb_policy.cu"), os.path.join(CSRC, "azb_a2c.cu"), os.path.join(CSRC, "azb_update.cu"), os.path.join(CSRC, "azb_variant.cu")]
HEADERS = [os.path.join(CSRC, "azb_rules.cuh"), os.path.join(CSRC, "azb_tc.cuh"), os.path.join(CSRC, "azb_mbar.cuh"), os.path.join(CSRC, "azb_variant.cuh"), os.path.join(CSRC, "azb_internal.h"), os.path.join(CSRC, "azb_queue.cuh"), os.path.join(os.path.dirname(PKG_DIR), "include", "azb.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",   # B200 only: no other arch, no PTX fallback
    "-lineinfo", "-O3", "-std=c++17",
    "-shared", "-Xcompiler", "-fPIC",
]


def find_nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found (set NVCC=/path/to/nvcc)")


def needs_build():
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    return any(os.path.getmtime(p) > t for p in SOURCES + HEADERS)


def build(force=False, verbose=False):
    """Compile libazb.so if missing or stale; returns its path.  Each translation unit is compiled to an object file
    under csrc/_obj (only when it or a header changed), all of them in parallel, then linked."""
    if not (force or needs_build()):
        return LIB_PATH
    nvcc = find_nvcc()
    obj_dir = os.path.join(CSRC, "_obj")
    os.makedirs(obj_dir, exist_ok=True)
    flags = [f for f in NVCC_FLAGS if f != "-shared"]
    newest_header = max(os.path.getmtime(h) for h in HEADERS)
    procs, objs = [], []
    for src in SOURCES:
        obj = os.path.join(obj_dir, os.path.basename(src)[:-3] + ".o")
        objs.append(obj)
        if force or not os.path.exists(obj) or os.path.getmtime(obj) < max(os.path.getmtime(src), newest_header):
            cmd = [nvcc] + flags + (["-Xptxas", "-v"] if verbose else []) + ["-c", "-o", obj, src]
            procs.append((cmd, subprocess.Popen(cmd)))
    for cmd, pr in procs:
        if pr.wait() != 0:
            raise subprocess.CalledProcessError(pr.returncode, cmd)
    # the link step gets the same -gencode: without it nvcc embeds an (empty) default-architecture device image
    subprocess.check_call([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", LIB_PATH] + objs)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force=True, verbose=True))
