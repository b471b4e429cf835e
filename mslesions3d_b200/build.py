"""Build ``libssd3d_b200.so`` (the C-ABI CUDA library, ``include/ssd3d_b200.h``) in-tree with nvcc.

    python -m mslesions3d_b200.build [--force]

Every ``csrc/*.cu`` is compiled for sm_100a only (``-gencode arch=compute_100a,code=sm_100a``; the
``a`` suffix is required for tcgen05/TMEM) with ``-lineinfo`` so that ncu's source page maps back to
the kernels.  nvcc cross-compiles, so this runs in the GPU-less build container; the resulting ``.so``
is git-ignored and travels to the GPU box with the working tree.
"""
from __future__ import annotations

import concurrent.futures
import os
import shutil
import subprocess
import sys

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, "csrc")
ROOT = os.path.dirname(PKG_DIR)
OBJ_DIR = os.path.join(ROOT, "build", "obj")
LIB_PATH = os.path.join(PKG_DIR, "libssd3d_b200.so")

ARCH_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON_FLAGS = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "-Xcompiler", "-O2",
                "--expt-relaxed-constexpr", "--expt-extended-lambda"]
# integer-exact kernels: never let the compiler contract a*b+c (boxes.cuh already uses *_rn intrinsics)
PER_FILE_FLAGS = {"detect.cu": ["-fmad=false"], "match_loss.cu": ["-fmad=false"], "box_ops.cu": ["-fmad=false"],
                  "metrics.cu": ["-fmad=false"], "augment.cu": ["-fmad=false"],
                  "windows.cu": ["-fmad=false"]}


def _nvcc() -> str:
    cand = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "nvcc")
    if os.path.isfile(cand):
        return cand
    found = shutil.which("nvcc")
    if not found:
        raise RuntimeError("nvcc not found (set CUDA_HOME)")
    return found


def _sources():
    return sorted(f for f in os.listdir(CSRC) if f.endswith(".cu"))


def _deps_mtime() -> float:
    m = 0.0
    for f in os.listdir(CSRC):
        m = max(m, os.path.getmtime(os.path.join(CSRC, f)))
    m = max(m, os.path.getmtime(os.path.join(ROOT, "include", "ssd3d_b200.h")))
    return m


def is_current() -> bool:
    return os.path.isfile(LIB_PATH) and os.path.getmtime(LIB_PATH) >= _deps_mtime()


def _compile_one(nvcc: str, src: str) -> str:
    obj = os.path.join(OBJ_DIR, src[:-3] + ".o")
    cmd = [nvcc, *ARCH_FLAGS, *COMMON_FLAGS, *PER_FILE_FLAGS.get(src, []), "-c", os.path.join(CSRC, src), "-o", obj]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed for %s:\n%s\n%s" % (src, r.stdout, r.stderr))
    return obj


def build(force: bool = False, verbose: bool = True) -> str:
    """Compile and link the library if it is missing or older than its sources; return its path."""
    if not force and is_current():
        return LIB_PATH
    nvcc = _nvcc()
    os.makedirs(OBJ_DIR, exist_ok=True)
    srcs = _sources()
    if verbose:
        print("[ssd3d_b200] nvcc sm_100a: %s" % " ".join(srcs), file=sys.stderr)
    with concurrent.futures.ThreadPoolExecutor(max_workers=min(8, len(srcs))) as ex:
        objs = list(ex.map(lambda s: _compile_one(nvcc, s), srcs))
    tmp = LIB_PATH + ".tmp"
    cmd = [nvcc, *ARCH_FLAGS, "-shared", "-cudart", "static", "-o", tmp, *objs]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n%s\n%s" % (r.stdout, r.stderr))
    os.replace(tmp, LIB_PATH)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv))
