"""In-tree nvcc build of librbm_b200.so (sm_100a only).

    python -m rigid_body_manipulation_b200.build [--force] [--verbose]

nvcc cross-compiles without a GPU; the resulting .so sits next to this file (git-ignored, but it travels to
the GPU box with the gpurun snapshot).  No torch, no pybind: the library exports the plain C ABI declared in
include/rbm_b200.h and is loaded with ctypes (rigid_body_manipulation_b200/_lib.py).
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
CSRC = os.path.join(PKG, "csrc")
OBJ = os.path.join(PKG, "_build")
LIB = os.path.join(PKG, "librbm_b200.so")
SOURCES = ["rbm_abi.cu", "rbm_rnea.cu", "rbm_regressor.cu", "rbm_linearize.cu", "rbm_setup.cu", "rbm_nccl.cu"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "--expt-relaxed-constexpr",
    "-Xcompiler", "-fPIC",
    "-Xcompiler", "-fvisibility=hidden",
    "-I", os.path.join(ROOT, "include"),
]


def _nvcc() -> str:
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found: the CUDA toolkit is required to build librbm_b200.so")
    return exe


def have_nvcc() -> bool:
    return bool(shutil.which("nvcc")) or os.path.exists("/usr/local/cuda/bin/nvcc")


def is_fresh() -> bool:
    """True when librbm_b200.so exists and was built from the sources and flags that are in the tree now."""
    stamp = os.path.join(OBJ, "fingerprint")
    return os.path.exists(LIB) and os.path.exists(stamp) and open(stamp).read() == _fingerprint()


def _sources():
    return [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]


def _fingerprint() -> str:
    h = hashlib.sha256()
    h.update(" ".join(NVCC_FLAGS).encode())
    for name in sorted(os.listdir(CSRC)) + ["../../include/rbm_b200.h"]:
        path = os.path.join(CSRC, name)
        if os.path.isfile(path):
            h.update(name.encode())
            with open(path, "rb") as f:
                h.update(f.read())
    return h.hexdigest()


def build_library(force: bool = False, verbose: bool = False) -> str:
    """Compile (if stale) and return the path of librbm_b200.so."""
    os.makedirs(OBJ, exist_ok=True)
    stamp = os.path.join(OBJ, "fingerprint")
    fp = _fingerprint()
    if not force and os.path.exists(LIB) and os.path.exists(stamp) and open(stamp).read() == fp:
        return LIB
    nvcc = _nvcc()
    objs = []
    procs = []
    for src in _sources():
        obj = os.path.join(OBJ, src.replace(".cu", ".o"))
        cmd = [nvcc, *NVCC_FLAGS, "-Xptxas", "-v", "-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    log = []
    for src, cmd, p in procs:
        out, _ = p.communicate()
        log.append(f"$ {' '.join(cmd)}\n{out}")
        if p.returncode != 0:
            sys.stderr.write(log[-1])
            raise RuntimeError(f"nvcc failed on {src}")
    with open(os.path.join(OBJ, "ptxas.log"), "w") as f:
        f.write("\n".join(log))
    if verbose:
        print("\n".join(log))
    link = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB, *objs, "-ldl"]
    r = subprocess.run(link, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout)
        raise RuntimeError("link failed")
    with open(stamp, "w") as f:
        f.write(fp)
    return LIB


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
