"""Builds libgnode_b200.so (hand-written sm_100a CUDA + the C ABI) in-tree with nvcc.

No torch headers are involved: the library's boundary is plain C (include/gnode_b200.h).
"""
import os
import shutil
import subprocess

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, "csrc")
LIB_PATH = os.path.join(PKG_DIR, "libgnode_b200.so")
SOURCES = ["gnode_graph.cu", "gnode_forward.cu", "gnode_backward.cu", "gnode_loss.cu", "gnode_mc.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared"]


def _nvcc():
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: libgnode_b200.so cannot be built")


def is_stale(out=LIB_PATH):
    if not os.path.exists(out):
        return True
    t = os.path.getmtime(out)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)]
    deps.append(os.path.join(os.path.dirname(PKG_DIR), "include", "gnode_b200.h"))
    return any(os.path.getmtime(d) > t for d in deps)


def build_library(force=False, extra_flags=(), verbose=False, out=LIB_PATH):
    """Compile every .cu of the package for sm_100a into `out` (default LIB_PATH). Returns `out`."""
    if not force and not is_stale(out):
        return out
    cmd = [_nvcc()] + NVCC_FLAGS + list(extra_flags) + ["-o", out] + [os.path.join(CSRC, s) for s in SOURCES]
    if verbose:
        print(" ".join(cmd))
    res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + res.stdout)
    if verbose and res.stdout:
        print(res.stdout)
    return out
