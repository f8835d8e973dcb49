"""In-tree build of the C-ABI library (libmsw_b200.so) for sm_100a.

    python -m minesweeper_ppo_b200.build [--force] [--verbose]

nvcc cross-compiles without a GPU; the .so stays next to this file (git-ignored)
so it travels with the working tree to the GPU box.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG, "csrc")
INCLUDE = os.path.join(os.path.dirname(PKG), "include")
LIB = os.path.join(PKG, "libmsw_b200.so")
SOURCES = ["msw_capi.cu", "msw_env.cu", "msw_gae.cu", "msw_sampler.cu", "msw_gn.cu", "msw_heads.cu", "msw_heads_tc.cu", "msw_conv_tc.cu", "msw_cnn_fwd.cu", "msw_avoid.cu", "msw_eval.cu", "msw_host_expand.cpp"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "--shared", "-Xcompiler", "-fPIC",
    "-Xptxas", "-v", "-diag-suppress", "186",
    "-cudart", "static",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; the CUDA toolkit is required to build libmsw_b200.so")


def _deps():
    out = [os.path.join(INCLUDE, "msw_b200.h"), os.path.abspath(__file__)]
    for f in os.listdir(CSRC):
        out.append(os.path.join(CSRC, f))
    return out


def is_stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(d) > t for d in _deps())


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not is_stale():
        return LIB
    srcs = [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    cmd = [_nvcc(), *NVCC_FLAGS, "-I", INCLUDE, "-o", LIB, *srcs]
    env = dict(os.environ)
    env.pop("CC", None), env.pop("CXX", None)       # use nvcc's default host compiler (gcc on PATH)
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, env=env)
    if verbose or r.returncode != 0:
        print(r.stdout)
    if r.returncode != 0:
        raise RuntimeError(f"nvcc failed ({r.returncode}): {' '.join(cmd)}")
    with open(os.path.join(PKG, "build_ptxas.log"), "w") as f:
        f.write(r.stdout)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv or "-v" in sys.argv))
