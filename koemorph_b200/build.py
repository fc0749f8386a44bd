"""Build the C-ABI shared library (in-tree, sm_100a only).

    python -m koemorph_b200.build            # incremental
    python -m koemorph_b200.build --force

Output: koemorph_b200/csrc/libkoemorph_b200.so (git-ignored; travels to the GPU box with the snapshot).
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

CSRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "csrc")
LIB = os.path.join(CSRC, "libkoemorph_b200.so")
SOURCES = ["api.cu", "logmel.cu", "dual_stream.cu", "dual_stream_tc.cu", "session.cu", "stream_pool.cu", "staging.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr"]


def _nvcc() -> str:
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found: the koemorph_b200 CUDA library cannot be built")
    return exe


def _stale(target: str, deps) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    nvcc = _nvcc()
    # everything a source may include: headers and the generated tables (melbank_default.inc)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h", ".inc"))]
    headers.append(os.path.join(os.path.dirname(CSRC), "..", "include", "koemorph_b200.h"))
    objs = []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        if not os.path.exists(s):
            continue
        o = s[:-3] + ".o"
        objs.append(o)
        if force or _stale(o, [s] + headers):
            cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", s, "-o", o]
            print(" ".join(cmd), flush=True)
            subprocess.check_call(cmd)
    if force or _stale(LIB, objs):
        cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB] + objs + ["-lcuda"]
        print(" ".join(cmd), flush=True)
        subprocess.check_call(cmd)
    return LIB


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print(LIB)
