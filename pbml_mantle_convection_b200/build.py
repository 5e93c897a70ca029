"""Build recipe for libpbmc.so (the C-ABI CUDA library).  sm_100a only; built in-tree so the
.so travels with the repo snapshot to the GPU box (it is git-ignored, not gpurun-ignored)."""
from __future__ import annotations

import hashlib
import os
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
CSRC = os.path.join(PKG, "csrc")
INCLUDE = os.path.join(ROOT, "include")
LIB = os.path.join(PKG, "libpbmc.so")
STAMP = os.path.join(PKG, "csrc", ".build_stamp")
SOURCES = ["api.cu", "conv_ffma.cu", "conv_umma.cu", "conv_row.cu", "conv_mux.cu", "conv_trunk.cu", "conv_edge9.cu", "pyramid.cu", "head.cu", "stencil.cu", "clock.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "--use_fast_math=false",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-O2", "--expt-relaxed-constexpr"]


def _nvcc():
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    raise RuntimeError("nvcc not found")


def _digest():
    h = hashlib.sha256()
    files = [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC)) if f.endswith((".cu", ".cuh", ".h"))]
    files.append(os.path.join(INCLUDE, "pbmc.h"))
    for f in files:
        with open(f, "rb") as fh:
            h.update(f.encode() + b"\0" + fh.read())
    h.update((" ".join(NVCC_FLAGS) + os.environ.get("PBMC_EXTRA_NVCC_FLAGS", "")).encode())
    return h.hexdigest()


def build(force=False, verbose=False):
    """Compile every .cu for sm_100a and link libpbmc.so.  No-op when sources are unchanged."""
    dig = _digest()
    if not force and os.path.exists(LIB) and os.path.exists(STAMP) and open(STAMP).read().strip() == dig:
        return LIB
    nvcc = _nvcc()
    flags = [f for f in NVCC_FLAGS if f != "--use_fast_math=false"] + os.environ.get("PBMC_EXTRA_NVCC_FLAGS", "").split()
    objs = []
    procs = []
    for s in SOURCES:
        o = os.path.join(CSRC, s.replace(".cu", ".o"))
        cmd = [nvcc, *flags, "-I", INCLUDE, "-I", CSRC, "-c", os.path.join(CSRC, s), "-o", o]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((s, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(o)
    failed = False
    for s, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode != 0:
            sys.stderr.write(f"--- nvcc {s}\n{out}\n")
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed (see output above)")
    subprocess.check_call([nvcc, "-shared", "-o", LIB, *objs, "-gencode", "arch=compute_100a,code=sm_100a", "-lcudart"])
    with open(STAMP, "w") as fh:
        fh.write(dig)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
