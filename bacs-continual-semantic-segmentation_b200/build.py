"""Builds libbacs_b200.so (sm_100a only) in-tree with nvcc.

``python -m bacs_b200.build`` or ``build_library()``; used by ``__graft_entry__.build()``.
The library is rebuilt only when a source is newer than the .so."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
CSRC = os.path.join(PKG, "csrc")
INCLUDE = os.path.join(ROOT, "include")
LIB = os.path.join(PKG, "libbacs_b200.so")
SOURCES = ["labels.cu", "prototypes.cu", "seen.cu", "pixel_loss.cu", "pixel_fast_bf16.cu", "pixel_fast_f32.cu",
           "pixel_fast_f16.cu", "distill.cu", "distill_tc.cu", "misc.cu", "peer.cu", "class_distance.cu", "pseudo.cu"]


NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=default"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; libbacs_b200.so cannot be built")


def _stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(INCLUDE, "bacs_b200.h"), __file__]
    return any(os.path.getmtime(d) > t for d in deps)


def build_library(force: bool = False, verbose: bool = False) -> str:
    if not force and not _stale():
        return LIB
    nvcc = _nvcc()
    objdir = os.path.join(PKG, "build")
    os.makedirs(objdir, exist_ok=True)
    procs = []
    for src in SOURCES:
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        cmd = [nvcc, *NVCC_FLAGS, *os.environ.get("BACS_NVCC_EXTRA", "").split(), "-I", INCLUDE, "-I", CSRC, "-c",
               os.path.join(CSRC, src), "-o", obj]      # BACS_NVCC_EXTRA: diagnostics builds (-DBACS_DTC_PROFILE ...)
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((src, obj, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    objs = []
    for src, obj, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode != 0:
            sys.stderr.write(out)
        if p.returncode != 0:
            raise RuntimeError("nvcc failed on %s" % src)
        objs.append(obj)
    cmd = [nvcc, "-shared", "-o", LIB, *objs, "-gencode", "arch=compute_100a,code=sm_100a", "-lcudart"]
    subprocess.run(cmd, check=True)
    return LIB


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose="-v" in sys.argv))
