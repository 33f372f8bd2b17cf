"""Builds ``librg_cuda.so`` (the C-ABI CUDA library, include/rg_cuda.h) in-tree for sm_100a.

nvcc cross-compiles without a GPU, so this runs on the CPU build box; the resulting ``.so`` is
git-ignored but travels with the source tree to the GPU machine.
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys

_HERE = os.path.dirname(os.path.abspath(__file__))
PKG_ROOT = os.path.abspath(os.path.join(_HERE, "..", ".."))          # robot-gym_b200/
REPO_ROOT = os.path.abspath(os.path.join(PKG_ROOT, ".."))
CSRC = os.path.join(PKG_ROOT, "csrc")
INCLUDE = os.path.join(REPO_ROOT, "include")
LIB_PATH = os.environ.get("RG_CUDA_LIB") or os.path.join(_HERE, "librg_cuda.so")   # override: A/B builds while tuning
STAMP_PATH = LIB_PATH + ".stamp"

SOURCES = ("rg_api.cu", "rg_mpc.cu", "rg_robot.cu")
NVCC_FLAGS = (
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "--fmad=true",          # the bit-exact gait arithmetic uses explicit __dmul_rn/__dadd_rn
    "-Xcompiler", "-fPIC",
    "-Xcompiler", "-O2",
)


def _extra_flags():
    # RG_DEBUG_TRACE=1: per-phase cycle counters of one env (intrusive); =2: only the per-CTA start / end stamps
    mode = os.environ.get("RG_DEBUG_TRACE")
    flags = ("-DRG_DEBUG_TRACE",) if mode == "1" else (("-DRG_DEBUG_TRACE", "-DRG_DEBUG_TIMELINE_ONLY") if mode == "2" else ())
    if os.environ.get("RG_EXTRA_NVCC_FLAGS"):          # experiments and checks, e.g. -DRG_DEBUG_POISON_SMEM=0xa5
        flags += tuple(os.environ["RG_EXTRA_NVCC_FLAGS"].split())
    return flags


def _nvcc() -> str:
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found: the CUDA library cannot be built on this machine")
    return exe


def _source_digest() -> str:
    h = hashlib.sha256()
    files = [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC))] + [os.path.join(INCLUDE, "rg_cuda.h")]
    for path in files:
        with open(path, "rb") as fh:
            h.update(path.encode())
            h.update(fh.read())
    h.update(" ".join(NVCC_FLAGS + _extra_flags()).encode())
    return h.hexdigest()


def is_current() -> bool:
    if not (os.path.exists(LIB_PATH) and os.path.exists(STAMP_PATH)):
        return False
    with open(STAMP_PATH) as fh:
        return fh.read().strip() == _source_digest()


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every .cu under csrc/ into librg_cuda.so; returns the library path."""
    if not force and is_current():
        return LIB_PATH
    nvcc = _nvcc()
    objs = []
    build_dir = os.path.join(PKG_ROOT, "build")
    os.makedirs(build_dir, exist_ok=True)
    procs = []
    for src in SOURCES:
        obj = os.path.join(build_dir, src.replace(".cu", ".o"))
        cmd = [nvcc, *NVCC_FLAGS, *_extra_flags(), "-I", INCLUDE, "-I", CSRC, "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
            print(" ".join(cmd), file=sys.stderr)
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    for src, proc in procs:
        out, _ = proc.communicate()
        if verbose and out:
            print(out, file=sys.stderr)
        if proc.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{out}")
    cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB_PATH, *objs]   # static cudart (nvcc default)
    res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if res.returncode != 0:
        raise RuntimeError(f"link failed:\n{res.stdout}")
    with open(STAMP_PATH, "w") as fh:
        fh.write(_source_digest())
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
