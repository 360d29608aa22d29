"""Builds libskillshot_b200.so (sm_100a only) in-tree with nvcc.

    python skillshot_learning_b200/build.py [--force] [-v]

(run as a script: importing the package needs the library this produces)

The .so is git-ignored but travels to the GPU box with the repo snapshot.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libskillshot_b200.so")
BUILD_DIR = os.path.join(HERE, "build")

ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "-Xcompiler", "-fno-strict-aliasing"]

# translation unit -> extra flags.  ss_env.cu must not contract a*b+c into an
# FMA: the reference is CPython float arithmetic (SURVEY.md hard part 3).
UNITS = {
    "ss_env.cu": ["-fmad=false"],
    "ss_learner.cu": [],
    "ss_mlp_tc.cu": [],      # (NOT -fmad=false: it costs the noise staging's sqrtf / fast-math sequences 18 %; the per-player env tick
                             #  it inlines, ss_env_pp.cuh, is written with explicit _rn intrinsics and needs no flag)
    "ss_mlp_grad_tc.cu": [],
    "ss_peer.cu": [],
    "ss_update.cu": [],
    "ss_frames_tc.cu": [],
    "ss_frames_grad_tc.cu": [],
    "ss_probe.cu": [],
    "ss_match.cu": [],
    "ss_league.cu": [],
    "ss_pool.cu": [],
}


def nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def _stale(target: str, deps: list[str]) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(BUILD_DIR, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    headers.append(os.path.join(HERE, "..", "include", "skillshot_b200.h"))
    headers.append(os.path.abspath(__file__))
    objs = []
    for unit, extra in UNITS.items():
        src = os.path.join(CSRC, unit)
        obj = os.path.join(BUILD_DIR, unit.replace(".cu", ".o"))
        if force or _stale(obj, [src] + headers):
            cmd = [nvcc()] + ARCH + COMMON + extra + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj]
            if verbose:
                print(" ".join(cmd), file=sys.stderr)
            subprocess.run(cmd, check=True)
        objs.append(obj)
    if force or _stale(OUT, objs):
        subprocess.run([nvcc()] + ARCH + ["-shared", "-o", OUT] + objs, check=True)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
