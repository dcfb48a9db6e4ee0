"""Builds libpime_b200.so in-tree with nvcc for sm_100a (no other arch, no JIT cache).

    python build.py            # incremental
    python build.py --force    # rebuild everything
"""
from __future__ import annotations

import concurrent.futures as cf
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "build")
LIB = os.path.join(HERE, "libpime_b200.so")
INCLUDE = os.path.join(os.path.dirname(HERE), "include")

SOURCES = ["common.cu", "step.cu", "actor.cu", "learner.cu", "learner_tc.cu", "rollout_wt_f32.cu", "rollout_wt_f64.cu", "rollout_ph_f32.cu", "rollout_ph_f64.cu",
           "rollout_track_wt_f32.cu", "rollout_track_wt_f64.cu", "rollout_track_ph_f32.cu", "rollout_track_ph_f64.cu",
           "rollout_gain_wt_f32.cu", "rollout_gain_wt_f64.cu", "rollout_gain_ph_f32.cu", "rollout_gain_ph_f64.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC",
              "--expt-relaxed-constexpr", "-Xptxas", "-v", "-I", INCLUDE]


def nvcc() -> str:
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found; libpime_b200 cannot be built (there is no CPU fallback)")
    return exe


def _deps_mtime() -> float:
    files = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    files.append(os.path.join(INCLUDE, "pime_b200.h"))
    return max(os.path.getmtime(f) for f in files)


def _compile(src: str, force: bool, hdr_mtime: float) -> str:
    s = os.path.join(CSRC, src)
    o = os.path.join(OBJ, src.replace(".cu", ".o"))
    if not force and os.path.exists(o) and os.path.getmtime(o) >= max(os.path.getmtime(s), hdr_mtime):
        return o
    cmd = [nvcc(), *NVCC_FLAGS, "-c", s, "-o", o]
    res = subprocess.run(cmd, capture_output=True, text=True)
    with open(o + ".log", "w") as f:
        f.write(" ".join(cmd) + "\n" + res.stdout + res.stderr)
    if res.returncode != 0:
        raise RuntimeError(f"nvcc failed on {src}:\n{res.stdout}\n{res.stderr}")
    return o


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(OBJ, exist_ok=True)
    hdr = _deps_mtime()
    with cf.ThreadPoolExecutor(max_workers=min(8, len(SOURCES))) as ex:
        objs = list(ex.map(lambda s: _compile(s, force, hdr), SOURCES))
    if force or not os.path.exists(LIB) or os.path.getmtime(LIB) < max(os.path.getmtime(o) for o in objs):
        cmd = [nvcc(), "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB, *objs, "-cudart", "static"]
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError(f"link failed:\n{res.stdout}\n{res.stderr}")
    if verbose:
        print(LIB)
    return LIB


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose=True)
