"""Builds libmbpo_b200.so (sm_100a) in-tree with nvcc.

One translation unit per compiled horizon (csrc/plan_inst.cu with -DMBPO_INST_H=<h>) plus the
C-ABI units (csrc/mbpo_b200.cu, csrc/replay.cu, csrc/collection.cu) and the any-horizon plan (csrc/plan_rt.cu); units compile in parallel and are skipped when up to date.
Usage:  python model-based-policy-optimizers_b200/build.py [--force]
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
INCLUDE = os.path.join(os.path.dirname(HERE), "include")
OBJ_DIR = os.path.join(HERE, "build")
LIB_PATH = os.path.join(HERE, "mbpo_b200", "libmbpo_b200.so")
HORIZONS = (5, 8, 15, 20, 30, 50)          # keep in sync with MBPO_FOR_EACH_H (csrc/host_util.h)

NVCC_FLAGS = ["-std=c++17", "-O3", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
              "-Xcompiler", "-fPIC", "-I", INCLUDE] + os.environ.get("MBPO_EXTRA_NVCC_FLAGS", "").split()


def _nvcc() -> str:
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found: cannot build libmbpo_b200.so")
    return nvcc


def _sources_mtime() -> float:
    paths = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(INCLUDE, "mbpo_b200.h"), __file__]
    return max(os.path.getmtime(p) for p in paths)


def _compile(job):
    src, obj, defs = job
    cmd = [_nvcc(), *NVCC_FLAGS, *defs, "-c", src, "-o", obj]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed: %s\n%s\n%s" % (" ".join(cmd), res.stdout, res.stderr))
    return obj


def build(force: bool = False, verbose: bool = True) -> str:
    newest = _sources_mtime()
    if not force and os.path.exists(LIB_PATH) and os.path.getmtime(LIB_PATH) >= newest:
        return LIB_PATH
    os.makedirs(OBJ_DIR, exist_ok=True)
    jobs = [(os.path.join(CSRC, "mbpo_b200.cu"), os.path.join(OBJ_DIR, "mbpo_b200.o"), []),
            (os.path.join(CSRC, "replay.cu"), os.path.join(OBJ_DIR, "replay.o"), []),
            (os.path.join(CSRC, "collection.cu"), os.path.join(OBJ_DIR, "collection.o"), []),
            (os.path.join(CSRC, "plan_rt.cu"), os.path.join(OBJ_DIR, "plan_rt.o"), [])]
    for h in HORIZONS:
        jobs.append((os.path.join(CSRC, "plan_inst.cu"), os.path.join(OBJ_DIR, "plan_h%d.o" % h),
                     ["-DMBPO_INST_H=%d" % h]))
    todo = [j for j in jobs if force or not os.path.exists(j[1]) or os.path.getmtime(j[1]) < newest]
    if verbose:
        print("[build] compiling %d translation unit(s) for sm_100a" % len(todo), flush=True)
    with ThreadPoolExecutor(max_workers=min(8, max(1, os.cpu_count() or 1))) as pool:
        list(pool.map(_compile, todo))
    cmd = [_nvcc(), "-shared", "-o", LIB_PATH, *[j[1] for j in jobs], "-cudart", "static"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("link failed: %s\n%s\n%s" % (" ".join(cmd), res.stdout, res.stderr))
    if verbose:
        print("[build] wrote %s" % LIB_PATH, flush=True)
    return LIB_PATH


if __name__ == "__main__":
    build(force="--force" in sys.argv)
