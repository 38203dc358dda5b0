"""Builds libseqdiff_b200.so (CUDA kernels + C ABI) in-tree with nvcc for sm_100a.

    python e3-invaraint-diffusion-model_b200/build.py [--force]

nvcc cross-compiles without a GPU; the .so is git-ignored but travels with gpurun snapshots.
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
# SEQDIFF_VARIANT=<name> with SEQDIFF_EXTRA_FLAGS="-D..." builds an experiment library libseqdiff_b200_<name>.so next to the product one
# (own object directory); python loads it when SEQDIFF_LIB names its path (_cabi.py).  A/B measurements only.
VARIANT = os.environ.get("SEQDIFF_VARIANT", "")
OBJ = os.path.join(HERE, "build" + ("_dbg" if os.environ.get("SEQDIFF_DEBUG_BOUNDS") == "1" else "") + (f"_{VARIANT}" if VARIANT else ""))
LIB = os.path.join(HERE, f"libseqdiff_b200_{VARIANT}.so" if VARIANT else ("libseqdiff_b200_dbg.so" if os.environ.get("SEQDIFF_DEBUG_BOUNDS") == "1" else "libseqdiff_b200.so"))
SOURCES = ["gemm.cu", "rowwise.cu", "attention.cu", "attention_pipe.cu", "reverse_step.cu", "gauss_step.cu", "decode_loss.cu", "collate.cu", "train_kernels.cu", "attention_train.cu", "attention_train_tc.cu", "attention_bwd_pipe.cu", "train.cu", "model.cu", "cabi.cu"]
# SEQDIFF_DEBUG_BOUNDS=1: device-side bounds / invariant asserts in every kernel (the stand-in for compute-sanitizer, which the GPU
# pool does not allow); it changes the object directory and the library name, not the sources.
DEBUG_BOUNDS = os.environ.get("SEQDIFF_DEBUG_BOUNDS") == "1"
HEADERS = ["common.cuh", "kernels.h", "model.cuh", "philox.cuh", "skew.cuh", os.path.join("..", "..", "include", "seqdiff_b200.h")]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden", "-Xptxas", "-v",
]
FLAGS += os.environ.get("SEQDIFF_EXTRA_FLAGS", "").split()
if DEBUG_BOUNDS:
    FLAGS.append("-DSEQDIFF_DEBUG_BOUNDS")


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(OBJ, exist_ok=True)
    hdrs = [os.path.join(CSRC, h) for h in HEADERS] + [os.path.abspath(__file__)]
    jobs = []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(OBJ, src.replace(".cu", ".o"))
        if force or _stale(o, [s] + hdrs):
            jobs.append((s, o))

    def cc(job):
        s, o = job
        r = subprocess.run([NVCC, *FLAGS, "-c", s, "-o", o], capture_output=True, text=True)
        return s, r

    if jobs:
        with ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 4)) as ex:
            for s, r in ex.map(cc, jobs):
                if verbose or r.returncode != 0:
                    sys.stderr.write(r.stdout + r.stderr)
                if r.returncode != 0:
                    raise RuntimeError(f"nvcc failed on {s}")
                with open(os.path.join(OBJ, os.path.basename(s) + ".ptxas.log"), "w") as f:
                    f.write(r.stderr)
    objs = [os.path.join(OBJ, s.replace(".cu", ".o")) for s in SOURCES]
    if force or jobs or _stale(LIB, objs):
        r = subprocess.run([NVCC, "-shared", "-o", LIB, *objs, "-gencode", "arch=compute_100a,code=sm_100a", "-lcudart"],
                           capture_output=True, text=True)
        if r.returncode != 0:
            sys.stderr.write(r.stdout + r.stderr)
            raise RuntimeError("link failed")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
