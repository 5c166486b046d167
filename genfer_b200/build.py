"""Builds libgenfer_taylor.so in-tree with nvcc for sm_100a (no JIT cache, the .so travels with the repo)."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libgenfer_taylor.so")
SOURCES = ["api.cu", "api_uni.cu", "group.cu", "eval_api.cpp", "kernels_elem.cu", "kernels_mul.cu", "kernels_mul_blk.cu", "kernels_mul_slide.cu", "kernels_mul_box.cu", "kernels_mul_axis.cu", "kernels_rec.cu", "kernels_wave.cu", "kernels_horner.cu", "interval_api.cu",
           "univariate.cu"]
HEADERS = ["common.hpp", "kernels.cuh", "device_sync.cuh", "interval.cuh", os.path.join("..", "..", "include", "genfer_taylor.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "--cudart=static", "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=default"]


def nvcc() -> str:
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def _stale(target: str, deps: list[str]) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    import glob
    hdrs = [os.path.join(CSRC, h) for h in HEADERS] + [os.path.abspath(__file__)]
    hdrs += glob.glob(os.path.join(CSRC, "evaluator", "*.hpp"))
    objs, procs = [], []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(objdir, src.replace(".cu", ".o").replace(".cpp", ".o"))
        objs.append(o)
        if force or _stale(o, [s] + hdrs):
            cmd = [nvcc(), *NVCC_FLAGS, "-c", s, "-o", o]
            if verbose:
                cmd.insert(1, "-Xptxas=-v")
            procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write(f"--- nvcc {src} ---\n{out}\n")
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed")
    if procs or force or _stale(LIB, objs):
        cmd = [nvcc(), "-shared", "--cudart=static", "-o", LIB, *objs, "-lpthread", "-ldl", "-lrt"]   # NCCL is dlopen'ed (group.cu), never linked
        subprocess.run(cmd, check=True)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
