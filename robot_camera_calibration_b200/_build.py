"""In-tree build of the CUDA library (sm_100a only) with nvcc.

`python -m robot_camera_calibration_b200._build` or `build()`; the resulting
librcc_ba.so sits next to this file so it travels with the repo snapshot.
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "librcc_ba.so")
SOURCES = ["assemble.cu", "assemble_equidistant.cu", "assemble_target.cu", "assemble_target_equidistant.cu",
           "evaluate.cu", "evaluate_target.cu", "schur.cu", "dense.cu", "problem.cu", "pnp.cu", "prior.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
CFLAGS = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC,-fopenmp,-O3", "-Xptxas", "-v",
          "--expt-relaxed-constexpr"]


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    srcs = [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".h", ".cuh"))]
    headers.append(os.path.join(HERE, "..", "include", "rcc_ba.h"))
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    objs, jobs = [], []
    for s in srcs:
        src = os.path.join(CSRC, s)
        obj = os.path.join(objdir, s.replace(".cu", ".o"))
        objs.append(obj)
        if force or _stale(obj, [src] + headers):
            jobs.append((src, obj))

    def compile_one(job):
        src, obj = job
        cmd = [NVCC] + ARCH + CFLAGS + ["-c", src, "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        log = os.path.join(objdir, os.path.basename(obj) + ".log")
        with open(log, "w") as f:
            f.write(" ".join(cmd) + "\n" + r.stdout + r.stderr)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            sys.stderr.write(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=4) as ex:
        list(ex.map(compile_one, jobs))
    if jobs or force or _stale(LIB, objs):
        cmd = [NVCC] + ARCH + ["-shared", "-o", LIB] + objs + [
            "-Xcompiler", "-fopenmp", "-lcusolver", "-lcublas", "-lnccl", "-lgomp",
            "-Xlinker", "-rpath,/usr/local/cuda/lib64"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
