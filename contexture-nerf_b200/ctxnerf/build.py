"""Build libctxnerf.so (hand-written sm_100a kernels + C-ABI) in-tree with nvcc.

    python -m ctxnerf.build            # from contexture-nerf_b200/
    python contexture-nerf_b200/ctxnerf/build.py

The library is written next to this file so that it travels with the repo
snapshot to the GPU box.  nvcc cross-compiles without a GPU.
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(os.path.dirname(PKG_DIR), "csrc")
BUILD_DIR = os.path.join(CSRC, "build")
LIB_PATH = os.path.join(PKG_DIR, "libctxnerf.so")
DIAG_LIB_PATH = os.path.join(PKG_DIR, "libctxnerf_diag.so")   # diagnostics build (include/ctxnerf_diag.h)
DIAG_DIR = os.path.join(CSRC, "diag")
DIAG_VARIANT = {"mlp_fwd.cu", "mlp_dgrad.cu"}     # product sources that carry #ifdef CTXNERF_DIAG sections

ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr",
          "-Xptxas", "-v"]
# Files whose fp32 arithmetic must match eager PyTorch bit for bit: no FMA contraction.
NO_FMAD = {"raygen.cu", "resample.cu"}


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; libctxnerf.so cannot be built")


def sources():
    return sorted(f for f in os.listdir(CSRC) if f.endswith(".cu"))


def _digest() -> str:
    h = hashlib.sha256()
    for d in (CSRC, DIAG_DIR):
        for f in sorted(os.listdir(d)):
            if f.endswith((".cu", ".cuh", ".h")):
                h.update(f.encode())
                with open(os.path.join(d, f), "rb") as fh:
                    h.update(fh.read())
    inc = os.path.join(os.path.dirname(os.path.dirname(PKG_DIR)), "include", "ctxnerf.h")
    if os.path.exists(inc):
        with open(inc, "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(BUILD_DIR, exist_ok=True)
    stamp = os.path.join(BUILD_DIR, "stamp.sha256")
    dig = _digest()
    if (not force and os.path.exists(LIB_PATH) and os.path.exists(DIAG_LIB_PATH) and os.path.exists(stamp)
            and open(stamp).read().strip() == dig):
        return LIB_PATH
    nvcc = _nvcc()
    inc = os.path.join(os.path.dirname(os.path.dirname(PKG_DIR)), "include")
    logs = []

    def compile_one(job):
        src_dir, src, diag = job
        obj = os.path.join(BUILD_DIR, src[:-3] + ("_diag.o" if diag else ".o"))
        cmd = [nvcc, "-c", os.path.join(src_dir, src), "-o", obj, "-I", inc, "-I", CSRC] + ARCH + COMMON
        if src in NO_FMAD:
            cmd.append("-fmad=false")
        if diag:
            cmd.append("-DCTXNERF_DIAG")
        r = subprocess.run(cmd, capture_output=True, text=True)
        logs.append((src + (" [diag]" if diag else ""), r.stdout + r.stderr))
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{r.stdout}\n{r.stderr}")
        return obj

    # product objects, then the extra objects of the diagnostics build: the sources with CTXNERF_DIAG sections
    # compiled a second time with the macro, and the micro-benchmarks / self-tests of csrc/diag
    jobs = [(CSRC, s, False) for s in sources()]
    diag_jobs = [(CSRC, s, True) for s in sorted(DIAG_VARIANT)] + \
                [(DIAG_DIR, f, True) for f in sorted(os.listdir(DIAG_DIR)) if f.endswith(".cu")]
    with ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1)) as ex:
        all_objs = list(ex.map(compile_one, jobs + diag_jobs))
    objs, diag_objs = all_objs[:len(jobs)], all_objs[len(jobs):]
    for out, members in ((LIB_PATH, objs),
                         (DIAG_LIB_PATH, [o for o, j in zip(objs, jobs) if j[1] not in DIAG_VARIANT] + diag_objs)):
        r = subprocess.run([nvcc, "-shared", "-o", out] + members + ARCH, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    with open(os.path.join(BUILD_DIR, "ptxas.log"), "w") as fh:
        for src, log in sorted(logs):
            fh.write(f"==== {src} ====\n{log}\n")
    with open(stamp, "w") as fh:
        fh.write(dig)
    if verbose:
        print(open(os.path.join(BUILD_DIR, "ptxas.log")).read())
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
