"""Build libbayes_portfolio.so (sm_100a) in-tree with nvcc.

    python -m incorporating_different_sources_b200.build [--force] [--verbose]

nvcc cross-compiles without a GPU; the .so sits next to this file so that it travels to the
GPU box with the repository snapshot (it is git-ignored, not gpurun-ignored).
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libbayes_portfolio.so")
SOURCES = ["bp_api.cu", "batch_plan.cu", "stream_kernels.cu", "gram_dmma.cu", "chol_solve.cu", "chol_cluster.cu", "chol_rcond.cu", "loop_kernels.cu", "eval_kernels.cu", "band_prep.cu", "estimators.cu", "jeffreys_chain.cu"]
HEADERS = ["batch_plan.h", "chol_panel.cuh", "common.cuh", "jorion_math.cuh", "kernels.h", os.path.join("..", "..", "include", "bayes_portfolio.h")]
NVCC_FLAGS = [
    "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
    "-Xcompiler", "-fPIC", "-Xptxas", "-v",
] + os.environ.get("BP_NVCC_EXTRA", "").split()


def _nvcc() -> str:
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found: cannot build libbayes_portfolio.so")
    return exe


def _stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS if os.path.exists(os.path.join(CSRC, s))]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not _stale():
        return LIB
    nvcc = _nvcc()
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    srcs = [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]

    def compile_one(src):
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        cmd = [nvcc, *NVCC_FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        return src, obj, r

    with ThreadPoolExecutor(max_workers=len(srcs)) as ex:
        results = list(ex.map(compile_one, srcs))
    log = []
    for src, obj, r in results:
        log.append(f"== {src}\n{r.stderr}")
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{r.stdout}\n{r.stderr}")
    with open(os.path.join(objdir, "ptxas.log"), "w") as f:
        f.write("\n".join(log))
    if verbose:
        print("\n".join(log))
    link = [nvcc, "-shared", "-o", LIB, *[o for _, o, _ in results], "-gencode", "arch=compute_100a,code=sm_100a"]
    r = subprocess.run(link, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return LIB


if __name__ == "__main__":
    path = build(force="--force" in sys.argv, verbose="--verbose" in sys.argv)
    print(path)
