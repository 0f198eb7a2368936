"""Builds libsfod_b200.so (hand-written sm_100a kernels behind the C ABI of include/sfod_b200.h).

In-tree build with plain nvcc: the resulting .so sits next to this file, is git-ignored, and travels
to the GPU box with the repo snapshot.  No torch headers are involved: the library is torch-agnostic.
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libsfod_b200.so")
SOURCES = ["ema.cu", "roi.cu", "detect.cu", "bn.cu", "image.cu", "augment.cu", "resize.cu", "linear.cu", "evaluate.cu"]
# -fmad=false: parity-critical arithmetic must not be contracted into FMAs; kernels that want FMAs call fmaf().
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-fmad=false", "-std=c++17",
              "-Xcompiler", "-fPIC,-fvisibility=hidden", "--threads", "2"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def _stale() -> bool:
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "sfod_b200.h"), __file__]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not _stale():
        return OUT
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    nvcc = _nvcc()

    def compile_one(src: str) -> str:
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        cmd = [nvcc, *NVCC_FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            print(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=4) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    cmd = [nvcc, "-shared", "-o", OUT, *objs, "-gencode", "arch=compute_100a,code=sm_100a", "--cudart", "shared"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
