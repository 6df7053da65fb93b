"""Build libvcl.so (the C-ABI CUDA library) in-tree with nvcc for sm_100a.

    python video-llava_b200/build.py [--force] [--verbose]

Objects and the shared library land next to the sources (video-llava_b200/csrc/*.o,
video-llava_b200/libvcl.so); both are git-ignored but travel to the GPU box with the snapshot.
nvcc cross-compiles without a GPU, so this also serves as the CPU-side "does it build" check.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libvcl.so")
SOURCES = ["vcl_api.cu", "gemm_tc.cu", "gemv.cu", "gemv_tc.cu", "gemv_tcw.cu", "gemv_mma.cu", "attention.cu", "attention_tc.cu", "attention_prefill_tc.cu", "decode_attention.cu", "elementwise.cu", "st_pool.cu", "sample.cu"]
HEADERS = ["common.cuh", "kernels.h", os.path.join("..", "..", "include", "vcl.h")]

ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
CFLAGS = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC",
          "--expt-relaxed-constexpr"]


def _nvcc() -> str:
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
    nvcc = _nvcc()
    hdrs = [os.path.join(CSRC, h) for h in HEADERS] + [os.path.abspath(__file__)]
    jobs = []
    objs = []
    for s in SOURCES:
        src = os.path.join(CSRC, s)
        obj = src[:-3] + ".o"
        objs.append(obj)
        if force or _stale(obj, [src] + hdrs):
            cmd = [nvcc, *ARCH, *CFLAGS, "-c", src, "-o", obj]
            if verbose:
                cmd.insert(1, "-Xptxas=-v")
            jobs.append(cmd)

    def run(cmd):
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + r.stdout + r.stderr)
        return r.stdout + r.stderr

    if jobs:
        with ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 1)) as ex:
            for out in ex.map(run, jobs):
                if verbose and out.strip():
                    print(out)
    if force or jobs or _stale(LIB, objs):
        # static cudart: the library is self-contained and loads on a machine without a GPU
        run([nvcc, *ARCH, "-shared", "-o", LIB, *objs, "-cudart", "static"])
    return LIB


if __name__ == "__main__":
    path = build(force="--force" in sys.argv, verbose="--verbose" in sys.argv)
    print(path)
