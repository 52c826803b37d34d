"""Build libsearchlite_gpu.so for sm_100a with nvcc (in-tree, so that it travels with gpurun)."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_DIR = os.path.join(HERE, "lib")
LIB_PATH = os.path.join(LIB_DIR, "libsearchlite_gpu.so")
SOURCES = ["slg_engine.cu", "slg_search.cu", "slg_rerank.cu", "slg_launch_tiles.cu", "slg_launch_warp.cu", "slg_launch_items.cu"]
HEADERS = ["slg_kernels.cuh", "slg_phrase.cuh", "slg_segfiles.h", "slg_warp_kernel.cuh", "slg_items_kernel.cuh", "slg_stream_kernel.cuh", "slg_scan_kernel.cuh",
           "slg_residency.cuh", "slg_async.cuh",
           "slg_host.h", "slg_dispatch.h", "slg_launch.h", "slg_filter.cuh", "slg_postimage.cuh", "slg_rerank.cuh",
           os.path.join("..", "..", "include", "searchlite_gpu.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC,-ffp-contract=off,-fno-fast-math,-pthread",
    "--fmad=false",            # never contract a*b+c: the reference's f32 arithmetic is unfused
]


def _nvcc() -> str:
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def needs_build() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    for f in SOURCES + HEADERS:
        if os.path.getmtime(os.path.join(CSRC, f)) > t:
            return True
    return False


def _compile_one(job):
    src, obj, verbose = job
    cmd = [_nvcc()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", "-o", obj, src]
    res = subprocess.run(cmd, capture_output=True, text=True)
    return src, res.returncode, res.stdout + res.stderr


def build(force: bool = False, verbose: bool = False) -> str:
    """every translation unit is compiled on its own thread (nvcc -c), then linked into the shared library"""
    if not force and not needs_build():
        return LIB_PATH
    from concurrent.futures import ThreadPoolExecutor
    os.makedirs(LIB_DIR, exist_ok=True)
    obj_dir = os.path.join(LIB_DIR, f"obj.{os.getpid()}")
    os.makedirs(obj_dir, exist_ok=True)
    jobs = [(os.path.join(CSRC, s), os.path.join(obj_dir, s.replace(".cu", ".o")), verbose) for s in SOURCES]
    try:
        with ThreadPoolExecutor(max_workers=len(jobs)) as ex:
            results = list(ex.map(_compile_one, jobs))
        failed = [r for r in results if r[1] != 0]
        if failed:
            for src, _, log in failed:
                sys.stderr.write(f"--- {src}\n{log}")
            raise RuntimeError("nvcc failed building libsearchlite_gpu.so")
        if verbose:
            for _, _, log in results:
                sys.stderr.write(log)
        tmp = LIB_PATH + f".{os.getpid()}.tmp"  # link next to the target, then rename: readers never see a partial library
        res = subprocess.run([_nvcc(), "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC,-pthread", "-o", tmp] +
                             [j[1] for j in jobs], capture_output=True, text=True)
        if res.returncode != 0:
            sys.stderr.write(res.stdout + res.stderr)
            if os.path.exists(tmp):
                os.remove(tmp)
            raise RuntimeError("linking libsearchlite_gpu.so failed")
        os.replace(tmp, LIB_PATH)
    finally:
        shutil.rmtree(obj_dir, ignore_errors=True)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
