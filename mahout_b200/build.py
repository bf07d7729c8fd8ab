"""In-tree nvcc build of libmahout_b200.so (sm_100a only).

`python -m mahout_b200.build` or `mahout_b200.build.build()`.  Objects go to
mahout_b200/csrc/build/, the library to mahout_b200/libmahout_b200.so (git-ignored, but it
travels to the GPU box with the gpurun snapshot).
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(CSRC, "build")
LIB = os.path.join(HERE, "libmahout_b200.so")
INCLUDE = os.path.join(os.path.dirname(HERE), "include")

SOURCES = ["runtime.cu", "sketch.cu", "group.cu", "route.cu", "synth.cu", "cosine.cu", "ingest.cu", "job.cu", "recommend.cu",
           "cmsized.cu", "sized_multi.cu", "itembased_multi.cu"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr",
    "-DMB200_BUILDING", "-I", INCLUDE,
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: libmahout_b200.so cannot be built")


def _deps_mtime() -> float:
    m = 0.0
    for root in (CSRC, INCLUDE):
        for f in os.listdir(root):
            if f.endswith((".cuh", ".h", ".hpp")):
                m = max(m, os.path.getmtime(os.path.join(root, f)))
    return m


def build(force: bool = False, verbose: bool = False) -> str:
    nvcc = _nvcc()
    os.makedirs(OBJ, exist_ok=True)
    hdr = _deps_mtime()
    srcs = [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    jobs = []
    for s in srcs:
        src = os.path.join(CSRC, s)
        obj = os.path.join(OBJ, s.replace(".cu", ".o"))
        stale = (force or not os.path.exists(obj)
                 or os.path.getmtime(obj) < max(os.path.getmtime(src), hdr))
        jobs.append((src, obj, stale))

    def compile_one(job):
        src, obj, stale = job
        if not stale:
            return
        cmd = [nvcc, *NVCC_FLAGS, "-c", src, "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
            print(" ".join(cmd), flush=True)
        r = subprocess.run(cmd, capture_output=True, text=True)
        if verbose and r.stderr:
            print(r.stderr)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")

    with ThreadPoolExecutor(max_workers=4) as ex:
        list(ex.map(compile_one, jobs))
    objs = [j[1] for j in jobs]
    if (force or not os.path.exists(LIB)
            or any(os.path.getmtime(o) > os.path.getmtime(LIB) for o in objs)):
        cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB, *objs,
               "-Xlinker", "--no-undefined"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    _build_cli(force)
    return LIB


CLI_SRC = os.path.join(CSRC, "cli_itemsimilarity.cpp")
CLI_BIN = os.path.join(HERE, "bin", "mahout_b200_itemsimilarity")


def _build_cli(force: bool = False) -> str:
    """the native host-side driver (C++, C ABI only) next to the library it drives"""
    os.makedirs(os.path.dirname(CLI_BIN), exist_ok=True)
    stale = (force or not os.path.exists(CLI_BIN)
             or os.path.getmtime(CLI_BIN) < max(os.path.getmtime(CLI_SRC), os.path.getmtime(LIB)))
    if stale:
        cxx = shutil.which("g++") or "g++"
        cmd = [cxx, "-O2", "-std=c++17", "-Wall", CLI_SRC, "-o", CLI_BIN, "-L", HERE, "-lmahout_b200",
               "-Wl,-rpath,$ORIGIN/.."]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"g++ failed for {CLI_SRC}:\n{r.stdout}\n{r.stderr}")
    return CLI_BIN


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
