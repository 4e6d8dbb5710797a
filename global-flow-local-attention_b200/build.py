"""Build libgfla_warp.so (sm_100a only) in-tree with nvcc.

    python -m gfla_b200.build          (or  __graft_entry__.build())

The library is a plain C-ABI shared object (include/gfla_warp.h): it does not
link against torch or libcuda (the driver entry point needed for TMA
descriptors is fetched at run time through the CUDA runtime), so it
cross-compiles on a box without a GPU and travels to the GPU box as a file.
"""
from __future__ import annotations

import concurrent.futures as cf
import hashlib
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "build")
LIB_DIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIB_DIR, "libgfla_warp.so")
INCLUDE = os.path.join(os.path.dirname(HERE), "include")

ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "-I", INCLUDE]
# per-file extras: the unfused ops keep IEEE mul/add separate so that their fp32 /
# fp64 forward is bit-identical to the (uncontracted) CPU oracle.
EXTRA = {"block_extract.cu": ["-fmad=false"], "resample2d.cu": ["-fmad=false"], "resample2d_nhwc.cu": ["-fmad=false"]}


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found (needed to build libgfla_warp.so for sm_100a)")


def _digest(paths) -> str:
    h = hashlib.sha256()
    for p in sorted(paths):
        with open(p, "rb") as f:
            h.update(p.encode() + b"\0" + f.read())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(OBJ, exist_ok=True)
    os.makedirs(LIB_DIR, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    headers.append(os.path.join(INCLUDE, "gfla_warp.h"))
    sources = sorted(f for f in os.listdir(CSRC) if f.endswith(".cu"))
    nvcc = _nvcc()
    jobs = []
    for src in sources:
        path = os.path.join(CSRC, src)
        obj = os.path.join(OBJ, src[:-3] + ".o")
        stamp = obj + ".sha"
        flags = ARCH + COMMON + EXTRA.get(src, []) + (["-DGFLA_TC_PROFILE"] if os.environ.get("GFLA_BUILD_PROFILE") == "1" else []) + (["-DGFLA_TC_KNOBS_ON"] if os.environ.get("GFLA_BUILD_KNOBS") == "1" else []) \
            + ([f"-DGFLA_TC_WAIT_CYCLES={int(os.environ['GFLA_TC_WAIT_CYCLES'])}LL"] if os.environ.get("GFLA_TC_WAIT_CYCLES") else [])
        dig = _digest([path] + headers) + " " + " ".join(flags)
        if not force and os.path.exists(obj) and os.path.exists(stamp) and open(stamp).read() == dig:
            continue
        jobs.append((src, [nvcc] + flags + ["-c", path, "-o", obj], stamp, dig))

    def run(job):
        src, cmd, stamp, dig = job
        if verbose:
            print(" ".join(cmd), flush=True)
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{r.stdout}\n{r.stderr}")
        with open(stamp, "w") as f:
            f.write(dig)
        return src

    if jobs:
        with cf.ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 4)) as ex:
            list(ex.map(run, jobs))
    objs = [os.path.join(OBJ, s[:-3] + ".o") for s in sources]
    if jobs or force or not os.path.exists(LIB):
        cmd = [nvcc] + ARCH + ["-shared", "-o", LIB] + objs
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
