"""Builds csrc/ into `_lib/libsot_b200.so` with nvcc for sm_100a (cross-compiles without a GPU).

In-tree on purpose: the built library travels with the repository snapshot to the GPU box.
Usage: `python -m sot_b200.build [--force]`, or `build()` from Python / `__graft_entry__.build()`.
"""
from __future__ import annotations

import concurrent.futures as cf
import glob
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ_DIR = os.path.join(HERE, "build")
LIB_DIR = os.path.join(HERE, "_lib")
LIB_PATH = os.path.join(LIB_DIR, "libsot_b200.so")
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xptxas", "-v"]


def _nvcc() -> str:
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found: the CUDA extension cannot be built (there is no CPU fallback)")
    return exe


def _sources():
    return sorted(glob.glob(os.path.join(CSRC, "*.cu")))


def _deps():
    return _sources() + sorted(glob.glob(os.path.join(CSRC, "*.cuh"))) + [
        os.path.join(os.path.dirname(HERE), "include", "sot_b200.h")]


def is_stale() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    return any(os.path.getmtime(p) > t for p in _deps() if os.path.exists(p))


def _compile(src: str) -> str:
    obj = os.path.join(OBJ_DIR, os.path.basename(src)[:-3] + ".o")
    cmd = [_nvcc(), *NVCC_FLAGS, "-c", src, "-o", obj]
    res = subprocess.run(cmd, capture_output=True, text=True)
    with open(obj[:-2] + ".ptxas.log", "w") as f:
        f.write(res.stdout + res.stderr)
    if res.returncode != 0:
        raise RuntimeError(f"nvcc failed for {src}:\n{res.stdout}\n{res.stderr}")
    return obj


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile (if stale or forced) and return the path of the shared library."""
    if not force and not is_stale():
        return LIB_PATH
    os.makedirs(OBJ_DIR, exist_ok=True)
    os.makedirs(LIB_DIR, exist_ok=True)
    # one builder at a time across processes (every rank of a torchrun job can find the library stale at once);
    # whoever gets the lock second finds it fresh and returns
    import fcntl
    with open(os.path.join(LIB_DIR, ".build.lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        if not force and not is_stale():
            return LIB_PATH
        return _build_locked(verbose)


def _build_locked(verbose: bool) -> str:
    wanted = {os.path.basename(src)[:-3] for src in _sources()}
    for old in glob.glob(os.path.join(OBJ_DIR, "*")):  # objects of configurations that no longer exist
        if os.path.basename(old).split(".")[0] not in wanted:
            os.remove(old)
    with cf.ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1)) as pool:
        objs = list(pool.map(_compile, _sources()))
    tmp = f"{LIB_PATH}.{os.getpid()}.tmp"
    cmd = [_nvcc(), "-shared", "-o", tmp, *objs, "-gencode", "arch=compute_100a,code=sm_100a"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError(f"link failed:\n{res.stdout}\n{res.stderr}")
    os.replace(tmp, LIB_PATH)
    if verbose:
        print(f"built {LIB_PATH}", file=sys.stderr)
    return LIB_PATH


def resource_report():
    """(kernel, registers, spill bytes) parsed from the ptxas logs of the last build."""
    import re
    rows = []
    for log in sorted(glob.glob(os.path.join(OBJ_DIR, "*.ptxas.log"))):
        name = None
        spill = 0
        for line in open(log):
            mm = re.search(r"Compiling entry function '(\S+)'", line)
            if mm:
                name = mm.group(1)
            mm = re.search(r"(\d+) bytes spill stores", line)
            if mm:
                spill = int(mm.group(1))
            mm = re.search(r"Used (\d+) registers", line)
            if mm and name:
                rows.append((name, int(mm.group(1)), spill))
                name = None
    return rows


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose=True)
    for name, regs, spill in resource_report():
        print(f"{regs:4d} regs {spill:5d} B spill  {name}")
