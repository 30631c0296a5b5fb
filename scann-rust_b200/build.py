"""Builds libscann_b200.so in-tree with nvcc for sm_100a (no JIT cache, the .so travels with gpurun)."""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIBDIR, "libscann_b200.so")
SOURCES = ["runtime.cu", "partition.cu", "select.cu", "treeah.cu", "taps.cu", "brute_force.cu", "tc_gemm.cu", "ivf.cu", "tcscan.cu", "build_index.cu", "kmtree.cu"]
HEADERS = ["common.cuh", "kernels.h", "lut16_device.cuh", "lut16_scan_kernel.cuh", "lut_f32_device.cuh", "lut_f32_scan_kernel.cuh", "tcscan.h", os.path.join("..", "..", "include", "scann_b200.h")]

NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-fmad=false",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-Wall", "--expt-relaxed-constexpr", "-diag-suppress", "177",
]


def _newer(target: str, deps) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    """Idempotent and safe under torchrun: ranks serialise on a file lock, objects and the library are written to a
    temporary name and renamed into place, so a concurrent loader never sees a half-written file."""
    import fcntl

    os.makedirs(LIBDIR, exist_ok=True)
    with open(os.path.join(LIBDIR, ".build.lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            return _build_locked(force, verbose)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)


def _build_locked(force: bool, verbose: bool) -> str:
    objdir = os.path.join(LIBDIR, "obj")
    os.makedirs(objdir, exist_ok=True)
    hdrs = [os.path.join(CSRC, h) for h in HEADERS]
    jobs = []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(objdir, src.replace(".cu", ".o"))
        if force or _newer(o, [s] + hdrs):
            cmd = [NVCC] + FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", s, "-o", o + ".tmp.o"]
            jobs.append(cmd)

    def run(cmd):
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode == 0:
            os.replace(cmd[-1], cmd[-1][:-len(".tmp.o")])
        return cmd, r
    if jobs:
        with ThreadPoolExecutor(max_workers=min(len(jobs), 6)) as ex:
            for cmd, r in ex.map(run, jobs):
                if verbose or r.returncode != 0:
                    sys.stderr.write(" ".join(cmd) + "\n" + r.stdout + r.stderr + "\n")
                if r.returncode != 0:
                    raise RuntimeError("nvcc failed for " + cmd[-3])
    objs = [os.path.join(objdir, s.replace(".cu", ".o")) for s in SOURCES]
    if force or jobs or _newer(LIB, objs):
        tmp = LIB + ".tmp"
        cmd = [NVCC, "-shared", "-o", tmp] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-cudart", "static"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            sys.stderr.write(r.stdout + r.stderr)
            raise RuntimeError("link failed")
        os.replace(tmp, LIB)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
