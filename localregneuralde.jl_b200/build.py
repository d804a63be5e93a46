"""Builds libLRNDE.so (nvcc, sm_100a) and liblrnde_hostcheck.so (g++, CPU) in-tree.

    python localregneuralde.jl_b200/build.py [--force]

The CUDA library is the product; the host-check library only re-exports the scalar
step-size logic of csrc/lrnde_controller.h and the save plan of csrc/lrnde_saveplan.h so
the CPU test-suite can pin them against the oracle without a GPU.
"""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
ROOT = os.path.dirname(HERE)
LIB = os.path.join(HERE, "libLRNDE.so")
HOSTCHECK = os.path.join(HERE, "liblrnde_hostcheck.so")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "--expt-relaxed-constexpr", "-Xcompiler", "-fPIC", "-shared",
]


def _newer(target, sources):
    if not os.path.exists(target):
        return False
    t = os.path.getmtime(target)
    return all(os.path.getmtime(s) <= t for s in sources)


def _sources():
    out = []
    for d in (CSRC, os.path.join(ROOT, "include")):
        for f in sorted(os.listdir(d)):
            if f.endswith((".cu", ".cuh", ".h", ".cpp")):
                out.append(os.path.join(d, f))
    out.append(os.path.abspath(__file__))
    return out


def _deps(path, seen=None):
    """The file and every quoted #include it reaches (object files are rebuilt only when these change)."""
    seen = seen if seen is not None else set()
    if path in seen or not os.path.exists(path):
        return seen
    seen.add(path)
    for line in open(path, errors="ignore"):
        line = line.strip()
        if line.startswith("#include \""):
            inc = line.split("\"")[1]
            _deps(os.path.normpath(os.path.join(os.path.dirname(path), inc)), seen)
    return seen


def build(force: bool = False, verbose: bool = False) -> str:
    srcs = _sources()
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    cus = [s for s in srcs if s.endswith(".cu")]
    flags = [f for f in NVCC_FLAGS if f != "-shared"]
    if os.environ.get("LRNDE_TRACE"):
        flags.append("-DLRNDE_UMMA_TRACE")
    if os.environ.get("LRNDE_WATCHDOG"):
        flags.append("-DLRNDE_WATCHDOG")
    if verbose:
        flags += ["-Xptxas", "-v"]
    procs, objs = [], []
    for cu in cus:  # one translation unit per .cu, compiled in parallel
        obj = os.path.join(objdir, os.path.basename(cu)[:-3] + ".o")
        objs.append(obj)
        if force or not _newer(obj, sorted(_deps(cu)) + [os.path.abspath(__file__)]):
            procs.append((cu, subprocess.Popen([nvcc, *flags, "-c", "-o", obj, cu], cwd=CSRC)))
    failed = [cu for cu, pr in procs if pr.wait() != 0]
    if failed:
        raise subprocess.CalledProcessError(1, "nvcc " + " ".join(failed))
    if force or procs or not _newer(LIB, objs):
        subprocess.run([nvcc, "-shared", "-o", LIB, *objs, "-lcuda"], check=True, cwd=CSRC)
    if force or not _newer(HOSTCHECK, srcs):
        cpps = [s for s in srcs if s.endswith(".cpp")]
        cmd = ["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-o", HOSTCHECK, *cpps]
        subprocess.run(cmd, check=True, cwd=CSRC)
    return LIB


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print(LIB)
