"""Build libldso_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python -m ldso_b200.build [--force]
"""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIBDIR, "libldso_b200.so")
# development aid: LDSO_B200_CFLAGS adds nvcc flags (e.g. -DK3V_...=0), LDSO_B200_LIB redirects the output / the library capi loads
EXTRA = os.environ.get("LDSO_B200_CFLAGS", "").split()
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC", "-shared"]


def sources():
    out = [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC)) if f.endswith((".cu", ".cuh", ".h"))]
    out.append(os.path.join(os.path.dirname(HERE), "include", "ldso_b200.h"))
    return out


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(s) > t for s in sources())


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB
    os.makedirs(LIBDIR, exist_ok=True)
    out = os.environ.get("LDSO_B200_LIB", LIB)
    # one object per .cu unit, compiled side by side; trace.cu (immature-point trace) keeps separate multiply/add roundings:
    # it is built with -fmad=false
    base = [f for f in FLAGS if f != "-shared"] + EXTRA + (["-Xptxas", "-v"] if verbose else [])
    objs, procs = [], []
    for src in sorted(f for f in os.listdir(CSRC) if f.endswith(".cu")):
        obj = os.path.join(LIBDIR, src[:-3] + ".o")
        mad = ["-fmad=false"] if src == "trace.cu" else []
        procs.append(subprocess.Popen([NVCC] + base + mad + ["-c", os.path.join(CSRC, src), "-o", obj]))
        objs.append(obj)
    failed = [p.args for p in procs if p.wait() != 0]
    if failed:
        raise subprocess.CalledProcessError(1, failed[0])
    subprocess.check_call([NVCC] + FLAGS + EXTRA + objs + ["-o", out])
    return out


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
