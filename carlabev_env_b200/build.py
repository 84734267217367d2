"""Build libcbev.so (the C-ABI CUDA library) in-tree with nvcc for sm_100a."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libcbev.so")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr"]
# sim.cu must evaluate a*b+c unfused, like the reference's NumPy / CPython scalars
SOURCES = [("api.cu", []), ("sim.cu", ["-fmad=false"]), ("render.cu", []), ("scenegen.cu", ["-fmad=false"]),
           ("snapshot.cu", [])]


def nvcc_path() -> str:
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; the CUDA engine cannot be built")


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(os.path.dirname(HERE), "include", "cbev.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB
    nvcc = nvcc_path()
    objs = []
    out_dir = os.path.join(HERE, "build")
    os.makedirs(out_dir, exist_ok=True)
    for src, extra in SOURCES:
        obj = os.path.join(out_dir, src.replace(".cu", ".o"))
        cmd = [nvcc, *ARCH, *COMMON, *extra, "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        subprocess.run(cmd, check=True)
        objs.append(obj)
    subprocess.run([nvcc, *ARCH, "-shared", "-Xcompiler", "-fPIC", *objs, "-o", LIB, "-lcudart"], check=True)
    return LIB


if __name__ == "__main__":
    print(build(force=True, verbose="-v" in sys.argv))
