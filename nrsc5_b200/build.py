"""Builds libnrsc5_b200.so (hand-written sm_100a CUDA + C ABI) in-tree with nvcc.

No torch extension machinery: the product boundary is a plain C-ABI shared
library (include/nrsc5_b200.h) that ctypes, cgo or the reference's own C host
code can bind.
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libnrsc5_b200.so")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = (["-DNB_DEBUG"] if os.environ.get("NB_DEBUG") else []) + ["-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr"]

# (source, extra flags).  engine.cu keeps the reference's float operation order in the acquisition /
# sync arithmetic, so FMA contraction is off there (the FFT uses explicit FMAs).
UNITS = [
    ("frontend.cu", []),
    ("engine.cu", ["-fmad=false"]),
    ("channelizer.cu", []),
]


def _newer(src_paths, out):
    if not os.path.exists(out):
        return True
    t = os.path.getmtime(out)
    return any(os.path.getmtime(p) > t for p in src_paths)


def build(verbose=False, force=False):
    # nvcc from $NVCC, else PATH, else the toolkit under $CUDA_HOME (a login shell need not put it on PATH)
    nvcc = (os.environ.get("NVCC") or shutil.which("nvcc")
            or os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "nvcc"))
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "nrsc5_b200.h")]
    if not force and not _newer(deps, OUT):
        return OUT
    objs = []
    for src, extra in UNITS:
        obj = os.path.join(CSRC, src.replace(".cu", ".o"))
        cmd = [nvcc, *ARCH, *COMMON, *extra, "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
            print(" ".join(cmd), flush=True)
        subprocess.run(cmd, check=True)
        objs.append(obj)
    cmd = [nvcc, *ARCH, "-shared", "-o", OUT, *objs, "-lcudart"]
    subprocess.run(cmd, check=True)
    return OUT


if __name__ == "__main__":
    print(build(verbose="-v" in sys.argv, force=True))
