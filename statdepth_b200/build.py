"""Build libsdepth.so (the sm_100a CUDA kernels + C ABI) in-tree with nvcc.

    python -m statdepth_b200.build [--force]

nvcc cross-compiles for sm_100a without a GPU; the .so is git-ignored but travels with the
working tree.  Per-file flags: the geometric kernels are compiled with -fmad=false so that their
float64 decisions are bit-identical to the CPU oracle (see csrc/simplex_pred.cuh).
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "_build")
LIB = os.path.join(HERE, "libsdepth%s.so" % os.environ.get("SD_LIB_SUFFIX", ""))
OBJ_SUFFIX = os.environ.get("SD_LIB_SUFFIX", "")
EXTRA = os.environ.get("SD_EXTRA_NVCC_FLAGS", "").split()
INCLUDE = os.path.join(os.path.dirname(HERE), "include")

ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC",
          "-I", INCLUDE]
SOURCES = {
    "ctx.cu": [],
    "api.cu": [],
    "mbd.cu": [],
    "bd_bits.cu": [],
    "bd_gemm.cu": [],
    "bd_match.cu": [],
    "oos.cu": [],
    "reference.cu": [],
    "reference_proj.cu": ["-fmad=false"],
    "extremal.cu": [],
    "halfspace.cu": [],
    "projection.cu": ["-fmad=false"],
    "outliers.cu": ["-fmad=false"],
    "pointcloud.cu": ["-fmad=false"],
    "simplicial_count.cu": ["-fmad=false"],
    "spatial.cu": [],
}
EXPORT_MAP = os.path.join(CSRC, "exports.map")


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.sep not in cand or os.path.exists(cand)):
            return cand
    raise RuntimeError("nvcc not found")


def _deps_mtime():
    m = 0.0
    for root in (CSRC, INCLUDE):
        for f in os.listdir(root):
            if f.endswith((".cu", ".cuh", ".h", ".map")):
                m = max(m, os.path.getmtime(os.path.join(root, f)))
    return m


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and os.path.exists(LIB) and os.path.getmtime(LIB) >= _deps_mtime():
        return LIB
    os.makedirs(OBJ, exist_ok=True)
    nvcc = _nvcc()
    headers_m = max(os.path.getmtime(os.path.join(CSRC, f)) for f in os.listdir(CSRC) if f.endswith(".cuh"))
    headers_m = max(headers_m, os.path.getmtime(os.path.join(INCLUDE, "statdepth_b200.h")))

    def compile_one(item):
        src, extra = item
        s = os.path.join(CSRC, src)
        o = os.path.join(OBJ, src.replace(".cu", OBJ_SUFFIX + ".o"))
        if not force and os.path.exists(o) and os.path.getmtime(o) >= max(os.path.getmtime(s), headers_m):
            return o
        cmd = [nvcc] + ARCH + COMMON + extra + EXTRA + ["-c", s, "-o", o]
        if verbose:
            print(" ".join(cmd), flush=True)
        subprocess.check_call(cmd)
        return o

    with ThreadPoolExecutor(max_workers=min(6, os.cpu_count() or 1)) as ex:
        objs = list(ex.map(compile_one, SOURCES.items()))
    cmd = [nvcc] + ARCH + ["-shared", "-o", LIB] + objs + ["-Xlinker", "--version-script=" + EXPORT_MAP,
                                                           "-cudart", "static"]
    if verbose:
        print(" ".join(cmd), flush=True)
    subprocess.check_call(cmd)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
