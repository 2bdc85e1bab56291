"""Builds lib/libssp_b200.so (the C-ABI library, include/ssp_b200.h) with nvcc for sm_100a.

No torch dependency: the library links only the static CUDA runtime, so it loads on a box without a
driver (symbol checks) and takes raw device pointers from any host language.
"""
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_DIR = os.path.join(HERE, "lib")
# SSP_TRACE=1 selects the instrumented variant (timeline trace of the tcgen05 kernels, scripts/trace_desc.py): its own
# object directory and library name, so the product library is never the traced one
TRACE = os.environ.get("SSP_TRACE") == "1"
LIB_PATH = os.path.join(LIB_DIR, "libssp_b200_trace.so" if TRACE else "libssp_b200.so")
OBJ_DIR = os.path.join(HERE, "build_trace" if TRACE else "build")

SOURCES = ["api.cu", "warp.cu", "detector.cu", "semantic.cu", "match.cu", "match_tc.cu", "heatmap.cu", "nms.cu", "subpixel.cu", "desc_common.cu", "desc_simt.cu", "desc_tc.cu", "exchange.cu", "labels.cu", "sparse.cu", "homography.cu", "eval.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "--use_fast_math=false",
]


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; the ssp_b200 CUDA library cannot be built")


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build_library(force=False, verbose=False):
    """Compile every CUDA source for sm_100a and link the shared library. Returns its path."""
    os.makedirs(LIB_DIR, exist_ok=True)
    os.makedirs(OBJ_DIR, exist_ok=True)
    nvcc = _nvcc()
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    flags = [f for f in NVCC_FLAGS if f != "--use_fast_math=false"] + (["-DSSP_TRACE"] if TRACE else [])

    def compile_one(src):
        obj = os.path.join(OBJ_DIR, src.replace(".cu", ".o"))
        path = os.path.join(CSRC, src)
        if force or _stale(obj, [path] + headers):
            cmd = [nvcc] + flags + ["-c", path, "-o", obj]
            if verbose:
                print(" ".join(cmd), file=sys.stderr)
            r = subprocess.run(cmd, capture_output=True, text=True)
            if r.returncode != 0:
                raise RuntimeError("nvcc failed for %s:\n%s\n%s" % (src, r.stdout, r.stderr))
        return obj

    with ThreadPoolExecutor(max_workers=min(8, len(SOURCES))) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    if force or _stale(LIB_PATH, objs):
        cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-cudart", "static", "-o", LIB_PATH] + objs
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("link failed:\n%s\n%s" % (r.stdout, r.stderr))
    return LIB_PATH


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose=True))
