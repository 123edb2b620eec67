"""Builds ``libzoomvit.so`` in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python -m zoomearth_b200.build [--force]

The shared object is git-ignored but travels with the tree to the GPU box; nothing is JIT-compiled at run
time and there is no fallback if it is missing (``zoomearth_b200._lib`` raises).
"""
import concurrent.futures
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
INCLUDE = os.path.join(os.path.dirname(HERE), "include")
LIB = os.path.join(HERE, "libzoomvit.so")
OBJ_DIR = os.path.join(HERE, "_build")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
SOURCES = ["zv_host.cpp", "zv_handoff.cpp", "zv_handoff.cu", "zv_k1.cu", "zv_gemm.cu", "zv_attn_tc.cu", "zv_attn_win_tc.cu", "zv_tower.cu", "zv_timing.cu"]
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-I", INCLUDE, "-I", CSRC,
          "-Xcompiler", "-fPIC,-fvisibility=hidden,-ffp-contract=off,-Wall,-Wno-unused-function"]
# build-time only: extra nvcc flags for the compile-time debug variants (e.g. ZV_NVCC_EXTRA="-DZV_DEBUG_K1_NO_TC" for an A/B run)
COMMON += os.environ.get("ZV_NVCC_EXTRA", "").split()


def _deps():
    return [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(INCLUDE, "zoomvit.h"), __file__]


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(d) > t for d in _deps())


def _compile(src):
    obj = os.path.join(OBJ_DIR, src + ".o")          # zv_handoff.cpp and zv_handoff.cu both build
    cmd = [NVCC] + ARCH + COMMON + ["-x", "cu", "-c", os.path.join(CSRC, src), "-o", obj]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode:
        raise RuntimeError(f"nvcc failed on {src}:\n{r.stdout}\n{r.stderr}")
    return obj


def build(force=False, verbose=False):
    if not force and not needs_build():
        return LIB
    os.makedirs(OBJ_DIR, exist_ok=True)
    with concurrent.futures.ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        objs = list(ex.map(_compile, SOURCES))
    cmd = [NVCC] + ARCH + ["-shared", "-o", LIB] + objs + ["-ldl", "-Xlinker", "--exclude-libs,ALL"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    if verbose:
        print("built", LIB)
    return LIB


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose=True)
