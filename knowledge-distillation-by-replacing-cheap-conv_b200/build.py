"""Builds libkdcc.so (the C-ABI CUDA library, include/kdcc.h) in-tree with nvcc for sm_100a.

    python knowledge-distillation-by-replacing-cheap-conv_b200/build.py [--force]

nvcc cross-compiles without a GPU.  The shared object sits next to this file so that it travels
to the GPU box with the repo snapshot; it is git-ignored.  No torch dependency: plain CUDA runtime
(static) and a run-time lookup of the driver's TMA descriptor encoder.
"""
import concurrent.futures
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "build")
LIB = os.path.join(HERE, "libkdcc.so")

SOURCES = ["loss_kernels.cu", "ce_kernels.cu", "layout_convert.cu", "metrics.cu", "tta.cu", "optim.cu", "dw_direct.cu", "dw_tma.cu", "dw_nhwc3.cu", "dw_tc.cu", "dw_tc2.cu", "dw_tc_wgrad.cu", "dw_tc_wgrad2.cu", "dw_tc_wgrad3.cu", "dw_api.cu", "pw_gemm_sm100.cu", "pw_gemm_simt.cu",
           "pw_api.cu", "tma_host.cu", "api_misc.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC,-fvisibility=hidden", "--expt-relaxed-constexpr"]


def _nvcc():
    return os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc" if os.path.exists("/usr/local/cuda/bin/nvcc") else "nvcc")


def _deps_mtime():
    m = 0.0
    for root in (CSRC, os.path.join(HERE, "..", "include")):
        for fn in os.listdir(root):
            if fn.endswith((".cu", ".cuh", ".h")):
                m = max(m, os.path.getmtime(os.path.join(root, fn)))
    return m


def _compile(src):
    obj = os.path.join(OBJ, src.replace(".cu", ".o"))
    cmd = [_nvcc()] + NVCC_FLAGS + ["-c", os.path.join(CSRC, src), "-o", obj]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed for %s:\n%s\n%s" % (src, r.stdout, r.stderr))
    return obj


def build(force=False, verbose=False):
    if not force and os.path.exists(LIB) and os.path.getmtime(LIB) >= _deps_mtime():
        return LIB
    os.makedirs(OBJ, exist_ok=True)
    with concurrent.futures.ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1)) as ex:
        objs = list(ex.map(_compile, SOURCES))
    cmd = [_nvcc(), "-shared", "-o", LIB] + objs + ["-cudart", "static", "-Xlinker", "--no-undefined", "-ldl", "-lpthread", "-lrt"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n%s\n%s" % (r.stdout, r.stderr))
    if verbose:
        print("built", LIB, os.path.getsize(LIB), "bytes")
    return LIB


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose=True)
