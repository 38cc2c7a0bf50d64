"""Builds librg_b200.so (sm_100a) in-tree with nvcc.  No torch involved: the boundary is a plain C ABI."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "librg_b200.so")
SOURCES = ["librg_b200.cu"]
HEADERS = ["ctx.cu", "f_api.cu", "pnp_api.cu", "geom_api.cu", "geom_kernels.cuh", "gs_api.cu", "gs_kernels.cuh", "ba_api.cu", "ba_kernels.cuh", "nccl_api.cu", "p2p_api.cu", "philox.cuh", "microbench.cu", "common.cuh", "score_core.cuh", "f_kernels.cuh", "jacobi.cuh", "pnp_kernels.cuh", "pnp_refine_api.cu", "pnp_refine_kernels.cuh", "tall.cuh", "plan.cuh", "bounded.cuh"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared", "-Xptxas", "-v", "-ldl"]


def _stale() -> bool:
    if not os.path.isfile(LIB):
        return True
    t = os.path.getmtime(LIB)
    for f in SOURCES + HEADERS:
        p = os.path.join(CSRC, f)
        if os.path.isfile(p) and os.path.getmtime(p) > t:
            return True
    return os.path.getmtime(os.path.abspath(__file__)) > t


LIB_DEBUG = os.path.join(HERE, "librg_b200_debug.so")


def build_debug(force: bool = False) -> str:
    """The same library with -DRG_DEBUG: device-side bounds / invariant assertions (RG_ASSERT) compiled in.  Loaded by
    tests/test_gpu_debug_build.py through RG_LIB; never the default."""
    if not force and os.path.isfile(LIB_DEBUG) and os.path.getmtime(LIB_DEBUG) >= max(
            os.path.getmtime(os.path.join(CSRC, f)) for f in SOURCES + HEADERS if os.path.isfile(os.path.join(CSRC, f))):
        return LIB_DEBUG
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    flags = [f for f in NVCC_FLAGS if f not in ("-Xptxas", "-v")]
    cmd = [nvcc] + flags + ["-DRG_DEBUG"] + [os.path.join(CSRC, f) for f in SOURCES] + ["-o", LIB_DEBUG]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
        raise RuntimeError("nvcc failed building librg_b200_debug.so")
    return LIB_DEBUG


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not _stale():
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    srcs = [os.path.join(CSRC, f) for f in SOURCES if os.path.isfile(os.path.join(CSRC, f))]
    cmd = [nvcc] + NVCC_FLAGS + srcs + ["-o", LIB]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed building librg_b200.so")
    with open(os.path.join(HERE, "build_ptxas.log"), "w") as f:
        f.write(res.stdout + res.stderr)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
    if "--debug" in sys.argv:
        print(build_debug(force="--force" in sys.argv))
