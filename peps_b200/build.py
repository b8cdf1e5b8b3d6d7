"""Builds libpeps_b200.so (CUDA, sm_100a) in-tree, and -- for CPU-side tests only -- the host simulation
library tests/hostsim/libpeps_hostsim.so (same engine/C ABI, device ops replaced by plain loops)."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libpeps_b200.so")
HOSTSIM_DIR = os.path.join(ROOT, "tests", "hostsim")
HOSTSIM_LIB = os.path.join(HOSTSIM_DIR, "libpeps_hostsim.so")

NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
CUDA_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared", "-x", "cu"]


def _newer(target, sources):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in sources)


def _sources():
    hdr = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".h")] + [os.path.join(ROOT, "include", "peps_b200.h")]
    return hdr


def build_cuda(force=False, verbose=False):
    srcs = [os.path.join(CSRC, f) for f in ("backend_cuda.cu", "engine.cpp", "c_api.cpp")]
    if not force and not _newer(LIB, srcs + _sources()):
        return LIB
    extra = os.environ.get("PEPS_NVCC_EXTRA", "").split()       # e.g. -DPEPS_KERNEL_CLOCKS (development builds)
    cmd = [NVCC] + CUDA_FLAGS + extra + (["-Xptxas", "-v"] if verbose else []) + srcs + ["-o", LIB, "-lcudart"]
    subprocess.check_call(cmd)
    return LIB


def build_hostsim(force=False):
    srcs = [os.path.join(HOSTSIM_DIR, f) for f in ("backend_host.cpp", "backend_host_minsr.cpp")] + \
        [os.path.join(CSRC, "engine.cpp"), os.path.join(CSRC, "c_api.cpp")]
    if not force and not _newer(HOSTSIM_LIB, srcs + _sources()):
        return HOSTSIM_LIB
    cmd = ["g++", "-O2", "-std=c++17", "-fPIC", "-shared"] + srcs + ["-o", HOSTSIM_LIB]
    subprocess.check_call(cmd)
    return HOSTSIM_LIB


if __name__ == "__main__":
    build_cuda(force="--force" in sys.argv, verbose="-v" in sys.argv)
    build_hostsim(force="--force" in sys.argv)
    print("built", LIB, "and", HOSTSIM_LIB)
