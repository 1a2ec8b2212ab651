"""Builds the in-tree native library (CUDA kernels for sm_100a + C++ host) and the `modkit` CLI.

    python -m modkit_b200.build            # libmodkit_b200.so + modkit
nvcc cross-compiles without a GPU. The .so stays in-tree (git-ignored, shipped by gpurun).
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "_build")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]


def _newer(target, sources):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in sources)


def build(force=False, verbose=False):
    os.makedirs(OUT, exist_ok=True)
    csrc = os.path.join(HERE, "csrc")
    host = os.path.join(csrc, "host")
    inc = os.path.join(os.path.dirname(HERE), "include", "mkp.h")
    dev_src = [os.path.join(csrc, "mkp_device.cu"), os.path.join(csrc, "mkp_kernels.cuh"), os.path.join(csrc, "mkp_ingest.cuh"), os.path.join(csrc, "mkp_fused.cuh"), os.path.join(csrc, "mkp_tile.cuh"), os.path.join(csrc, "mkp_hemi.cuh"), inc]
    host_src = [os.path.join(host, f) for f in ("capi.cpp", "bam_reader.hpp", "pileup_host.hpp", "pileup_run.hpp", "pileup_hemi.hpp")] + [inc]
    lib = os.path.join(OUT, "libmodkit_b200.so")
    exe = os.path.join(OUT, "modkit")
    common = ["-O3", "-std=c++17", "-lineinfo", "--fmad=false", "-Xcompiler", "-fPIC,-O3,-pthread,-ffp-contract=off"]
    if force or _newer(lib, dev_src + host_src):
        cmd = [NVCC] + ARCH + common + (["-Xptxas", "-v"] if verbose else []) + ["-shared", dev_src[0], host_src[0], "-o", lib, "-lz", "-lcudart"]
        subprocess.check_call(cmd)
    if force or _newer(exe, [lib, os.path.join(host, "main.cpp")]):
        cmd = ["g++", "-O2", "-std=c++17", "-pthread", os.path.join(host, "main.cpp"), "-o", exe, "-L" + OUT, "-lmodkit_b200",
               "-Wl,-rpath,$ORIGIN", "-L/usr/local/cuda/lib64", "-Wl,-rpath,/usr/local/cuda/lib64", "-lz"]
        subprocess.check_call(cmd)
    return lib


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
