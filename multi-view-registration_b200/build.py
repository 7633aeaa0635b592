"""Build recipe for libmvr_b200.so (CUDA kernels + C ABI + C++ host driver), sm_100a only.

Run as `python multi-view-registration_b200/build.py` or through __graft_entry__.build().
nvcc cross-compiles without a GPU; the .so is kept in-tree (git-ignored) so it travels with gpurun.
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
HOST = os.path.join(HERE, "host")
LIB = os.path.join(HERE, "libmvr_b200.so")

CU_SOURCES = ["index.cu", "pair_index.cu", "cell_nn.cu", "icp.cu", "normals.cu", "denoise.cu", "score.cu", "features.cu", "api.cu"]
HOST_SOURCES = ["registrator.cpp", "lum.cpp", "capi.cpp", "multi.cpp", "global.cpp"]

NVCC_FLAGS = [
    "-O3", "-std=c++17",
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo",
    "-Xcompiler", "-fPIC",
    "-fmad=false",          # IEEE add/mul everywhere: the device-side solves match the host arithmetic bit for bit
    "-Xcompiler", "-fno-fast-math",
]


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: the CUDA path cannot be built (there is no CPU fallback)")


def sources():
    srcs = [os.path.join(CSRC, f) for f in CU_SOURCES]
    srcs += [os.path.join(HOST, f) for f in HOST_SOURCES if os.path.exists(os.path.join(HOST, f))]
    return srcs


def deps():
    out = []
    for d in (CSRC, HOST, os.path.join(os.path.dirname(HERE), "include")):
        if os.path.isdir(d):
            out += [os.path.join(d, f) for f in os.listdir(d)]
    return out


def stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(p) > t for p in deps())


def build(force=False, verbose=False, out=None):
    if out is None and not force and not stale():
        return LIB
    cmd = [_nvcc()] + NVCC_FLAGS + ["-shared", "-o", out or LIB, "-x", "cu"] + sources() + ["-ldl"]
    if verbose:
        cmd += ["-Xptxas", "-v"]
        print(" ".join(cmd))
    env = dict(os.environ)
    # the image exports CXX=/opt/gcc/bin/g++ (no OpenMP specs); nvcc should use the system g++
    res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, env=env)
    if verbose or res.returncode != 0:
        sys.stderr.write(res.stdout)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed building libmvr_b200.so")
    return out or LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
