"""Builds marl_llm_b200/lib/libswarm_b200.so (sm_100a only) with nvcc; no JIT, no torch extension machinery.

The .so is built in-tree so that it travels with the repo snapshot to the GPU box.  A `libAssemblyEnv.so` symlink
is placed beside it: that is the file name the reference's c_lib.py:14-21 loads (see INTEGRATION.md)."""
import os
import shutil
import subprocess

PKG = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(PKG, "csrc", "swarm_abi.cu")
SRCS = [SRC, os.path.join(PKG, "csrc", "rollout_abi.cu"), os.path.join(PKG, "csrc", "policy_abi.cu")]
DEPS = SRCS + [os.path.join(PKG, "csrc", "swarm_kernels.cuh"), os.path.join(PKG, "csrc", "render_kernels.cuh"), os.path.join(PKG, "csrc", "state_kernels.cuh"), os.path.join(PKG, "csrc", "rollout_kernels.cuh"), os.path.join(PKG, "csrc", "policy_kernels.cuh"),
        os.path.join(os.path.dirname(PKG), "include", "swarm_b200.h")]
LIB_DIR = os.path.join(PKG, "lib")
LIB = os.path.join(LIB_DIR, "libswarm_b200.so")
LEGACY_NAME = os.path.join(LIB_DIR, "libAssemblyEnv.so")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",   # B200 only
    "-lineinfo", "-O3", "-std=c++17",
    "-fmad=false",                                   # parity: the reference is FMA-free fp64
    "-shared", "-Xcompiler", "-fPIC",
]


def nvcc_path():
    cand = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.isfile(cand):
        raise RuntimeError("nvcc not found")
    return cand


def is_stale():
    if not os.path.isfile(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(d) > t for d in DEPS)


def build_library(force=False, verbose=False):
    if not (force or is_stale()):
        return LIB
    os.makedirs(LIB_DIR, exist_ok=True)
    extra = os.environ.get("SWARM_NVCC_EXTRA", "").split()
    cmd = [nvcc_path()] + NVCC_FLAGS + extra + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB] + SRCS
    env = dict(os.environ)
    env.pop("CC", None); env.pop("CXX", None)        # the image exports a gcc without libgomp specs
    subprocess.check_call(cmd, env=env)
    if os.path.islink(LEGACY_NAME) or os.path.exists(LEGACY_NAME):
        os.remove(LEGACY_NAME)
    os.symlink(os.path.basename(LIB), LEGACY_NAME)
    return LIB


if __name__ == "__main__":
    print(build_library(force=True, verbose=True))
