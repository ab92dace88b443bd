"""Builds marl_llm_b200/lib/libswarm_b200.so (sm_100a only) with nvcc; no JIT, no torch extension machinery.

The .so is built in-tree so that it travels with the repo snapshot to the GPU box.  A `libAssemblyEnv.so` symlink
is placed beside it: that is the file name the reference's c_lib.py:14-21 loads (see INTEGRATION.md)."""
import os
import shutil
import subprocess

PKG = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(PKG, "csrc", "swarm_abi.cu")
SRCS = [SRC, os.path.join(PKG, "csrc", "rollout_abi.cu"), os.path.join(PKG, "csrc", "policy_abi.cu"), os.path.join(PKG, "csrc", "prior_abi.cu")]
# the prior-program header is compiled into the library as text (prior_abi.cu hands it to NVRTC): regenerated on every build
PRIOR_API = os.path.join(os.path.dirname(PKG), "include", "swarm_prior_api.cuh")
DEPS = SRCS + [os.path.join(PKG, "csrc", "swarm_kernels.cuh"), os.path.join(PKG, "csrc", "render_kernels.cuh"), os.path.join(PKG, "csrc", "state_kernels.cuh"), os.path.join(PKG, "csrc", "rollout_kernels.cuh"), os.path.join(PKG, "csrc", "policy_kernels.cuh"),
        os.path.join(PKG, "csrc", "prior_program.h"), os.path.join(os.path.dirname(PKG), "include", "swarm_b200.h"), PRIOR_API]
LIB_DIR = os.path.join(PKG, "lib")
LIB = os.path.join(LIB_DIR, "libswarm_b200.so")
LEGACY_NAME = os.path.join(LIB_DIR, "libAssemblyEnv.so")
GEN_DIR = os.path.join(LIB_DIR, "gen")

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


def write_prior_api_text():
    """GEN_DIR/swarm_prior_api.inc: the bytes of include/swarm_prior_api.cuh as a C initializer list (prior_abi.cu)."""
    os.makedirs(GEN_DIR, exist_ok=True)
    data = open(PRIOR_API, "rb").read()
    rows = [", ".join(str(b - 256 if b > 127 else b) for b in data[k:k + 32]) for k in range(0, len(data), 32)]   # as signed char
    with open(os.path.join(GEN_DIR, "swarm_prior_api.inc"), "w") as f:
        f.write(",\n".join(rows) + "\n")


def build_library(force=False, verbose=False):
    if not (force or is_stale()):
        return LIB
    os.makedirs(LIB_DIR, exist_ok=True)
    write_prior_api_text()
    extra = os.environ.get("SWARM_NVCC_EXTRA", "").split()
    cmd = [nvcc_path()] + NVCC_FLAGS + ["-I", GEN_DIR] + extra + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB] + SRCS
    env = dict(os.environ)
    env.pop("CC", None); env.pop("CXX", None)        # the image exports a gcc without libgomp specs
    subprocess.check_call(cmd, env=env)
    if os.path.islink(LEGACY_NAME) or os.path.exists(LEGACY_NAME):
        os.remove(LEGACY_NAME)
    os.symlink(os.path.basename(LIB), LEGACY_NAME)
    return LIB


if __name__ == "__main__":
    print(build_library(force=True, verbose=True))
