"""Builds the sm_100a CUDA library in-tree (flatland-marl_b200/csrc/libflatland_b200.so).

nvcc cross-compiles without a GPU; the built .so is git-ignored but travels to the GPU box."""
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SRC = os.path.join(HERE, "csrc", "flatland_b200.cu")
HDR = os.path.join(ROOT, "include", "flatland_b200.h")
LIB = os.path.join(HERE, "csrc", "libflatland_b200.so")
POLICY_DIR = os.path.join(HERE, "csrc", "policy")
POLICY_SRC = os.path.join(POLICY_DIR, "policy.cu")
POLICY_HDR = os.path.join(ROOT, "include", "flatland_policy_b200.h")
POLICY_LIB = os.path.join(POLICY_DIR, "libflatland_policy_b200.so")

# (nvcc's --split-compile cuts the build from 3 min to 1, but its output differs from run to run — in size by tens of per
# cent; the shipped libraries are built without it so that a rebuild from these sources gives the same bytes.  Development
# builds may set FL_NVCC_SPLIT=1.)
NVCC_FLAGS = (["--split-compile", "0"] if os.environ.get("FL_NVCC_SPLIT") == "1" else []) + \
             ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "--expt-extended-lambda", "-Xcompiler", "-fPIC", "-shared"]


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    srcs = [os.path.join(HERE, "csrc", f) for f in os.listdir(os.path.join(HERE, "csrc")) if f.endswith((".cu", ".cuh", ".h"))]
    return any(os.path.getmtime(p) > t for p in srcs + [HDR])


def policy_needs_build():
    if not os.path.exists(POLICY_LIB):
        return True
    t = os.path.getmtime(POLICY_LIB)
    srcs = [os.path.join(POLICY_DIR, f) for f in os.listdir(POLICY_DIR) if f.endswith((".cu", ".cuh"))]
    return any(os.path.getmtime(p) > t for p in srcs + [POLICY_HDR])


def build(force=False, verbose=False):
    """Both libraries: the step/observation path (libflatland_b200.so) and the policy forward pass
    (policy/libflatland_policy_b200.so, tcgen05 kernels)."""
    nvcc = os.environ.get("NVCC", "nvcc")
    extra = ["-Xptxas", "-v"] if verbose else []
    if force or needs_build():
        subprocess.check_call([nvcc] + NVCC_FLAGS + extra + ["-I", os.path.join(ROOT, "include"), "-o", LIB, SRC])
    if force or policy_needs_build():
        subprocess.check_call([nvcc] + NVCC_FLAGS + extra + ["-I", os.path.join(ROOT, "include"), "-o", POLICY_LIB, POLICY_SRC])
    return LIB


if __name__ == "__main__":
    print(build(force=True, verbose=True))
