"""Builds libdekf_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
SO = os.path.join(HERE, "libdekf_b200.so")
SOURCES = ["dekf_api.cu"]
DEPS = ["dekf_api.cu", "solve_tma.cuh", "box_solve.cuh", "box_team.cuh", "foot_team.cuh", "foot_window.cuh", "box_window.cuh", "footstate.cuh", "estimator_core.cuh", "smallmat.cuh", "kinematics.cuh", "host_setup.hpp"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-shared",
              "-Xcompiler", "-fPIC", "--use_fast_math=false"]


def needs_build():
    if not os.path.exists(SO):
        return True
    t = os.path.getmtime(SO)
    deps = [os.path.join(CSRC, d) for d in DEPS] + [os.path.join(HERE, "..", "include", "dekf_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False, defines=(), out=None):
    """`defines` / `out`: tuning variants of the library (tools/, never the product default)."""
    target = out or SO
    if not force and out is None and not needs_build():
        return SO
    nvcc = os.environ.get("NVCC", "nvcc")
    flags = [f for f in NVCC_FLAGS if not f.startswith("--use_fast_math")]
    cmd = [nvcc] + flags + [f"-D{d}" for d in defines] + (["-Xptxas", "-v"] if verbose else []) + ["-o", target] + [
        os.path.join(CSRC, s) for s in SOURCES]
    subprocess.check_call(cmd)
    return target


if __name__ == "__main__":
    import sys
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
