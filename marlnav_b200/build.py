"""marlnav_b200/build.py -- compile libmarlnav_b200.so in-tree with nvcc for sm_100a.

    python -m marlnav_b200.build [--force] [--verbose]

nvcc cross-compiles without a GPU.  -fmad=false is REQUIRED: the kernels spell
every fused multiply-add explicitly (__fmaf_rn) and rely on plain `a*b+c` staying
unfused to reproduce torch-CPU's float32 results bit for bit (SURVEY.md Appendix A).
"""
import os
import subprocess
import sys

_HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(_HERE, "csrc", "marlnav_kernels.cu")
SRC2 = os.path.join(_HERE, "csrc", "marlnav_rollout.cu")
DEPS = [SRC, SRC2, os.path.join(_HERE, "csrc", "marlnav_math.cuh"), os.path.join(_HERE, "csrc", "marlnav_actor.cuh"),
        os.path.join(_HERE, "csrc", "marlnav_launch.cuh"),
        os.path.join(os.path.dirname(_HERE), "include", "marlnav_b200.h"),
        os.path.join(os.path.dirname(_HERE), "include", "marlnav_b200_typed.h"),
        os.path.join(os.path.dirname(_HERE), "include", "marlnav_b200_rollout_typed.h"),
        os.path.join(os.path.dirname(_HERE), "include", "marlnav_b200_final.h")]
LIB = os.path.join(_HERE, "libmarlnav_b200.so")

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-fmad=false", "-prec-div=true", "-prec-sqrt=true", "-ftz=false",
              "-Xcompiler", "-fPIC,-mfma,-ffp-contract=off", "-shared", "-cudart", "static"]


def nvcc_path():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def build(force=False, verbose=False):
    """Compile when the library is missing or older than its sources; returns its path."""
    if not force and os.path.exists(LIB) and all(os.path.getmtime(LIB) >= os.path.getmtime(d) for d in DEPS):
        return LIB
    cmd = [nvcc_path()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB, SRC, SRC2]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed building libmarlnav_b200.so (see stderr)")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
