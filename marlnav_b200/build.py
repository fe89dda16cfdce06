"""marlnav_b200/build.py -- compile libmarlnav_b200.so in-tree with nvcc for sm_100a.

    python -m marlnav_b200.build [--force] [--verbose]

nvcc cross-compiles without a GPU.  -fmad=false is REQUIRED: the kernels spell
every fused multiply-add explicitly (__fmaf_rn) and rely on plain `a*b+c` staying
unfused to reproduce torch-CPU's float32 results bit for bit (SURVEY.md Appendix A).

Every csrc/*.cu is one unit, compiled by its own nvcc process, all at the same time, into a
temporary directory; the objects are then linked once.  The library is rebuilt when any
csrc/*.cu, csrc/*.cuh or include/*.h is newer than it.
"""
import glob
import os
import subprocess
import sys
import tempfile

_HERE = os.path.dirname(os.path.abspath(__file__))
SOURCES = sorted(glob.glob(os.path.join(_HERE, "csrc", "*.cu")))
DEPS = SOURCES + sorted(glob.glob(os.path.join(_HERE, "csrc", "*.cuh")) +
                        glob.glob(os.path.join(os.path.dirname(_HERE), "include", "*.h")))
LIB = os.path.join(_HERE, "libmarlnav_b200.so")

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-fmad=false", "-prec-div=true", "-prec-sqrt=true", "-ftz=false",
              "-Xcompiler", "-fPIC,-mfma,-ffp-contract=off"]
LINK_FLAGS = ["-shared", "-cudart", "static"]


def nvcc_path():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def compile_library(out_path, extra_flags=(), verbose=False):
    """Compile every unit with NVCC_FLAGS + extra_flags in parallel and link them into out_path."""
    nvcc, flags = nvcc_path(), NVCC_FLAGS + list(extra_flags) + (["-Xptxas", "-v"] if verbose else [])
    with tempfile.TemporaryDirectory(prefix="marlnav_build_") as tmp:
        objs = [os.path.join(tmp, os.path.basename(src) + ".o") for src in SOURCES]
        # each unit's output goes to a file: a pipe nobody reads yet would stall that nvcc
        logs = [open(obj + ".log", "w+") for obj in objs]
        procs = [subprocess.Popen([nvcc] + flags + ["-c", "-o", obj, src], stdout=log, stderr=subprocess.STDOUT)
                 for src, obj, log in zip(SOURCES, objs, logs)]
        failed = []
        for src, proc, log in zip(SOURCES, procs, logs):
            proc.wait()
            log.seek(0)
            if verbose or proc.returncode != 0:
                sys.stderr.write(log.read())
            log.close()
            if proc.returncode != 0:
                failed.append(os.path.basename(src))
        if failed:
            raise RuntimeError(f"nvcc failed compiling {', '.join(failed)} (see stderr)")
        # with the same -gencode as the units, or nvcc adds a device-link stub for its default arch
        res = subprocess.run([nvcc] + flags + LINK_FLAGS + ["-o", out_path] + objs, capture_output=True, text=True)
        if verbose or res.returncode != 0:
            sys.stderr.write(res.stdout + res.stderr)
        if res.returncode != 0:
            raise RuntimeError(f"nvcc failed linking {out_path} (see stderr)")
    return out_path


def build(force=False, verbose=False):
    """Compile when the library is missing or older than its sources; returns its path."""
    if not force and os.path.exists(LIB) and all(os.path.getmtime(LIB) >= os.path.getmtime(d) for d in DEPS):
        return LIB
    return compile_library(LIB, verbose=verbose)


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
