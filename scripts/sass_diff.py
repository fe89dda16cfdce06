"""Compare the SASS of two builds of the library, kernel by kernel.

    python scripts/sass_diff.py A.so B.so

Runs `cuobjdump -sass` on both, splits the listings at "Function :" and compares each kernel's
instructions by mangled name.  Prints the kernels only one build has and those whose SASS differs;
exits 0 only when both builds hold the same kernels with identical SASS.  A host-side refactor
should leave every kernel identical.  Needs no GPU.
"""
import os
import re
import subprocess
import sys


def cuobjdump():
    cand = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "cuobjdump")
    return cand if os.path.exists(cand) else "cuobjdump"


def kernels(lib):
    """{mangled name: SASS lines} of every function in `lib`."""
    out = subprocess.run([cuobjdump(), "-sass", lib], capture_output=True, text=True, check=True).stdout
    funcs = {}
    for part in out.split("Function : ")[1:]:
        name, _, body = part.partition("\n")
        lines = []
        for ln in body.splitlines():
            if re.match(r"\s*(\.{5,}|Fatbin )", ln):    # end of the function: a separator or the next
                break                                   # fatbin's banner, which names the source paths
            if ln.strip():
                lines.append(ln.strip())
        funcs[name.strip()] = lines
    return funcs


def main(argv):
    if len(argv) != 3:
        sys.exit(__doc__)
    a, b = kernels(argv[1]), kernels(argv[2])
    only_a, only_b = sorted(a.keys() - b.keys()), sorted(b.keys() - a.keys())
    differ = sorted(k for k in a.keys() & b.keys() if a[k] != b[k])
    for k in only_a:
        print(f"only in {argv[1]}: {k}")
    for k in only_b:
        print(f"only in {argv[2]}: {k}")
    for k in differ:
        print(f"SASS differs: {k} ({len(a[k])} vs {len(b[k])} instruction lines)")
    same = len(a.keys() & b.keys()) - len(differ)
    print(f"{len(a)} vs {len(b)} kernels; {same} identical, {len(differ)} differ, "
          f"{len(only_a)} + {len(only_b)} unmatched")
    return 0 if not (only_a or only_b or differ) else 1


if __name__ == "__main__":
    sys.exit(main(sys.argv))
