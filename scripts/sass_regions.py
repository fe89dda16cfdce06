"""Static instruction accounting of one step-kernel instance, per source region, without a GPU.

    python scripts/sass_regions.py LIB_OR_CUBIN [--kernel SUBSTRING ...] [--source FILE] [--top N]

Disassembles the named instance from a built library (or a cubin) with line information (the
library is compiled with -lineinfo), maps every instruction to the line of the kernel's source
file it was inlined into, and cuts the kernel at the phase markers of that source (comment lines
`// ---- <name>`, e.g. `// ---- P2a: ...`; code before the first one is the prologue).  For each
region it prints the static instruction count, its loops (backward branches: the loop head's
address, the body's size) and the opcode mix; then the registers, stack frame and shared memory
ptxas gave the instance.

Static counts times trip counts are how the step's executed instructions are accounted here: the
thread-per-env kernel's P2b runs A times per env, a no-reset step skips the guarded fallback, P4a
and P4b.  The default instance is the benchmark's: step_env_kernel<3, 3> with the reference's
division profile and float32 observations.
"""
import argparse
import collections
import os
import re
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CUDA_BIN = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin")
HEADLINE = "_ZN2mn15step_env_kernelILi3ELi3ELb0ENS_8DivModesILi3ELi2ELi1ELi2ELi3ELi1EEELb0EfEEvNS_8StepArgsE"

INS_RE = re.compile(r"^\s+(?:\{\s*)?/\*([0-9a-f]{4,})\*/\s+(?:@!?U?P[T0-9]+\s+)?([A-Z][A-Z0-9_]*)([^;]*);")
LINE_RE = re.compile(r'^\s*//## File "([^"]+)", line (\d+)(?: inlined at "([^"]+)", line (\d+))?')


def tool(name):
    path = os.path.join(CUDA_BIN, name)
    return path if os.path.exists(path) else name


def symbols(cubin):
    """name -> symbol index of every function in an ELF cubin (.symtab parsed directly)."""
    import struct
    data = open(cubin, "rb").read()
    assert data[:4] == b"\x7fELF" and data[4] == 2, "64-bit ELF expected"
    shoff, = struct.unpack_from("<Q", data, 0x28)
    shentsize, shnum = struct.unpack_from("<HH", data, 0x3A)
    secs = [struct.unpack_from("<IIQQQQIIQQ", data, shoff + i * shentsize) for i in range(shnum)]
    out = {}
    for s in secs:
        if s[1] != 2:                                   # SHT_SYMTAB
            continue
        strtab = secs[s[6]]
        for i in range(s[5] // 24):
            st_name, st_info = struct.unpack_from("<IB", data, s[4] + 24 * i)
            if st_info & 0xF != 2:                      # STT_FUNC
                continue
            o = strtab[4] + st_name
            out[data[o:data.index(b"\0", o)].decode()] = i
    return out


def find_instance(path, patterns, tmp):
    """(cubin, symbol index, name) of the one function whose name contains every pattern."""
    cubins = [path]
    if not path.endswith(".cubin"):
        subprocess.run([tool("cuobjdump"), "-xelf", "all", os.path.abspath(path)], cwd=tmp, check=True,
                       stdout=subprocess.DEVNULL)
        cubins = sorted(os.path.join(tmp, f) for f in os.listdir(tmp) if f.endswith(".cubin"))
    hits = []
    for c in cubins:
        for name, idx in symbols(c).items():
            if all(p in name for p in patterns):
                hits.append((c, idx, name))
    exact = [h for h in hits if h[2] in patterns]          # a full name wins over the subroutines named after it
    hits = exact or hits
    if len(hits) != 1:
        names = sorted({h[2] for h in hits})
        sys.exit(f"{len(names)} functions match {patterns}" + (":\n  " + "\n  ".join(names[:20]) if names else ""))
    return hits[0]


def markers(source):
    """[(line, region name)] of the `// ---- <name>` phase markers of the kernel source."""
    out = []
    for n, text in enumerate(open(source), 1):
        m = re.match(r"\s*// ---- (P[0-9A-Za-z]+)", text)
        if m:
            out.append((n, m.group(1)))
    return out


def disassemble(cubin, idx, source):
    """[(address, opcode, operands, kernel source line or None)] in address order, and
    {label: index of the instruction it marks}."""
    text = subprocess.run([tool("nvdisasm"), "-gi", "-c", "-fun", str(idx), cubin], check=True,
                          capture_output=True, text=True).stdout
    base = os.path.basename(source)
    out, line, labels = [], None, {}
    for raw in text.splitlines():
        m = re.match(r"^(\.L_x_\d+):", raw)
        if m:
            labels[m.group(1)] = len(out)
            continue
        m = LINE_RE.match(raw)
        if m:
            # the block's last plain `File` entry is the outermost frame: a line of the kernel
            if m.group(3) is None and os.path.basename(m.group(1)) == base:
                line = int(m.group(2))
            elif m.group(3) is not None and os.path.basename(m.group(3)) == base:
                line = int(m.group(4))
            continue
        m = INS_RE.match(raw)
        if m:
            out.append((int(m.group(1), 16), m.group(2), m.group(3), line))
    return out, labels


def resources(path, name):
    res = subprocess.run([tool("cuobjdump"), "-res-usage", path], capture_output=True, text=True).stdout
    lines = res.splitlines()
    for i, l in enumerate(lines):
        if name in l and i + 1 < len(lines):
            return lines[i + 1].strip()
    return "(not found)"


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("lib", help="built library (.so) or cubin")
    ap.add_argument("--kernel", nargs="+", default=[HEADLINE], help="substrings of the mangled instance name")
    ap.add_argument("--source", default=os.path.join(ROOT, "marlnav_b200", "csrc", "marlnav_step_env.cu"))
    ap.add_argument("--top", type=int, default=12, help="opcodes listed per region")
    args = ap.parse_args()

    with tempfile.TemporaryDirectory(prefix="sass_regions_") as tmp:
        cubin, idx, name = find_instance(args.lib, args.kernel, tmp)
        ins, labels = disassemble(cubin, idx, args.source)
        res = resources(cubin, name)
    marks = markers(args.source)

    def region(line):
        r = "prologue"
        for n, nm in marks:
            if line is not None and line >= n:
                r = nm
        return r
    # an instruction without a kernel line (e.g. the trailing BRA-to-self) stays in the previous region
    regions, order, cur = collections.defaultdict(list), [], "prologue"
    for k, (addr, op, opnds, line) in enumerate(ins):
        if line is not None:
            cur = region(line)
        if cur not in regions:
            order.append(cur)
        regions[cur].append(k)
    # loops: a branch back to a lower address; the body is [target, branch]
    loops = []
    for k, (addr, op, opnds, _) in enumerate(ins):
        m = re.search(r"(\.L_x_\d+)", opnds) if op == "BRA" else None
        if m and m.group(1) in labels and labels[m.group(1)] <= k:
            loops.append((labels[m.group(1)], k))

    print(name)
    print(f"{len(ins)} static instructions; {res}")
    print(f"{'region':<10}{'static':>8}  loops (head: body)   opcode mix")
    for r in order:
        ks = regions[r]
        kset = set(ks)
        lps = [f"{ins[s][0]:#06x}: {e - s + 1}" for s, e in loops if s in kset]
        ops = collections.Counter(ins[k][1] for k in ks)
        mix = ops.most_common(args.top)
        local = f" LDL:{ops['LDL']} STL:{ops['STL']}" if ops["LDL"] or ops["STL"] else ""
        print(f"{r:<10}{len(ks):>8}  {', '.join(lps) or '-':<20} " + " ".join(f"{o}:{c}" for o, c in mix) + local)


if __name__ == "__main__":
    main()
