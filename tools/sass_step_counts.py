#!/usr/bin/env python3
"""FP64, shuffle and local-memory instruction counts of the step loops of one trajectory-kernel instantiation, from its SASS.

    python tools/sass_step_counts.py "TileLane<2, 1, 1>, 1, 2, 4, 0, 8"              # compile that one instantiation
    python tools/sass_step_counts.py "TileLane<2, 1, 1>, 1, 2, 4, 0, 8" --lib        # juqbox_b200/lib/libjuqbox_b200.so
    python tools/sass_step_counts.py "TileLane<2, 1, 1>, 1, 2, 4, 0, 8" --lib path/to/lib.so

The argument is the template argument list of jq_traj_kernel (LaneT, UPL, MINB, JT, OBJ, GLT, NW, PIPE, SEG), as passed to
traj_inst; trailing defaults may be left out.  Without --lib the instantiation is compiled alone from juqbox_b200/csrc with the
build's nvcc flags, which gives the same code as the library build.  Needs nvcc / cuobjdump, no GPU.

A loop is a backward branch; the step loops are the innermost loops of at least --min-len instructions (default 500): the time
loops of the forward sweep -- one copy with the history stores, one without -- and of the backward sweep.  The control-table fills
(about 300 instructions each) and the hand-over waits are smaller; lower --min-len for layouts with few elements per lane.  Counts are static: instructions in the loop body, i.e. per lane per time step for the unrolled
step code.  Also prints the registers and spill bytes ptxas reports for the compiled kernel (not with --lib).
"""
import argparse
import collections
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)
OPS = ["DFMA", "DMUL", "DADD", "SHFL", "STL", "LDL"]
DEFAULTS = ["1", "0", "0", "0", "TRAJ_WARPS", "0", "false"]        # MINB, JT, OBJ, GLT, NW, PIPE, SEG


def split_args(s):
    out, depth, cur = [], 0, ""
    for ch in s:
        depth += ch == "<"
        depth -= ch == ">"
        if ch == "," and depth == 0:
            out.append(cur.strip())
            cur = ""
        else:
            cur += ch
    return out + [cur.strip()] if cur.strip() else out


def compile_one(args):
    from juqbox_b200 import build
    csrc = os.path.join(os.path.abspath(ROOT), "juqbox_b200", "csrc")
    with tempfile.TemporaryDirectory() as d:
        cu, obj = os.path.join(d, "one.cu"), os.path.join(d, "one.o")
        with open(cu, "w") as f:
            f.write(f'#include "{csrc}/jq_traj_kernels.cuh"\n'
                    f"const Inst kOne[] = {{ traj_inst<{args}>() }};\n"
                    "const InstPart kInstD = inst_part(kOne);\n")
        flags = [x for x in build.NVCC_FLAGS if x not in ("--threads", "0")]
        r = subprocess.run([build._nvcc(), *flags, "-Xptxas", "-v", "-c", cu, "-o", obj], capture_output=True, text=True)
        if r.returncode != 0:
            sys.exit(r.stderr)
        ptxas = [re.sub(r"^ptxas info\s*:\s*", "", l.strip()) for l in r.stderr.splitlines() if re.search(r"spill stores|Used \d+ registers", l)]
        sass = subprocess.run(["cuobjdump", "-sass", obj], capture_output=True, text=True, check=True).stdout
    return sass, ptxas


def function_from_lib(lib, args):
    sass = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout
    blocks = re.split(r"\n\s*Function : (\S+)\n", sass)
    names = blocks[1::2]
    dem = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True).stdout.splitlines()
    want = re.sub(r"\s+", "", f"jq_traj_kernel<{args}>")
    hits = [i for i, d in enumerate(dem) if want in re.sub(r"\s+", "", d.replace("(anonymous namespace)::", ""))]
    if len(hits) != 1:
        sys.exit(f"{len(hits)} kernels match {want!r} in {lib}")
    return blocks[2 + 2 * hits[0]]


def step_loops(sass, min_len):
    ins = []
    for line in sass.splitlines():
        m = re.match(r"\s+/\*([0-9a-f]{4,})\*/\s+(.*?);", line)
        if m:
            op = re.match(r"(@!?U?P\w+\s+)?([A-Z0-9_]+)", m.group(2)).group(2)
            ins.append((int(m.group(1), 16), op, m.group(2)))
    loops = []
    for a, op, txt in ins:
        m = re.search(r"BRA\b.*?0x([0-9a-f]+)", txt) if op == "BRA" else None
        if m and int(m.group(1), 16) < a:
            loops.append((int(m.group(1), 16), a))
    big = [(t, a) for t, a in loops if sum(1 for x in ins if t <= x[0] <= a) >= min_len]
    inner = [(t, a) for t, a in big if not any((t2, a2) != (t, a) and t <= t2 and a2 <= a for t2, a2 in big)]
    out = []
    for t, a in sorted(set(inner)):
        c = collections.Counter(x[1] for x in ins if t <= x[0] <= a)
        out.append((t, a, sum(c.values()), c))
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("inst", help='template arguments of jq_traj_kernel, e.g. "TileLane<2, 1, 1>, 1, 2, 4, 0, 8"')
    ap.add_argument("--lib", nargs="?", const="", default=None, help="count in the built library (default path when no value)")
    ap.add_argument("--min-len", type=int, default=500, help="smallest loop body, in instructions, that counts as a step loop")
    a = ap.parse_args()
    args = split_args(a.inst)
    if len(args) < 2:
        sys.exit("need at least LaneT and UPL")
    if a.lib is None:
        sass, ptxas = compile_one(", ".join(args))
        for l in ptxas:
            print("ptxas:", l)
    else:
        from juqbox_b200 import build
        full = args + DEFAULTS[len(args) - 2:]
        full = [x.replace("TRAJ_WARPS", "4") for x in full]
        sass = function_from_lib(a.lib or build.LIB, ", ".join(full))
    print("loop [first, last] address | instructions | " + " ".join(f"{o:>5s}" for o in OPS) + " | FP64")
    for t, e, n, c in step_loops(sass, a.min_len):
        print(f"[{t:#07x}, {e:#07x}] | {n:5d} | " + " ".join(f"{c[o]:5d}" for o in OPS) + f" | {c['DFMA'] + c['DMUL'] + c['DADD']:5d}")


if __name__ == "__main__":
    main()
