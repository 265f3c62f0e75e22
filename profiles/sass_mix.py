#!/usr/bin/env python3
"""Static instruction mix of the middle scan's hot loop (CPU only, no GPU needed).

Compiles tgsfilter_b200/csrc/tgsf_cuda.cu for sm_100a to a cubin (nvcc -cubin -Xptxas -v), disassembles one
k_mid_scan_dyn<NW, AP> instantiation (cuobjdump -sass) and finds its loops that load 16 bases per iteration
(LDG.E.128): the halo loop and the tracked loop, which is the hot one.  Prints, per adapter-column (one loop
iteration is 16 columns for each of the AP adapters), the instructions of each such loop by pipe and by opcode,
and the registers / stack / spills ptxas reports for the kernel.  `--packed` does the same for k_mid_scan_packed,
which scans a pair of adapters of <= 50 bp as one 96-bit vector (2 adapter-columns per column).

The pipe of an opcode follows NVIDIA's instruction-set notes: LOP3, IADD3, SHF, ISETP, LEA, SEL, PRMT and the
integer min/max ops issue to the ALU pipe; IMAD in all its forms (.X, .MOV, .SHL, .IADD) to the FMA pipe.  The
count is static: every instruction of the loop body once, including the few that only a rare branch executes.

    python profiles/sass_mix.py                 # k_mid_scan_dyn<1,2>, the benchmark's instantiation
    python profiles/sass_mix.py --nw 4 --ap 1
    python profiles/sass_mix.py --packed        # k_mid_scan_packed, what the benchmark's adapter pair runs now
    python profiles/sass_mix.py --cubin x.cubin --ptxas-log x.log   # reuse an earlier compile
"""
from __future__ import annotations

import argparse
import collections
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tgsfilter_b200", "csrc", "tgsf_cuda.cu")

PIPES = [
    ("alu", {"LOP3", "LOP", "IADD3", "IADD", "VIADD", "SHF", "SHL", "SHR", "ISETP", "SEL", "LEA", "PLOP3", "IMNMX", "VIMNMX",
             "VIMNMX3", "VIADDMNMX", "PRMT", "BMSK", "SGXT", "P2R", "R2P", "IABS", "FSEL", "FSETP", "FMNMX"}),
    ("fma", {"IMAD", "IMUL", "FFMA", "FMUL", "FADD", "HFMA2"}),
    ("popc/flo", {"POPC", "FLO", "BREV"}),
    ("lsu", {"LDS", "LDG", "STS", "STG", "LD", "ST", "LDL", "STL", "ATOM", "ATOMS", "ATOMG", "RED", "LDC"}),
    ("uniform", {"S2UR", "R2UR", "ULDC"}),
    ("control", {"BRA", "BSSY", "BSYNC", "CALL", "RET", "EXIT", "WARPSYNC", "NOP", "BAR", "YIELD", "BREAK"}),
]

LINE = re.compile(r"^\s*/\*([0-9a-f]{4,})\*/\s+(?:@!?U?P[0-9T]\s+)?([A-Z0-9_]+)((?:\.[A-Z0-9_]+)*)\s*(.*?);")


def pipe_of(op: str) -> str:
    for name, ops in PIPES:
        if op in ops:
            return name
    if op.startswith("U"):
        return "uniform"
    return "other"


def compile_cubin(out_dir: str) -> tuple[str, str]:
    cubin = os.path.join(out_dir, "tgsf_cuda.cubin")
    nvcc = os.environ.get("NVCC", "nvcc")
    cmd = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-cubin", "-Xptxas", "-v",
           "-o", cubin, SRC]
    r = subprocess.run(cmd, check=True, capture_output=True, text=True, cwd=ROOT)
    return cubin, r.stdout + r.stderr


def function_sass(cubin: str, mangled_prefix: str) -> tuple[str, list[tuple[int, str, str, str]]]:
    sass = subprocess.run(["cuobjdump", "-sass", cubin], check=True, capture_output=True, text=True).stdout
    name, body = None, []
    for line in sass.splitlines():
        if "Function :" in line:
            if name is not None:
                break
            fn = line.split("Function :", 1)[1].strip()
            if fn.startswith(mangled_prefix):
                name = fn
            continue
        if name is not None:
            m = LINE.match(line)
            if m:
                body.append((int(m.group(1), 16), m.group(2), m.group(3), m.group(4)))
    if name is None:
        sys.exit(f"no function {mangled_prefix}* in {cubin}")
    return name, body


def loops_with_wide_loads(body):
    """(start, end) address ranges of the innermost backward-branch loops that contain an LDG.E.128."""
    loops = []
    for addr, op, mods, args in body:
        if op == "BRA":
            m = re.search(r"0x([0-9a-f]+)", args)
            if m and int(m.group(1), 16) <= addr:
                loops.append((int(m.group(1), 16), addr))
    inner = [lp for lp in loops if not any(o != lp and lp[0] <= o[0] and o[1] <= lp[1] for o in loops)]
    return [lp for lp in inner
            if any(lp[0] <= a <= lp[1] and op == "LDG" and ".128" in mods for a, op, mods, _ in body)]


def ptxas_resources(log: str, name: str) -> str:
    lines = log.splitlines()
    for i, line in enumerate(lines):
        if "Compiling entry function" in line and f"'{name}'" in line:
            out = []
            for l in lines[i + 1:i + 6]:
                if "Compiling entry function" in l:
                    break
                if "stack frame" in l or "Used" in l:
                    out.append(l.split("info    :")[-1].strip())
            return "; ".join(out)
    return "not found in the ptxas log"


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--nw", type=int, default=1, help="Myers words per adapter (template NW)")
    ap.add_argument("--ap", type=int, default=2, help="adapters per thread (template AP)")
    ap.add_argument("--packed", action="store_true", help="k_mid_scan_packed (a pair in one 96-bit vector)")
    ap.add_argument("--cubin", help="use this cubin instead of compiling")
    ap.add_argument("--ptxas-log", help="with --cubin: the -Xptxas -v output of that compile")
    args = ap.parse_args()

    with tempfile.TemporaryDirectory(prefix="sass_mix_") as tmp:
        if args.cubin:
            cubin = args.cubin
            log = open(args.ptxas_log).read() if args.ptxas_log else ""
        else:
            cubin, log = compile_cubin(tmp)
        if args.packed:
            args.ap = 2
            name, body = function_sass(cubin, "_Z17k_mid_scan_packed")
        else:
            name, body = function_sass(cubin, f"_Z14k_mid_scan_dynILi{args.nw}ELi{args.ap}E")

    cols = 16 * args.ap
    print(f"k_mid_scan_packed  ({name})" if args.packed else f"k_mid_scan_dyn<{args.nw},{args.ap}>  ({name})")
    if log:
        print(f"  ptxas: {ptxas_resources(log, name)}")
    loops = sorted(loops_with_wide_loads(body), key=lambda lp: lp[1] - lp[0])
    if not loops:
        sys.exit("no loop with a 16-byte load found")
    for i, (lo, hi) in enumerate(loops):
        label = "hot loop (tracked columns)" if i == len(loops) - 1 else "halo loop"
        ins = [(op, mods) for a, op, mods, _ in body if lo <= a <= hi]
        by_op = collections.Counter(op + (".X" if op in ("IADD3", "IMAD") and ".X" in mods else "")
                                    + (".MOV" if op == "IMAD" and ".MOV" in mods else "")
                                    + (".SHL" if op == "IMAD" and ".SHL" in mods else "")
                                    + (".HI" if op == "IMAD" and ".HI" in mods else "") for op, mods in ins)
        by_pipe = collections.Counter()
        for op, _ in ins:
            by_pipe[pipe_of(op)] += 1
        print(f"\n  {label}: 0x{lo:x}..0x{hi:x}, {len(ins)} instructions = {len(ins) / cols:.2f} per adapter-column "
              f"({cols} adapter-columns per iteration)")
        for pipe, n in sorted(by_pipe.items(), key=lambda kv: -kv[1]):
            print(f"    {pipe:10s} {n:5d}  {n / cols:6.2f} per adapter-column  {n * args.ap / cols:6.2f} per column")
        print("    by opcode: " + ", ".join(f"{op} {n / cols:.2f}" for op, n in by_op.most_common()))


if __name__ == "__main__":
    main()
