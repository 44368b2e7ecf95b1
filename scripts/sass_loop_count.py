#!/usr/bin/env python3
"""Instruction count and opcode mix of a kernel's walk loops, from `cuobjdump -sass` of the built library (no GPU needed).

A loop is the span from a backward branch's target to the branch.  The walk loops are the innermost loops that issue at
least --min-loads global loads; every step of a walk gathers one voxel, so a loop body's step count is its number of LDG
and "per step" is the body's instruction count over that.  Each major-axis instantiation of the sensitivities walk is a
loop of its own (three per kernel).

    python scripts/sass_loop_count.py --kernel 'siddon_sens_slab_kernel<8, 16, 8, 8, false>'
    python scripts/sass_loop_count.py --kernel siddon_sens_slab_kernel --max-per-step 24   # exit 1 above the budget
    python scripts/sass_loop_count.py --md5          # md5 of every function's instruction text, to diff two builds
"""
from __future__ import annotations

import argparse
import collections
import hashlib
import os
import re
import shutil
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEFAULT_LIB = os.path.join(ROOT, "diffdrr_b200", "libb200drr.so")
_INSN = re.compile(r"^\s*/\*([0-9a-f]{4,})\*/\s+(.*?)\s*;")
_BRA = re.compile(r"\bBRA\s+(?:`\(\.L_x_\d+\)|0x([0-9a-f]+))")


def _tool(name: str) -> str:
    path = shutil.which(name) or os.path.join("/usr/local/cuda/bin", name)
    if not os.path.exists(path):
        sys.exit(f"{name} not found (CUDA toolkit)")
    return path


def functions(binary: str) -> dict[str, list[tuple[int, str]]]:
    """mangled name -> [(address, instruction text without encoding)]"""
    text = subprocess.run([_tool("cuobjdump"), "-sass", binary], check=True, capture_output=True, text=True).stdout
    out: dict[str, list[tuple[int, str]]] = {}
    cur = None
    for line in text.splitlines():
        if line.strip().startswith("Function :"):
            cur = line.split(":", 1)[1].strip()
            out[cur] = []
        elif cur is not None:
            m = _INSN.match(line)
            if m:
                out[cur].append((int(m.group(1), 16), " ".join(m.group(2).split())))
    return out


def demangle(names: list[str]) -> dict[str, str]:
    res = subprocess.run([_tool("cu++filt")], input="\n".join(names), check=True, capture_output=True, text=True).stdout
    # cu++filt spells template arguments "(int)8" and "(bool)0": print them as written in the source
    pretty = [n.replace("(int)", "").replace("(bool)0", "false").replace("(bool)1", "true") for n in res.splitlines()]
    return dict(zip(names, pretty))


def opcode(insn: str) -> str:
    """opcode with its modifiers, '@P' prefix kept as a marker of predication: '@P FFMA', 'LDG.E.CONSTANT'"""
    parts = insn.split()
    pred = parts[0].startswith("@")
    op = parts[1] if pred else parts[0]
    return ("@P " if pred else "") + op


def walk_loops(insns: list[tuple[int, str]], min_loads: int) -> list[tuple[int, int, list[str]]]:
    addr_idx = {a: i for i, (a, _) in enumerate(insns)}
    loops = []
    for i, (a, t) in enumerate(insns):
        m = _BRA.search(t)
        if not m or not m.group(1):
            continue
        tgt = int(m.group(1), 16)
        if tgt > a or tgt not in addr_idx:
            continue
        body = [x for _, x in insns[addr_idx[tgt]: i + 1]]
        loops.append((tgt, a, body))
    # innermost only: drop loops that contain another loop
    inner = [lp for lp in loops if not any(o is not lp and lp[0] <= o[0] and o[1] <= lp[1] for o in loops)]
    return [lp for lp in inner if sum(opcode(x).split(".")[0].endswith("LDG") for x in lp[2]) >= min_loads]


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("binary", nargs="?", default=DEFAULT_LIB, help="library or cubin (default: the in-tree libb200drr.so)")
    ap.add_argument("--kernel", default="siddon_sens_slab_kernel<8, 16, 8, 8, false>",
                    help="substring of the demangled kernel name (default: the production sensitivities kernel)")
    ap.add_argument("--min-loads", type=int, default=4, help="a walk loop issues at least this many LDG (default 4)")
    ap.add_argument("--max-per-step", type=float, default=None, help="exit 1 if a walk loop needs more per step")
    ap.add_argument("--md5", action="store_true", help="print md5 of each function's instruction text and exit")
    args = ap.parse_args()

    funcs = functions(args.binary)
    names = demangle(sorted(funcs))
    if args.md5:
        for mangled in sorted(funcs, key=lambda n: names[n]):
            h = hashlib.md5("\n".join(t for _, t in funcs[mangled]).encode()).hexdigest()
            print(f"{h}  {names[mangled]}")
        return 0

    worst = 0.0
    found = False
    for mangled in sorted(funcs, key=lambda n: names[n]):
        if args.kernel not in names[mangled]:
            continue
        found = True
        print(names[mangled])
        for lo, hi, body in walk_loops(funcs[mangled], args.min_loads):
            hist = collections.Counter(opcode(x) for x in body)
            steps = sum(n for op, n in hist.items() if op.split()[-1].startswith("LDG"))
            per = len(body) / steps
            worst = max(worst, per)
            print(f"  loop 0x{lo:04x}-0x{hi:04x}: {len(body)} instructions, {steps} steps, {per:.2f} per step")
            for op, n in hist.most_common():
                print(f"    {n:4d}  {n / steps:5.2f}/step  {op}")
    if not found:
        print(f"no function matches {args.kernel!r}", file=sys.stderr)
        return 2
    if args.max_per_step is not None and worst > args.max_per_step:
        print(f"FAIL: {worst:.2f} instructions per step > {args.max_per_step}")
        return 1
    return 0


if __name__ == "__main__":
    sys.exit(main())
