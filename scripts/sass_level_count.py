#!/usr/bin/env python3
"""Instructions per hash-grid level in one kernel's SASS, by opcode class.

Compiles a CUDA source for sm_100a (the library's flags), disassembles it with cuobjdump and splits the chosen kernel at its
8-byte table gathers (LDG.E.64), 8 loads (corners) per level in program order.  A level's segment runs from its first load
to the first load of the next level; the last level of a region ends at the first store or barrier after it, so it also holds
whatever code follows (the next path's set-up, for instance): read the levels before it.  The compiler interleaves the blend
of one level with the geometry of the next, so a segment is a level's worth of work, not the instructions of one level in
source order.  Counts are static: code that a segment branches over (such as the `% size` fallback of a hashed level whose
size is not a power of two) is counted as well.

usage: python scripts/sass_level_count.py instance_nerf_b200/csrc/render_fused.cu --kernel 'k_render_fusedILi1E'
       [--nvcc-arg=-DFOO ...] [--all]
"""
from __future__ import annotations

import argparse
import os
import re
import subprocess
import sys
import tempfile
from collections import Counter

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
CUOBJDUMP = os.path.join(os.path.dirname(NVCC), "cuobjdump")
FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "--expt-relaxed-constexpr", "-cubin"]

# opcode class of a SASS mnemonic (first match wins; matched against the full dotted mnemonic)
CLASSES = [
    ("gather", r"^LDG\.E\.64"),
    ("other load", r"^LD"),
    ("address", r"^(LEA|IMAD\.WIDE|IMAD\.X|IADD3\.X|IADD\.64|IADD3\.64)"),
    ("logic", r"^LOP3"),
    ("int", r"^(IADD3|VIADD|IMAD|SHF|SHL|SHR|ISETP|SEL|IABS|IMNMX|VIMNMX|MOV|PRMT|I2F|F2I\.U32\.TRUNC|F2I\.FTZ|MUFU)"),
    ("blend", r"^(HADD2|HFMA2|HMUL2|F2FP|FMUL2|FFMA2|FADD2)"),
    ("fp32", r"^(FADD|FMUL|FFMA|FRND|F2I|FSETP|FSEL|FMNMX)"),
    ("control", r"^(BRA|BSSY|BSYNC|WARPSYNC|BAR|EXIT|RET|CALL|NOP|YIELD|PLOP3|VOTE|BREAK)"),
]
STORE_OR_BARRIER = re.compile(r"^(STTM|STS|STG|ST\.|BAR|SYNCS|EXIT|RET|WARPSYNC)")
INSN = re.compile(r"/\*([0-9a-f]{4,})\*/\s+(@!?U?P\w+\s+)?([A-Z][A-Z0-9_.]*)")


def classify(op: str) -> str:
    for name, pat in CLASSES:
        if re.match(pat, op):
            return name
    return "other"


def compile_sass(src: str, extra: list[str]) -> str:
    with tempfile.TemporaryDirectory() as td:
        cubin = os.path.join(td, "k.cubin")
        inc = ["-I", os.path.join(ROOT, "include"), "-I", os.path.dirname(os.path.abspath(src))]
        subprocess.run([NVCC, *FLAGS, *inc, *extra, "-o", cubin, src], check=True)
        return subprocess.run([CUOBJDUMP, "-sass", cubin], check=True, capture_output=True, text=True).stdout


def functions(sass: str) -> dict[str, list[str]]:
    out: dict[str, list[str]] = {}
    name = None
    for line in sass.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            name = m.group(1)
            out[name] = []
            continue
        if name is None:
            continue
        m = INSN.search(line)
        if m:
            out[name].append(m.group(3))
    return out


def level_segments(ops: list[str], gap: int) -> list[tuple[int, int, int, int]]:
    """(region, start, end, loads) per level.  A region is a run of table gathers with less than `gap` instructions between
    consecutive loads (one code path over consecutive levels); a region whose load count is a multiple of 8 is cut into levels
    of 8 loads in program order (the compiler hoists a few loads of the next level into the previous one)."""
    loads = [i for i, op in enumerate(ops) if op.startswith("LDG.E.64")]
    regions: list[list[int]] = []
    for i in loads:
        if regions and i - regions[-1][-1] <= gap:
            regions[-1].append(i)
        else:
            regions.append([i])
    segs = []
    for r, reg in enumerate(regions):
        end = next((j for j in range(reg[-1] + 1, len(ops)) if STORE_OR_BARRIER.match(ops[j])), len(ops))
        n = 8 if len(reg) % 8 == 0 else len(reg)
        starts = reg[::n]
        for k, s in enumerate(starts):
            segs.append((r, s, starts[k + 1] if k + 1 < len(starts) else end, n))
    return segs


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("source")
    ap.add_argument("--kernel", required=True, help="regex matched against the mangled function names; the first match is used")
    ap.add_argument("--nvcc-arg", action="append", default=[], help="extra nvcc argument (repeatable)")
    ap.add_argument("--gap", type=int, default=320, help="loads closer than this many instructions belong to one region")
    ap.add_argument("--all", action="store_true", help="also print regions whose loads are not levels (single 8-byte loads)")
    a = ap.parse_args()

    funcs = functions(compile_sass(a.source, a.nvcc_arg))
    names = [n for n in funcs if re.search(a.kernel, n)]
    if not names:
        print(f"no function matches {a.kernel!r}; functions: {list(funcs)}", file=sys.stderr)
        return 1
    name = names[0]
    ops = funcs[name]
    cols = [c for c, _ in CLASSES] + ["other"]
    print(f"{name}: {len(ops)} instructions")
    print(f"{'region':>6} {'start':>6} " + " ".join(f"{c:>10}" for c in cols) + f" {'total':>6}")
    for r, s, e, n in level_segments(ops, a.gap):
        if n != 8 and not a.all:
            continue
        cnt = Counter(classify(op) for op in ops[s:e])
        print(f"{r:>6} {s:>6} " + " ".join(f"{cnt[c]:>10}" for c in cols) + f" {e - s:>6}")
    return 0


if __name__ == "__main__":
    sys.exit(main())
