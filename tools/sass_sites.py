#!/usr/bin/env python
"""Static SASS of the wavefront kernels: per kernel, the opcode histogram and where the control-flow instructions
(BRA, BSSY, BSYNC) come from, per source file and per source line (nvdisasm -g). Needs nvcc / nvdisasm, not a GPU.

    python tools/sass_sites.py                          # cross-compiles webp-decoder_b200/csrc/vp8_pairs.cu for sm_100a
    python tools/sass_sites.py --cubin k.cubin          # an existing cubin
    python tools/sass_sites.py --kernel 'vp8_mb_lockstep<(int)4, (bool)1, (bool)1>' --lines 40
    python tools/sass_sites.py --src /path/to/other/csrc/vp8_pairs.cu --summary   # e.g. a checkout of another commit

--summary prints one line per kernel: static instructions, BRA, BSSY, BSYNC, NOP.
Static counts say what the compiler emitted, not how often it runs: executed counts need a profiler on the GPU."""
from __future__ import annotations

import argparse
import collections
import os
import re
import shutil
import subprocess
import sys
import tempfile
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
SRC = ROOT / "webp-decoder_b200" / "csrc" / "vp8_pairs.cu"
FLOW = ("BRA", "BSSY", "BSYNC")


def tool(name: str) -> str:
    for cand in (shutil.which(name), f"/usr/local/cuda/bin/{name}"):
        if cand and Path(cand).exists():
            return cand
    sys.exit(f"{name} not found")


def compile_cubin(src: Path, out: Path, defines: list[str]) -> None:
    cmd = [tool("nvcc"), "-cubin", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
           f"-I{ROOT / 'include'}", *[f"-D{d}" for d in defines], "-o", str(out), str(src)]
    subprocess.run(cmd, check=True)


def demangle(names: list[str]) -> dict[str, str]:
    filt = shutil.which("cu++filt") or "/usr/local/cuda/bin/cu++filt"
    if not Path(filt).exists():
        return {n: n for n in names}
    out = subprocess.run([filt], input="\n".join(names), capture_output=True, text=True, check=True).stdout.splitlines()
    return {n: re.sub(r"\(anonymous namespace\)::", "", d) for n, d in zip(names, out)}


def parse(cubin: Path) -> dict[str, list[tuple[str, int, str]]]:
    """kernel (mangled) -> [(file, line, opcode)] for every instruction of its .text section."""
    text = subprocess.run([tool("nvdisasm"), "-g", "-c", str(cubin)], capture_output=True, text=True, check=True).stdout
    kernels: dict[str, list[tuple[str, int, str]]] = {}
    cur, where = None, ("?", 0)
    sec = re.compile(r"^//-+ \.text\.(\S+) -+")
    loc = re.compile(r'^\s*//## File "([^"]+)", line (\d+)')
    ins = re.compile(r"^\s*/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P[T0-9]+\s+)?([A-Z][A-Z0-9_.]*)")
    for ln in text.splitlines():
        m = sec.match(ln)
        if m:
            cur, where = m.group(1), ("?", 0)
            kernels[cur] = []
            continue
        if cur is None:
            continue
        m = loc.match(ln)
        if m:
            where = (os.path.basename(m.group(1)), int(m.group(2)))
            continue
        m = ins.match(ln)
        if m:
            kernels[cur].append((where[0], where[1], m.group(1)))
    return kernels


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--cubin", type=Path, help="disassemble this cubin instead of compiling")
    ap.add_argument("--src", type=Path, default=SRC, help="source to cross-compile (default: the repository's vp8_pairs.cu)")
    ap.add_argument("-D", dest="defines", action="append", default=[], help="preprocessor define for the compile")
    ap.add_argument("--kernel", default="", help="only kernels whose demangled name contains this text")
    ap.add_argument("--lines", type=int, default=25, help="source lines to list per kernel (most control-flow sites first)")
    ap.add_argument("--summary", action="store_true", help="one line per kernel")
    a = ap.parse_args()

    with tempfile.TemporaryDirectory() as tmp:
        cubin = a.cubin
        if cubin is None:
            cubin = Path(tmp) / "k.cubin"
            compile_cubin(a.src.resolve(), cubin, a.defines)
        kernels = parse(cubin)
    names = demangle(list(kernels))
    for mangled, code in sorted(kernels.items(), key=lambda kv: names[kv[0]]):
        name = names[mangled]
        if a.kernel not in name or not code:
            continue
        ops = collections.Counter(op.split(".")[0] for _, _, op in code)
        # BRA.DIV: the divergence test the compiler puts in front of a warp-collective operation (vote, shuffle, __syncwarp)
        # where it cannot prove the warp converged; it branches to an out-of-line copy of the operation
        div = sum(op == "BRA.DIV" for _, _, op in code)
        if a.summary:
            print(f"{name}: {len(code)} instructions, BRA {ops['BRA']} (BRA.DIV {div}), BSSY {ops['BSSY']}, BSYNC {ops['BSYNC']}, NOP {ops['NOP']}")
            continue
        print(f"== {name}: {len(code)} instructions static (sm_100a), {div} of the BRA are BRA.DIV")
        print("opcode histogram:")
        for op, n in ops.most_common():
            print(f"  {op:12s} {n:6d} {100 * n / len(code):5.1f}%")
        per_file = collections.defaultdict(collections.Counter)
        per_line = collections.defaultdict(collections.Counter)
        for f, line, op in code:
            op = op.split(".")[0]
            if op in FLOW:
                per_file[f][op] += 1
                per_line[(f, line)][op] += 1
        print("control flow per source file:" + "".join(f"{o:>7s}" for o in FLOW))
        for f, c in sorted(per_file.items(), key=lambda kv: -sum(kv[1].values())):
            print(f"  {f:30s}" + "".join(f"{c[o]:7d}" for o in FLOW))
        print(f"control flow per source line (top {a.lines}):" + "".join(f"{o:>7s}" for o in FLOW))
        for (f, line), c in sorted(per_line.items(), key=lambda kv: (-sum(kv[1].values()), kv[0]))[:a.lines]:
            print(f"  {f + ':' + str(line):36s}" + "".join(f"{c[o]:7d}" for o in FLOW))
        print()


if __name__ == "__main__":
    main()
