"""Static instruction mix of every step_fast_kernel instantiation, without a GPU.

Compiles humanoid_b200/csrc/phc_kernels.cu for sm_100a with the flags of build() (into a temporary directory) and
prints, per instantiation: registers, stack frame and spills (ptxas -v), the static SASS instruction count and the
histogram of fp32 opcodes.  It also checks that the SASS counts of FFMA2 / FMUL2 / FADD2 equal the PTX counts of
fma.rn.f32x2 / mul.rn.f32x2 / add.rn.f32x2: ptxas fuses a packed multiply and add into one FFMA2 even under
-fmad=false, which changes results, so a mismatch (fusing or duplication) exits non-zero.

    python profiles/sass_mix.py [--root <tree>]
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
FLAGS = ["-O3", "-std=c++17", "-lineinfo", "-fmad=false"]
FP_OPS = ("FFMA", "FMUL", "FADD", "FFMA2", "FMUL2", "FADD2", "FMNMX", "FSEL", "FSETP", "MUFU")
PAIRS = (("FFMA2", "fma.rn.f32x2"), ("FMUL2", "mul.rn.f32x2"), ("FADD2", "add.rn.f32x2"))
KERNEL = "step_fast_kernel"


def demangle_args(name: str) -> str:
    """_ZN3phc16step_fast_kernelILi4ELi8ELb0ELb0ELb0ELb1ELb1EEEv... -> <4,8,0,0,0,1,1>"""
    m = re.search(r"step_fast_kernelI(.*?)EEv", name)
    vals = re.findall(r"L[ib](\d+)E?", m.group(1)) if m else []
    return "<" + ",".join(vals) + ">"


def compile_tree(root: str, tmp: str) -> tuple[str, str, str]:
    src = os.path.join(root, "humanoid_b200", "csrc", "phc_kernels.cu")
    cubin, ptx = os.path.join(tmp, "k.cubin"), os.path.join(tmp, "k.ptx")
    arch = ["-gencode", "arch=compute_100a,code=sm_100a"]
    r = subprocess.run(["nvcc", *FLAGS, *arch, "-cubin", "-Xptxas", "-v", "-o", cubin, src], capture_output=True,
                       text=True, check=True)  # fmt: skip
    subprocess.run(["nvcc", *FLAGS, "-arch=compute_100a", "-ptx", "-o", ptx, src], check=True)
    sass = subprocess.run(["cuobjdump", "-sass", cubin], capture_output=True, text=True, check=True).stdout
    with open(ptx) as f:
        return r.stderr, sass, f.read()


def ptxas_info(log: str) -> dict[str, dict]:
    out, cur = {}, None
    for line in log.splitlines():
        m = re.search(r"Compiling entry function '(\w+)'", line)
        if m:
            cur = m.group(1)
            out[cur] = {}
            continue
        if cur is None:
            continue
        m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m:
            out[cur].update(stack=int(m.group(1)), spill_st=int(m.group(2)), spill_ld=int(m.group(3)))
        m = re.search(r"Used (\d+) registers", line)
        if m:
            out[cur]["regs"] = int(m.group(1))
    return out


def sass_functions(sass: str) -> dict[str, collections.Counter]:
    out, cur = {}, None
    for line in sass.splitlines():
        m = re.match(r"\s+Function : (\w+)", line)
        if m:
            cur = out.setdefault(m.group(1), collections.Counter())
            continue
        m = re.match(r"\s+/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P\w+\s+)?([A-Z][A-Z0-9_]*)", line)
        if m and cur is not None:
            cur[m.group(1)] += 1
    return out


def ptx_entries(ptx: str) -> dict[str, str]:
    parts = re.split(r"\.entry\s+(\w+)\(", ptx)
    return {parts[i]: parts[i + 1] for i in range(1, len(parts) - 1, 2)}


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--root", default=ROOT, help="source tree to compile (default: this repository)")
    a = ap.parse_args()
    with tempfile.TemporaryDirectory() as tmp:
        log, sass, ptx = compile_tree(os.path.abspath(a.root), tmp)
    info, funcs, entries = ptxas_info(log), sass_functions(sass), ptx_entries(ptx)
    bad = 0
    print(f"| `{KERNEL}` | regs | stack | spill st/ld | SASS | " + " | ".join(FP_OPS) + " | PTX f32x2 fma/mul/add |")
    print("|---" * (6 + len(FP_OPS)) + "|")
    for name in sorted(n for n in funcs if KERNEL in n):
        c, i, body = funcs[name], info.get(name, {}), entries.get(name, "")
        nptx = [len(re.findall(re.escape(op) + r"\s", body)) for _, op in PAIRS]
        for (sop, pop), k in zip(PAIRS, nptx):
            if c[sop] != k:
                bad += 1
                print(f"MISMATCH {demangle_args(name)}: {c[sop]} {sop} in SASS, {k} {pop} in PTX", file=sys.stderr)
        row = [demangle_args(name), i.get("regs"), i.get("stack"), f"{i.get('spill_st')}/{i.get('spill_ld')}",
               sum(c.values()), *(c[o] for o in FP_OPS), "/".join(map(str, nptx))]  # fmt: skip
        print("| " + " | ".join(str(v) for v in row) + " |")
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
