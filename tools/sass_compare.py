r"""Compare the SASS of the kernels two builds of libazg.so have in common, modulo symbol names.

    python tools/sass_compare.py OLD.so NEW.so [--rename REGEX=REPLACEMENT ...]

Each kernel of OLD is paired with the kernel of NEW whose demangled name (spaces removed) equals OLD's after the --rename
substitutions (re.sub, in order; e.g. `k_qmlp2<\(int\)3,=k_qmlp2<env::Pendulum,` when a template parameter changed from a state
width to an env type).  Instructions are compared with addresses, encodings and symbol operands removed.  Prints one line
per pair and exits 1 if any pair differs or has no partner.  Runs on the CPU (cuobjdump and cu++filt of the CUDA toolkit).
"""
from __future__ import annotations

import argparse
import re
import shutil
import subprocess
import sys


def _tool(name: str) -> str:
    return shutil.which(name) or f"/usr/local/cuda/bin/{name}"


def kernels(lib: str) -> dict:
    out = subprocess.run([_tool("cuobjdump"), "-sass", lib], capture_output=True, text=True, check=True).stdout
    funcs, cur = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1)
            funcs[cur] = []
            continue
        if cur is None:
            continue
        m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s+(.*?)\s*;", line)
        if m:
            ins = re.sub(r"\(\*\"[^\"]*\"\*\)", "", m.group(1))            # (*"symbol"*) operands
            ins = re.sub(r"`\([^)]*\)", "`()", ins)                          # branch targets by label name
            ins = re.sub(r"\b_Z\w+", "SYM", ins)                            # mangled names in operands
            funcs[cur].append(" ".join(ins.split()))
    names = list(funcs)
    dem = subprocess.run([_tool("cu++filt")], input="\n".join(names), capture_output=True, text=True, check=True).stdout.split("\n")
    return {d.replace(" ", ""): funcs[n] for n, d in zip(names, dem)}


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("old")
    ap.add_argument("new")
    ap.add_argument("--rename", action="append", default=[])
    a = ap.parse_args()
    old, new = kernels(a.old), kernels(a.new)
    ren = [r.split("=", 1) for r in a.rename]
    bad = 0
    for name, ins in sorted(old.items()):
        target = name
        for x, y in ren:
            target = re.sub(x, y, target)
        if target not in new:
            print(f"MISSING  {name} -> {target}")
            bad += 1
            continue
        same = new[target] == ins
        bad += not same
        print(f"{'same   ' if same else 'DIFFERS'}  {len(ins):6d} instructions  {name}" + ("" if target == name else f"  ->  {target}"))
    print(f"{len(old)} kernels compared, {bad} differ or are missing; {len(new) - len(old)} kernels only in {a.new}")
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
