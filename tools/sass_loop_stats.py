"""Instruction count and opcode histogram of the PGS sweep loops of a kernel, from `cuobjdump -sass`.

A sweep loop is an innermost loop (the span from a backward branch's target to the branch) that holds a VOTE: every
sweep loop ends with the ballot of Bullet's exit test.  Runs without a GPU on the cross-compiled library.

Usage: python tools/sass_loop_stats.py LIB_OR_CUBIN KERNEL [KERNEL ...]
  KERNEL is a substring of the mangled name or of the short demangled form, e.g.
  'step_kernel<3,1,4,1,0,0,0,1>' (the latency build's solo12 kernel with joint limits, as bench.py runs it).
  --all lists every function with a sweep loop."""
import argparse
import re
import shutil
import subprocess
import sys
from collections import Counter

_RE_FUNC = re.compile(r"^\s*Function\s*:\s*(\S+)")
_RE_INS = re.compile(r"^\s*/\*([0-9a-f]{4,})\*/\s+(.*?)\s*;")
_RE_BRA = re.compile(r"^(?:@!?U?P\w+\s+)?BRA(?:\.\S+)?\s+(?:!?U?P\w+,\s*)?(?:\S+,\s*)?0x([0-9a-f]+)")


def _tool(name):
    return shutil.which(name) or f"/usr/local/cuda/bin/{name}"


def short_names(mangled):
    """['_ZN4solo11step_kernelILi3E...'] -> {mangled: 'step_kernel<3,1,4,1,0,0,0,1>'}"""
    dem = subprocess.run([_tool("cu++filt")], input="\n".join(mangled) + "\n", capture_output=True,
                         text=True).stdout.splitlines()
    out = {}
    for m, d in zip(mangled, dem):
        d = re.sub(r"\((?:int|bool|unsigned int)\)", "", d)
        d = d.split("(")[0].replace("solo::", "").replace(" ", "")
        out[m] = d[4:] if d.startswith("void") else d
    return out


def functions(path):
    """{mangled name: [(address, instruction text)]}"""
    out = subprocess.run([_tool("cuobjdump"), "-sass", path], capture_output=True, text=True, check=True).stdout
    funcs, cur = {}, None
    for line in out.splitlines():
        m = _RE_FUNC.match(line)
        if m:
            cur = funcs.setdefault(m.group(1), [])
            continue
        m = _RE_INS.match(line)
        if m and cur is not None:
            cur.append((int(m.group(1), 16), m.group(2)))
    return funcs


def opcode(text):
    t = re.sub(r"^@!?U?P\w+\s+", "", text)
    return t.split()[0].split(".")[0]


def sweep_loops(ins):
    """innermost backward-branch spans that hold a VOTE: [(first index, last index)]"""
    idx = {a: i for i, (a, _) in enumerate(ins)}
    spans = []
    for i, (a, t) in enumerate(ins):
        m = _RE_BRA.match(t)
        if m and int(m.group(1), 16) <= a and int(m.group(1), 16) in idx:
            spans.append((idx[int(m.group(1), 16)], i))
    inner = [s for s in spans if not any(o != s and s[0] <= o[0] and o[1] <= s[1] for o in spans)]
    return [s for s in inner if any(opcode(ins[k][1]) == "VOTE" for k in range(s[0], s[1] + 1))]


def report(name, short, ins):
    loops = sweep_loops(ins)
    print(f"{short}  ({name})")
    if not loops:
        print("  no sweep loop")
    for lo, hi in loops:
        hist = Counter(opcode(t) for _, t in ins[lo:hi + 1])
        spill = hist.get("STL", 0) + hist.get("LDL", 0)
        print(f"  loop {ins[lo][0]:#x}..{ins[hi][0]:#x}: {hi - lo + 1} instructions, {spill} STL/LDL")
        print("   " + "  ".join(f"{c} {op}" for op, c in hist.most_common()))


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("lib")
    ap.add_argument("kernel", nargs="*")
    ap.add_argument("--all", action="store_true")
    a = ap.parse_args()
    funcs = functions(a.lib)
    shorts = short_names(list(funcs))
    found = False
    for name, ins in funcs.items():
        short = shorts[name]
        if a.all:
            hit = bool(sweep_loops(ins))
        else:
            hit = any(k in name or k.replace(" ", "") in short for k in a.kernel)
        if hit:
            found = True
            report(name, short, ins)
    if not found:
        print("no matching kernel", file=sys.stderr)
        sys.exit(1)


if __name__ == "__main__":
    main()
