"""Static SASS budget of one kernel of the built library -- runs without a GPU (cuobjdump + c++filt).

Prints, for one instantiation (default: the headline `changepoint_sliced_kernel<2,4,true>`), the number of SASS
instructions (the NOP padding after the kernel's end excluded), the counts of the branch / reconvergence, select,
shuffle and fp64 opcodes, and the registers and local-memory frame.  With --base it prints a second library (e.g. a
build of the parent commit) beside it, with the difference.

    python scripts/cp_sass_budget.py
    python scripts/cp_sass_budget.py --base /tmp/parent/libriemann_b200.so --kernel 'changepoint_sliced_kernel<2,4,false>'

Static counts weigh every instruction once, however often it runs: they show what a change removed from the code, not
what it saved per step (that needs the per-instruction execution counts of a profiler, or the bench)."""
import argparse
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "riemann_b200", "libriemann_b200.so")

# (label, opcode regex on the mnemonic without its modifiers)
CLASSES = [("BRA", r"BRA"), ("BSSY", r"BSSY"), ("BSYNC", r"BSYNC"), ("FSEL", r"FSEL"), ("SEL", r"SEL"),
           ("SHFL", r"SHFL"), ("fp64 (DADD DMUL DFMA DSETP DMNMX)", r"DADD|DMUL|DFMA|DSETP|DMNMX")]
INSN = re.compile(r"^\s+/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P[T0-9]+\s+)?([A-Z][A-Z0-9_]*)((?:\.[A-Z0-9_]+)*)", re.M)


def _run(cmd):
    return subprocess.run(cmd, capture_output=True, text=True, check=True).stdout


def _norm(name):
    name = re.sub(r"^void\s+|\(anonymous namespace\)::|\(.*$", "", name.strip())
    return re.sub(r"\s+", "", name)


def find_kernel(lib, kernel):
    """mangled name, registers, stack bytes of the kernel whose demangled name (without arguments) is `kernel`"""
    txt = _run(["cuobjdump", "-res-usage", lib])
    rows = re.findall(r"Function (\S+):\s*\n\s*REG:(\d+) STACK:(\d+)", txt)
    names = _run(["c++filt"] + [r[0] for r in rows]).splitlines()
    want = _norm(kernel)
    hits = [r for n, r in zip(names, rows) if _norm(n).split("::")[-1] == want]
    if len(hits) != 1:
        sys.exit("%d kernels named %s in %s" % (len(hits), kernel, lib))
    return hits[0][0], int(hits[0][1]), int(hits[0][2])


def budget(lib, kernel):
    mangled, reg, stack = find_kernel(lib, kernel)
    sass = _run(["cuobjdump", "-sass", "-fun", mangled, lib])
    insns = [(m.group(1), m.group(2)) for m in INSN.finditer(sass) if m.group(1) != "NOP"]
    ops = [o for o, _ in insns]
    out = {"instructions": len(ops)}
    for label, pat in CLASSES:
        out[label] = sum(1 for o in ops if re.fullmatch(pat, o))
    out["fp64 conversions (F2F I2F F2I .F64)"] = sum(1 for o, mod in insns if o in ("F2F", "I2F", "F2I") and ".F64" in mod)
    out["BRA+BSSY+BSYNC"] = out["BRA"] + out["BSSY"] + out["BSYNC"]
    out["FSEL+SEL"] = out["FSEL"] + out["SEL"]
    out["registers"] = reg
    out["frame (B)"] = stack
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--lib", default=LIB, help="library to read (default: the built one)")
    ap.add_argument("--base", help="a second library printed beside it (e.g. the parent commit's build)")
    ap.add_argument("--kernel", default="changepoint_sliced_kernel<2,4,true>")
    a = ap.parse_args()
    cur = budget(a.lib, a.kernel)
    base = budget(a.base, a.kernel) if a.base else None
    print("# Static SASS of `%s` (sm_100a, `cuobjdump -sass`)\n" % _norm(a.kernel))
    if base:
        print("| | base | this build | change |\n|---|---|---|---|")
        for key in cur:
            print("| %s | %d | %d | %+d |" % (key, base[key], cur[key], cur[key] - base[key]))
    else:
        print("| | count |\n|---|---|")
        for key in cur:
            print("| %s | %d |" % (key, cur[key]))


if __name__ == "__main__":
    main()
