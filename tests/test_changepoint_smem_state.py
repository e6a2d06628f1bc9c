"""
The time-sliced changepoint kernel keeps the accepted state's rows (cpx, cpv and the cached run boundaries) in shared
memory (riemann_b200/csrc/changepoint.cu, cp_block), which lets it run six resident blocks of 128 threads per SM
(RMN_CP_MINBLOCKS_SLICED = 6, DESIGN.md 4.1).  CPU checks on the built library:

* every GL = 4 instantiation of changepoint_sliced_kernel fits 80 registers (65,536 / (6 x 128) = 85, allocated in
  units of 8), and nothing is spilled inside its T loop: the at most 8 B frame holds one value that is stored and loaded
  only around a time slice;
* its static shared memory holds the 10 KB of state rows (4 rows x 128 threads x (8 + 8 + 4) B), and six blocks of it
  plus the bench data's staged tables (12,880 B) fit the 228 KB of shared memory of a B200 SM.
"""
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "riemann_b200", "libriemann_b200.so")
SLICED = ["changepoint_sliced_kernel<%d,4,%s>" % (d, g) for d in (1, 2) for g in ("true", "false")]
STATE_ROWS = 4 * 128 * (8 + 8 + 4)
BENCH_TABLES = 12880            # (XP + 2 M + 2) * 8 + G * 20 at M = 100, G = 512
SM_SMEM, BLOCK_RESERVED = 228 * 1024, 1024


def _need_tools():
    if not os.path.exists(LIB) or shutil.which("cuobjdump") is None or shutil.which("c++filt") is None:
        pytest.skip("needs the built library, cuobjdump and c++filt")


def _usage():
    """demangled name -> (mangled, registers, stack bytes, static shared bytes) of the sliced GL = 4 kernels"""
    txt = subprocess.run(["cuobjdump", "-res-usage", LIB], capture_output=True, text=True, check=True).stdout
    rows = re.findall(r"Function (\S+):\s*\n\s*REG:(\d+) STACK:(\d+) SHARED:(\d+)", txt)
    names = subprocess.run(["c++filt"] + [r[0] for r in rows], capture_output=True, text=True, check=True).stdout
    out = {}
    for name, (mangled, reg, stack, shared) in zip(names.splitlines(), rows):
        m = re.search(r"(changepoint_sliced_kernel<[^>]*>)", name)
        if m:
            out[m.group(1).replace(" ", "")] = (mangled, int(reg), int(stack), int(shared))
    missing = [k for k in SLICED if k not in out]
    assert not missing, (missing, sorted(out))
    return out


def test_sliced_kernels_fit_six_blocks_per_sm():
    _need_tools()
    usage = _usage()
    over = {k: usage[k][1:3] for k in SLICED if usage[k][1] > 80 or usage[k][2] > 8}
    assert not over, over


def test_sliced_kernels_spill_nothing_inside_the_t_loop():
    _need_tools()
    usage = _usage()
    insn = re.compile(r"/\*([0-9a-f]{4,})\*/\s+(?:@!?U?P[T0-9]+\s+)?([A-Z][A-Z0-9_.]*)(.*?);")
    for k in SLICED:
        sass = subprocess.run(["cuobjdump", "-sass", "-fun", usage[k][0], LIB], capture_output=True, text=True,
                              check=True).stdout
        loops, spills = [], []
        for m in insn.finditer(sass):
            addr, op = int(m.group(1), 16), m.group(2)
            if op.startswith("BRA"):
                tgt = re.search(r"0x([0-9a-f]+)", m.group(3))
                if tgt and int(tgt.group(1), 16) < addr:
                    loops.append((int(tgt.group(1), 16), addr))
            if op.startswith(("STL", "LDL")):
                spills.append(addr)
        # the two longest loops: the loop over work items, and the T loop inside it
        loops.sort(key=lambda r: r[1] - r[0], reverse=True)
        assert len(loops) >= 2, (k, loops)
        t0, t1 = loops[1]
        assert loops[0][0] < t0 and t1 < loops[0][1], (k, loops[:2])
        inside = [hex(a) for a in spills if t0 <= a <= t1]
        assert not inside, (k, inside)


def test_state_rows_are_in_static_shared_memory_and_six_blocks_fit():
    _need_tools()
    usage = _usage()
    for k in SLICED:
        shared = usage[k][3]
        assert shared >= STATE_ROWS, (k, shared)
        assert 6 * (shared + BENCH_TABLES + BLOCK_RESERVED) <= SM_SMEM, (k, shared)
