"""Instruction budget of the headline kernel from a saved `ncu --set full --import-source on` report (no GPU needed):
executed warp-instructions per warp-step, by how often each instruction runs (1.0 = every step, 0.82 = the
trans-dimensional block, 0.25 = the thinned diagnostics ...), by opcode, and by source file:line region.

    python scripts/ncu_instruction_budget.py gpurun_out/r22_changepoint_full.ncu-rep 8192 1000 > profiles/r1_changepoint_instruction_budget.md

(8192 = warps of the launch, 1000 = MH iterations of the launch: one warp-step = 8 chain-steps at 4 lanes per chain.)"""
import collections
import csv
import io
import re
import subprocess
import sys

# Source regions are found by ANCHOR text in the current sources (the capture must be of the same commit): a region
# runs from its anchor line to the line before the next anchor of the same file.
ANCHORS = {
    "common.cuh": [("__device__ __forceinline__ uint4 philox4x32_10", "Philox4x32-10 rounds"),
                   ("// uniform on (0,1): (x + 0.5)", "Box-Muller normals / uniforms"),
                   ("// Metropolis-Hastings accept rule", "accept rule helpers")],
    "changepoint.cuh": [("// #{i : x_i <= c}", "run boundaries (bucket table / binary search)"),
                        ("// uniform on (0,1) from 32 random bits", "fast uniforms")],
    "changepoint.cu": [("__device__ __forceinline__ unsigned gballot", "group ballot / butterfly sums"),
                       ("// value of element e-1 for every row", "shift_prev / shift_next (neighbour element)"),
                       ("// value of element e + off, off in", "shift_by (insert / delete gather)"),
                       ("// a[idx] for a per-chain element index", "elem_at / count_below"),
                       ("__device__ __forceinline__ void cp_terms", "likelihood / prior sums (cp_terms)"),
                       ("// log of four per-chain arguments with one call", "batched log (log4)"),
                       ("__device__ __forceinline__ double cp_assemble", "log-posterior assembly (cp_assemble)"),
                       ("// full evaluation (pointwise entry", "full evaluation helper"),
                       ("__device__ __forceinline__ void cp_block(", "prologue (state load, caches, Philox prefetch)"),
                       ("    for (int64_t t = t_begin; t < t_end; ++t) {", "per-step randoms and move selection"),
                       ("        // What the warp as a whole needs this step", "warp votes"),
                       ("        // normals of the block moves", "normals (Box-Muller calls, second Philox block)"),
                       ("        // ---- build the proposal by selection", "fixed-dimension proposal by selection"),
                       ("        if (any3) {", "birth / death arithmetic and rebuild"),
                       ("        // run boundaries only move when a location moves", "run-boundary search"),
                       ("        if (!INJ) rA = rk.block(step + 1", "Philox prefetch"),
                       ("        // ---- log-posterior of the proposal from the pieces", "evaluation calls"),
                       ("        // sampler.py:83-84 with Python's min(0, nan) == 0", "accept, state update"),
                       ("        if ((step % RMN_CP_DIAG_EVERY) == 0) {", "thinned diagnostics"),
                       ("        if (live && tracing) {", "trace stores + epilogue"),
                       ("changepoint_kernel(const __grid_constant__ CPParams P", "kernel wrappers (data staging, time slices)"),
                       ("// evaluate n states given in the canonical layout", "(other kernels)")],
}


def find_regions(root):
    import os
    out = []
    for fname, anchors in ANCHORS.items():
        lines = open(os.path.join(root, "riemann_b200", "csrc", fname)).read().splitlines()
        pos = []
        for text, label in anchors:
            hits = [i + 1 for i, l in enumerate(lines) if text in l]
            if not hits:
                raise SystemExit("anchor not found in %s: %r" % (fname, text))
            pos.append((hits[0], label))
        for k, (lo, label) in enumerate(pos):
            hi = pos[k + 1][0] - 1 if k + 1 < len(pos) else len(lines)
            out.append((fname, lo, hi, label))
    return out


def main():
    import os
    rep, warps, iters = sys.argv[1], int(sys.argv[2]), int(sys.argv[3])
    REGIONS = find_regions(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    base = float(warps * iters)
    txt = subprocess.run(["ncu", "-i", rep, "--page", "source", "--print-source", "cuda,sass", "--csv"],
                         capture_output=True, text=True).stdout
    rows = list(csv.reader(io.StringIO(txt)))
    path, line = "", 0
    seen = {}                                # address -> [count, sass, [(file, line), ...]]: inlined code is listed once
    for r in rows:                           # per frame of its inline stack, so every address is counted ONCE
        if len(r) == 2 and r[0] == "File Path":
            path = r[1].split("/")[-1]
            continue
        if len(r) < 8 or r[0] in ("Line No", "Function Name"):
            continue
        if r[0] != "":                       # a source line header; its SASS rows follow
            line = int(r[0]) if r[0].isdigit() else 0
            continue
        if not r[2].startswith("0x"):
            continue
        try:
            n = int(r[7])
        except ValueError:
            continue
        seen.setdefault(r[2], [n, r[3], []])[2].append((path, line))
    by_freq, by_op, by_region = (collections.Counter() for _ in range(3))
    static_freq = collections.Counter()
    total = 0
    rank = {"changepoint.cu": 3, "changepoint.cuh": 2, "common.cuh": 1}
    for n, sass_txt, frames in seen.values():
        total += n
        f = round(n / base, 2)
        by_freq[f] += n
        static_freq[f] += 1
        sass = sass_txt.split()
        op = sass[1] if sass and sass[0].startswith("@") else (sass[0] if sass else "?")
        by_op[op.split(".")[0]] += n
        # attribute to the outermost frame ncu lists inside our sources (helpers are defined above their callers)
        fpath, fline = max(frames, key=lambda fr: (rank.get(fr[0], 0) if fr[1] > 0 else -1, fr[1]))
        label = "other (inlined math library: log, division, sqrt slow paths; intrinsics headers)"
        for suffix, lo, hi, lab in REGIONS:
            if fpath == suffix and lo <= fline <= hi:
                label = lab
                break
        by_region[label] += n
    print("# Instruction budget of the changepoint kernel (`cp_block<0,2,4>`; from `%s`)\n" % rep.split("/")[-1])
    print("%.3e executed warp-instructions = **%.0f per warp-step = %.0f per chain-step** (8 chains per warp).\n"
          % (total, total / base, total / base / 8))
    print("## By how often an instruction runs\n\n| runs on this fraction of warp-steps | static instructions | executed per warp-step | share |\n|---|---|---|---|")
    for f, n in sorted(by_freq.items(), key=lambda kv: -kv[1])[:10]:
        print("| %.2f | %d | %.0f | %.1f %% |" % (f, static_freq[f], n / base, 100.0 * n / total))
    print("\n## By source region\n\n| region | executed per warp-step | share |\n|---|---|---|")
    for lab, n in sorted(by_region.items(), key=lambda kv: -kv[1]):
        print("| %s | %.0f | %.1f %% |" % (lab, n / base, 100.0 * n / total))
    print("\n## By opcode\n\n| opcode | executed per warp-step | share |\n|---|---|---|")
    for op, n in by_op.most_common(16):
        print("| `%s` | %.0f | %.1f %% |" % (op, n / base, 100.0 * n / total))


if __name__ == "__main__":
    main()
