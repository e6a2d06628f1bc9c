#!/usr/bin/env python
"""Cost of the rung summaries of parallel tempering on the changepoint model (PTSampler.set_posterior_summary,
cp_tempered_summary_kernel) against cp_tempered_kernel without them.  Two ladder shapes of bench.py's changepoint
problem -- 13,107 ladders x 5 and 8,192 ladders x 8 temperatures (betas 0.5**i) -- each with summaries off, on at
every = 16 and on at every = 64 (rung 0, a 201-point grid over [xmin, xmax], 128 value bins).  Runs of 1,000 steps,
device-timed with CUDA events around the kernel launches alone (enough launches per window for >= --min-seconds), the six
configurations alternated round by round in one process so that clock and neighbour drift hit them alike.  Prints the
card's name, power limit and max SM clock beside the chain-steps/s (all rungs) of every round.

    python scripts/bench_cp_pt_summary.py [--rounds 3] [--iters 1000] [--min-seconds 1.0] [--out results/cp_pt_summary.json]
"""
import argparse
import json
import math
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except Exception:
        return "unknown"


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--iters", type=int, default=1000)
    ap.add_argument("--min-seconds", type=float, default=1.0)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    from riemann_b200 import PTSampler, synthetic
    from riemann_b200.models.changepoint import ChangepointParams, ChangepointRegression1D
    from riemann_b200.proposals.changepoint import ChangepointRegression1DProp
    c = synthetic.changepoint_problem()
    model = ChangepointRegression1D(c["x"], c["y"], c["xmin"], c["xmax"], c["lamb"], c["kmax"], c["alpha"], c["beta"])
    prop = ChangepointRegression1DProp(model, c["hscale"])
    grid = np.linspace(c["xmin"], c["xmax"], 201)
    vr = (float(np.min(c["y"])) - 1.0, float(np.max(c["y"])) + 1.0)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def window(flat, reps):
        torch.cuda.synchronize()
        ev0.record()
        for _ in range(reps):
            flat._run_device(a.iters, 0, 1, 0)        # the kernel launch alone: no state download in the window
        ev1.record()
        torch.cuda.synchronize()
        return ev0.elapsed_time(ev1) * 1e-3

    runs = {}
    for L, nt in ((13107, 5), (8192, 8)):
        for every in (None, 16, 64):
            name = "%dx%d %s" % (L, nt, "off" if every is None else "every=%d" % every)
            pt = PTSampler(model, prop, ChangepointParams(*c["theta0"]), betas=0.5 ** np.arange(nt), K=L, seed=1)
            if every:
                pt.set_posterior_summary(grid, vr, 128, every, rung=0)
            flat = pt._sampler
            flat.enable_kernel_timing()
            pt.run(a.iters, trace=False)                 # warm-up
            dt = window(flat, 1)
            runs[name] = dict(pt=pt, flat=flat, chains=L * nt, reps=max(1, math.ceil(a.min_seconds / dt)),
                              kernel=flat.kernel_timing()["kernel"])
    rates = {n: [] for n in runs}
    for _ in range(a.rounds):
        for name, r in runs.items():
            dt = window(r["flat"], r["reps"])
            rates[name].append(r["chains"] * a.iters * r["reps"] / dt)
    med = {n: float(np.median(v)) for n, v in rates.items()}
    out = {"card (name, power limit, max SM clock)": card(), "iters": a.iters, "grid": len(grid), "value_bins": 128,
           "rung": 0, "kernel": {n: r["kernel"] for n, r in runs.items()},
           "launches_per_window": {n: r["reps"] for n, r in runs.items()},
           "chain_steps_per_s (all rungs)": rates,
           "median_vs_off": {n: med[n] / med[n.split()[0] + " off"] for n in runs}}
    print(json.dumps(out, indent=1))
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
