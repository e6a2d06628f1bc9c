#!/usr/bin/env python
"""Cost of the changepoint sampler's posterior summaries (Sampler.set_posterior_summary) at the headline shape:
65,536 chains of bench.py's changepoint problem, runs of 1,000 steps (bench.py's --iters), device-timed with CUDA events
around each run.  Three configurations -- summaries off, on at every = 16 and on at every = 64 (a 201-point grid over
[xmin, xmax], 128 value bins) -- are timed in one process, alternated round by round so that clock and neighbour drift
hit them alike.  Prints the card's name, power limit and max SM clock beside the chain-steps/s of every round.

    python scripts/bench_cp_summary.py [--rounds 3] [--iters 1000] [--warmup 2] [--out results/cp_summary.json]
"""
import argparse
import json
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
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--chains", type=int, default=65536)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    from riemann_b200 import Sampler, synthetic
    from riemann_b200.models.changepoint import ChangepointParams, ChangepointRegression1D
    from riemann_b200.proposals.changepoint import ChangepointRegression1DProp
    c = synthetic.changepoint_problem()
    model = ChangepointRegression1D(c["x"], c["y"], c["xmin"], c["xmax"], c["lamb"], c["kmax"], c["alpha"], c["beta"])
    prop = ChangepointRegression1DProp(model, c["hscale"])
    grid = np.linspace(c["xmin"], c["xmax"], 201)
    vr = (float(np.min(c["y"])) - 1.0, float(np.max(c["y"])) + 1.0)
    configs = {"off": None, "every=16": 16, "every=64": 64}
    samplers = {}
    for name, every in configs.items():
        s = Sampler(model, prop, ChangepointParams(*c["theta0"]), K=a.chains, seed=1)
        if every:
            s.set_posterior_summary(grid, vr, 128, every)
        s.enable_kernel_timing()
        for _ in range(a.warmup):
            s.run(a.iters, trace=False)
        s.kernel_timing()
        samplers[name] = s
    rates = {n: [] for n in configs}
    kernels = {}
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(a.rounds):
        for name, s in samplers.items():
            torch.cuda.synchronize()
            ev0.record()
            s._run_device(a.iters, 0, 1, 0)           # the kernel launch alone: no state download in the window
            ev1.record()
            torch.cuda.synchronize()
            rates[name].append(a.chains * a.iters / (ev0.elapsed_time(ev1) * 1e-3))
            kernels[name] = s.kernel_timing()["kernel"]
    base = float(np.median(rates["off"]))
    out = {"card (name, power limit, max SM clock)": card(), "chains": a.chains, "iters": a.iters,
           "grid": len(grid), "value_bins": 128, "kernel": kernels,
           "chain_steps_per_s": rates, "median_vs_off": {n: float(np.median(r)) / base for n, r in rates.items()}}
    print(json.dumps(out, indent=1))
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
