"""Parallel tempering on the changepoint model (cp_tempered_kernel) against the untempered one-slice kernel, on one GPU.

Prints the card's name, power limit and max SM clock, then:
  * rates: the untempered one-slice kernel (RMN_CP_SLICED=0) at 65,536 chains, tempered 13,107 ladders x 5 and
    8,192 ladders x 8; CUDA events around the kernel launch, a warm-up first, every timed run >= 1 s, 3 runs per
    configuration alternated.  Chain-steps/s over all rungs and beta = 1 chain-steps/s.
  * mixing: 512 ladders x 5 against 512 untempered chains, tau of k and sigma at rung 0 from thinned traces
    (riemann_b200.diagnostics.integrated_time_chains), ESS per beta = 1 chain-step and per second; for the ladders
    also the swap statistics after the burn-in (PTSampler.swap_statistics): acceptance per pair of neighbouring
    rungs, round trips per ladder per 1,000 steps and the up-moving fraction per rung.

    python scripts/bench_cp_tempering.py [--runs 3] [--min-seconds 1.0]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def problem():
    from oracle import riemann_port as port
    from riemann_b200.models.changepoint import ChangepointParams, ChangepointRegression1D
    from riemann_b200.proposals.changepoint import ChangepointRegression1DProp
    pm, pp, _, _ = port.make_changepoint_problem()
    dm = ChangepointRegression1D(pm.x, pm.y, pm.xmin, pm.xmax, pm.lamb, int(pm.kmax), pm.alpha, pm.beta)
    return dm, ChangepointRegression1DProp(dm, pp.hscale), ChangepointParams([2.0], [1.0, 3.0], 0.1)


def make(kind, dm, dp, th0, seed=1):
    from riemann_b200 import PTSampler, Sampler
    if kind[0] == "plain":
        os.environ["RMN_CP_SLICED"] = "0"            # read when the sampler is created: the one-slice kernel
        try:
            s = Sampler(dm, dp, th0, K=kind[1], seed=seed)
        finally:
            del os.environ["RMN_CP_SLICED"]
        return s, s, kind[1]
    L, nt = kind[1], kind[2]
    pt = PTSampler(dm, dp, th0, betas=0.5 ** np.arange(nt), K=L, seed=seed)
    return pt, pt._sampler, L


def timed(flat, T):
    import torch
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    flat._run_device(T, 0, 1, 0)
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / 1e3


def rates(dm, dp, th0, runs, min_s):
    configs = [("plain", 65536), ("pt", 13107, 5), ("pt", 8192, 8)]
    made = [make(c, dm, dp, th0) for c in configs]
    steps = []
    for (_, flat, _), c in zip(made, configs):
        flat._run_device(300, 0, 1, 0)               # warm-up (module load, data staging)
        t = timed(flat, 2000)
        steps.append(int(np.ceil(2000 * 1.2 * min_s / t / 1000.0)) * 1000)
    res = {c: [] for c in configs}
    for _ in range(runs):                            # alternated
        for (_, flat, _), c, T in zip(made, configs, steps):
            dt = timed(flat, T)
            res[c].append((flat.K * T / dt, T, dt))
    out = []
    for (_, flat, beta1), c in zip(made, configs):
        r = np.array([x[0] for x in res[c]])
        name = "untempered one-slice, K = {}".format(c[1]) if c[0] == "plain" else \
            "tempered {} ladders x {}".format(c[1], c[2])
        out.append(dict(config=name, chains=flat.K, beta1_chains=beta1, steps=res[c][0][1],
                        seconds=[float(x[2]) for x in res[c]],
                        chain_steps_per_s=[float(v) for v in r],
                        beta1_chain_steps_per_s=[float(v * beta1 / flat.K) for v in r]))
    return out


def mixing(dm, dp, th0, burn=6000, T=40000, thin=40):
    from riemann_b200.diagnostics import integrated_time_chains
    out = []
    for kind in (("plain", 512), ("pt", 512, 5)):
        obj, flat, beta1 = make(kind, dm, dp, th0, seed=3)
        flat.run(burn, trace=False)
        flat.reset_diagnostics()                     # the swap statistics cover the 2 T steps after the burn-in
        import time
        import torch
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        flat._run_device(T, 0, 1, 0)
        torch.cuda.synchronize()
        dt_plain = time.perf_counter() - t0           # the untraced time of T steps (for ESS per second)
        flat.run(T, 0, thin)                         # the same number of steps again, traced and thinned
        tr = flat._chain_thetas
        nt = 1 if kind[0] == "plain" else kind[2]
        k = tr.k[1:, ::nt].astype(np.float64)        # rung 0 of every ladder: [rec, 512]
        sig = tr.sig[1:, ::nt]
        tau = integrated_time_chains(np.stack([k, sig], axis=2)) * thin     # in MH steps
        ess_per_step = 1.0 / tau                     # per beta = 1 chain-step
        rec = dict(config="untempered" if kind[0] == "plain" else "tempered x {}".format(nt),
                   tau_k=float(tau[0]), tau_sig=float(tau[1]),
                   ess_per_beta1_chain_step=[float(v) for v in ess_per_step],
                   seconds_for_T=dt_plain,
                   ess_per_s=[float(beta1 * T / dt_plain / t) for t in tau])
        if kind[0] == "pt":
            sw = obj.swap_statistics(allreduce=False)
            rec.update(swap_steps=sw.steps, swap_acceptance=[float(v) for v in sw.acceptance],
                       round_trips=sw.round_trips,
                       round_trips_per_ladder_per_1000_steps=1000.0 * sw.round_trips / (sw.ladders * sw.steps),
                       up_fraction=[float(v) for v in sw.up_fraction])
        out.append(rec)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--min-seconds", type=float, default=1.0)
    args = ap.parse_args()
    from riemann_b200 import _lib
    _lib.require_cuda()
    print("card: " + card(), flush=True)
    dm, dp, th0 = problem()
    for r in rates(dm, dp, th0, args.runs, args.min_seconds):
        print(json.dumps(r), flush=True)
    for r in mixing(dm, dp, th0):
        print(json.dumps(r), flush=True)


if __name__ == "__main__":
    main()
