#!/usr/bin/env python
"""
Device version of the reference's examples/test_changepoint.py: synthetic piecewise-constant data from the model's
own generator (5 true changepoints, 100 points), the 4-way mixture proposal (moves of the changepoint locations /
the step heights / the noise scale, birth-death), started from one changepoint -- first as ONE chain with the
reference's list-of-ChangepointParams history, then as 65,536 chains.  The reference plots the chain; this prints
the same summaries (acceptance fraction, posterior over the number of changepoints, noise scale, the posterior
predictive step function on a grid).  Needs a B200 (no CPU fallback).
"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from riemann_b200 import Sampler                                                        # noqa: E402
from riemann_b200.models.changepoint import ChangepointParams, ChangepointRegression1D  # noqa: E402
from riemann_b200.proposals.changepoint import ChangepointRegression1DProp              # noqa: E402


def main():
    np.random.seed(42)
    Ncpx, Ndata = 5, 100
    xmin, xmax, hmin, hmax = 1.0, 3.0, 1.0, 3.0
    theta_true = ChangepointParams(np.sort(np.random.uniform(xmin, xmax, size=Ncpx)),
                                   np.random.uniform(hmin, hmax, size=Ncpx + 1), 0.1)
    model = ChangepointRegression1D([], [], xmin, xmax, 1.0 * Ncpx, 2 * Ncpx, 1, 1)
    model.x, model.y = model.generate_synthetic_data(theta_true, Ndata)
    proposal = ChangepointRegression1DProp(model, hmax - hmin)
    theta0 = ChangepointParams([0.5 * (xmin + xmax)], [hmin, hmax], 0.1)
    print("true changepoints", np.round(theta_true.cpx, 3), "heights", np.round(theta_true.cpv, 3))

    # one chain, the reference's API and history
    sampler = Sampler(model, proposal, theta0)
    sampler.run(20000)
    lp = np.array(sampler._chain_logpost)
    ks = np.array([len(th.cpx) for th in sampler._chain_thetas])
    print("one chain: %d states, acceptance fraction %.3f, k after burn-in: mean %.2f, histogram %s"
          % (len(ks), np.mean(lp[1:] != lp[:-1]), ks[10000:].mean(), np.bincount(ks[10000:]).tolist()))
    best = sampler._chain_thetas[int(np.argmax(lp))]
    print("           highest-posterior state: cpx", np.round(best.cpx, 3), "cpv", np.round(best.cpv, 3),
          "sig %.3f" % float(best.sig))

    # many chains: device-resident, only the final states and the diagnostics come back
    K = 65536
    many = Sampler(model, proposal, theta0, K=K, seed=1)
    many.run(10000, trace=False)
    many.reset_diagnostics()
    # posterior summaries of the second half on the device: the predictive band on a grid, changepoint locations, k
    grid = np.linspace(xmin, xmax, 101)
    many.set_posterior_summary(grid, value_range=(hmin - 1.0, hmax + 1.0), value_bins=200, every=16)
    many.run(10000, trace=False)
    d = many.diagnostics()
    final = many._chain_thetas                      # ChangepointTrace: arrays indexed [record, chain]; one record here
    kfin = np.asarray(final.k[-1])
    print("%d chains x %d steps: acceptance %.3f, overflows %d, mean sigma %.4f, mean k %.2f (tracked functionals: "
          "sigma, k, prediction at 6 grid points)" % (d["chains"], d["steps"], d["accept_rate"], d["overflows"],
                                                     d["mean"][0], d["mean"][1]))
    print("           posterior-predictive mean at the tracked points", np.round(d["mean"][2:], 3))
    print("           k over the final states: histogram", np.bincount(kfin).tolist())
    first = final[-1, 0]                            # one state as ChangepointParams, like the reference's history items
    print("           chain 0 ends at cpx", np.round(first.cpx, 3), "cpv", np.round(first.cpv, 3))
    ps = many.posterior_summary()
    band = ps.yhat_quantiles([0.05, 0.5, 0.95])
    print("posterior summary: %d sampled chain-steps, posterior over k %s" % (ps.nsamples,
                                                                           np.round(ps.khist / ps.nsamples, 3).tolist()))
    for g in range(0, len(grid), 20):
        print("           predictive band at x = %.2f: 5%% %.3f  50%% %.3f  95%% %.3f" % (grid[g], *band[:, g]))
    top = np.argsort(ps.cpxhist)[::-1][:5]
    cells = ["[%.2f, %.2f): %.3f" % (grid[i - 1], grid[i], ps.cpxhist[i] / ps.nsamples) for i in sorted(top) if 0 < i < len(grid)]
    print("           most likely changepoint cells (changepoints per state):", "; ".join(cells))


if __name__ == "__main__":
    main()
