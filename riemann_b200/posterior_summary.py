"""
Posterior summaries of the changepoint sampler, accumulated on the device (rmn_sampler_cp_set_summary; for one rung of
PTSampler's tempering ladders, rmn_sampler_cp_set_rung_summary): integer histograms of the number of changepoints, of
the changepoint locations on a grid, and of the posterior predictive ŷ(x) = ChangepointRegression1D.predict(theta, x)
at every grid point, binned on a value range.  The counts are exact and
do not depend on how a run is split into calls, kernels, time slices or chain shards; the means and quantiles derived
from them here are binned estimates.
"""
import numpy as np

from .sampling_errors import ParameterError

GMAX = HMAX = 1024


def check_summary_args(grid, value_range, value_bins, every):
    """-> (grid as a float64 array, vlo, vhi, H, every), or ParameterError; the library checks the same again."""
    g = np.ascontiguousarray(np.asarray(grid, dtype=np.float64).reshape(-1))
    if not 1 <= g.size <= GMAX:
        raise ParameterError("posterior summary: need 1 to {} grid points (got {})".format(GMAX, g.size))
    if not np.all(np.isfinite(g)):
        raise ParameterError("posterior summary: the grid must be finite")
    if np.any(np.diff(g) <= 0):
        raise ParameterError("posterior summary: the grid must be strictly increasing")
    try:
        vlo, vhi = (float(v) for v in value_range)
    except (TypeError, ValueError):
        raise ParameterError("posterior summary: value_range must be a pair (vlo, vhi)")
    if not (np.isfinite(vlo) and np.isfinite(vhi) and vlo < vhi):
        raise ParameterError("posterior summary: need a finite value range vlo < vhi")
    if int(value_bins) != value_bins or not 1 <= int(value_bins) <= HMAX:
        raise ParameterError("posterior summary: need 1 to {} value bins".format(HMAX))
    if int(every) != every or not 1 <= int(every) <= 2 ** 62:
        raise ParameterError("posterior summary: need every >= 1")
    return g, vlo, vhi, int(value_bins), int(every)


class PosteriorSummary(object):
    """
    Counts since the last reset (Sampler.posterior_summary, PTSampler.posterior_summary):
      grid [G], value_edges [H + 1] (bin b = 1..H of yhist covers [value_edges[b-1], value_edges[b])),
      khist [16] (number of changepoints 0..15), cpxhist [G + 1] (cell i holds changepoints x with
      grid[i-1] <= x < grid[i], cell 0 those below grid[0] and cell G those at or above grid[-1]),
      yhist [G, H + 2] (bin 0: ŷ below value_edges[0]; bin H + 1: at or above value_edges[-1]), nsamples (sampled
      chain-steps; every row of yhist and khist sums to it).
    yhat_mean, yhat_quantiles(q): binned estimates, off by up to one bin width.
    """

    def __init__(self, grid, vlo, vhi, khist, cpxhist, yhist, nsamples):
        self.grid = np.asarray(grid, dtype=np.float64)
        H = yhist.shape[1] - 2
        self.value_edges = vlo + (vhi - vlo) * np.arange(H + 1) / H
        self.khist, self.cpxhist, self.yhist = khist, cpxhist, yhist
        self.nsamples = int(nsamples)

    @property
    def underflow(self):
        """samples per grid point whose ŷ lies below the value range"""
        return self.yhist[:, 0]

    @property
    def overflow(self):
        """samples per grid point whose ŷ lies at or above the top of the value range"""
        return self.yhist[:, -1]

    @property
    def yhat_mean(self):
        """posterior-predictive mean per grid point from the bin centres of the in-range samples (binned estimate, off by
        up to one bin width); the samples outside the range are left out, not guessed at (see underflow / overflow)"""
        c = self.yhist[:, 1:-1].astype(np.float64)
        mid = 0.5 * (self.value_edges[1:] + self.value_edges[:-1])
        n = c.sum(1)
        with np.errstate(invalid="ignore", divide="ignore"):
            return np.where(n > 0, (c * mid).sum(1) / n, np.nan)

    def yhat_quantiles(self, q):
        """posterior-predictive quantiles per grid point, [len(q), G]: the per-point CDF interpolated linearly inside
        a bin (binned estimate, off by up to one bin width).  A quantile that falls among the samples below / above
        the value range is -inf / +inf."""
        q = np.atleast_1d(np.asarray(q, dtype=np.float64))
        if np.any((q < 0) | (q > 1)):
            raise ParameterError("quantiles must lie in [0, 1]")
        e, w = self.value_edges, self.value_edges[1] - self.value_edges[0]
        H = len(e) - 1
        out = np.full((len(q), len(self.grid)), np.nan)
        for g in range(len(self.grid)):
            cnt = self.yhist[g].astype(np.float64)
            cum = np.cumsum(cnt)
            N = cum[-1]
            if N == 0:
                continue
            for a, qa in enumerate(q):
                t = qa * N
                b = int(np.searchsorted(cum, t, "left")) if t > 0 else int(np.searchsorted(cum, 0.0, "right"))
                if b == 0:
                    out[a, g] = -np.inf
                elif b == H + 1:
                    out[a, g] = np.inf
                else:
                    out[a, g] = e[b - 1] + w * (t - cum[b - 1]) / cnt[b]
        return out

    @property
    def k_mean(self):
        """posterior mean of the number of changepoints (exact: khist is not binned)"""
        return float((np.arange(len(self.khist)) * self.khist).sum() / max(self.nsamples, 1))
