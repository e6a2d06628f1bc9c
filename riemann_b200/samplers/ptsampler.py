"""
Parallel tempering -- riemann/samplers/ptsampler.py:11-127 ("next" row N3 of SURVEY.md section 8f).

The reference builds one `Sampler` per temperature around `TemperedModel(model, beta)` (likelihood * beta,
prior untouched) and, every step and sequentially along the ladder, lets each chain either take a within-chain
MH step or -- with probability `Pswap` -- propose a swap with the next chain down the ladder.  Here the ladder
lies along the chain axis of the device engine: chains l*Nt .. l*Nt+Nt-1 are ladder l, the swap is a warp shuffle
inside the MH kernel on the small-d path (riemann_b200/csrc/small_gauss.cu) and an exchange of the two chain rows by the
initiator's warp on the dense-Gaussian path (d > 8, riemann_b200/csrc/dense.cu) and on the logistic model
(riemann_b200/csrc/logistic.cu; the prior is not tempered, :33-37) -- `rmn_sampler_set_tempering` -- and
`K` independent ladders run side by side.  On the changepoint model (ChangepointRegression1D with the shared,
non-adaptive ChangepointRegression1DProp) a ladder of at most 8 temperatures lives inside one warp of the changepoint
kernel (riemann_b200/csrc/changepoint.cu, cp_tempered_kernel) and a swap exchanges the two chains' register rows by
shuffle; `theta0` is then a ChangepointParams (every chain), a list of K (one per ladder) or of K*Nt, and the
histories are lists of ChangepointParams (K = 1) or ChangepointTrace objects [record, ladder] (K > 1).

Reference behaviours kept: the default ladder `0.5**arange(5)`; the selection uniform is drawn for every chain,
swapped or not (:104); the last chain never initiates (:107); `mhratio = min(1, exp(...))` with Python's `min`
(nan -> 1); `run(Nsamples, Nburn, Nthin)` ignores `Nburn`/`Nthin` and exposes the history of the beta = betas[0]
chain as `_chain_thetas` / `_chain_logpost` (:83-90).  Reference defects not reproduced: passing `betas=` raises
in the reference (`isinstance(betas, np.array)`, :62) -- here an explicit ladder is used as given, which is what
that branch intends; `sample()` returns `np.array(zip(...))` there (:127) and the states here.
The reference shares ONE proposal object between all temperatures (:81), so only non-adaptive proposals make
sense; the device engine enforces that (MetropolisRandomWalk, pCN; Gaussian models of any dimension, logistic model;
ChangepointRegression1DProp on the changepoint model).
"""
import ctypes as C

import numpy as np

from .. import _lib
from ..models.changepoint import ChangepointParams, ChangepointRegression1D, unpack_state
from ..models.model import Model
from ..posterior_summary import check_summary_args
from ..sampling_errors import ParameterError
from .sampler import ChangepointTrace, Sampler


class TemperedModel(Model):
    """ptsampler.py:11-38 -- host-side protocol object (the device kernel applies beta itself)."""

    def __init__(self, base_model, beta):
        if not (beta >= 0 and beta <= 1):
            raise ParameterError("beta = {} must be a number between 0 and 1".format(beta))
        self.base_model = base_model
        self.beta = beta

    def set_beta(self, beta):
        self.beta = beta

    def log_likelihood(self, theta):
        return (self.base_model.log_likelihood(theta)) * self.beta

    def log_prior(self, theta):
        return self.base_model.log_prior(theta)


class _TemperatureView(object):
    """`pt.samplers[i]`: the history of temperature i (what the reference keeps in its i-th Sampler)."""

    def __init__(self, pt, i):
        self._pt, self._i = pt, i
        self.model = TemperedModel(pt.model, pt.betas[i])

    @property
    def _chain_thetas(self):
        return self._pt._history_of(self._i)[0]

    @property
    def _chain_logpost(self):
        return self._pt._history_of(self._i)[1]

    def current_state(self):
        th, lp = self._pt._history_of(self._i)
        return th[-1], lp[-1]


class SwapStatistics(object):
    """Swap statistics of the changepoint tempering ladders since the last reset (PTSampler.swap_statistics), pooled
    over the ladders: int64 counts and the rates derived from them.

    proposed[i], accepted[i]  (Nt-1,)  swaps rung i initiated with rung i+1 / swaps taken
    acceptance                (Nt-1,)  accepted / proposed (nan where nothing was proposed)
    up[i], down[i]            (Nt,)    at every step s with s % 16 == 0 (the diagnostics' cadence, after the step's
                                       swaps), chains at rung i whose replica last touched rung 0 / rung Nt-1
    up_fraction               (Nt,)    up / (up + down) (nan where neither): the fraction of replicas moving up, whose
                                       steep drops show where the ladder needs another temperature (Katzgraber et
                                       al. 2006); 1 at rung 0 and 0 at rung Nt-1 by construction
    round_trips                        replicas that went from rung 0 to rung Nt-1 and back to rung 0
    ladders, steps                     the ladders counted and the PT steps per chain since the reset, so that
                                       round_trips / (ladders * steps) is the round-trip rate per ladder-step
    """

    def __init__(self, proposed, accepted, up, down, round_trips, ladders, steps):
        self.proposed, self.accepted = proposed, accepted
        self.up, self.down = up, down
        self.round_trips, self.ladders, self.steps = int(round_trips), int(ladders), int(steps)
        self.acceptance = np.where(proposed > 0, accepted / np.maximum(proposed, 1), np.nan)
        n = up + down
        self.up_fraction = np.where(n > 0, up / np.maximum(n, 1), np.nan)

    def __repr__(self):
        return "SwapStatistics(acceptance={}, round_trips={}, up_fraction={}, ladders={}, steps={})".format(
            np.round(self.acceptance, 4).tolist(), self.round_trips, np.round(self.up_fraction, 4).tolist(),
            self.ladders, self.steps)


class PTSampler(object):
    """Same constructor as the reference (ptsampler.py:47) plus `K` = number of independent ladders, the Philox seed,
    the global id of the first ladder (`chain_offset`, in ladders) and, on the changepoint model, the move schedule
    (`Sampler`'s `move_schedule`; with "group" the ladders of a warp share the move-type draws)."""

    def __init__(self, model, proposal, theta0, betas=None, Pswap=0.1, K=1, seed=0, chain_offset=0, move_schedule=None):
        self.betas = 0.5 ** np.arange(5) if betas is None else np.asarray(betas, dtype=np.float64)
        if self.betas.ndim != 1 or not (2 <= len(self.betas) <= 32):
            raise ParameterError("betas must be a 1-d ladder of 2..32 temperatures")
        if not (Pswap > 0 and Pswap < 1):
            raise ParameterError("Pswap must be a number between 0 and 1")
        self.Pswap, self.model, self.proposal = Pswap, model, proposal
        self.K, self.Nt = int(K), len(self.betas)
        self._is_cp = isinstance(model, ChangepointRegression1D)
        if self._is_cp:
            if isinstance(theta0, ChangepointParams):
                th0 = [theta0] * (self.K * self.Nt)                    # every temperature starts at theta0 (:80-81)
            else:
                th0 = list(theta0)
                if len(th0) == self.K:
                    th0 = [th for th in th0 for _ in range(self.Nt)]
                elif len(th0) != self.K * self.Nt:
                    raise ParameterError("theta0 must be a ChangepointParams or a list of K or K*Nt of them")
        else:
            th0 = np.atleast_1d(np.asarray(theta0, dtype=np.float64))
            if th0.ndim == 1:
                th0 = np.tile(th0, (self.K * self.Nt, 1))              # every temperature starts at theta0 (:80-81)
            elif th0.shape[0] == self.K:
                th0 = np.repeat(th0, self.Nt, axis=0)
            elif th0.shape[0] != self.K * self.Nt:
                raise ParameterError("theta0 must be (d,), (K, d) or (K*Nt, d)")
        self._sampler = Sampler(model, proposal, th0, K=self.K * self.Nt, seed=seed, chain_offset=chain_offset * self.Nt,
                                _tempering=(self.betas, Pswap), move_schedule=move_schedule)
        self._summary, self.summary_rung = None, None
        self.d = self._sampler.d
        self._thetas, self._logpost = [], []
        self._take_record(0)
        self.samplers = [_TemperatureView(self, i) for i in range(self.Nt)]
        self._publish()

    def _take_record(self, r):
        """Append record r of the flat sampler's history as [ladder][temperature] arrays (the changepoint model: a
        tuple k, cpx, cpv, sig)."""
        th, lp = self._sampler._chain_thetas, np.asarray(self._sampler._chain_logpost)
        shape = (self.K, self.Nt)
        if self._is_cp:
            self._thetas.append(tuple(getattr(th, n)[r].reshape(shape + getattr(th, n).shape[2:])
                                      for n in ("k", "cpx", "cpv", "sig")))
        else:
            self._thetas.append(np.asarray(th[r]).reshape(shape + (self.d,)))
        self._logpost.append(lp[r].reshape(shape))

    # history [record][ladder][temperature]
    def _history_of(self, i):
        lp = np.stack([l[:, i] for l in self._logpost])                # [rec, K]
        if self._is_cp:
            k, cpx, cpv, sig = (np.stack([t[n][:, i] for t in self._thetas]) for n in range(4))
            if self.K == 1:
                return [unpack_state(k[r, 0], cpx[r, 0], cpv[r, 0], sig[r, 0]) for r in range(k.shape[0])], \
                    list(lp[:, 0])
            return ChangepointTrace(k, cpx, cpv, sig), lp
        th = np.stack([t[:, i] for t in self._thetas])                 # [rec, K, d]
        if self.K == 1:
            return list(th[:, 0]), list(lp[:, 0])
        return th, lp

    def _publish(self):
        self._chain_thetas, self._chain_logpost = self._history_of(0)

    def _absorb(self, ex=None):
        for r in range(1, len(self._sampler._chain_logpost)):         # record 0 is the state we already hold
            self._take_record(r)
        self._publish()
        return ex

    def run(self, Nsamples, Nburn=0, Nthin=1, trace=True):
        """ptsampler.py:83-90: Nsamples PT steps; Nburn / Nthin are accepted and ignored like there.
        `trace=False` keeps only the final state (many ladders, long runs)."""
        if trace:
            self._sampler.run(int(Nsamples), 0, 1)
            self._absorb()
        else:
            self._sampler.run(int(Nsamples), trace=False)
            self._thetas, self._logpost = [], []
            self._take_record(-1)
            self._publish()

    def run_injected(self, usel, xi=None, u=None, tape=None):
        """Parity mode: usel[T, K*Nt], xi[T, K*Nt, d], u[T, K*Nt] in the reference's per-chain draw order; the
        changepoint model takes tape[T, K*Nt, NSLOT] instead of xi and u (a swap initiator's swap uniform in the
        RMN_CP_SLOT_ACC slot)."""
        if self._is_cp:
            ex = self._sampler.run_injected(tape=tape, usel=usel)
        else:
            ex = self._sampler.run_injected(xi=xi, u=u, usel=usel)
        return self._absorb(ex)

    def sample(self):
        self.run(1)
        return [s.current_state() for s in self.samplers]

    def reset_diagnostics(self):
        """Zero the device accumulators of every rung: the diagnostics, the posterior-summary counts and, on the
        changepoint model, the swap counts of `swap_statistics` (the replicas' directions stay, so a round trip in
        progress still completes)."""
        self._sampler.reset_diagnostics()

    # ------------------------------------------------------------------ swap statistics (changepoint model)
    def swap_statistics(self, allreduce=True):
        """
        How the ladders mix since the last reset, counted in the tempered kernel (rmn_sampler_cp_get_swap_stats), as a
        SwapStatistics: per pair of neighbouring rungs the swaps proposed and accepted, the replicas' round trips
        from rung 0 to rung Nt-1 and back, and per rung the up / down flow histogram.  A replica's direction travels
        with its state; set_state starts the walk (rung 0 up, rung Nt-1 down).  With torch.distributed initialised
        the int64 counts are summed over the ranks (their ladders are disjoint).  Changepoint model only; the chains
        are unchanged by the counting.
        """
        if not self._is_cp:
            raise ParameterError("swap statistics are counted on the changepoint model only")
        torch, nt = self._sampler._torch, self.Nt
        # [ladders | proposed (nt-1) | accepted (nt-1) | up (nt) | down (nt) | round trips]
        buf = torch.zeros(1 + 2 * (nt - 1) + 2 * nt + 1, dtype=torch.int64, device="cuda")
        at = lambda i: C.c_void_p(buf.data_ptr() + 8 * i)
        _lib.check(_lib.load().rmn_sampler_cp_get_swap_stats(
            self._sampler._handle, at(1), at(nt), at(2 * nt - 1), at(3 * nt - 1), at(4 * nt - 1), _lib.stream_ptr()))
        buf[0] = self.K
        steps = int(self._sampler.diagnostics_block()[4].item())       # PT steps per chain since the reset
        if allreduce:
            from ..distributed import reduce_counts
            buf = reduce_counts(buf)
        c = buf.cpu().numpy()
        return SwapStatistics(c[1:nt], c[nt:2 * nt - 1], c[2 * nt - 1:3 * nt - 1], c[3 * nt - 1:4 * nt - 1],
                              c[4 * nt - 1], c[0], steps)

    # ------------------------------------------------------------------ posterior summaries (changepoint model)
    def set_posterior_summary(self, grid, value_range=None, value_bins=128, every=16, rung=0):
        """
        Accumulate the posterior summaries of `Sampler.set_posterior_summary` (riemann_b200/posterior_summary.py) for the
        chains of ONE temperature, inverse temperature betas[rung], of every ladder (rmn_sampler_cp_set_rung_summary):
        after every PT step whose global index is a multiple of `every`, each ladder's rung-`rung` state -- as it
        stands after that step's swaps -- adds to the integer histograms of the number of changepoints, of the
        changepoint locations over the cells of `grid`, and of ChangepointRegression1D.predict(theta, grid[g]) over
        `value_bins` bins of `value_range` = (vlo, vhi) plus an under- and an overflow bin.  No trace is kept.  The
        default rung 0 is the beta = betas[0] chain, the one this sampler exposes as `_chain_thetas` and whose moments
        `diagnostics()` reports; the other rungs sample tempered distributions.  The counts are reset now and by
        reset_diagnostics.  grid=None turns the summaries off.  Changepoint model only; the chains are unchanged bit
        for bit.
        """
        if not self._is_cp:
            raise ParameterError("posterior summaries are available on the changepoint model only")
        lib = _lib.load()
        if grid is None:
            _lib.check(lib.rmn_sampler_cp_set_rung_summary(self._sampler._handle, 0, 0, None, 0.0, 0.0, 0, 0))
            self._summary = None
            return
        if isinstance(rung, bool) or int(rung) != rung or not 0 <= int(rung) < self.Nt:
            raise ParameterError("rung must be an integer in 0..{} (got {})".format(self.Nt - 1, rung))
        g, vlo, vhi, H, every = check_summary_args(grid, value_range, value_bins, every)
        _lib.check(lib.rmn_sampler_cp_set_rung_summary(self._sampler._handle, int(rung), len(g), _lib.ptr(g), vlo, vhi,
                                                       H, every))
        self._summary = (g, vlo, vhi, H)
        self.summary_rung = int(rung)

    def posterior_summary(self, allreduce=True):
        """
        The summary counts of rung `summary_rung` (0: the beta = betas[0] chains of `_chain_thetas` and `diagnostics()`)
        since the last reset, as a PosteriorSummary; nsamples counts ladders x sampled steps.  With torch.distributed
        initialised the int64 counts are summed over the ranks: ladders on different ranks are disjoint replicas, so
        the sum is the pooled summary.
        """
        if self._summary is None:
            raise ParameterError("no posterior summary is set (set_posterior_summary)")
        return self._sampler._read_summary(self._summary, allreduce)

    def diagnostics(self, allreduce=True):
        """Posterior summaries of the beta = betas[0] chains ONLY (one per ladder): the device accumulators hold every
        rung of every ladder, and pooling the tempered rungs (beta < 1) would inflate the variance.  Built from the
        per-chain moments (`Sampler.chain_moments`), rank-local (`allreduce` is accepted for interface symmetry:
        ladders on other ranks are independent replicas, combine their summaries on the host if needed).
        `accept_rate` is that of the flat engine -- accepted within-chain moves per chain-step over all temperatures,
        a swap step counting as no move -- and is reported as `accept_rate_all_rungs`; `swap_fraction` = Pswap.
        On the changepoint model `swap_acceptance` is the accepted fraction of the swaps proposed between rung i and
        i+1 (`swap_statistics`)."""
        from ..distributed import summarize_block
        flat = self._sampler.diagnostics(allreduce=False)
        m, v = self._sampler.chain_moments()                      # [nd, K * Nt], chain fastest
        m0, v0 = m[:, ::self.Nt], v[:, ::self.Nt]                 # rung 0 of every ladder
        nd = m0.shape[0]
        blk = np.zeros(6 + 3 * nd)
        blk[0], blk[1], blk[4] = self.K, flat["samples"], flat["steps"]
        blk[6:6 + nd] = m0.sum(axis=1)
        blk[6 + nd:6 + 2 * nd] = (m0 * m0).sum(axis=1)
        blk[6 + 2 * nd:] = v0.sum(axis=1)
        out = summarize_block(blk)
        out.pop("accept_rate", None)
        out["accept_rate_all_rungs"] = flat["accept_rate"]
        out["swap_fraction"] = float(self.Pswap)
        out["temperatures"] = self.Nt
        if self._is_cp:                                           # per pair of neighbouring rungs, rank-local like the rest
            out["swap_acceptance"] = self.swap_statistics(allreduce=False).acceptance
        return out
