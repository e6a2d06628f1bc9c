"""
Posterior summaries of one rung of the tempering ladders on the changepoint model (PTSampler.set_posterior_summary,
rmn_sampler_cp_set_rung_summary; riemann_b200/csrc/changepoint.cu, cp_tempered_summary_kernel).

CPU: the six cp_tempered_summary_kernel instantiations fit the tempered kernel's budget (at most 128 registers, no
local-memory frame, no spill instructions); the library refuses a null sampler; the host checks the model and the rung.
GPU: the device counts EQUAL the numpy reference (summary_reference of test_gpu_changepoint_summary) over the states of
the chosen rung -- the replayed fixture ladder and traced Philox ladders of 3, 5 and 8 temperatures; summaries leave the
chains, the accept / overflow counts and the diagnostics bit-identical; shards' counts sum to the full run's; the counts
agree with the base rung's diagnostics; unsupported set-ups are refused.
"""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from test_gpu_changepoint_summary import _bench_problem, _grid, _search_problem, summary_reference
from test_gpu_changepoint_tempering import _check_replay, _device_problem

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "riemann_b200", "libriemann_b200.so")
L = 16
DIAG_EVERY = 16          # RMN_CP_DIAG_EVERY


def _counts(ps):
    return ps.khist, ps.cpxhist, ps.yhist, ps.nsamples


def _assert_counts_equal(a, b):
    for u, v in zip(a, b):
        assert np.array_equal(np.asarray(u), np.asarray(v))


# ------------------------------------------------------------------------------------------------------------- CPU
def test_tempered_summary_kernels_fit_the_tempered_budget():
    import __graft_entry__ as ge
    ge.build()
    if shutil.which("cuobjdump") is None or shutil.which("c++filt") is None:
        pytest.skip("needs cuobjdump and c++filt")
    txt = subprocess.run(["cuobjdump", "-res-usage", LIB], capture_output=True, text=True, check=True).stdout
    rows = re.findall(r"Function (\S+):\s*\n\s*REG:(\d+) STACK:(\d+)", txt)
    names = subprocess.run(["c++filt"] + [r[0] for r in rows], capture_output=True, text=True, check=True).stdout
    found = {}
    for name, (mangled, reg, stack) in zip(names.splitlines(), rows):
        m = re.search(r"(cp_tempered_summary_kernel<[^>]*>)", name)
        if m:
            found[m.group(1).replace(" ", "")] = (mangled, int(reg), int(stack))
    want = ["cp_tempered_summary_kernel<%s,%d>" % (i, d) for i in ("false", "true") for d in (0, 1, 2)]
    assert sorted(found) == sorted(want), sorted(found)
    for name, (mangled, reg, stack) in found.items():
        assert stack == 0 and reg <= 128, (name, reg, stack)
        sass = subprocess.run(["cuobjdump", "-sass", "-fun", mangled, LIB], capture_output=True, text=True,
                              check=True).stdout
        assert not re.search(r"\b(STL|LDL)\b", sass), name


def test_null_sampler_is_refused_by_the_library():
    import __graft_entry__ as ge
    ge.build()
    from riemann_b200 import _lib
    g = np.linspace(0, 1, 4)
    assert _lib.load().rmn_sampler_cp_set_rung_summary(None, 0, 4, _lib.ptr(g), 0.0, 1.0, 8, 1) == _lib.RMN_ERR_PARAM


def test_host_checks_the_model_and_the_rung():
    import __graft_entry__ as ge
    ge.build()
    from riemann_b200 import ParameterError, PTSampler
    good = dict(grid=np.linspace(1, 3, 5), value_range=(0.0, 4.0), value_bins=16, every=4)
    for is_cp, rung in ((False, 0), (True, -1), (True, 5), (True, 1.5), (True, True)):
        pt = PTSampler.__new__(PTSampler)
        pt._is_cp, pt.Nt, pt._sampler = is_cp, 5, None            # no device sampler: nothing may reach the library
        with pytest.raises(ParameterError):
            pt.set_posterior_summary(rung=rung, **good)
    pt = PTSampler.__new__(PTSampler)
    pt._summary = None
    with pytest.raises(ParameterError):
        pt.posterior_summary()


# ------------------------------------------------------------------------------------------------------------- GPU
def _pt(problem, K, betas, Pswap=0.3, seed=3, chain_offset=0, schedule="group"):
    from riemann_b200 import PTSampler
    from riemann_b200.models.changepoint import ChangepointParams, ChangepointRegression1D
    from riemann_b200.proposals.changepoint import ChangepointRegression1DProp
    x, y, xmin, xmax, lamb, kmax, alpha, beta, hscale = problem
    dm = ChangepointRegression1D(x, y, xmin, xmax, lamb, int(kmax), alpha, beta)
    dp = ChangepointRegression1DProp(dm, hscale)
    return PTSampler(dm, dp, ChangepointParams([2.0], [1.0, 3.0], 0.1), betas=betas, Pswap=Pswap, K=K, seed=seed,
                     chain_offset=chain_offset, move_schedule=schedule)


@pytest.mark.gpu
@pytest.mark.parametrize("every", [1, 7])
def test_fixture_replay_counts_the_rung_states(golden, every):
    """The replayed fixture ladder: every rung still reproduces it, and the counts of rung 0 / nt - 1 are those of the
    fixture's states of that rung after the sampled steps (record t + 1 = state after step t)."""
    from riemann_b200 import PTSampler
    g = golden("pt_changepoint")
    dm, dp, th0 = _device_problem()
    nt, T = len(g["betas"]), g["usel"].shape[0]
    grid, (vlo, vhi, H) = _grid(_bench_problem()), (0.5, 3.5, 24)
    rec = np.arange(T)[np.arange(T) % every == 0] + 1
    for rung in (0, nt - 1):
        pt = PTSampler(dm, dp, th0)
        pt.set_posterior_summary(grid, (vlo, vhi), H, every, rung=rung)
        ex = pt.run_injected(g["usel"], tape=g["tape"])
        _check_replay(pt, ex, g)
        ref = summary_reference(g["k"][rung, rec], g["cpx"][rung, rec], g["cpv"][rung, rec], grid, vlo, vhi, H)
        ps = pt.posterior_summary(allreduce=False)
        assert ps.nsamples == len(rec)
        _assert_counts_equal(_counts(ps), ref)


@pytest.mark.gpu
@pytest.mark.parametrize("data", ["bench", "search"])
@pytest.mark.parametrize("schedule", ["group", "chain"])
@pytest.mark.parametrize("nt", [3, 5, 8])
def test_philox_counts_equal_reference_over_the_traced_rung(data, schedule, nt):
    """Traced Philox ladders (nt = 3: two ladders per warp; 8: no idle groups), bench data (bucket table) and binary-
    search data: the counts of rung 0 and of the hottest rung equal the reference over pt.samplers[rung]'s trace."""
    problem = _bench_problem() if data == "bench" else _search_problem()
    grid, (vlo, vhi, H) = _grid(problem), (0.5, 3.5, 20)
    K, T, every = 97, 400, 3
    betas = 0.6 ** np.arange(nt)
    rec = np.arange(T)[np.arange(T) % every == 0] + 1
    for rung in (0, nt - 1):
        pt = _pt(problem, K, betas, seed=40 + nt, schedule=schedule)
        pt.set_posterior_summary(grid, (vlo, vhi), H, every, rung=rung)
        pt.run(T)
        tr = pt.samplers[rung]._chain_thetas                               # [rec, K]
        ref = summary_reference(tr.k[rec], tr.cpx[rec], tr.cpv[rec], grid, vlo, vhi, H)
        ps = pt.posterior_summary(allreduce=False)
        assert ps.nsamples == K * len(rec)
        _assert_counts_equal(_counts(ps), ref)


@pytest.mark.gpu
def test_rung_summaries_do_not_perturb_the_chains():
    """4,096 ladders x 5 untraced over two run calls: states, log-posteriors, accept / overflow counts, the diagnostics
    block and the per-chain moments are bit-identical with summaries on and off."""
    out = {}
    for on in (False, True):
        pt = _pt(_bench_problem(), 4096, 0.5 ** np.arange(5), Pswap=0.1, seed=1)
        if on:
            pt.set_posterior_summary(np.linspace(1.0, 3.0, 101), (0.0, 4.0), 64, every=16, rung=0)
        pt.run(700, trace=False)
        pt.run(310, trace=False)
        s = pt._sampler
        out[on] = (s._download_state(), s.diagnostics_block().cpu().numpy(), s.chain_moments())
    (a_st, a_lp), a_blk, a_m = out[False]
    (b_st, b_lp), b_blk, b_m = out[True]
    for x, y in zip(a_st, b_st):
        assert np.array_equal(x, y)
    assert np.array_equal(a_lp, b_lp)
    assert np.array_equal(a_blk, b_blk)
    assert np.array_equal(a_m[0], b_m[0]) and np.array_equal(a_m[1], b_m[1])


@pytest.mark.gpu
@pytest.mark.parametrize("schedule", ["group", "chain"])
def test_counts_of_two_shards_sum_to_the_full_run(schedule):
    """40 ladders x 3 split at ladder offsets 0 and 13 (13: the middle of a two-ladder schedule group)."""
    grid, vr = _grid(_bench_problem()), (0.5, 3.5)
    kw = dict(betas=[1.0, 0.5, 0.2], Pswap=0.3, seed=17, schedule=schedule)
    for rung in (0, 1):
        full = _pt(_bench_problem(), 40, **kw)
        full.set_posterior_summary(grid, vr, 20, every=3, rung=rung)
        full.run(600, trace=False)
        want = _counts(full.posterior_summary(allreduce=False))
        got = None
        for off, n in ((0, 13), (13, 27)):
            part = _pt(_bench_problem(), n, chain_offset=off, **kw)
            part.set_posterior_summary(grid, vr, 20, every=3, rung=rung)
            part.run(600, trace=False)
            c = _counts(part.posterior_summary(allreduce=False))
            got = c if got is None else tuple(u + v for u, v in zip(got, c))
        _assert_counts_equal(got, want)
        assert want[3] == 40 * len(range(0, 600, 3))


@pytest.mark.gpu
def test_rung0_summaries_agree_with_the_diagnostics():
    """every = RMN_CP_DIAG_EVERY, rung 0, a grid with the diagnostics' 6 query points: nsamples = ladders x samples,
    khist's mean is PTSampler.diagnostics()'s k mean, and the binned yhat mean is within half a bin of its means."""
    problem = _bench_problem()
    xmin, xmax = problem[2], problem[3]
    xq = xmin + (xmax - xmin) * (np.arange(6) + 0.5) / 6.0
    grid = np.unique(np.concatenate([xq, np.linspace(xmin, xmax, 13)]))
    K = 2048
    pt = _pt(problem, K, 0.5 ** np.arange(5), Pswap=0.1, seed=5)
    pt.run(1000, trace=False)
    pt.reset_diagnostics()
    pt.set_posterior_summary(grid, (-2.0, 6.0), 200, every=DIAG_EVERY, rung=0)
    pt.run(2000, trace=False)
    d = pt.diagnostics(allreduce=False)
    ps = pt.posterior_summary(allreduce=False)
    assert d["samples"] > 0 and ps.nsamples == K * d["samples"]
    assert abs(ps.k_mean - d["mean"][1]) <= 1e-12 * abs(d["mean"][1])
    at = np.searchsorted(grid, xq)
    assert np.all(ps.underflow[at] == 0) and np.all(ps.overflow[at] == 0)
    w = ps.value_edges[1] - ps.value_edges[0]
    assert np.all(np.abs(ps.yhat_mean[at] - d["mean"][2:8]) <= 0.5 * w + 1e-12)
    pt.reset_diagnostics()
    ps0 = pt.posterior_summary(allreduce=False)
    assert ps0.nsamples == 0 and ps0.khist.sum() == 0 and ps0.yhist.sum() == 0 and ps0.cpxhist.sum() == 0


@pytest.mark.gpu
def test_refusals_and_bookkeeping():
    from riemann_b200 import ParameterError, PTSampler, Sampler
    from riemann_b200 import _lib
    from riemann_b200.models import benchmarks
    from riemann_b200.models.changepoint import ChangepointParams, ChangepointRegression1D
    from riemann_b200.proposals.changepoint import ChangepointRegression1DProp
    from riemann_b200.proposals.randomwalk import MetropolisRandomWalk
    lib, grid = _lib.load(), np.linspace(1.0, 3.0, 9)
    pt = _pt(_bench_problem(), 16, 0.5 ** np.arange(4))
    with pytest.raises(ParameterError):
        pt.posterior_summary()                                          # nothing set yet
    for rung in (-1, 4):
        with pytest.raises(ParameterError):
            pt.set_posterior_summary(grid, (0.0, 4.0), rung=rung)
        assert lib.rmn_sampler_cp_set_rung_summary(pt._sampler._handle, rung, 9, _lib.ptr(grid), 0.0, 4.0, 8, 1) == \
            _lib.RMN_ERR_PARAM
    # a tempered Gaussian ladder
    gpt = PTSampler(benchmarks.benchmark_gauss2d_corr, MetropolisRandomWalk(0.5 * np.eye(2)), np.ones(2), K=16)
    with pytest.raises(ParameterError):
        gpt.set_posterior_summary(grid, (0.0, 1.0))
    assert lib.rmn_sampler_cp_set_rung_summary(gpt._sampler._handle, 0, 9, _lib.ptr(grid), 0.0, 1.0, 8, 1) == \
        _lib.RMN_ERR_UNSUPPORTED
    # the rung entry on an untempered changepoint sampler
    x, y, xmin, xmax, lamb, kmax, alpha, beta, hscale = _bench_problem()
    dm = ChangepointRegression1D(x, y, xmin, xmax, lamb, int(kmax), alpha, beta)
    s = Sampler(dm, ChangepointRegression1DProp(dm, hscale), ChangepointParams([2.0], [1.0, 3.0], 0.1), K=64)
    assert lib.rmn_sampler_cp_set_rung_summary(s._handle, 0, 9, _lib.ptr(grid), 0.0, 4.0, 8, 1) == \
        _lib.RMN_ERR_UNSUPPORTED
    # the untempered entry still refuses the tempered sampler
    assert lib.rmn_sampler_cp_set_summary(pt._sampler._handle, 9, _lib.ptr(grid), 0.0, 4.0, 8, 1) == \
        _lib.RMN_ERR_UNSUPPORTED
    # on, then off: the runs go through the summary kernel, then the plain tempered kernel again
    pt._sampler.enable_kernel_timing()
    pt.set_posterior_summary(grid, (0.0, 4.0), every=2, rung=3)
    assert pt.summary_rung == 3
    pt.run(10, trace=False)
    assert pt._sampler.kernel_timing()["kernel"] == "cp_tempered_summary_kernel"
    assert pt.posterior_summary().nsamples == 16 * 5
    pt.set_posterior_summary(None)
    with pytest.raises(ParameterError):
        pt.posterior_summary()
    pt.run(10, trace=False)
    assert pt._sampler.kernel_timing()["kernel"] == "cp_tempered_kernel"
