"""
Posterior summaries of the changepoint sampler accumulated on the device (Sampler.set_posterior_summary,
rmn_sampler_cp_set_summary; riemann_b200/csrc/changepoint.cu, CPSummary and the cp_summary kernels).

CPU: the numpy reference of the four summaries against a brute-force ChangepointRegression1D.predict loop; the host
validation; the exact int64 rank sum over two gloo ranks; no spill in the summary kernels.
GPU: the device counts EQUAL the numpy reference over traced / replayed states; a summary run leaves the chains, the
accept / overflow counts and the diagnostics bit-identical; the counts do not depend on the time slicing, the kernel or
the sharding; they agree with the diagnostics block and with the reference sampler's chains; unsupported set-ups are
refused.
"""
import os
import re
import shutil
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "riemann_b200", "libriemann_b200.so")
L = 16
P_MIN = 1e-3


def summary_reference(k, cpx, cpv, grid, vlo, vhi, H, chunk=1 << 16):
    """khist [16], cpxhist [G + 1], yhist [G, H + 2], nsamples of the states (k [n], cpx / cpv [n, 16]) with the
    semantics of rmn_sampler_cp_set_summary: i = searchsorted(grid, cpx[j], 'right') per changepoint j < k,
    yhat = cpv[searchsorted(cpx[:k], grid)] (ChangepointRegression1D.predict), bin 1 + floor((yhat - vlo) * inv) with
    inv = H / (vhi - vlo) clamped to [0, H + 1] (NaN -> 0)."""
    grid = np.asarray(grid, dtype=np.float64)
    k = np.asarray(k).astype(np.int64).reshape(-1)
    cpx = np.asarray(cpx, dtype=np.float64).reshape(len(k), -1)
    cpv = np.asarray(cpv, dtype=np.float64).reshape(len(k), -1)
    G, W = len(grid), H + 2
    inv = H / (vhi - vlo)
    khist = np.bincount(k, minlength=L).astype(np.int64)
    cpxhist = np.zeros(G + 1, np.int64)
    yhist = np.zeros(G * W, np.int64)
    for a in range(0, len(k), chunk):
        kk, xx, vv = k[a:a + chunk], cpx[a:a + chunk], cpv[a:a + chunk]
        live = np.arange(xx.shape[1])[None, :] < kk[:, None]
        cpxhist += np.bincount(np.searchsorted(grid, xx[live], "right"), minlength=G + 1)
        idx = np.zeros((len(kk), G), np.int64)
        for j in range(xx.shape[1]):
            idx += live[:, j, None] & (xx[:, j, None] < grid[None, :])
        y = np.take_along_axis(vv, idx, 1)
        with np.errstate(invalid="ignore"):
            t = (y - vlo) * inv
            b = np.where(t >= 0, np.where(t < H, 1 + np.floor(np.where(t < H, t, 0)), H + 1), 0).astype(np.int64)
        yhist += np.bincount((np.arange(G)[None, :] * W + b).ravel(), minlength=G * W)
    return khist, cpxhist, yhist.reshape(G, W), len(k)


# ------------------------------------------------------------------------------------------------------------- CPU
def _random_states(rng, n, xmin, xmax, vlo, vhi, grid):
    k = rng.integers(0, L, n)
    k[:4] = (0, 15, 1, 15)
    cpx = np.zeros((n, L))
    cpv = np.zeros((n, L))
    for c in range(n):
        pool = np.concatenate([rng.uniform(xmin, xmax, 40), grid[(grid >= xmin) & (grid <= xmax)]])
        cpx[c, :k[c]] = np.sort(rng.choice(pool, k[c], replace=False))       # some changepoints ON grid points
        h = rng.uniform(vlo - 1.0, vhi + 1.0, k[c] + 1)                      # some heights outside the range
        edges = vlo + (vhi - vlo) * np.arange(9) / 8
        on = rng.random(k[c] + 1) < 0.3
        h[on] = rng.choice(np.concatenate([edges, [vlo, vhi]]), on.sum())    # some exactly on bin edges
        cpv[c, :k[c] + 1] = h
    return k, cpx, cpv


def test_numpy_reference_matches_brute_force_predict():
    from riemann_b200.models.changepoint import ChangepointRegression1D, unpack_state
    rng = np.random.default_rng(5)
    xmin, xmax, vlo, vhi, H = 1.0, 3.0, 0.5, 3.5, 8
    grid = np.concatenate([[-1.0, 0.5, xmin], np.linspace(1.1, 2.9, 17), [xmax, 3.2, 7.0]])   # points outside too
    model = ChangepointRegression1D([], [], xmin, xmax, 5.0, 10, 1.0, 1.0)
    k, cpx, cpv = _random_states(rng, 300, xmin, xmax, vlo, vhi, grid)
    kh, ch, yh, n = summary_reference(k, cpx, cpv, grid, vlo, vhi, H)
    G, inv = len(grid), H / (vhi - vlo)
    kb, cb, yb = np.zeros(L, int), np.zeros(G + 1, int), np.zeros((G, H + 2), int)
    for c in range(len(k)):
        th = unpack_state(k[c], cpx[c], cpv[c], 0.1)
        kb[len(th.cpx)] += 1
        for x in th.cpx:
            cb[int(np.sum(grid <= x))] += 1
        for g, xg in enumerate(grid):
            y = float(model.predict(th, xg))
            b = 1 + int(np.floor((y - vlo) * inv))
            yb[g, min(max(b, 0), H + 1)] += 1
    assert n == len(k) and np.array_equal(kh, kb) and np.array_equal(ch, cb) and np.array_equal(yh, yb)
    assert (yh[:, 0] > 0).all() and (yh[:, -1] > 0).all()       # under- and overflow both exercised
    assert np.all(yh.sum(1) == n) and kh.sum() == n


def test_host_validation_refuses_bad_input():
    from riemann_b200 import ParameterError
    from riemann_b200.posterior_summary import check_summary_args
    from riemann_b200.samplers.sampler import Sampler
    good = dict(grid=np.linspace(0, 1, 5), value_range=(0.0, 1.0), value_bins=16, every=4)
    g, vlo, vhi, H, every = check_summary_args(**good)
    assert len(g) == 5 and (vlo, vhi, H, every) == (0.0, 1.0, 16, 4)
    bad = [dict(grid=[0.0, 2.0, 1.0]), dict(grid=[0.0, 1.0, 1.0]), dict(grid=[0.0, np.nan]), dict(grid=[0.0, np.inf]),
           dict(grid=[]), dict(grid=np.arange(1025.0)), dict(value_bins=0), dict(value_bins=1025),
           dict(value_range=(1.0, 1.0)), dict(value_range=(2.0, 1.0)), dict(value_range=(0.0, np.inf)),
           dict(value_range=(np.nan, 1.0)), dict(every=0), dict(every=-3)]
    for b in bad:
        with pytest.raises(ParameterError):
            check_summary_args(**dict(good, **b))
    # the model family and tempering are checked before anything reaches the library
    for is_cp, tempered in ((False, False), (True, True)):
        s = Sampler.__new__(Sampler)
        s._is_cp, s._tempered = is_cp, tempered
        with pytest.raises(ParameterError):
            s.set_posterior_summary(**good)


def test_null_sampler_is_refused_by_the_library():
    import __graft_entry__ as ge
    ge.build()
    from riemann_b200 import _lib
    lib = _lib.load()
    g = np.linspace(0, 1, 4)
    assert lib.rmn_sampler_cp_set_summary(None, 4, _lib.ptr(g), 0.0, 1.0, 8, 1) == _lib.RMN_ERR_PARAM
    assert lib.rmn_sampler_cp_get_summary(None, None, None, None, None, None) == _lib.RMN_ERR_PARAM


_GLOO = r"""
import sys, numpy as np, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from riemann_b200.distributed import reduce_counts
dist.init_process_group("gloo")
r = dist.get_rank()
big = (1 << 60) + 12345                              # beyond fp64's 53-bit integers: the sum must stay int64
parts = [np.array([big, 7, 0, -3, 5], np.int64), np.array([3, 1 << 40, 11, 3, 0], np.int64)]
out = reduce_counts(torch.tensor(parts[r]))
assert out.dtype == torch.int64
assert np.array_equal(out.numpy(), parts[0] + parts[1]), out
dist.barrier(); dist.destroy_process_group()
print("rank", r, "ok")
"""


def test_count_rank_sum_two_ranks_gloo(tmp_path):
    script = tmp_path / "gloo_counts.py"
    script.write_text(_GLOO)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29641", str(script), ROOT],
                       capture_output=True, text=True, timeout=240, env=env)
    assert r.returncode == 0, r.stdout + r.stderr
    assert r.stdout.count("ok") == 2


def test_summary_kernels_spill_nothing():
    """The summary kernels (one-slice at 4 resident blocks per SM, time-sliced at 5) keep their T loops free of
    local-memory traffic: no STL / LDL anywhere in them, and a 0-byte frame."""
    import __graft_entry__ as ge
    ge.build()
    if shutil.which("cuobjdump") is None or shutil.which("c++filt") is None:
        pytest.skip("needs cuobjdump and c++filt")
    txt = subprocess.run(["cuobjdump", "-res-usage", LIB], capture_output=True, text=True, check=True).stdout
    rows = re.findall(r"Function (\S+):\s*\n\s*REG:(\d+) STACK:(\d+)", txt)
    names = subprocess.run(["c++filt"] + [r[0] for r in rows], capture_output=True, text=True, check=True).stdout
    found = {}
    for name, (mangled, reg, stack) in zip(names.splitlines(), rows):
        m = re.search(r"(cp_summary_(?:sliced_)?kernel<[^>]*>)", name)
        if m:
            found[m.group(1).replace(" ", "")] = (mangled, int(reg), int(stack))
    want = ["cp_summary_kernel<%s,%d,%s>" % (i, d, g) for d in (0, 1, 2)
            for i, g in (("false", "true"), ("false", "false"), ("true", "true"))]
    want += ["cp_summary_sliced_kernel<%d,%s>" % (d, g) for d in (1, 2) for g in ("true", "false")]
    assert sorted(found) == sorted(want), sorted(found)
    for name, (mangled, reg, stack) in found.items():
        assert stack == 0, (name, stack)
        assert reg <= (96 if "sliced" in name else 128), (name, reg)
        sass = subprocess.run(["cuobjdump", "-sass", "-fun", mangled, LIB], capture_output=True, text=True,
                              check=True).stdout
        assert not re.search(r"\b(STL|LDL)\b", sass), name


# ------------------------------------------------------------------------------------------------------------- GPU
def _bench_problem():
    from oracle import riemann_port as port
    pm, pp, _, _ = port.make_changepoint_problem()
    return pm.x, pm.y, pm.xmin, pm.xmax, pm.lamb, pm.kmax, pm.alpha, pm.beta, pp.hscale


def _search_problem():
    """data with three equal x in a row: no bucket table fits (a bucket holds at most 2 points), so run boundaries
    come from the binary search (DATA = 1)"""
    rng = np.random.default_rng(2)
    xmin, xmax = 1.0, 3.0
    x = np.repeat(np.sort(rng.uniform(xmin, xmax, 34)), 3)[:100]
    y = np.where(x < 1.7, 1.2, np.where(x < 2.4, 2.6, 1.8)) + 0.1 * rng.standard_normal(100)
    return x, y, xmin, xmax, 5.0, 10, 1.0, 1.0, 2.0


def _sampler(problem, K, seed=3, chain_offset=0, schedule="group"):
    from riemann_b200 import Sampler
    from riemann_b200.models.changepoint import ChangepointParams, ChangepointRegression1D
    from riemann_b200.proposals.changepoint import ChangepointRegression1DProp
    x, y, xmin, xmax, lamb, kmax, alpha, beta, hscale = problem
    dm = ChangepointRegression1D(x, y, xmin, xmax, lamb, int(kmax), alpha, beta)
    dp = ChangepointRegression1DProp(dm, hscale)
    return Sampler(dm, dp, ChangepointParams([2.0], [1.0, 3.0], 0.1), K=K, seed=seed, chain_offset=chain_offset,
                   move_schedule=schedule)


def _grid(problem):
    x, xmin, xmax = problem[0], problem[2], problem[3]
    inside = np.linspace(xmin + 0.013, xmax - 0.017, 29)
    return np.unique(np.concatenate([[xmin - 0.5, xmin], x[5:95:9], inside, [xmax, xmax + 0.25]]))


def _counts(ps):
    return ps.khist, ps.cpxhist, ps.yhist, ps.nsamples


def _assert_counts_equal(a, b):
    for u, v in zip(_counts(a) if not isinstance(a, tuple) else a, _counts(b) if not isinstance(b, tuple) else b):
        assert np.array_equal(np.asarray(u), np.asarray(v))


@pytest.mark.gpu
@pytest.mark.parametrize("data", ["bench", "search"])
@pytest.mark.parametrize("schedule", ["group", "chain"])
def test_counts_equal_reference_over_the_traced_states(data, schedule):
    problem = _bench_problem() if data == "bench" else _search_problem()
    grid = _grid(problem)
    assert np.any(np.isin(grid, problem[0])) and grid[0] < problem[2] and grid[-1] > problem[3]
    K, T, vlo, vhi, H = 4096, 600, 0.5, 3.5, 24
    for every in (1, 16):
        s = _sampler(problem, K, schedule=schedule)
        s.set_posterior_summary(grid, (vlo, vhi), H, every)
        s.run(T)                                       # trace of every step: record t + 1 = state after step t
        tr = s._chain_thetas
        rec = np.arange(T)[np.arange(T) % every == 0] + 1
        ref = summary_reference(tr.k[rec], tr.cpx[rec], tr.cpv[rec], grid, vlo, vhi, H)
        ps = s.posterior_summary(allreduce=False)
        _assert_counts_equal(ps, ref)


@pytest.mark.gpu
def test_injected_replay_still_matches_the_fixture_and_counts_its_states(golden):
    from gpu_helpers import relerr
    from riemann_b200 import Sampler
    from riemann_b200.models.changepoint import ChangepointParams, ChangepointRegression1D
    from riemann_b200.proposals.changepoint import ChangepointRegression1DProp
    g = golden("changepoint")
    xmin, xmax, lamb, kmax, alpha, beta, hscale = g["hyper"]
    dm = ChangepointRegression1D(g["x"], g["y"], xmin, xmax, lamb, int(kmax), alpha, beta)
    dp = ChangepointRegression1DProp(dm, hscale)
    nch, T = g["tape"].shape[:2]
    th0 = [ChangepointParams(g["cpx"][c, 0, :g["k"][c, 0]], g["cpv"][c, 0, :g["k"][c, 0] + 1], g["sig"][c, 0])
           for c in range(nch)]
    grid = np.concatenate([[xmin - 1.0], np.linspace(xmin, xmax, 41), g["x"][10:90:20], [xmax + 1.0]])
    grid = np.unique(grid)
    vlo, vhi, H = float(np.min(g["y"])), float(np.max(g["y"])), 32
    s = Sampler(dm, dp, th0)
    s.set_posterior_summary(grid, (vlo, vhi), H, every=1)
    s.run_injected(tape=np.transpose(g["tape"], (1, 0, 2)))
    tr = s._chain_thetas
    assert np.array_equal(tr.k.T, g["k"])
    assert relerr(s._chain_logpost.T, g["logpost"]) < 1e-9
    ref = summary_reference(g["k"][:, 1:].ravel(), g["cpx"][:, 1:].reshape(-1, L), g["cpv"][:, 1:].reshape(-1, L),
                            grid, vlo, vhi, H)
    _assert_counts_equal(s.posterior_summary(allreduce=False), ref)


@pytest.mark.gpu
def test_summaries_do_not_perturb_the_chains():
    """65,536 chains untraced (time-sliced kernels): states, log-posteriors, accept / overflow counts and the whole
    diagnostics block are bit-identical with summaries on and off."""
    out = {}
    for on in (False, True):
        s = _sampler(_bench_problem(), 65536, seed=1)
        if on:
            s.set_posterior_summary(np.linspace(1.0, 3.0, 101), (0.0, 4.0), 64, every=16)
        s.run(700, trace=False)
        s.run(310, trace=False)
        out[on] = (s._download_state(), s.diagnostics_block().cpu().numpy(), s.chain_moments())
    (a_st, a_lp), a_blk, a_m = out[False]
    (b_st, b_lp), b_blk, b_m = out[True]
    for x, y in zip(a_st, b_st):
        assert np.array_equal(x, y)
    assert np.array_equal(a_lp, b_lp)
    assert np.array_equal(a_blk, b_blk)
    assert np.array_equal(a_m[0], b_m[0]) and np.array_equal(a_m[1], b_m[1])


@pytest.mark.gpu
def test_counts_do_not_depend_on_slicing_or_kernel(monkeypatch):
    """30,000 chains: 938 blocks, more than the summary kernels' resident slots and not a whole number of waves, so
    RMN_CP_SLICED=1 runs cp_summary_sliced_kernel and RMN_CP_SLICED=0 cp_summary_kernel."""
    out = {}
    for mode, kernel in (("0", "cp_summary_kernel"), ("1", "cp_summary_sliced_kernel")):
        monkeypatch.setenv("RMN_CP_SLICED", mode)
        s = _sampler(_bench_problem(), 30000, seed=3, chain_offset=13)
        s.set_posterior_summary(_grid(_bench_problem()), (0.5, 3.5), 48, every=16)
        s.enable_kernel_timing()
        s.run(450, trace=False)
        s.run(230, trace=False)
        assert s.kernel_timing()["kernel"] == kernel
        out[mode] = (s.posterior_summary(allreduce=False), s._download_state())
    _assert_counts_equal(out["0"][0], out["1"][0])
    assert out["0"][0].nsamples == 30000 * len(range(0, 680, 16))
    for x, y in zip(out["0"][1][0], out["1"][1][0]):
        assert np.array_equal(x, y)


@pytest.mark.gpu
@pytest.mark.parametrize("schedule", ["group", "chain"])
def test_counts_of_two_shards_sum_to_the_full_run(schedule):
    grid, vr = _grid(_bench_problem()), (0.5, 3.5)
    full = _sampler(_bench_problem(), 96, seed=11, schedule=schedule)
    full.set_posterior_summary(grid, vr, 20, every=3)
    full.run(400, trace=False)
    want = _counts(full.posterior_summary(allreduce=False))
    got = None
    for off, n in ((0, 37), (37, 59)):                    # 37: not a multiple of the 8-chain schedule groups
        part = _sampler(_bench_problem(), n, seed=11, chain_offset=off, schedule=schedule)
        part.set_posterior_summary(grid, vr, 20, every=3)
        part.run(400, trace=False)
        c = _counts(part.posterior_summary(allreduce=False))
        got = c if got is None else tuple(u + v for u, v in zip(got, c))
    _assert_counts_equal(got, want)


@pytest.mark.gpu
def test_summaries_agree_with_the_diagnostics():
    """Grid with the diagnostics' 6 query points, every = 16 (the diagnostics' thinning): the binned mean of yhat is
    within half a bin width of the diagnostics' mean there, and khist's mean is the diagnostics' k mean."""
    problem = _bench_problem()
    xmin, xmax = problem[2], problem[3]
    xq = xmin + (xmax - xmin) * (np.arange(6) + 0.5) / 6.0
    grid = np.unique(np.concatenate([xq, np.linspace(xmin, xmax, 13)]))
    s = _sampler(problem, 8192, seed=5)
    s.run(1000, trace=False)
    s.reset_diagnostics()
    s.set_posterior_summary(grid, (-2.0, 6.0), 200, every=16)
    s.run(2000, trace=False)
    d = s.diagnostics(allreduce=False)
    ps = s.posterior_summary(allreduce=False)
    assert ps.nsamples == 8192 * d["samples"]
    assert abs(ps.k_mean - d["mean"][1]) <= 1e-12 * abs(d["mean"][1])
    at = np.searchsorted(grid, xq)
    assert np.all(ps.underflow[at] == 0) and np.all(ps.overflow[at] == 0)
    w = ps.value_edges[1] - ps.value_edges[0]
    assert np.all(np.abs(ps.yhat_mean[at] - d["mean"][2:8]) <= 0.5 * w + 1e-12)
    # a reset zeroes the counts together with the diagnostics
    s.reset_diagnostics()
    ps0 = s.posterior_summary(allreduce=False)
    assert ps0.nsamples == 0 and ps0.khist.sum() == 0 and ps0.yhist.sum() == 0 and ps0.cpxhist.sum() == 0


@pytest.mark.gpu
def test_summaries_agree_with_the_reference_sampler(golden):
    """One sample per chain (the final states of 4,096 chains after the reference run's length) against the
    reference's thinned chains (tests/golden/changepoint_marginals.npz), chi-square gates of test_gpu_ks_marginals:
    k, and yhat at the tracked points binned by the summary's own rule; quantiles against the reference's."""
    from scipy import stats
    g = golden("changepoint_marginals")
    problem = _bench_problem()
    xmin, xmax = problem[2], problem[3]
    xq = xmin + (xmax - xmin) * (g["query"] + 0.5) / 6.0
    vlo, vhi, H = -1.0, 5.0, 24
    K, T = 4096, int(g["T"])
    s = _sampler(problem, K, seed=77)
    s.run(T - 1, trace=False)
    s.set_posterior_summary(xq, (vlo, vhi), H, every=1)
    s.run(1, trace=False)                                  # samples the state after the last step only
    ps = s.posterior_summary(allreduce=False)
    assert ps.nsamples == K and np.array_equal(ps.khist, np.bincount(s._chain_thetas.k[-1], minlength=L))
    ref_k = g["k"][:, ::2].ravel()
    lo, hi = 4, 10
    dev_h = np.array([ps.khist[:lo + 1].sum()] + list(ps.khist[lo + 1:hi]) + [ps.khist[hi:].sum()], float)
    ref_h = np.histogram(np.clip(ref_k, lo, hi), np.arange(lo, hi + 2))[0].astype(float)
    assert stats.chi2_contingency(np.array([dev_h, ref_h]))[1] > P_MIN
    for qi in range(len(xq)):
        ry = g["yq"][:, ::2, qi].ravel()
        rb = summary_reference(np.zeros(len(ry), int), np.zeros((len(ry), L)),
                               np.pad(ry[:, None], ((0, 0), (0, L - 1))), [xq[qi]], vlo, vhi, H)[2][0]
        keep = (ps.yhist[qi] + rb) >= 10
        tab = np.array([np.append(ps.yhist[qi][keep], ps.yhist[qi][~keep].sum()),
                        np.append(rb[keep], rb[~keep].sum())], float)
        tab = tab[:, tab.sum(0) > 0]
        assert stats.chi2_contingency(tab)[1] > P_MIN
        dq = ps.yhat_quantiles([0.05, 0.5, 0.95])[:, qi]
        rq = np.quantile(ry, [0.05, 0.5, 0.95])
        assert np.all(np.abs(dq - rq) <= 0.25 * (rq[2] - rq[0]) + (vhi - vlo) / H), (dq, rq)


@pytest.mark.gpu
def test_unsupported_set_ups_are_refused(monkeypatch):
    from riemann_b200 import ParameterError, PTSampler, Sampler
    from riemann_b200 import _lib
    from riemann_b200.models import benchmarks
    from riemann_b200.models.changepoint import ChangepointParams, ChangepointRegression1D
    from riemann_b200.proposals.changepoint import ChangepointRegression1DProp
    from riemann_b200.proposals.randomwalk import MetropolisRandomWalk
    lib, grid = _lib.load(), np.linspace(1.0, 3.0, 9)
    gs = Sampler(benchmarks.benchmark_gauss2d_corr, MetropolisRandomWalk(0.5 * np.eye(2)), np.ones(2), K=64)
    with pytest.raises(ParameterError):
        gs.set_posterior_summary(grid, (0.0, 1.0))
    assert lib.rmn_sampler_cp_set_summary(gs._handle, 9, _lib.ptr(grid), 0.0, 1.0, 8, 1) == _lib.RMN_ERR_UNSUPPORTED
    x, y, xmin, xmax, lamb, kmax, alpha, beta, hscale = _bench_problem()
    dm = ChangepointRegression1D(x, y, xmin, xmax, lamb, int(kmax), alpha, beta)
    dp = ChangepointRegression1DProp(dm, hscale)
    pt = PTSampler(dm, dp, ChangepointParams([2.0], [1.0, 3.0], 0.1), betas=0.5 ** np.arange(4), K=16)
    with pytest.raises(ParameterError):
        pt._sampler.set_posterior_summary(grid, (0.0, 4.0))
    assert lib.rmn_sampler_cp_set_summary(pt._sampler._handle, 9, _lib.ptr(grid), 0.0, 4.0, 8, 1) == \
        _lib.RMN_ERR_UNSUPPORTED
    monkeypatch.setenv("RMN_CP_GL", "8")
    s8 = _sampler(_bench_problem(), 64)
    with pytest.raises(ParameterError):
        s8.set_posterior_summary(grid, (0.0, 4.0))
    monkeypatch.delenv("RMN_CP_GL")
    s4 = _sampler(_bench_problem(), 64)
    with pytest.raises(ParameterError):
        s4.posterior_summary()                             # nothing set yet
    s4.set_posterior_summary(grid, (0.0, 4.0), every=2)
    s4.run(10, trace=False)
    assert s4.posterior_summary().nsamples == 64 * 5
    s4.set_posterior_summary(None)
    with pytest.raises(ParameterError):
        s4.posterior_summary()
