"""
Run boundaries of the changepoint likelihood on adversarial data (riemann_b200/csrc/changepoint.cuh: run_boundary).

A run boundary is #{i : x_i <= c} for a changepoint location c.  rmn_model_changepoint_create builds a bucket table when
no bucket of its grid holds more than two data points and the kernels then look the boundary up in it; other data keeps
the binary search (here: "clustered" and "triplicates").  Each case evaluates the log-likelihood (rmn_model_cp_logpost, which = 1) of many one- and
three-changepoint states and compares it with the numpy oracle at 1e-12 relative.  The heights differ by O(1) from the
data, so a boundary off by one changes the value by about 1 / M relative, far above the tolerance.

The query locations cover every data point, its neighbouring doubles, bucket edges of every power-of-two grid up to
2,048 buckets and their neighbours, points outside [xmin, xmax], +-inf, -0.0 and +-1e308.  A NaN location gets
boundary 0, the same as -inf (numpy's searchsorted would put a NaN last), so it is compared with the oracle at -inf.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
TOL = 1e-12


def _edge_grid(xmin, xmax):
    q = []
    for g in (2 ** p for p in range(1, 12)):
        e = xmin + np.arange(g + 1) * ((xmax - xmin) / g)
        q += [e, np.nextafter(e, np.inf), np.nextafter(e, -np.inf)]
    return np.concatenate(q)


def _queries(x, xmin, xmax, rng):
    span = xmax - xmin
    return np.concatenate([x, np.nextafter(x, np.inf), np.nextafter(x, -np.inf), _edge_grid(xmin, xmax),
                           rng.uniform(xmin - 0.2 * span, xmax + 0.2 * span, 500),
                           [xmin - span, xmax + span, -np.inf, np.inf, -0.0, 0.0, 1e308, -1e308]])


def _cases():
    rng = np.random.default_rng(11)
    edges = np.arange(64) / 64.0                                            # one point on every edge of 64 buckets
    sub = np.sort(rng.choice(1024, 300, replace=False)) / 1024.0            # points on edges of a finer grid
    return {
        "duplicates": (np.repeat(np.linspace(0.0, 1.0, 40), 2), 0.0, 1.0),   # pairs of equal x
        "clustered": (np.sort(np.concatenate([1.5 + 1e-12 * np.arange(30), np.linspace(0.0, 3.0, 40)])), 0.0, 3.0),
        "triplicates": (np.sort(np.concatenate([np.full(3, 0.25), np.linspace(0.0, 1.0, 20)])), 0.0, 1.0),
        "on_edges": (edges, 0.0, 1.0),
        "on_finer_edges": (sub, 0.0, 1.0),
        "outside_range": (np.concatenate([[-0.3], np.linspace(0.01, 0.99, 50), [1.2]]), 0.0, 1.0),
        "single_point": (np.array([0.5]), 0.0, 1.0),
        "bench_like": (np.sort(1.0 + 2.0 * rng.uniform(size=100)), 1.0, 3.0),
    }


def _models(x, xmin, xmax, seed):
    from oracle import riemann_port as port
    from riemann_b200.models.changepoint import ChangepointRegression1D
    y = np.random.default_rng(seed).uniform(0.0, 1.0, len(x))
    args = (x, y, xmin, xmax, 3.0, 10, 1.0, 1.0)
    return ChangepointRegression1D(*args), port.ChangepointRegression1D(*args)


@pytest.mark.parametrize("case", sorted(_cases()))
def test_boundaries_match_searchsorted(case):
    from oracle import riemann_port as port
    from riemann_b200.models.changepoint import ChangepointParams
    x, xmin, xmax = _cases()[case]
    dm, om = _models(x, xmin, xmax, 5)
    rng = np.random.default_rng(7)
    q = _queries(x, xmin, xmax, rng)
    states = [((c,), (0.0 + 3.0 * (i % 2), 5.0 - 3.0 * (i % 2)), 0.4) for i, c in enumerate(q)]
    for _ in range(300):                                                    # three sorted locations
        states.append((tuple(np.sort(rng.choice(q, 3))), (0.0, 4.0, -2.0, 3.0), 0.7))
    states.append(((np.nan,), (0.0, 5.0), 0.4))                             # NaN location: boundary 0, as -inf
    states.append(((np.nan, 0.6 * xmin + 0.4 * xmax), (0.0, 5.0, -1.0), 0.4))
    got = dm._eval_states([ChangepointParams(np.array(c), np.array(v), s) for c, v, s in states], 1)
    want = []
    with np.errstate(all="ignore"):
        for c, v, s in states:
            c = np.where(np.isnan(c), -np.inf, c)
            want.append(om.log_likelihood(port.ChangepointParams(c, np.array(v), s)))
    want = np.array(want)
    assert np.all(np.isfinite(want))
    bad = np.flatnonzero(np.abs(got - want) > TOL * np.abs(want))
    assert bad.size == 0, [(states[i][0], got[i], want[i]) for i in bad[:5]]


@pytest.mark.parametrize("case", ["clustered", "on_edges"])
def test_sampler_carries_fresh_log_posteriors(case):
    """Short runs on data that keeps the binary search (clustered) and on data that gets the bucket table: one wave
    (one-slice kernel) and 938 blocks at GL = 4 (time-sliced); the carried log-posteriors must equal a fresh pointwise
    evaluation of the final states."""
    import torch
    from riemann_b200 import Sampler, _lib
    from riemann_b200.models.changepoint import ChangepointParams
    from riemann_b200.proposals.changepoint import ChangepointRegression1DProp
    x, xmin, xmax = _cases()[case]
    dm, _ = _models(x, xmin, xmax, 9)
    dp = ChangepointRegression1DProp(dm, 1.0)
    mid = 0.5 * (xmin + xmax)
    for K in (64, 30000):
        s = Sampler(dm, dp, ChangepointParams([mid], [0.3, 0.7], 0.3), K=K, seed=3)
        s.run(240, trace=False)
        (k, cpx, cpv, sig), lp = s._download_state()
        assert np.all(np.isfinite(lp))
        dk, dx, dv, ds = (torch.as_tensor(a, device="cuda") for a in (k, cpx, cpv, sig))
        out = torch.empty(K, dtype=torch.float64, device="cuda")
        _lib.check(_lib.load().rmn_model_cp_logpost(dm._handle, 0, K, _lib.ptr(dk), _lib.ptr(dx), _lib.ptr(dv),
                                                    _lib.ptr(ds), _lib.ptr(out), _lib.stream_ptr()))
        assert np.allclose(out.cpu().numpy(), lp, rtol=1e-12, atol=1e-9)
