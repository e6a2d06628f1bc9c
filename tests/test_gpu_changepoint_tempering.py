"""
Parallel tempering on the changepoint model: riemann_b200.PTSampler / rmn_sampler_set_tempering on
ChangepointRegression1D with the shared ChangepointRegression1DProp (riemann/samplers/ptsampler.py:41-127), run by
cp_tempered_kernel (riemann_b200/csrc/changepoint.cu).

* CPU: the oracle port replays tests/golden/pt_changepoint.npz (recorded by tests/pt_changepoint_fixture.py; `source` says whether
  the reference or the port recorded it) exactly; the fixture regenerates bit for bit from the unmodified reference
  where that tree is available; the tempered entry points have no local-memory frame.
* GPU: every rung's state, log-posterior and swap decision at every step of the replayed stream; many ladders and
  ladders of 3 and 8 temperatures against the port; Philox mode: rung 0 samples the posterior, every rung carries
  log_prior + beta * log_likelihood of its state, shards reproduce the full run bit for bit; refusals; diagnostics.

Tolerance 1e-9 (fp64 device vs fp64 numpy), 1e-10 relative for carried vs fresh evaluation on the device.
"""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from gpu_helpers import relerr
from pt_changepoint_fixture import PTSlotTapeDraws, pt_changepoint_arrays

TOL = 1e-9
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "riemann_b200", "libriemann_b200.so")
P_MIN = 1e-3


def _fixture_states(g):
    """[nt][T+1] states of the fixture as (k, cpx, cpv, sig) arrays."""
    return g["k"], g["cpx"], g["cpv"], g["sig"]


def _port_replay(g):
    from oracle import riemann_port as port
    pm, pp, th0, _ = port.make_changepoint_problem()
    pt = port.PTSampler(pm, pp, th0, betas=g["betas"], Pswap=float(g["pswap"]),
                        draws=PTSlotTapeDraws(g["usel"], g["tape"]))
    with np.errstate(all="ignore"):
        pt.run(g["usel"].shape[0])
    return pt


def _pack(states):
    from oracle.gen_golden import _cp_pack_state
    st = [_cp_pack_state(th) for th in states]
    return (np.array([s[0] for s in st]), np.array([s[1] for s in st]), np.array([s[2] for s in st]),
            np.array([s[3] for s in st]))


# ---------------------------------------------------------------------------------------------------------- CPU tests
def test_oracle_replays_the_fixture(golden):
    g = golden("pt_changepoint")
    pt = _port_replay(g)
    k, cpx, cpv, sig = _fixture_states(g)
    for i in range(len(g["betas"])):
        pk, px, pv, ps = _pack(pt.samplers[i]._chain_thetas)
        assert np.array_equal(pk, k[i]) and np.array_equal(px, cpx[i])
        assert np.array_equal(pv, cpv[i]) and np.array_equal(ps, sig[i])
        assert np.array_equal(np.array(pt.samplers[i]._chain_logpost, dtype=np.float64), g["logpost"][i])
    assert int((g["kind"] == 1).sum()) > 100


def test_fixture_regenerates_from_the_reference(golden):
    from oracle import refshim
    if not refshim.reference_available():
        pytest.skip("reference tree not available (the committed fixture records its source)")
    g = golden("pt_changepoint")
    out = pt_changepoint_arrays(refshim.load_reference())
    for name, v in out.items():
        assert np.array_equal(v, g[name]), name


def test_tempered_kernels_have_no_local_memory_frame():
    if not os.path.exists(LIB) or shutil.which("cuobjdump") is None or shutil.which("c++filt") is None:
        pytest.skip("needs the built library, cuobjdump and c++filt")
    txt = subprocess.run(["cuobjdump", "-res-usage", LIB], capture_output=True, text=True, check=True).stdout
    rows = re.findall(r"Function (\S+):\s*\n\s*REG:(\d+) STACK:(\d+)", txt)
    names = subprocess.run(["c++filt"] + [r[0] for r in rows], capture_output=True, text=True, check=True).stdout
    found = {}
    for name, (_, reg, stack) in zip(names.splitlines(), rows):
        m = re.search(r"(cp_tempered_kernel<[^>]*>)", name)
        if m:
            found[m.group(1).replace(" ", "")] = (int(reg), int(stack))
    assert len(found) == 6, found                                     # INJ x DATA
    for name, (reg, stack) in found.items():
        assert stack == 0 and reg <= 128, (name, reg, stack)


# ---------------------------------------------------------------------------------------------------------- GPU tests
def _device_problem():
    from oracle import riemann_port as port
    from riemann_b200.models.changepoint import ChangepointParams, ChangepointRegression1D
    from riemann_b200.proposals.changepoint import ChangepointRegression1DProp
    pm, pp, th0, _ = port.make_changepoint_problem()
    dm = ChangepointRegression1D(pm.x, pm.y, pm.xmin, pm.xmax, pm.lamb, int(pm.kmax), pm.alpha, pm.beta)
    return dm, ChangepointRegression1DProp(dm, pp.hscale), ChangepointParams(th0.cpx, th0.cpv, th0.sig)


def _trace_arrays(tr):
    """K = 1 history (list of ChangepointParams) -> packed arrays."""
    from riemann_b200.models.changepoint import pack_states
    return pack_states(tr)


def _check_replay(pt, ex, g, T=None):
    k, cpx, cpv, sig = _fixture_states(g)
    T = g["usel"].shape[0] if T is None else T
    nt = len(g["betas"])
    for i in range(nt):
        dk, dx, dv, ds = _trace_arrays(pt.samplers[i]._chain_thetas)
        assert np.array_equal(dk, k[i, :T + 1])
        assert relerr(dx, cpx[i, :T + 1]) < TOL and relerr(dv, cpv[i, :T + 1]) < TOL
        assert relerr(ds, sig[i, :T + 1]) < TOL
        assert relerr(np.array(pt.samplers[i]._chain_logpost), g["logpost"][i, :T + 1]) < TOL
    dk0, dx0, _, _ = _trace_arrays(pt._chain_thetas)                   # ptsampler.py:89-90: rung 0
    assert np.array_equal(dk0, k[0, :T + 1]) and relerr(dx0, cpx[0, :T + 1]) < TOL
    # swap decisions: an accepted swap shows as both partners changing state at a swap step, or as a swap of two
    # identical states (every rung starts at theta0)
    kind = g["kind"][:T]
    st = np.concatenate([k[:, :T + 1, None], cpx[:, :T + 1], cpv[:, :T + 1], sig[:, :T + 1, None]], axis=2)
    moved = np.any(st[:, 1:] != st[:, :-1], axis=2).T                      # [T][nt]
    same_next = np.zeros((T, nt), dtype=bool)
    same_next[:, :-1] = np.all(st[:-1, :-1] == st[1:, :-1], axis=2).T    # rung i and i+1 equal before step t
    same_prev = np.zeros((T, nt), dtype=bool)
    same_prev[:, 1:] = same_next[:, :-1]
    acc = ex["accepted"].astype(bool)[:T]
    assert np.array_equal(acc[kind == 1], (moved | same_next)[kind == 1])
    assert np.array_equal(acc[kind == 2], (moved | same_prev)[kind == 2])


@pytest.mark.gpu
def test_injected_ladder_matches_the_fixture(golden):
    from riemann_b200 import PTSampler
    g = golden("pt_changepoint")
    dm, dp, th0 = _device_problem()
    pt = PTSampler(dm, dp, th0)
    assert np.array_equal(pt.betas, g["betas"]) and pt.Pswap == float(g["pswap"])
    ex = pt.run_injected(g["usel"], tape=g["tape"])
    _check_replay(pt, ex, g)
    # a participant's proposal record is its partner's state, with logqratio = 0
    kind = g["kind"]
    assert np.all(ex["logqratio"][kind != 0] == 0.0)
    assert np.array_equal(ex["prop_k"][kind == 1], g["k"][1:, :-1].T[kind[:, :-1] == 1])


def _port_run(betas, Pswap, T, seed):
    from oracle import riemann_port as port
    return pt_changepoint_arrays(port, T=T, seed=seed, betas=np.asarray(betas, dtype=np.float64), Pswap=Pswap)


@pytest.mark.gpu
def test_many_ladders_each_replay_the_stream(golden):
    """13 ladders x 5 temperatures fed the same stream: every ladder reproduces it."""
    from riemann_b200 import PTSampler
    g = golden("pt_changepoint")
    dm, dp, th0 = _device_problem()
    K, T = 13, 500
    pt = PTSampler(dm, dp, th0, K=K)
    rep = lambda a: np.concatenate([a[:T]] * K, axis=1)
    pt.run_injected(rep(g["usel"]), tape=rep(g["tape"]))
    for rung in (0, 3, 4):
        tr, lp = pt.samplers[rung]._chain_thetas, pt.samplers[rung]._chain_logpost   # [rec, K]
        for l in (0, 6, 12):
            assert np.array_equal(tr.k[:, l], g["k"][rung, :T + 1])
            assert relerr(tr.cpx[:, l], g["cpx"][rung, :T + 1]) < TOL
            assert relerr(tr.sig[:, l], g["sig"][rung, :T + 1]) < TOL
            assert relerr(lp[:, l], g["logpost"][rung, :T + 1]) < TOL


@pytest.mark.gpu
@pytest.mark.parametrize("betas,Pswap", [([1.0, 0.4, 0.1], 0.3),                     # S = 4: two ladders per warp
                                         (list(0.7 ** np.arange(8)), 0.2)])          # S = 8: no idle groups
def test_explicit_ladders_match_the_port(betas, Pswap):
    from riemann_b200 import PTSampler
    T = 800
    ref = _port_run(betas, Pswap, T, seed=610 + len(betas))
    dm, dp, th0 = _device_problem()
    pt = PTSampler(dm, dp, th0, betas=betas, Pswap=Pswap)
    ex = pt.run_injected(ref["usel"], tape=ref["tape"])
    _check_replay(pt, ex, ref)
    assert int((ref["kind"] == 1).sum()) > 50


@pytest.fixture(scope="module")
def philox_ladders():
    """2,048 ladders x 5 in Philox mode from the start state of the reference's marginal chains, 6,000 + 4,000 steps
    (diagnostics reset in between, like changepoint_posterior.npz's window)."""
    from riemann_b200 import PTSampler
    from riemann_b200.models.changepoint import ChangepointParams
    dm, dp, _ = _device_problem()
    K = 2048
    pt = PTSampler(dm, dp, ChangepointParams([2.0], [1.0, 3.0], 0.1), K=K, seed=91)
    pt.run(6000, trace=False)
    pt._sampler.reset_diagnostics()
    pt.run(4000, trace=False)
    return dm, pt


@pytest.mark.gpu
def test_philox_rung0_samples_the_posterior(golden, philox_ladders):
    from scipy import stats
    from oracle import riemann_port as port
    from riemann_b200.models.changepoint import unpack_state
    dm, pt = philox_ladders
    g = golden("changepoint_marginals")
    assert int(g["T"]) == 10000
    pm, _, _, _ = port.make_changepoint_problem()
    k, cpx, cpv, sig = pt._thetas[-1]                                         # [K, nt, ...]
    K, nt = k.shape
    k0, x0, v0, s0 = k[:, 0], cpx[:, 0], cpv[:, 0], sig[:, 0]
    assert stats.ks_2samp(s0, g["sig"][:, ::2].ravel()).pvalue > P_MIN
    for qi, q in enumerate(g["query"]):
        xq = pm.xmin + (pm.xmax - pm.xmin) * (q + 0.5) / 6.0
        yq = np.array([v0[c, np.searchsorted(x0[c, :k0[c]], xq)] for c in range(K)])
        assert stats.ks_2samp(yq, g["yq"][:, ::2, qi].ravel()).pvalue > P_MIN
    lo, hi = 4, 10
    bins = np.arange(lo, hi + 2)
    dev_h = np.histogram(np.clip(k0, lo, hi), bins)[0].astype(float)
    ref_h = np.histogram(np.clip(g["k"][:, ::2].ravel(), lo, hi), bins)[0].astype(float)
    assert stats.chi2_contingency(np.array([dev_h, ref_h]))[1] > P_MIN
    # every rung carries combine(log_prior, beta_i * log_likelihood) of the state it holds
    states = [unpack_state(k[l, i], cpx[l, i], cpv[l, i], sig[l, i]) for l in range(K) for i in range(nt)]
    ll = dm._eval_states(states, 1).reshape(K, nt)
    lpr = dm._eval_states(states, 2).reshape(K, nt)
    with np.errstate(all="ignore"):
        tl = ll * pt.betas[None, :]
        ref = np.where(np.isfinite(lpr) & np.isfinite(tl), lpr + tl, -np.inf)
    lp = pt._logpost[-1]
    fin = np.isfinite(ref)
    assert np.array_equal(np.isfinite(lp), fin)
    assert np.max(np.abs(lp[fin] - ref[fin]) / np.abs(ref[fin])) < 1e-10
    # tempering changes something: the hot rungs hold states with other numbers of changepoints
    assert np.any(k[:, 0] != k[:, nt - 1])
    assert k[:, nt - 1].mean() != k[:, 0].mean()


@pytest.mark.gpu
def test_diagnostics_report_the_base_rung(golden, philox_ladders):
    _, pt = philox_ladders
    ref = golden("changepoint_posterior")
    dg = pt.diagnostics()
    assert dg["chains"] == pt.K and dg["temperatures"] == 5
    assert ref["mean_k"].min() <= dg["mean"][1] <= ref["mean_k"].max(), (dg["mean"][1], ref["mean_k"])
    assert 0.0 < dg["accept_rate_all_rungs"] < 1.0


@pytest.mark.gpu
@pytest.mark.parametrize("schedule", ["group", "chain"])
def test_shards_reproduce_the_full_run(schedule):
    """40 ladders x 3 (two ladders per warp): shards at ladder offsets 0 and 13 equal the full run bit for bit; offset 13
    starts the shard in the middle of a two-ladder schedule group."""
    from riemann_b200 import PTSampler
    dm, dp, th0 = _device_problem()
    kw = dict(betas=[1.0, 0.5, 0.2], Pswap=0.3, seed=17, move_schedule=schedule)
    full = PTSampler(dm, dp, th0, K=40, **kw)
    full.run(600, trace=False)
    (fk, fx, fv, fs), flp = full._sampler._download_state()
    for off, n in ((0, 13), (13, 27)):
        part = PTSampler(dm, dp, th0, K=n, chain_offset=off, **kw)
        part.run(600, trace=False)
        (pk, px, pv, ps), plp = part._sampler._download_state()
        sl = slice(3 * off, 3 * (off + n))
        assert np.array_equal(pk, fk[sl]) and np.array_equal(px, fx[sl])
        assert np.array_equal(pv, fv[sl]) and np.array_equal(ps, fs[sl])
        assert np.array_equal(plp, flp[sl])
    assert np.any(fk[0::3] != fk[2::3])


@pytest.mark.gpu
def test_refusals(golden):
    from riemann_b200 import PTSampler, Sampler
    from riemann_b200.sampling_errors import ParameterError
    g = golden("pt_changepoint")
    dm, dp, th0 = _device_problem()
    with pytest.raises(ParameterError):
        PTSampler(dm, dp, th0, betas=0.8 ** np.arange(9))                   # nt <= 8 on this model
    with pytest.raises(ParameterError):
        Sampler(dm, dp, th0, K=15, chain_offset=4, _tempering=(0.5 ** np.arange(5), 0.1))   # chain_offset % nt != 0
    pt = PTSampler(dm, dp, th0)
    with pytest.raises(ParameterError):
        pt._sampler.run_injected(tape=g["tape"][:10])                       # no selection uniforms
    s = Sampler(dm, dp, th0, K=5, chain_offset=4)                           # untempered: nothing new is refused
    s.run_injected(tape=g["tape"][:10])
    s.run(20, trace=False)
