"""
Swap statistics of the changepoint tempering ladders (PTSampler.swap_statistics, rmn_sampler_cp_get_swap_stats;
riemann_b200/csrc/changepoint.cu, cp_block under TEMPER): swaps proposed / accepted per pair of neighbouring rungs, the
replicas' round trips from rung 0 to rung nt-1 and back, and the up / down flow histogram per rung.

CPU: the numpy reference `swap_stats_reference` on a hand-computed sequence and on the fixture's initiators; the twelve
tempered kernel instantiations that count stay within the tempered budget (at most 128 registers, no local-memory
frame, no spill instructions); the library refuses a null sampler; the host refuses other models.
GPU: the device counts EQUAL the reference walked through the swap decisions of the replayed fixture ladder and of the
port-recorded ladders of 3 and 8 temperatures; many ladders, split runs, resets, set_state, shards, rung summaries on
or off; known answers in Philox mode; refusals.
"""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "riemann_b200", "libriemann_b200.so")
DIAG_EVERY = 16          # RMN_CP_DIAG_EVERY
NONE, UP, DOWN = 0, 1, 2


def swap_stats_reference(kind, accepted, nt, step0=0):
    """Walk the replica labels of one ladder through its swap decisions.  kind[t, i]: 0 within-chain step, 1 rung i
    initiates a swap with rung i+1, 2 rung i is that partner; accepted[t, i] (read where kind == 1): the swap was taken.
    Step t has the global index step0 + t.  -> dict of the counts rmn_sampler_cp_get_swap_stats returns."""
    kind, accepted = np.asarray(kind), np.asarray(accepted, dtype=bool)
    lab = np.full(nt, NONE)
    lab[0], lab[nt - 1] = UP, DOWN
    out = dict(proposed=np.zeros(nt - 1, np.int64), accepted=np.zeros(nt - 1, np.int64), up=np.zeros(nt, np.int64),
               down=np.zeros(nt, np.int64), round_trips=0)
    for t in range(kind.shape[0]):
        for i in np.flatnonzero(kind[t] == 1):
            out["proposed"][i] += 1
            if accepted[t, i]:
                out["accepted"][i] += 1
                lab[i], lab[i + 1] = lab[i + 1], lab[i]
                if i == 0:
                    out["round_trips"] += int(lab[0] == DOWN)
                    lab[0] = UP
                if i + 1 == nt - 1:
                    lab[nt - 1] = DOWN
        if (step0 + t) % DIAG_EVERY == 0:
            out["up"] += lab == UP
            out["down"] += lab == DOWN
    return out


def fixture_decisions(g, T=None):
    """(kind, accepted) of a recorded ladder: an initiator's swap was taken where its state changed at the swap step,
    or where the two partners held the same state before it (as _check_replay of test_gpu_changepoint_tempering)."""
    T = g["usel"].shape[0] if T is None else T
    k, cpx, cpv, sig = g["k"], g["cpx"], g["cpv"], g["sig"]
    st = np.concatenate([k[:, :T + 1, None], cpx[:, :T + 1], cpv[:, :T + 1], sig[:, :T + 1, None]], axis=2)
    moved = np.any(st[:, 1:] != st[:, :-1], axis=2).T                      # [T][nt]
    same_next = np.zeros_like(moved)
    same_next[:, :-1] = np.all(st[:-1, :-1] == st[1:, :-1], axis=2).T
    return g["kind"][:T], moved | same_next


def _as_dict(s):
    return dict(proposed=s.proposed, accepted=s.accepted, up=s.up, down=s.down, round_trips=s.round_trips)


def _assert_stats_equal(got, want, scale=1):
    for name in ("proposed", "accepted", "up", "down"):
        assert np.array_equal(np.asarray(got[name]), scale * np.asarray(want[name])), (name, got[name], want[name])
    assert int(got["round_trips"]) == scale * int(want["round_trips"]), (got["round_trips"], want["round_trips"])


# ------------------------------------------------------------------------------------------------------------- CPU
def test_reference_counts_a_hand_computed_sequence():
    """nt = 3, 17 steps: a swap 0-1 (rung 0's NONE arrival becomes UP), a swap 1-2 (rung 2 gets UP, becomes DOWN), a
    rejected 0-1, a taken 0-1 that brings the DOWN replica back to rung 0 (one round trip); samples at steps 0 and 16."""
    kind, acc = np.zeros((17, 3), np.int8), np.zeros((17, 3), bool)
    kind[0], acc[0, 0] = (1, 2, 0), True
    kind[1], acc[1, 1] = (0, 1, 2), True
    kind[2] = (1, 2, 0)
    kind[3], acc[3, 0] = (1, 2, 0), True
    r = swap_stats_reference(kind, acc, 3)
    _assert_stats_equal(r, dict(proposed=[3, 1], accepted=[2, 1], up=[2, 2, 0], down=[0, 0, 2], round_trips=1))
    # the same sequence from step 1: step 16 (t = 15) is the only sampled one
    r = swap_stats_reference(kind, acc, 3, step0=1)
    _assert_stats_equal(r, dict(proposed=[3, 1], accepted=[2, 1], up=[1, 1, 0], down=[0, 0, 1], round_trips=1))


def test_reference_on_the_fixture(golden):
    g = golden("pt_changepoint")
    nt = len(g["betas"])
    kind, acc = fixture_decisions(g)
    r = swap_stats_reference(kind, acc, nt)
    assert np.array_equal(r["proposed"], (g["kind"] == 1).sum(0)[:-1])
    assert np.all(r["accepted"] <= r["proposed"]) and r["accepted"].sum() > 0
    assert np.all(r["up"] + r["down"] <= len(range(0, kind.shape[0], DIAG_EVERY)))
    assert r["down"][0] == 0 and r["up"][nt - 1] == 0


def test_counting_kernels_fit_the_tempered_budget():
    import __graft_entry__ as ge
    ge.build()
    if shutil.which("cuobjdump") is None or shutil.which("c++filt") is None:
        pytest.skip("needs cuobjdump and c++filt")
    txt = subprocess.run(["cuobjdump", "-res-usage", LIB], capture_output=True, text=True, check=True).stdout
    rows = re.findall(r"Function (\S+):\s*\n\s*REG:(\d+) STACK:(\d+)", txt)
    names = subprocess.run(["c++filt"] + [r[0] for r in rows], capture_output=True, text=True, check=True).stdout
    found = {}
    for name, (mangled, reg, stack) in zip(names.splitlines(), rows):
        m = re.search(r"(cp_tempered(?:_summary)?_kernel<[^>]*>)", name)
        if m:
            found[m.group(1).replace(" ", "")] = (mangled, int(reg), int(stack))
    want = ["%s<%s,%d>" % (k, i, d) for k in ("cp_tempered_kernel", "cp_tempered_summary_kernel")
            for i in ("false", "true") for d in (0, 1, 2)]
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
    assert _lib.load().rmn_sampler_cp_get_swap_stats(None, None, None, None, None, None, None) == _lib.RMN_ERR_PARAM


def test_host_refuses_other_models():
    import __graft_entry__ as ge
    ge.build()
    from riemann_b200 import ParameterError, PTSampler
    pt = PTSampler.__new__(PTSampler)
    pt._is_cp, pt.Nt, pt._sampler = False, 5, None            # no device sampler: nothing may reach the library
    with pytest.raises(ParameterError):
        pt.swap_statistics()


# ------------------------------------------------------------------------------------------------------------- GPU
def _pt(K, betas, Pswap=0.3, seed=3, chain_offset=0, schedule="group"):
    from riemann_b200 import PTSampler
    from riemann_b200.models.changepoint import ChangepointParams
    from test_gpu_changepoint_tempering import _device_problem
    dm, dp, _ = _device_problem()
    return PTSampler(dm, dp, ChangepointParams([2.0], [1.0, 3.0], 0.1), betas=betas, Pswap=Pswap, K=K, seed=seed,
                     chain_offset=chain_offset, move_schedule=schedule)


@pytest.mark.gpu
def test_fixture_replay_counts_equal_the_reference(golden):
    """The replayed fixture ladder (1,500 steps, 5 rungs) reproduces its states, and its counts are the reference's
    over the fixture's swap decisions."""
    from riemann_b200 import PTSampler
    from test_gpu_changepoint_tempering import _check_replay, _device_problem
    g = golden("pt_changepoint")
    pt = PTSampler(*_device_problem())
    ex = pt.run_injected(g["usel"], tape=g["tape"])
    _check_replay(pt, ex, g)
    s = pt.swap_statistics(allreduce=False)
    _assert_stats_equal(_as_dict(s), swap_stats_reference(*fixture_decisions(g), len(g["betas"])))
    assert s.ladders == 1 and s.steps == g["usel"].shape[0]
    assert s.up_fraction[0] == 1.0 and s.up_fraction[-1] == 0.0


@pytest.mark.gpu
@pytest.mark.parametrize("betas,Pswap", [([1.0, 0.4, 0.1], 0.3),                     # S = 4: two ladders per warp
                                         (list(0.7 ** np.arange(8)), 0.2)])          # S = 8: no idle groups
def test_explicit_ladders_count_the_reference(betas, Pswap):
    """The port-recorded ladders of test_explicit_ladders_match_the_port."""
    from riemann_b200 import PTSampler
    from test_gpu_changepoint_tempering import _check_replay, _device_problem, _port_run
    ref = _port_run(betas, Pswap, 800, seed=610 + len(betas))
    pt = PTSampler(*_device_problem(), betas=betas, Pswap=Pswap)
    ex = pt.run_injected(ref["usel"], tape=ref["tape"])
    _check_replay(pt, ex, ref)
    _assert_stats_equal(_as_dict(pt.swap_statistics(allreduce=False)),
                        swap_stats_reference(*fixture_decisions(ref), len(betas)))


@pytest.mark.gpu
def test_many_ladders_count_each_ladder(golden):
    """13 ladders fed the same stream: every count is 13 x the single ladder's."""
    from riemann_b200 import PTSampler
    from test_gpu_changepoint_tempering import _device_problem
    g = golden("pt_changepoint")
    K, T = 13, 500
    pt = PTSampler(*_device_problem(), K=K)
    rep = lambda a: np.concatenate([a[:T]] * K, axis=1)
    pt.run_injected(rep(g["usel"]), tape=rep(g["tape"]))
    s = pt.swap_statistics(allreduce=False)
    _assert_stats_equal(_as_dict(s), swap_stats_reference(*fixture_decisions(g, T), len(g["betas"])), scale=K)
    assert s.ladders == K


@pytest.mark.gpu
def test_split_runs_and_resets(golden):
    """700 + 800 steps count what one 1,500-step call counts (the labels persist across launches); with a reset in
    between, the second window counts the difference, and a trip begun before the reset still completes."""
    from riemann_b200 import PTSampler
    from test_gpu_changepoint_tempering import _device_problem
    g = golden("pt_changepoint")
    nt, T = len(g["betas"]), g["usel"].shape[0]
    full = swap_stats_reference(*fixture_decisions(g), nt)
    first = swap_stats_reference(*fixture_decisions(g, 700), nt)
    for reset in (False, True):
        pt = PTSampler(*_device_problem())
        pt.run_injected(g["usel"][:700], tape=g["tape"][:700])
        _assert_stats_equal(_as_dict(pt.swap_statistics(allreduce=False)), first)
        if reset:
            pt.reset_diagnostics()
            z = pt.swap_statistics(allreduce=False)
            assert z.proposed.sum() == 0 and z.up.sum() == 0 and z.round_trips == 0 and z.steps == 0
        pt.run_injected(g["usel"][700:], tape=g["tape"][700:])
        s = pt.swap_statistics(allreduce=False)
        want = {n: full[n] - first[n] for n in full} if reset else full
        _assert_stats_equal(_as_dict(s), want)
        assert s.steps == (T - 700 if reset else T)


@pytest.mark.gpu
def test_set_state_restarts_the_replica_walk():
    """After 500 steps, set_state(theta0) + reset + step 0: the next 500 steps count what a fresh sampler's first 500
    count (the labels are re-initialised with the states)."""
    from riemann_b200 import _lib
    from riemann_b200.models.changepoint import ChangepointParams
    kw = dict(betas=0.5 ** np.arange(5), Pswap=0.2, seed=8)
    fresh = _pt(64, **kw)
    fresh.run(500, trace=False)
    want = _as_dict(fresh.swap_statistics(allreduce=False))
    pt = _pt(64, **kw)
    pt.run(500, trace=False)
    pt._sampler.set_state([ChangepointParams([2.0], [1.0, 3.0], 0.1)] * (64 * 5))
    pt.reset_diagnostics()
    _lib.check(_lib.load().rmn_sampler_set_step(pt._sampler._handle, 0))
    pt.run(500, trace=False)
    _assert_stats_equal(_as_dict(pt.swap_statistics(allreduce=False)), want)
    assert want["proposed"].sum() > 0 and want["accepted"].sum() > 0


@pytest.mark.gpu
@pytest.mark.parametrize("schedule", ["group", "chain"])
def test_counts_of_two_shards_sum_to_the_full_run(schedule):
    """40 ladders x 3 split at ladder offsets 0 and 13 (13: the middle of a two-ladder schedule group)."""
    kw = dict(betas=[1.0, 0.5, 0.2], Pswap=0.3, seed=17, schedule=schedule)
    full = _pt(40, **kw)
    full.run(600, trace=False)
    want = _as_dict(full.swap_statistics(allreduce=False))
    got = None
    for off, n in ((0, 13), (13, 27)):
        part = _pt(n, chain_offset=off, **kw)
        part.run(600, trace=False)
        c = _as_dict(part.swap_statistics(allreduce=False))
        got = c if got is None else {k: got[k] + c[k] for k in c}
    _assert_stats_equal(got, want)
    assert want["proposed"].sum() > 0


@pytest.mark.gpu
def test_rung_summaries_do_not_change_the_counts():
    """The same seeded Philox run with the rung summaries off and on (cp_tempered_kernel, cp_tempered_summary_kernel):
    identical swap counts and identical chains."""
    out = {}
    for on in (False, True):
        pt = _pt(512, 0.5 ** np.arange(5), Pswap=0.1, seed=1)
        if on:
            pt.set_posterior_summary(np.linspace(1.0, 3.0, 101), (0.0, 4.0), 64, every=16, rung=0)
        pt.run(700, trace=False)
        pt.run(310, trace=False)
        out[on] = (_as_dict(pt.swap_statistics(allreduce=False)), pt._sampler._download_state())
    _assert_stats_equal(out[True][0], out[False][0])
    (a_st, a_lp), (b_st, b_lp) = out[False][1], out[True][1]
    for x, y in zip(a_st, b_st):
        assert np.array_equal(x, y)
    assert np.array_equal(a_lp, b_lp)


@pytest.mark.gpu
def test_known_answers_in_philox_mode():
    """betas = [1, 1, 1, 1]: the swap ratio is exp(0) = 1 up to the last bits of the carried log-posteriors and a
    Philox uniform never exceeds 1 - 2^-33, so every proposed swap is taken.  The default ladder on 2,048 ladders:
    every pair accepts some swaps and rejects others, replicas complete round trips, rung 0 holds only up-moving and
    rung nt-1 only down-moving replicas; diagnostics() reports the same per-pair acceptance."""
    flat = _pt(256, [1.0, 1.0, 1.0, 1.0], Pswap=0.3, seed=4)
    flat.run(500, trace=False)
    s = flat.swap_statistics(allreduce=False)
    assert np.all(s.proposed > 0) and np.array_equal(s.accepted, s.proposed)
    pt = _pt(2048, 0.5 ** np.arange(5), Pswap=0.1, seed=91)
    pt.run(6000, trace=False)
    s = pt.swap_statistics(allreduce=False)
    assert s.ladders == 2048 and s.steps == 6000
    assert np.all(s.acceptance > 0) and np.all(s.acceptance < 1)
    assert s.round_trips > 0
    assert s.up_fraction[0] == 1.0 and s.up_fraction[-1] == 0.0
    assert np.all(s.up + s.down <= 2048 * len(range(0, 6000, DIAG_EVERY)))
    assert np.array_equal(pt.diagnostics(allreduce=False)["swap_acceptance"], s.acceptance)


@pytest.mark.gpu
def test_refusals():
    from riemann_b200 import ParameterError, PTSampler, Sampler
    from riemann_b200 import _lib
    from riemann_b200.models import benchmarks
    from riemann_b200.proposals.randomwalk import MetropolisRandomWalk
    from test_gpu_changepoint_tempering import _device_problem
    lib = _lib.load()
    s = Sampler(*_device_problem(), K=10)                                    # untempered changepoint sampler
    assert lib.rmn_sampler_cp_get_swap_stats(s._handle, None, None, None, None, None, None) == _lib.RMN_ERR_UNSUPPORTED
    gpt = PTSampler(benchmarks.benchmark_gauss2d_corr, MetropolisRandomWalk(0.5 * np.eye(2)), np.ones(2), K=16)
    with pytest.raises(ParameterError):
        gpt.swap_statistics()
    assert lib.rmn_sampler_cp_get_swap_stats(gpt._sampler._handle, None, None, None, None, None, None) == \
        _lib.RMN_ERR_UNSUPPORTED
    gpt.run(10, trace=False)
    assert "swap_acceptance" not in gpt.diagnostics(allreduce=False)
