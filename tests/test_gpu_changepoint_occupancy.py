"""
The changepoint T-step kernels' occupancy targets (riemann_b200/csrc/changepoint.cu, RMN_CP_MINBLOCKS_SLICED and
RMN_CP_MINBLOCKS).

* Resource check (CPU): every GL = 4 instantiation of the time-sliced kernel fits 96 registers per thread, so five blocks
  of 128 threads are resident per SM; ptxas spills at most one value there, live only before and after the T loop (an
  8 B frame).  The one-slice kernel keeps four blocks per SM (128 registers) and spills nothing: at 96 registers ptxas
  spills inside its T loop (the prefetched Philox words), and traced runs measured slower there (DESIGN.md 4.1).
* Pinned Philox states (GPU): two 24,576-chain runs (shared and per-chain move schedule) at chain_offset = 3 -- the
  schedule groups are unaligned and the launch is time-sliced -- must reproduce, bit for bit, the states,
  log-posteriors, per-chain moments and diagnostics block recorded with the 128-register kernel.  The runs are made
  time-sliced (the default) and as one slice: the diagnostics sums are added sample by sample in time order, so they
  do not depend on how the launch is sliced either.
* Data near the default shared-memory limit (GPU): the staged tables plus the kernels' static shared memory exceed
  48 KB, so the sampler must raise the kernels' dynamic shared-memory limit.
"""
import hashlib
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "riemann_b200", "libriemann_b200.so")
# (registers, bytes of local-memory frame): 65,536 registers per SM / (5 blocks x 128 threads) = 102, allocated in units
# of 8 per thread -> 96; 4 blocks -> 128
LIMITS = {"changepoint_sliced_kernel": (96, 8), "changepoint_kernel": (128, 0)}


def _resource_usage():
    txt = subprocess.run(["cuobjdump", "-res-usage", LIB], capture_output=True, text=True, check=True).stdout
    rows = re.findall(r"Function (\S+):\s*\n\s*REG:(\d+) STACK:(\d+)", txt)
    names = subprocess.run(["c++filt"] + [r[0] for r in rows], capture_output=True, text=True, check=True).stdout
    out = {}
    for name, (_, reg, stack) in zip(names.splitlines(), rows):
        m = re.search(r"(changepoint(?:_sliced)?_kernel<[^>]*>)", name)
        if m:
            out[m.group(1).replace(" ", "")] = (int(reg), int(stack))
    return out


def test_gl4_kernels_fit_their_occupancy_targets():
    if not os.path.exists(LIB) or shutil.which("cuobjdump") is None or shutil.which("c++filt") is None:
        pytest.skip("needs the built library, cuobjdump and c++filt")
    usage = _resource_usage()
    want = ["changepoint_sliced_kernel<%d,4,%s>" % (d, g) for d in (1, 2) for g in ("true", "false")]
    want += ["changepoint_kernel<false,%d,4,%s>" % (d, g) for d in (0, 1, 2) for g in ("true", "false")]
    want += ["changepoint_kernel<true,%d,4,true>" % d for d in (0, 1, 2)]
    missing = [k for k in want if k not in usage]
    assert not missing, (missing, sorted(usage))
    over = {k: usage[k] for k in want
            if usage[k][0] > LIMITS[k.split("<")[0]][0] or usage[k][1] > LIMITS[k.split("<")[0]][1]}
    assert not over, over


# SHA-256 of each result array, recorded on a B200 with the 128-register kernel (4 blocks per SM) launched as one slice:
# that kernel added each launch's diagnostics sums into the chain's entries at the end of every time slice, so only its
# one-slice launch sums them in time order.  Its states and log-posteriors were the same sliced or not.
PINNED = {
    "group": {
        "k": "30725632688153b673dc167cc4130474d2e2802a80b8e6511ca0eeee4d11e7b4",
        "cpx": "6489b4d1c072ff1e1dd70a3d0b5027175bb3bea60d85e7f93653fe52ce2c5700",
        "cpv": "d3d62acad862e96c7bf42704283ff716faa6ccd5c7eba16cd4c2d710d36ac7a3",
        "sig": "23a5b8c759224eca4637c282cb7c4df53fe9eb701046bd63a1cfa5763c90182a",
        "logpost": "0790bf39d5d62c76960c405e84c0934e719764c83a8a314c3d7219a33fb1df1e",
        "mean": "c0c5943e86538f996ed2d1270e66a1ca7005af5068832bfaca03703e4e756393",
        "var": "7bbb468c5a8cd5253a9580c2944bb3387786b0aac2e2d4ef0b38e05a7fbd895e",
        "diagnostics": "5e674a922df01d6e9a42a70ffb02522d0444564297c867a7704d331f475250ce",
    },
    "chain": {
        "k": "30371b2b6fa58a13e423386ebc1c8c71c93d52f1fea4c82a83722426806ecf3a",
        "cpx": "bd08127cbe4eba4ce81c5fffc72d86be26da04b3755d3b7dd2b99df2aa88e9e0",
        "cpv": "aca09569f540b0aa411b6dd93ecf8c86f2d5f5712a08e5592fc1d50b394bbff2",
        "sig": "fccb96e4aa0863c1eced9a8df3be7f1c06c2fe0f95d9a7d0f26a620e1ed69706",
        "logpost": "6b79e38fe0ef08a199b6c41caa48e12921cd40a78032f6287dc1f1ae46a9e814",
        "mean": "5392b6cc6876d0f81437b277bf8d24446f9d2744a9049c2b6aba88d8761c2389",
        "var": "7b9508dcf222a8c6849e87cd506ab946b8ce81e705e2693dbd7e40910cb4672f",
        "diagnostics": "872d5a4dfa6a17a51e60f702c1aa92c09f896e48327980e938800dcb9b5b0fb9",
    },
}


def _digest(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def pinned_run(schedule):
    """1,000 burn-in steps, a diagnostics reset, 400 steps; every result as a SHA-256 digest."""
    from oracle import riemann_port as port
    from riemann_b200 import Sampler
    from riemann_b200.models.changepoint import ChangepointParams, ChangepointRegression1D
    from riemann_b200.proposals.changepoint import ChangepointRegression1DProp
    pm, pp, _, _ = port.make_changepoint_problem()
    dm = ChangepointRegression1D(pm.x, pm.y, pm.xmin, pm.xmax, pm.lamb, int(pm.kmax), pm.alpha, pm.beta)
    dp = ChangepointRegression1DProp(dm, pp.hscale)
    s = Sampler(dm, dp, ChangepointParams([2.0], [1.0, 3.0], 0.1), K=24576, seed=17, chain_offset=3,
                move_schedule=schedule)
    s.run(1000, trace=False)
    s.reset_diagnostics()
    s.run(400, trace=False)
    (k, cpx, cpv, sig), lp = s._download_state()          # canonical padding: cpx beyond k, cpv beyond k + 1 are 0
    mean, var = s.chain_moments()
    blk = s.diagnostics_block().cpu().numpy()              # [K, samples, accepts, overflows, steps, 0, sums...]
    arrays = {"k": k, "cpx": cpx, "cpv": cpv, "sig": sig, "logpost": lp, "mean": mean, "var": var, "diagnostics": blk}
    return {n: _digest(a) for n, a in arrays.items()}, blk


@pytest.mark.gpu
@pytest.mark.parametrize("sliced", ["1", "0"])
@pytest.mark.parametrize("schedule", ["group", "chain"])
def test_pinned_philox_states_are_bit_identical(schedule, sliced, monkeypatch):
    monkeypatch.setenv("RMN_CP_SLICED", sliced)
    got, blk = pinned_run(schedule)
    assert blk[0] == 24576 and blk[4] == 400
    assert got == PINNED[schedule], {n: (got[n], PINNED[schedule].get(n)) for n in got if got[n] != PINNED[schedule].get(n)}


@pytest.mark.gpu
@pytest.mark.parametrize("gl", ["4", "8", "16"])
def test_data_near_the_default_shared_memory_limit(gl, monkeypatch):
    """M = 1,800 data points: the staged tables take 45,200 B of dynamic shared memory, which with the kernel's static
    shared memory exceeds the 48 KB a kernel may use without raising its limit.  One-slice and time-sliced runs must
    launch, and the carried log-posteriors must equal a fresh pointwise evaluation of the final states."""
    import torch
    from riemann_b200 import Sampler, _lib
    from riemann_b200.models.changepoint import ChangepointParams, ChangepointRegression1D
    from riemann_b200.proposals.changepoint import ChangepointRegression1DProp
    monkeypatch.setenv("RMN_CP_GL", gl)
    rng = np.random.default_rng(4)
    M = 1800
    x = np.sort(rng.uniform(0.0, 10.0, M))
    y = np.where(x < 4.0, 1.0, 3.0) + 0.3 * rng.standard_normal(M)
    dm = ChangepointRegression1D(x, y, 0.0, 10.0, 3.0, 10, 1.0, 1.0)
    dp = ChangepointRegression1DProp(dm, 1.0)
    for K in (64, 30000):                       # one wave (one-slice kernel); at GL = 4, 938 blocks (time-sliced)
        s = Sampler(dm, dp, ChangepointParams([5.0], [1.0, 3.0], 0.3), K=K, seed=2)
        s.run(240, trace=False)
        (k, cpx, cpv, sig), lp = s._download_state()
        assert np.all(np.isfinite(lp))
        dk, dx, dv, ds = (torch.as_tensor(a, device="cuda") for a in (k, cpx, cpv, sig))
        out = torch.empty(K, dtype=torch.float64, device="cuda")
        _lib.check(_lib.load().rmn_model_cp_logpost(dm._handle, 0, K, _lib.ptr(dk), _lib.ptr(dx), _lib.ptr(dv),
                                                    _lib.ptr(ds), _lib.ptr(out), _lib.stream_ptr()))
        assert np.allclose(out.cpu().numpy(), lp, rtol=1e-12, atol=1e-9)
