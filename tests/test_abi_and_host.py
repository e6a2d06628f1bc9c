"""
CPU: the C-ABI library loads and exports every symbol include/riemann_b200.h declares
(no compute calls), plus the host-side logic (sharding, diagnostics maths, error mapping,
the 2-rank gloo all-reduce of the diagnostics block).
"""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as g
    g.build()
    from riemann_b200 import _lib
    return _lib


def test_every_declared_symbol_is_exported_and_bound(lib):
    hdr = open(os.path.join(ROOT, "include", "riemann_b200.h")).read()
    declared = set(re.findall(r"\b(rmn_[a-z0-9_]+)\s*\(", hdr))
    assert len(declared) >= 30
    L = lib.load()
    for name in sorted(declared):
        assert hasattr(L, name), "library does not export %s" % name
    assert declared == set(lib.SIGNATURES), declared ^ set(lib.SIGNATURES)
    assert L.rmn_version() == 100


def test_every_entry_point_is_documented_with_the_interface_it_replaces():
    """INTEGRATION.md section 2 holds one row per exported function (reference file:line or `(absent)`)."""
    hdr = open(os.path.join(ROOT, "include", "riemann_b200.h")).read()
    doc = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    missing = [n for n in sorted(set(re.findall(r"\b(rmn_[a-z0-9_]+)\s*\(", hdr))) if n not in doc]
    assert not missing, missing


def test_c99_consumer_compiles_links_and_gets_error_codes(tmp_path, lib):
    """The boundary is a C ABI: a -std=c99 -pedantic translation unit includes the header, links the shared
    library and sees RMN_ERR_PARAM + a message for bad arguments (no GPU involved)."""
    lib.load()
    exe = str(tmp_path / "abi_consumer")
    libdir = os.path.join(ROOT, "riemann_b200")
    r = subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"),
                        os.path.join(ROOT, "tests", "c", "abi_consumer.c"), "-o", exe, "-L", libdir,
                        "-l:libriemann_b200.so", "-Wl,-rpath," + libdir], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and "abi consumer ok" in r.stdout, r.stdout + r.stderr


def test_library_carries_tcgen05_tma_and_dmma_sass(lib):
    """Static evidence that the tensor-core paths are native sm_100a code (mnemonics per the B200 profiling recipe):
    tcgen05.mma = UTC*MMA, tcgen05.ld = LDTM, TMA = UTMALDG in the GEMM object; fp64 DMMA in the dense / logistic ones."""
    lib.load()
    import __graft_entry__ as ge
    import shutil
    if shutil.which("cuobjdump") is None or not os.path.exists(os.path.join(ge.OBJ, "tc_gemm.o")):
        pytest.skip("needs cuobjdump and the build objects")

    def sass(obj):
        return subprocess.run(["cuobjdump", "-sass", os.path.join(ge.OBJ, obj)], capture_output=True, text=True).stdout
    tc = sass("tc_gemm.o")
    assert "sm_100a" in tc
    for mnemonic in ("UTCHMMA", "LDTM", "UTMALDG", "SYNCS"):
        assert mnemonic in tc, mnemonic
    assert "DMMA" in sass("dense.o") and "DMMA" in sass("logistic.o")


def test_header_constants_match_host_and_oracle(lib):
    from oracle import riemann_port as port
    hdr = open(os.path.join(ROOT, "include", "riemann_b200.h")).read()
    val = lambda n: int(re.search(r"#define %s (\d+)" % n, hdr).group(1))
    assert val("RMN_CP_LANES") == lib.CP_LANES
    assert val("RMN_CP_SLOT_XI") == lib.CP_SLOT["xi"] == port.CP_SLOT_XI
    assert val("RMN_CP_SLOT_ACC") == lib.CP_SLOT["acc"] == port.CP_SLOT_ACC
    assert val("RMN_CP_SLOT_N") == port.CP_SLOT_N and val("RMN_CP_SLOT_S") == port.CP_SLOT_S
    assert lib.CP_NSLOT == port.cp_nslot(lib.CP_LANES)
    assert val("RMN_SMALL_D_MAX") == lib.SMALL_D_MAX


def test_bad_arguments_return_param_error_without_a_gpu(lib):
    import ctypes as C
    from riemann_b200 import ParameterError
    L = lib.load()
    h = C.c_void_p()
    # L with a non-positive diagonal -> RMN_ERR_PARAM -> ParameterError (host-only check)
    bad = np.zeros((2, 2))
    rc = L.rmn_proposal_rw_create(C.byref(h), 2, lib.ptr(bad), 0, 0.25)
    assert rc == lib.RMN_ERR_PARAM
    with pytest.raises(ParameterError):
        lib.check(rc)
    assert b"Cholesky" in L.rmn_last_error()
    assert L.rmn_proposal_hmc_create(C.byref(h), 2, -1.0, 1, None, None, None, 0, 0.75) == lib.RMN_ERR_PARAM
    assert L.rmn_proposal_mmala_create(C.byref(h), 0, 0.1) == lib.RMN_ERR_PARAM
    assert L.rmn_proposal_changepoint_create(C.byref(h), 2.0, None) == lib.RMN_OK
    assert L.rmn_proposal_destroy(h) == lib.RMN_OK
    # pooled covariance adaptation (SURVEY 8f N5): dense path only, sane schedule -- all host-side checks
    h12, h2 = C.c_void_p(), C.c_void_p()
    assert L.rmn_proposal_rw_create(C.byref(h12), 12, lib.ptr(np.eye(12)), 0, 0.25) == lib.RMN_OK
    assert L.rmn_proposal_rw_set_pooled_cov_adapt(h12, 0, 0.5, 1e-10, 0) == lib.RMN_ERR_PARAM          # t_adapt < 1
    assert L.rmn_proposal_rw_set_pooled_cov_adapt(h12, 10, -1.0, 1e-10, 0) == lib.RMN_ERR_PARAM        # sd <= 0
    assert L.rmn_proposal_rw_set_pooled_cov_adapt(h12, 10, 0.5, 1e-10, 0) == lib.RMN_OK
    assert L.rmn_proposal_rw_create(C.byref(h2), 2, lib.ptr(np.eye(2)), 0, 0.25) == lib.RMN_OK
    assert L.rmn_proposal_rw_set_pooled_cov_adapt(h2, 10, 0.5, 1e-10, 0) == lib.RMN_ERR_PARAM          # small-d path
    assert b"dense path" in L.rmn_last_error()
    assert L.rmn_proposal_destroy(h12) == lib.RMN_OK and L.rmn_proposal_destroy(h2) == lib.RMN_OK
    from riemann_b200.proposals.randomwalk import PooledAdaptCovRandomWalk
    with pytest.raises(ParameterError):
        PooledAdaptCovRandomWalk(np.eye(12), t_adapt=0)
    p = PooledAdaptCovRandomWalk(np.eye(12), t_adapt=50, stop_after=1000, adapt_scale=True)
    assert p._pooled_cov and p._adaptive and p.target_accept_rate == 0.25 and p.L.shape == (12, 12)


_NO_DEVICE = r"""
import sys, numpy as np
sys.path.insert(0, sys.argv[1])
from riemann_b200.models.gaussian import MultiGaussianDist
try:
    MultiGaussianDist(np.zeros(2), np.eye(2))
except RuntimeError as e:
    print(e)
"""


def test_no_cpu_fallback(lib):
    """Without a visible CUDA device (hidden from a child process, so this runs on a GPU machine too) the host classes
    refuse to work instead of computing on the CPU."""
    r = subprocess.run([sys.executable, "-c", _NO_DEVICE, ROOT], capture_output=True, text=True, timeout=240,
                       env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 0, r.stdout + r.stderr
    assert "no CPU fallback" in r.stdout, r.stdout + r.stderr


def test_product_never_imports_oracle():
    for dirpath, _, files in os.walk(os.path.join(ROOT, "riemann_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle", src, re.M), f


def test_grad_stand_in_refuses_arbitrary_callables():
    """riemann_b200.grad (for examples/riemann_ex1.py:237) only binds device-model methods."""
    from riemann_b200 import ParameterError, grad
    with pytest.raises(ParameterError):
        grad(lambda th: -0.5 * np.sum(th ** 2))
    with pytest.raises(ParameterError):
        grad(np.sum)


def test_bench_engine_arm_never_imports_oracle():
    """bench.py may execute oracle/ only in its CPU legs (cpu_baseline and --impl reference share _cpu_worker;
    cpu_kind asks refshim whether the staged reference copy is present)."""
    import ast
    tree = ast.parse(open(os.path.join(ROOT, "bench.py")).read())
    where = []
    for fn in ast.walk(tree):
        if isinstance(fn, (ast.FunctionDef, ast.Module)):
            for node in ast.iter_child_nodes(fn) if isinstance(fn, ast.Module) else ast.walk(fn):
                mods = ([a.name for a in node.names] if isinstance(node, ast.Import)
                        else [node.module or ""] if isinstance(node, ast.ImportFrom) else [])
                if any(m.split(".")[0] == "oracle" for m in mods):
                    where.append(getattr(fn, "name", "<module>"))
    assert where and set(where) <= {"_cpu_worker", "cpu_kind"} and "_cpu_worker" in where, where
    # the synthetic inputs both arms use come from one neutral numpy module
    from oracle import riemann_port as port
    from riemann_b200 import synthetic
    pm = port.make_changepoint_problem()[0]
    c = synthetic.changepoint_problem()
    assert np.array_equal(pm.x, c["x"]) and np.array_equal(pm.y, c["y"])


def test_shard_chains():
    from riemann_b200.distributed import shard_chains
    for K, G in [(65536, 8), (10, 3), (7, 8), (16384, 4)]:
        parts = [shard_chains(K, r, G) for r in range(G)]
        assert sum(k for _, k in parts) == K
        off = 0
        for o, k in parts:
            assert o == off
            off += k


def test_summarize_block_matches_oracle_estimator():
    from oracle import ess
    from riemann_b200.distributed import summarize_block
    rng = np.random.default_rng(1)
    K, n, d, phi = 300, 2000, 3, 0.7
    x = np.zeros((n, K, d))
    x[0] = rng.standard_normal((K, d))
    for t in range(1, n):
        x[t] = phi * x[t - 1] + np.sqrt(1 - phi ** 2) * rng.standard_normal((K, d))
    m = x.mean(0)
    v = x.var(0)
    blk = np.concatenate([[K, n, 0.3 * K * n, 0, n, 0], m.sum(0), (m * m).sum(0), v.sum(0)])
    out = summarize_block(blk)
    ess_o, tau_o, rhat_o = ess.ess_from_chain_moments(n, m, x.var(0, ddof=1))
    assert np.allclose(out["tau"], tau_o, rtol=1e-9)
    assert np.allclose(out["ess"], ess_o, rtol=1e-9)
    assert np.allclose(out["rhat"], rhat_o, rtol=1e-9)
    assert abs(out["accept_rate"] - 0.3) < 1e-12
    assert np.all(np.abs(out["tau"] - (1 + phi) / (1 - phi)) < 1.5)


_GLOO = r"""
import os, sys, numpy as np, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from riemann_b200.distributed import reduce_block, shard_chains, summarize_block
dist.init_process_group("gloo")
r, w = dist.get_rank(), dist.get_world_size()
K_total, n, nd = 10, 50, 2
off, k = shard_chains(K_total)
rng = np.random.default_rng(0)
m = rng.standard_normal((K_total, nd)); v = rng.uniform(0.5, 1.5, (K_total, nd))
mine = slice(off, off + k)
blk = np.concatenate([[k, n, 7.0 * k, 0, n, 0], m[mine].sum(0), (m[mine]**2).sum(0), v[mine].sum(0)])
out = reduce_block(torch.tensor(blk))
full = np.concatenate([[K_total, n, 7.0 * K_total, 0, n, 0], m.sum(0), (m**2).sum(0), v.sum(0)])
assert np.allclose(out.numpy(), full), (out.numpy(), full)
s = summarize_block(out.numpy())
assert s["chains"] == K_total and s["steps"] == n
dist.barrier(); dist.destroy_process_group()
print("rank", r, "ok")
"""


def test_diagnostics_allreduce_two_ranks_gloo(tmp_path):
    script = tmp_path / "gloo_worker.py"
    script.write_text(_GLOO)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1",
                        "--nproc-per-node=2", "--master-addr", "127.0.0.1", "--master-port", "29617",
                        str(script), ROOT], capture_output=True, text=True, timeout=240, env=env)
    assert r.returncode == 0, r.stdout + r.stderr
    assert r.stdout.count("ok") == 2


def _expected_cpu_kind():
    """The CPU arm times the unmodified reference package where its copy is staged (oracle/build_ref.py), and otherwise
    the numpy port (oracle/riemann_port.py, pinned to the reference by tests/golden/*.npz); the line must say which."""
    from oracle import refshim
    return "reference" if refshim.reference_available() else "port"


def test_reference_arm_under_torchrun_prints_one_line():
    """`bench.py --impl reference --gpus N` launches like the engine arm (torchrun, one process per GPU):
    rank 0 alone runs the CPU sampler and prints the line, the other ranks exit 0 without work and without output."""
    import json
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29633", os.path.join(ROOT, "bench.py"),
                        "--impl", "reference", "--gpus", "2", "--steps", "2", "--warmup", "1",
                        "--cpu-seconds-reference", "1.5", "--workload", "gauss2d_rw"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT, env=dict(os.environ, MASTER_ADDR="127.0.0.1"))
    assert r.returncode == 0, r.stdout + r.stderr
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["n_gpus"] == 2 and d["steps"] == 2 and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == _expected_cpu_kind() and d["e2e"]["h2d_bytes_per_step"] == 0 and d["gpu_launches"] == 0


def test_sokal_tau_matches_ar1_and_oracle():
    """riemann_b200.diagnostics (emcee-style integrated autocorrelation time) on AR(1) chains with the
    analytic tau = (1 + phi) / (1 - phi), against oracle/ess.py, and against the engine's moment-based
    many-chain estimator (summarize_block)."""
    from oracle import ess as oess
    from riemann_b200 import diagnostics as dg
    from riemann_b200.distributed import summarize_block
    rng = np.random.default_rng(0)
    N, K = 4000, 256
    for phi in (0.5, 0.9):
        e = rng.standard_normal((N + 500, K)) * np.sqrt(1 - phi * phi)
        x = np.zeros_like(e)
        for t in range(1, len(e)):
            x[t] = phi * x[t - 1] + e[t]
        x = x[500:]
        want = (1 + phi) / (1 - phi)
        tau_multi = dg.integrated_time_chains(x)[0]
        assert abs(tau_multi / want - 1) < 0.05
        one = dg.integrated_time(x[:, 0])[0]
        assert abs(one - oess.integrated_time(x[:, 0])[0]) < 1e-9             # same algorithm as the oracle
        assert abs(tau_multi - oess.integrated_time_multi(x[:, :, None])[0]) < 1e-9
        # the moment-based estimator of the diagnostics block on the same chains
        m, v = x.mean(0), x.var(0)
        blk = np.array([K, N, 0, 0, N, 0, m.sum(), (m * m).sum(), v.sum()])
        assert abs(summarize_block(blk)["tau"][0] / want - 1) < 0.25
        assert abs(dg.effective_sample_size(x)[0] / (N * K / want) - 1) < 0.05


def test_bench_line_contract():
    """The JSON line bench.py printed on a B200 in round 1 (tests/golden/bench_line_changepoint_r1.json,
    gpurun r60) against the measurement contract: every required key, its type and the internal consistency
    of the numbers.  bench.py's static tables must cover every workload it offers."""
    import importlib.util
    import json
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    with open(os.path.join(root, "tests", "golden", "bench_line_changepoint_r1.json")) as f:
        d = json.load(f)
    for k, t in (("metric", str), ("value", float), ("unit", str), ("n_gpus", int), ("steps", int), ("warmup", int),
                 ("ms_per_step", float), ("higher_is_better", bool), ("scaling", str), ("dtype", str), ("data", str),
                 ("config", dict), ("e2e", dict), ("gpu_launches", int), ("roofline", dict), ("cpu_baseline", dict),
                 ("clocks", dict)):
        assert isinstance(d[k], t), k
    assert d["vs_baseline"] is None and d["warmup"] >= 3 and d["gpu_launches"] > 0
    assert "workload" in d["config"] and "model" not in d["config"]
    for k in ("value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"):
        assert k in d["e2e"]
    assert d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0 and d["e2e"]["value"] != d["value"]
    r = d["roofline"]
    for k in ("bound", "achieved", "peak", "unit", "frac", "traffic", "kernel", "kernel_share_of_step"):
        assert k in r
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-12
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["value"] > 0 and cb["sample"]
    assert set(d["clocks"]) >= {"sm_mhz", "sm_max_mhz", "reasons"}
    K, T = d["config"]["chains_total"], d["config"]["iters_per_step"]
    assert abs(d["value"] - K * T / (d["ms_per_step"] * 1e-3)) < 1e-6 * d["value"]
    spec = importlib.util.spec_from_file_location("_bench", os.path.join(root, "bench.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    assert set(b.CHAINS_PER_GPU) == set(b.ALGO_FLOP)
    assert b.METRIC == d["metric"] and b.UNIT == d["unit"]


def test_bench_line_contract_round2():
    """The line the default `bench.py` invocation printed on a B200 in round 2 (tests/golden/bench_line_r2.json, gpurun
    r2by): the headline keys of the contract, the `configs` array with every BASELINE config at its own sharding, the
    ESS phase, and the consistency of each entry's numbers."""
    import importlib.util
    import json
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    with open(os.path.join(root, "tests", "golden", "bench_line_r2.json")) as f:
        d = json.load(f)
    spec = importlib.util.spec_from_file_location("_bench", os.path.join(root, "bench.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    assert d["metric"] == b.METRIC and d["unit"] == b.UNIT and d["vs_baseline"] is None and d["scaling"] == "weak"
    assert d["roofline"]["traffic"] is None and "profiled" in d["roofline"]          # static ncu numbers only under `profiled`
    assert d["roofline"]["algo_flop_per_chain_step"] == 350.0 and d["roofline"]["algo_compares_per_chain_step"] == 300.0
    assert d["cpu_baseline"]["kind"] == "reference"
    e = d["ess"]
    assert e["max_rhat"] < 1.05 and e["window_over_tau"] > 10 and d["min_ess_per_sec"] == e["min_ess_per_sec"] > 0
    assert len(e["tau_steps"]) == len(e["functionals"]) == 8
    keys = [c["key"] for c in d["configs"]]
    assert keys == [k for k, *_ in b.SUBCONFIGS]
    for c in d["configs"]:
        assert "error" not in c, c
        for k in ("value", "e2e", "dtype", "roofline", "diagnostics", "clocks", "cpu_baseline", "scaling", "ms_per_step"):
            assert k in c, (c["key"], k)
        T, K, steps = c["config"]["iters_per_step"], c["config"]["chains_total"], c["steps"]
        assert abs(c["value"] - K * T / (c["ms_per_step"] * 1e-3)) < 1e-6 * c["value"]
        assert c["e2e"]["h2d_bytes_per_step"] > 0 and c["e2e"]["value"] != c["value"]
        r = c["roofline"]
        assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-12 and r["kernel_launches"] > 0 and "timed_in" in r
    tot = {c["key"]: c["config"]["chains_total"] for c in d["configs"]}
    assert tot["gauss1000_mala_f64"] == tot["gauss1000_mala_tf32x3"] == 16384          # BASELINE.json's own chain counts
    assert tot["logistic_mala_f64"] == 8192 and tot["logistic_mmala_tf32x3"] == 4096 and tot["gauss2d_rw_k1"] == 1


def test_reference_arm_chains_continue_across_steps():
    """bench.py --impl reference: every core's chain of the UNMODIFIED reference runs through warm-up and timed segments
    without restarting, so the tau / ESS window is the whole timed region -- the window is the sum of the timed
    segments' steps, and the per-step throughputs average to the line's value."""
    import importlib
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    if root not in sys.path:
        sys.path.insert(0, root)
    b = importlib.import_module("bench")              # by its real name: the spawned workers unpickle bench._cpu_worker
    vals, cb = b.cpu_reference_segments("gauss2d_rw", 1, 3, 0.4, cores=2)
    assert cb["kind"] == _expected_cpu_kind() and cb["cores"] == 2 and len(vals) == 3 and all(v > 0 for v in vals)
    e = cb["ess"]
    assert e["chains"] == 2 and e["steps_per_chain"] >= 3 * 2000          # three timed segments of whole 2,000-step chunks
    assert min(vals) <= cb["value"] <= max(vals)
    assert "3 timed segments" in cb["sample"] and "after 1 untimed" in cb["sample"]
    assert ("min_ess_per_sec" in cb) and (cb["min_ess_per_sec"] is not None or "min_ess_per_sec_unreliable" in cb)


def test_split_rhat_sees_a_common_drift():
    """summarize_split: chains that all drift the same way have R-hat ~ 1 over the whole window (every chain mean
    is the same) but split-R-hat > 1; stationary AR(1) chains give ~1 and the right tau either way."""
    from riemann_b200.distributed import summarize_block, summarize_split
    rng = np.random.default_rng(3)
    K, n, phi = 512, 2000, 0.8

    def block(x):
        m, v = x.mean(0), x.var(0)
        return np.array([x.shape[1], x.shape[0], 0, 0, x.shape[0], 0, m.sum(), (m * m).sum(), v.sum()])

    e = rng.standard_normal((n + 200, K)) * np.sqrt(1 - phi * phi)
    x = np.zeros_like(e)
    for t in range(1, len(e)):
        x[t] = phi * x[t - 1] + e[t]
    x = x[200:]
    s = summarize_split(block(x[:n // 2]), block(x[n // 2:]))
    assert s["chains"] == 2 * K and abs(s["rhat"][0] - 1) < 0.01
    assert abs(s["tau"][0] / ((1 + phi) / (1 - phi)) - 1) < 0.2
    drift = x + np.linspace(-1.0, 1.0, n)[:, None]                 # every chain drifts alike
    whole = summarize_block(block(drift))
    split = summarize_split(block(drift[:n // 2]), block(drift[n // 2:]))
    assert abs(whole["rhat"][0] - 1) < 0.01 and split["rhat"][0] > 1.1
    with pytest.raises(ValueError):
        summarize_split(block(x[:100]), block(x[:200]))


_ROW_SCRIPT = r"""
import os, sys, ctypes, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from riemann_b200.distributed import exchange_unique_id, shard_rows
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
calls = []
def fake_id(buf, n):
    calls.append(n)
    ctypes.memmove(buf, bytes(range(128)), 128)
uid = exchange_unique_id(fake_id)
assert uid.raw == bytes(range(128)), "rank %d got a different id" % rank
assert len(calls) == (1 if rank == 0 else 0)          # only rank 0 asks NCCL for an id
off, n = shard_rows(1001)
assert (off, n) == ((0, 501) if rank == 0 else (501, 500))
print("rank %d ok" % rank, flush=True)
dist.destroy_process_group()
"""


def test_row_shard_host_logic_two_ranks_gloo(tmp_path):
    """The host side of the row-sharded data mode: one NCCL unique id reaches every rank, rows split contiguously."""
    script = tmp_path / "rows.py"
    script.write_text(_ROW_SCRIPT)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", "29544", str(script), ROOT],
                       capture_output=True, text=True, timeout=240, env=env)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "rank 0 ok" in r.stdout and "rank 1 ok" in r.stdout
