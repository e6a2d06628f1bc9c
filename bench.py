#!/usr/bin/env python
"""
bench.py -- MH chain-steps/sec and min-ESS/sec of the B200 engine on BASELINE.json's metric, next to the
CPU sampler timed on the same box.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
                    [--workload NAME [--precision P] [--chains C] [--iters T]] [--no-configs] [--no-cpu]

The line printed by the default invocation (the one the driver runs):

* headline = BASELINE.json configs[1]: the changepoint model of examples/test_changepoint.py, 4-way
  RW/birth/death Metropolis proposal, 65,536 chains per GPU (weak scaling).  One bench "step" = one launch of the
  hot path: T MH iterations of every chain (`--iters`, default 1000), device-resident.  `value` is device-timed
  with the state resident, `e2e` goes through the public API with host buffers.
* `configs` = one entry per remaining BASELINE config AT BASELINE'S OWN SHARDING (fixed total chain counts split
  over the N GPUs = strong scaling): gauss2d_rw (K = 1 latency as examples/test_randomwalk.py:39-40 runs it, and
  2^20 chains per GPU), gauss1000_mala (16,384 chains / N; f64 and tf32x3), logistic_mala (8,192 / N; f64 and
  tf32x3), logistic_mmala (4,096 / N; f64 and tf32x3).  Every entry carries value, e2e, dtype, a live roofline of
  its dominant kernel, diagnostics and (N = 1 only) a short CPU leg.
* `ess` (changepoint): min-ESS/sec as a MEASUREMENT -- a separate device-timed phase whose two half-windows are
  long enough for the slowest tracked functional (window_over_tau, split-R-hat < 1.05 required, else null with
  the reason), plus the Sokal-window estimator of examples/test_randomwalk.py:42 on a traced subset, the same
  estimator the CPU arm applies to its chains.
* `multi_gpu_checks` (N >= 2): chain-shard invariance of the Philox streams at N ranks (bitwise) and the
  row-sharded data mode replaying the reference-stream fixtures with the rows split over the N ranks.

`--workload NAME` prints the line of that single workload (profiling, DESIGN.md tables).

`--dump-outputs DIR` writes what the headline workload's last timed step computed (`dump_outputs`) as float64 .npy
files, so that two builds can be compared output for output: inputs, seeds and step counts depend on the arguments only.

Timing: W untimed warm-up steps, then K steps each bracketed by CUDA events on the launching stream, L2 flushed
(256 MiB write) between steps outside the event pairs, barrier + synchronize on both sides, MAX over ranks.
`roofline.achieved` is the algorithmic work of the timed region divided by the DOMINANT kernel's own time in it
(CUDA events around each of its launches, rmn_sampler_kernel_timing).

CPU arm (`--impl reference`, and `cpu_baseline` at N = 1): the UNMODIFIED reference sampler
(riemann/samplers/sampler.py:44-90, staged by oracle/build_ref.py under oracle/_ref/, imported through
oracle/refshim.py) for configs 1-3, `kind: "reference"`; the numpy port (oracle/riemann_port.py) for the two
models the reference does not contain (logistic regression: configs 4, 5), `kind: "port"`.  One chain per host core.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "mh_chain_steps_per_sec"
UNIT = "chain-steps/s"
SEED = 20261018
CHAINS_PER_GPU = {"changepoint": 65536, "gauss2d_rw": 1 << 20, "gauss1000_mala": 16384,
                  "logistic_mala": 1024, "logistic_mmala": 512, "gauss2d_pt": 5 * (1 << 17)}
# BASELINE.json's own chain counts ("16,384 chains sharded over 1/2/4/8", "8,192 chains over 8", "4,096 chains")
CHAINS_TOTAL = {"gauss1000_mala": 16384, "logistic_mala": 8192, "logistic_mmala": 4096}
ITERS = {"changepoint": 1000, "gauss2d_rw": 2000, "gauss1000_mala": 20, "logistic_mala": 2, "logistic_mmala": 2,
         "gauss2d_pt": 2000}
# SURVEY.md section 8d: algorithmic work per chain-step.  changepoint: 350 flop (+ 300 compares, reported
# separately as `algo_compares_per_chain_step`, not counted as flop).
ALGO_FLOP = {"changepoint": 350.0, "gauss2d_rw": 40.0, "gauss1000_mala": 2.0e6,
             "logistic_mala": 4.0e8, "logistic_mmala": 4.4e8, "gauss2d_pt": 40.0}
ALGO_COMPARES = {"changepoint": 300.0}

# The `configs` array of the default line: (key, workload, precision, sharding, iters/step); each is timed over --steps.
#   sharding "strong": BASELINE's total chain count split over the ranks; "weak": per-GPU count; "replica": K = 1.
SUBCONFIGS = [
    ("gauss2d_rw_k1", "gauss2d_rw", "f64", "replica", 10000),
    ("gauss2d_rw", "gauss2d_rw", "f64", "weak", 2000),
    ("gauss1000_mala_f64", "gauss1000_mala", "f64", "strong", 20),
    ("gauss1000_mala_tf32x3", "gauss1000_mala", "tf32x3", "strong", 20),
    ("logistic_mala_f64", "logistic_mala", "f64", "strong", 2),
    ("logistic_mala_tf32x3", "logistic_mala", "tf32x3", "strong", 4),
    ("logistic_mmala_f64", "logistic_mmala", "f64", "strong", 2),
    ("logistic_mmala_tf32x3", "logistic_mmala", "tf32x3", "strong", 4),
]

# From the committed ncu captures (`ncu --set full`, one launch of the dominant kernel): DRAM bytes per launch and
# pipe/issue utilisation.  STATIC evidence, reported under roofline.profiled only -- the live numbers of a run are
# `value`, `ms_per_step`, `roofline.achieved`.
PROFILED_FILE = os.path.join(ROOT, "profiles", "profiled_kernels.json")


def load_profiled():
    try:
        with open(PROFILED_FILE) as f:
            return json.load(f)
    except Exception:
        return {}


def load_peaks():
    """MEASURED_PEAKS.json (driver-written: HBM copy GB/s, bf16 cuBLAS TF/s) plus the figures it does
    not carry, measured here with the same method by scripts/peaks/measure_peaks.py and committed as
    profiles/measured_peaks_extra.json (fp64 DFMA / DMMA, TF32 cuBLAS).  Fallbacks are B200_PROFILING.md's."""
    d, src = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "sm_max_mhz": 1965.0}, "fallback"
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        src = "measured"
    x = os.path.join(ROOT, "profiles", "measured_peaks_extra.json")
    if os.path.exists(x):
        with open(x) as f:
            d["extra"] = json.load(f)
    return d, src


# ----------------------------------------------------------------------------
# CPU arm: the unmodified reference (oracle/_ref via refshim) or the numpy port, one chain per core
# ----------------------------------------------------------------------------
def cpu_kind(workload):
    """'reference' where the reference contains the model and its staged copy is present, else 'port'."""
    if workload in ("changepoint", "gauss2d_rw", "gauss1000_mala"):
        from oracle import refshim
        if refshim.reference_available():
            return "reference"
    return "port"


def _cp_functionals(thetas, xq):
    """sigma, k, y_hat(x_q) (changepoint.py:175-181) of a list of ChangepointParams -> [n, 2 + len(xq)]."""
    out = np.empty((len(thetas), 2 + len(xq)))
    for i, th in enumerate(thetas):
        cpx = np.atleast_1d(np.asarray(th.cpx, dtype=np.float64))
        cpv = np.atleast_1d(np.asarray(th.cpv, dtype=np.float64))
        out[i, 0] = float(np.squeeze(th.sig))
        out[i, 1] = len(cpx)
        out[i, 2:] = cpv[np.searchsorted(cpx, xq)]
    return out


def _vec_functionals(thetas):
    th = np.asarray(thetas, dtype=np.float64).reshape(len(thetas), -1)
    if th.shape[1] <= 8:
        return th
    return np.concatenate([th[:, :7], th.mean(axis=1, keepdims=True)], axis=1)


def _cpu_worker(args):
    workload, seed, budget_s, kind = args
    os.environ["OPENBLAS_NUM_THREADS"] = "1"
    os.environ["OMP_NUM_THREADS"] = "1"
    import numpy as np
    from riemann_b200 import synthetic
    np.random.seed(seed)
    quiet = None
    if kind == "reference":
        from oracle import refshim
        R = refshim.load_reference()
        quiet = refshim.quiet
        if workload == "changepoint":
            c = synthetic.changepoint_problem()
            model = R.ChangepointRegression1D(c["x"], c["y"], c["xmin"], c["xmax"], c["lamb"], c["kmax"],
                                              c["alpha"], c["beta"])
            prop = R.ChangepointRegression1DProp(model, c["hscale"])
            th0 = R.ChangepointParams(np.array(c["theta0"][0]), np.array(c["theta0"][1]), c["theta0"][2])
            chunk = 500
        elif workload == "gauss2d_rw":
            model = R.benchmarks.benchmark_gauss2d_corr
            prop = R.MetropolisRandomWalk(0.5 * np.eye(2))
            th0 = np.ones(2)
            chunk = 2000
        else:
            model = R.MultiGaussianDist(np.zeros(1000), 0.1 * np.eye(1000) + 0.9 * np.ones((1000, 1000)))
            prop = R.VanillaHMC(0.08, 1, model.grad_log_likelihood)         # = MALA (hamiltonian.py:55-91)
            th0 = np.zeros(1000)
            chunk = 2
        s = R.Sampler(model, prop, th0)
    else:
        from oracle import riemann_port as port
        if workload == "changepoint":
            model, prop, th0, _ = port.make_changepoint_problem()
            chunk = 500
        elif workload == "gauss2d_rw":
            model, prop, th0, chunk = port.benchmark_gauss(2), port.MetropolisRandomWalk(0.5 * np.eye(2)), np.ones(2), 2000
        elif workload == "gauss1000_mala":
            model = port.benchmark_gauss(1000)
            prop, th0, chunk = port.MALA(0.08, model.grad_log_likelihood), np.zeros(1000), 5
        else:
            N, d = (100000, 64) if workload == "logistic_mmala" else (1000000, 100)
            X, y, ts, pv = port.make_logistic_problem(N, d)
            model = port.LogisticRegression(X, y, pv)
            prop = (port.SimplifiedMMALA(0.5, model) if workload == "logistic_mmala"
                    else port.MALA(0.02, model.grad_log_posterior))
            th0, chunk = ts.copy(), 1
        s = port.Sampler(model, prop, th0)
    xq = None
    if workload == "changepoint":
        c = synthetic.changepoint_problem()
        xq = c["xmin"] + (c["xmax"] - c["xmin"]) * (np.arange(6) + 0.5) / 6.0
    import contextlib
    segments = []                                          # the chain CONTINUES from one segment into the next
    with np.errstate(all="ignore"), (quiet() if quiet else contextlib.nullcontext()):
        for seg_s in (budget_s if isinstance(budget_s, (list, tuple)) else [budget_s]):
            n, spent, funcs = 0, 0.0, []
            while spent < seg_s:
                t0 = time.perf_counter()
                s.run(chunk)                               # Sampler.run (sampler.py:44-54): chunk x Sampler.sample
                spent += time.perf_counter() - t0
                n += chunk
                new = s._chain_thetas[1:]                  # run() keeps [last state] + the chunk
                funcs.append(_cp_functionals(new, xq) if xq is not None else _vec_functionals(new))
            segments.append((n, spent, np.concatenate(funcs, axis=0)))
    return segments if isinstance(budget_s, (list, tuple)) else segments[0]


def chain_ess(funcs_list, wall, names):
    """Sokal-window tau (emcee's estimator, examples/test_randomwalk.py:42; riemann_b200/diagnostics.py) with the
    chains as walkers, and the moment-based tau = n B / W, of traced chains [n, chains, nf]."""
    from riemann_b200 import diagnostics as dgn
    n = min(f.shape[0] for f in funcs_list)
    if n < 64:
        return {"min_ess_per_sec": None, "reason": "only %d steps per chain in the sample" % n}
    x = np.stack([f[:n] for f in funcs_list], axis=1)                  # [n, chains, nf]
    with np.errstate(all="ignore"):
        tau = dgn.integrated_time_chains(x)
        m, v = x.mean(axis=0), x.var(axis=0, ddof=1)
        B, W = m.var(axis=0, ddof=1) if x.shape[1] > 1 else np.full(x.shape[2], np.nan), v.mean(axis=0)
        tau_m = n * B / W
    tmax = float(np.nanmax(tau))
    chains = x.shape[1]
    out = {"estimator": "Sokal window (c = 5), ACF averaged over the chains; tau in MH steps",
           "functionals": names, "sokal_tau_steps": [float(t) for t in tau],
           "moment_tau_steps": [float(t) for t in tau_m], "steps_per_chain": int(n), "chains": int(chains),
           "window_over_tau": n / tmax, "reliable": bool(n >= 50 * tmax),
           "min_ess": chains * n / tmax, "min_ess_per_sec": chains * n / tmax / wall}
    if chains > 1 and np.all(np.isfinite(tau_m)):
        # the GPU arm's `ess` estimator (tau = n B / W over the chains) on these few chains: B has chains - 1 degrees
        # of freedom, so this is a noisy figure (relative error ~ sqrt(2 / (chains - 1)))
        out["moment_min_ess_per_sec"] = chains * n / max(float(np.max(tau_m)), 1.0) / wall
    if not out["reliable"]:
        out["reason"] = "chain length is %.1f tau of the slowest functional (< 50 tau: emcee would refuse)" % (n / tmax)
    return out


FUNC_NAMES = {"changepoint": ["sigma", "k"] + ["yhat(xq%d)" % q for q in range(6)],
              "gauss2d_rw": ["theta0", "theta1"]}


def cpu_baseline(workload, budget_s=12.0, cores=None, with_ess=True):
    import multiprocessing as mp
    cores = cores or len(os.sched_getaffinity(0))
    if workload.startswith("logistic"):
        cores = min(cores, 16)                           # every worker builds its own copy of X (0.8 GB at config 4)
    kind = cpu_kind(workload)
    ctx = mp.get_context("spawn")
    with ctx.Pool(cores) as pool:
        res = pool.map(_cpu_worker, [(workload, 1000 + i, budget_s, kind) for i in range(cores)])
    steps = sum(r[0] for r in res)
    wall = max(r[1] for r in res)
    what = ("the UNMODIFIED reference (riemann/samplers/sampler.py:44-90 via oracle/refshim.py)" if kind == "reference"
            else "the numpy restatement of riemann's Sampler.sample (oracle/riemann_port.py; the reference has no such model)")
    out = {"value": steps / wall, "unit": UNIT, "cores": cores, "kind": kind,
           "sample": "%d independent chains (one per host core) of %s on the same synthetic %s problem, %.1f s each, "
                     "%d chain-steps total" % (cores, what, workload, budget_s, steps)}
    if with_ess:
        _attach_ess(out, workload, [r[2] for r in res], wall)
    return out


def _attach_ess(out, workload, funcs_list, wall):
    names = FUNC_NAMES.get(workload, ["theta%d" % j for j in range(7)] + ["mean(theta)"])
    e = chain_ess(funcs_list, wall, names[:funcs_list[0].shape[1]])
    out["ess"] = e
    out["min_ess_per_sec"] = e.get("min_ess_per_sec") if e.get("reliable") else None
    if out["min_ess_per_sec"] is None:
        out["min_ess_per_sec_unreliable"] = e.get("min_ess_per_sec")


def cpu_reference_segments(workload, warm, timed, per_s, cores=None):
    """The reference arm's timed region: every host core runs ONE chain through `warm` untimed and `timed` timed
    segments of `per_s` seconds, the chain continuing from segment to segment (the warm-up segments are its burn-in).
    Returns (per-segment chain-steps/s, cpu_baseline dict): throughput per segment = chain-steps of all chains / the
    slowest chain's time in it; tau / ESS from the concatenated timed segments of every chain."""
    import multiprocessing as mp
    cores = cores or len(os.sched_getaffinity(0))
    if workload.startswith("logistic"):
        cores = min(cores, 16)
    kind = cpu_kind(workload)
    ctx = mp.get_context("spawn")
    with ctx.Pool(cores) as pool:
        res = pool.map(_cpu_worker, [(workload, 1000 + i, [per_s] * (warm + timed), kind) for i in range(cores)])
    vals, walls, steps = [], [], 0
    for g in range(warm, warm + timed):
        n = sum(r[g][0] for r in res)
        w = max(r[g][1] for r in res)
        vals.append(n / w)
        walls.append(w)
        steps += n
    wall = float(sum(walls))
    what = ("the UNMODIFIED reference (riemann/samplers/sampler.py:44-90 via oracle/refshim.py)" if kind == "reference"
            else "the numpy restatement of riemann's Sampler.sample (oracle/riemann_port.py; the reference has no such model)")
    out = {"value": steps / wall, "unit": UNIT, "cores": cores, "kind": kind,
           "sample": "%d independent chains (one per host core) of %s on the same synthetic %s problem: %d timed "
                     "segments of %.1f s after %d untimed ones, each chain continuing across segments; %d chain-steps "
                     "in the timed segments" % (cores, what, workload, timed, per_s, warm, steps)}
    _attach_ess(out, workload, [np.concatenate([r[g][2] for g in range(warm, warm + timed)], axis=0) for r in res], wall)
    return vals, out


# ----------------------------------------------------------------------------
# clocks
# ----------------------------------------------------------------------------
class ClockSampler(object):
    """nvidia-smi sampled every 50 ms in the background; started BEFORE warm-up (the tool needs
    a few hundred ms to come up) and filtered to the wall-clock windows of the timed regions."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        self.rows = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                       "-lms", "50", "-i", str(gpu_index)], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        """Terminate the sampler and parse its log (call once, after the last timed region)."""
        import datetime
        self.rows = []
        if self.p is None:
            return
        time.sleep(0.12)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 8:
                continue
            try:
                ts = datetime.datetime.strptime(parts[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                self.rows.append((ts, float(parts[1]), float(parts[2]),
                                  [nm for nm, v in zip(names, parts[4:8]) if v.lower().startswith("active")]))
            except ValueError:
                continue
        self.f.close()
        os.unlink(self.f.name)

    def window(self, t0, t1):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        rows = self.rows or []
        use = [r for r in rows if t0 - 0.05 <= r[0] <= t1 + 0.05]
        if not use and rows:                                   # window shorter than the sampling period
            mid = 0.5 * (t0 + t1)
            use = sorted(rows, key=lambda r: abs(r[0] - mid))[:2]
            out["note"] = "timed window shorter than the 50 ms sampling period: nearest samples used"
        if use:
            out.update(sm_mhz=float(np.median([r[1] for r in use])), sm_max_mhz=float(max(r[2] for r in use)),
                       samples=len(use), reasons=sorted({x for r in use for x in r[3]}))
        return out


# ----------------------------------------------------------------------------
# workloads
# ----------------------------------------------------------------------------
_DATA_CACHE = {}


def _logistic_model(N, d):
    """One device copy of the synthetic design matrix per (N, d), shared by the precisions of a config."""
    from riemann_b200 import synthetic
    from riemann_b200.models.logistic import LogisticRegression
    key = ("logistic", N, d)
    if key not in _DATA_CACHE:
        X, y, ts, pv = synthetic.logistic_problem(N, d)
        _DATA_CACHE.clear()                                # at most one data set resident
        _DATA_CACHE[key] = (LogisticRegression(X, y, pv), ts)
    return _DATA_CACHE[key]


def build_workload(name, K, seed, chain_offset, precision="f64"):
    """Returns (sampler, description).  Start states are keyed by GLOBAL chain id, so a shard is the
    corresponding slice of the one-GPU problem."""
    from riemann_b200 import Sampler, synthetic    # synthetic-input recipes (SURVEY 8d); the engine arm never imports oracle/
    if name == "changepoint":
        from riemann_b200.models.changepoint import ChangepointParams, ChangepointRegression1D
        from riemann_b200.proposals.changepoint import ChangepointRegression1DProp
        c = synthetic.changepoint_problem()
        model = ChangepointRegression1D(c["x"], c["y"], c["xmin"], c["xmax"], c["lamb"], c["kmax"], c["alpha"], c["beta"])
        prop = ChangepointRegression1DProp(model, c["hscale"])
        s = Sampler(model, prop, ChangepointParams(*c["theta0"]), K=K, seed=seed,
                    chain_offset=chain_offset)
        return s, "changepoint regression (examples/test_changepoint.py recipe: M=100, 5 true changepoints)"
    if name == "gauss2d_rw":
        from riemann_b200.models import benchmarks
        from riemann_b200.proposals.randomwalk import MetropolisRandomWalk
        s = Sampler(benchmarks.benchmark_gauss2d_corr, MetropolisRandomWalk(0.5 * np.eye(2)), np.ones(2),
                    K=K, seed=seed, chain_offset=chain_offset)
        return s, "benchmark_gauss2d_corr, MetropolisRandomWalk(0.5 I)"
    if name == "gauss2d_pt":
        # "next" row N3: parallel tempering, ladders of 5 temperatures (ptsampler.py default) along the chain axis
        from riemann_b200 import PTSampler
        from riemann_b200.models import benchmarks
        from riemann_b200.proposals.randomwalk import MetropolisRandomWalk
        if K % 5:
            raise SystemExit("gauss2d_pt: chains per GPU must be a multiple of 5 (one ladder = 5 temperatures)")
        pt = PTSampler(benchmarks.benchmark_gauss2d_corr, MetropolisRandomWalk(0.5 * np.eye(2)), np.ones(2),
                       K=K // 5, seed=seed, chain_offset=chain_offset // 5)
        pt._sampler._pt_owner = pt                      # keep the wrapper alive
        return pt._sampler, ("benchmark_gauss2d_corr, PTSampler: %d ladders x 5 temperatures (0.5**arange(5)), "
                             "Pswap = 0.1, MetropolisRandomWalk(0.5 I)" % (K // 5))
    if name == "gauss1000_mala":
        from riemann_b200.models import benchmarks
        from riemann_b200.proposals.hamiltonian import MALA
        m = benchmarks.gauss_corr(1000)
        rng = np.random.Generator(np.random.Philox(key=[synthetic.SEED_BASE + 3, chain_offset]))
        th0 = rng.standard_normal((K, 1000))
        s = Sampler(m, MALA(0.08, m.grad_log_likelihood), th0, seed=seed, chain_offset=chain_offset,
                    precision=precision)
        return s, "dense Gaussian d=1000 (0.1 I + 0.9 11^T), MALA eps=0.08, precision " + precision
    if name in ("logistic_mala", "logistic_mmala"):
        from riemann_b200.proposals.hamiltonian import MALA, SimplifiedMMALA
        N, d = (100000, 64) if name == "logistic_mmala" else (1000000, 100)
        m, ts = _logistic_model(N, d)
        rng = np.random.Generator(np.random.Philox(key=[synthetic.SEED_BASE + 5, chain_offset]))
        th0 = ts[None, :] + 0.01 * rng.standard_normal((K, d))
        prop = SimplifiedMMALA(0.5, m) if name == "logistic_mmala" else MALA(0.02, m.grad_log_posterior)
        if precision == "tf32-metric" and name != "logistic_mmala":
            raise SystemExit("--precision tf32-metric applies to logistic_mmala only")
        s = Sampler(m, prop, th0, seed=seed, chain_offset=chain_offset, precision=precision)
        return s, "logistic regression N=%d d=%d, %s%s" % (
            N, d, "simplified mMALA" if "mm" in name else "MALA",
            {"f64": "", "tf32-metric": ", Fisher metric on tcgen05 (TF32 GEMM)",
             "tf32x3": ", likelihood sweep on tcgen05"}[precision])
    raise SystemExit("unknown workload %r" % name)


DTYPE_NOTE = {"f64": "f64",
              "tf32x3": "tf32x3 tensor-core products (fp32-accurate), f64 accept test",
              "tf32-metric": "f64 (proposal metric: tf32 tensor cores)"}


class Ctx(object):
    """Process-wide measurement context: rank / world, stream, L2 flush buffer, clock sampler."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
        import __graft_entry__ as ge
        if self.rank == 0 and not os.path.exists(ge.OUT):
            ge.build()
        if self.world > 1:
            dist.barrier()
        self.flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
        self.clocks = ClockSampler(self.local) if self.rank == 0 else None
        self.peaks, self.peak_src = load_peaks()
        self.profiled = load_profiled()
        self.windows = []

    def sync_all(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
            self.torch.cuda.synchronize()

    def max_over_ranks(self, v):
        t = self.torch.tensor([v], dtype=self.torch.float64, device="cuda")
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def close(self):
        if self.world > 1:
            self.dist.destroy_process_group()


def roofline_for(ctx, wl, precision, Kg, T, steps, kt, ms):
    """roofline.achieved = ALGORITHMIC work of the timed region / the dominant kernel's OWN time in it
    (CUDA events on the launching stream, rmn_sampler_kernel_timing); the kernel's share of the step is
    reported next to it and must agree with the ncu launch list under profiles/."""
    peaks, extra = ctx.peaks, ctx.peaks.get("extra", {})
    algo_flop_step = ALGO_FLOP[wl] * Kg * T              # per bench step, per GPU
    if wl == "logistic_mmala" and precision == "tf32-metric":
        algo_flop_step = 4.0 * 100000 * 64 * Kg * T      # lg_eval_kernel's part: logits + gradient, 4 N d
    kernel_ms = kt["total_ms"] if kt["launches"] > 0 else ms
    ach = algo_flop_step * steps / (kernel_ms * 1e-3) / 1e12
    computed_fp64 = 148 * 64 * 2 * peaks["sm_max_mhz"] * 1e6 / 1e12      # fp64 FMA lanes x clock
    if wl in ("changepoint", "gauss2d_rw", "gauss2d_pt"):
        peak = extra.get("fp64_dfma_tflops", computed_fp64)
        roof = {"bound": "alu", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak, "traffic": None,
                "algo_flop_per_chain_step": ALGO_FLOP[wl],
                "note": "issue-bound fp64/integer kernel (SURVEY 8d: not HBM, not tensor, ~0 algorithmic HBM bytes); achieved = "
                        "%.0f algorithmic flop/chain-step x rate against the fp64 DFMA rate %s; the binding resource is "
                        "the warp-instruction issue rate, see `profiled` (issue-slot utilisation, instructions per "
                        "chain-step from ncu)"
                        % (ALGO_FLOP[wl], "measured by scripts/peaks (profiles/measured_peaks_extra.json)"
                           if "fp64_dfma_tflops" in extra else "computed as 148 SM x 64 lanes x 2 x clocks.max.sm")}
        if wl in ALGO_COMPARES:
            roof["algo_compares_per_chain_step"] = ALGO_COMPARES[wl]
    elif precision == "tf32-metric" and wl == "logistic_mmala":
        peak = extra.get("fp64_dmma_tflops", computed_fp64)
        roof = {"bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak, "traffic": None,
                "note": "dominant kernel = lg_eval_kernel (fp64 DMMA, 4 N d = 2.6e7 flop per chain-step) against the "
                        "measured DMMA peak; the metric GEMM (4.2e8 flop per chain-step) runs on tcgen05 in TF32"}
    elif precision == "tf32x3" and wl == "logistic_mmala" and "gemm" in kt["kernel"]:
        bf16 = "bf16" in kt["kernel"]
        peak = peaks["bf16_tflops"] if bf16 else extra.get("tf32_cublas_tflops", 0.5 * peaks["bf16_tflops"])
        ach = 100000.0 * 64 * 65 * Kg * T * steps / (kernel_ms * 1e-3) / 1e12
        roof = {"bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak, "traffic": None,
                "note": "dominant kernel = the Fisher-metric GEMM of the proposal on tcgen05 (%s operands, fp32 accumulate): "
                        "N d (d+1) = 4.16e8 flop per chain-step (the symmetric half, SURVEY 8d) against the %s; the fused "
                        "likelihood sweep (4 N d flop) is the second kernel of the step"
                        % ("bf16" if bf16 else "TF32", "dense bf16 peak of MEASURED_PEAKS.json" if bf16 else "cuBLAS TF32 peak")}
    elif precision == "tf32x3" and wl.startswith("logistic"):
        peak = extra.get("tf32_cublas_tflops", 0.5 * peaks["bf16_tflops"])
        n_, d_ = (100000, 64) if wl == "logistic_mmala" else (1000000, 100)
        ach = 4.0 * n_ * d_ * Kg * T * steps / (kernel_ms * 1e-3) / 1e12
        roof = {"bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak, "traffic": None,
                "note": "likelihood sweep on tcgen05, timed as a whole (CUDA events around its launches); achieved counts "
                        "the ALGORITHMIC 4 N d flop per chain-step once (the fp32-accurate logits are one TF32 MMA plus two "
                        "bf16 MMAs of twice the depth for the correction terms, the gradient one bf16 MMA), against the "
                        "cuBLAS TF32 peak -- the rate of the product that carries the leading term"}
    elif precision == "tf32x3":
        peak = extra.get("tf32_cublas_tflops", 0.5 * peaks["bf16_tflops"])
        roof = {"bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak, "traffic": None,
                "note": "tcgen05 kind::tf32, 3 MMAs per product (fp32-accurate): achieved counts the ALGORITHMIC "
                        "2 d^2 flop per chain-step once, so 1/3 is the ceiling of this scheme; peak = %s"
                        % ("cuBLAS TF32 8192^3 measured by scripts/peaks (profiles/measured_peaks_extra.json)"
                           if "tf32_cublas_tflops" in extra else "half the %s bf16 figure of MEASURED_PEAKS.json" % ctx.peak_src)}
    else:
        peak = extra.get("fp64_dmma_tflops", computed_fp64)
        roof = {"bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak, "traffic": None,
                "note": "fp64 tensor path (DMMA m8n8k4); peak = %s"
                        % ("mma.sync.m8n8k4.f64 rate measured by scripts/peaks (profiles/measured_peaks_extra.json)"
                           if "fp64_dmma_tflops" in extra else "computed 148 SM x 64 lanes x 2 x clocks.max.sm")}
    roof["kernel"] = kt["kernel"]
    roof["kernel_launches"] = kt["launches"]
    roof["kernel_ms_per_launch"] = kernel_ms / max(kt["launches"], 1)
    roof["kernel_share_of_step"] = kernel_ms / ms if ms > 0 else None
    prof = ctx.profiled.get("%s/%s" % (wl, precision))
    if prof:
        roof["profiled"] = prof            # static ncu evidence (DRAM bytes per launch, pipe utilisation), with its source file
        if roof["bound"] == "alu" and prof.get("warp_inst_per_chain_step"):
            # the binding resource of an issue-bound kernel: warp-instructions issued per second (instruction count per
            # chain-step from the committed ncu capture x the LIVE chain-step rate of the kernel) against what the SMs can
            # issue (SMs x 4 schedulers x SM clock)
            rate = Kg * T * steps / (kernel_ms * 1e-3)
            issue_peak = 148 * 4 * peaks["sm_max_mhz"] * 1e6
            roof["issue_frac"] = prof["warp_inst_per_chain_step"] * rate / issue_peak
            roof["issue_note"] = ("%d warp-instructions per chain-step (static, %s) x %.3g chain-steps/s (live) / (148 SM x 4 "
                                  "schedulers x %.0f MHz)" % (prof["warp_inst_per_chain_step"], prof["source"].split(",")[0],
                                                              rate, peaks["sm_max_mhz"]))
    return roof


DUMP_BYTES = 60 << 20                                   # below 64 MB with the .npy headers


def dump_outputs(out_dir, s, blk, rank, world):
    """What the last timed step computed, as a caller of the sampler receives it: every chain's state and log-posterior
    and the all-reduced diagnostics block, as float64 DIR/<name>.npy (DIR/<name>_rank<r>.npy on several ranks).  The
    unused lanes of a changepoint state (cpx beyond k, cpv beyond k + 1) are 0, whatever the kernels left there, so
    every value is finite and the shapes are fixed.  Where the per-chain arrays exceed DUMP_BYTES in all, a fixed seeded
    sample of chains is written, their indices in chain_index.npy."""
    if s._is_cp:
        (k, cpx, cpv, sig), lp = s._download_state()
        lane = np.arange(cpx.shape[1])[None, :]
        out = {"k": k, "cpx": np.where(lane < k[:, None], cpx, 0.0), "cpv": np.where(lane <= k[:, None], cpv, 0.0),
               "sig": sig, "logpost": lp}
    else:
        th, lp = s._download_state()
        out = {"theta": th, "logpost": lp}
    out = {n: np.asarray(a, dtype=np.float64) for n, a in out.items()}
    diag = blk.cpu().numpy().astype(np.float64)
    K = len(lp)
    per_chain = sum(a.nbytes for a in out.values()) // K + 8          # + 8: its entry in chain_index
    n = min(K, (DUMP_BYTES - diag.nbytes) // per_chain)
    if n < K:
        idx = np.sort(np.random.default_rng(SEED).choice(K, n, replace=False))
        out = {name: a[idx] for name, a in out.items()}
        out["chain_index"] = idx.astype(np.float64)
    out["diagnostics"] = diag
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, (name if world == 1 else "%s_rank%d" % (name, rank)) + ".npy"), a)


def measure(ctx, wl, precision, Kg, T, steps, warmup, burn, chain_offset, K_total, scaling, cpu_seconds=0.0, e2e=True,
            dump_dir=None):
    """One workload on this rank's shard: burn-in, warm-up, `steps` timed launches (CUDA events, L2 flush between
    them), split-chain diagnostics over the two halves of the timed region, the end-to-end leg, roofline.  dump_dir:
    dump_outputs() of the last timed step, before the roofline and end-to-end legs run the chains further."""
    torch = ctx.torch
    from riemann_b200 import _lib
    from riemann_b200.distributed import reduce_block, summarize_block, summarize_split
    s, desc = build_workload(wl, Kg, SEED, chain_offset, precision)
    stream = torch.cuda.current_stream()
    lib = _lib.load()
    s.run(burn, trace=False)
    for _ in range(max(warmup, 3)):
        s.run(T, trace=False)
        blk = reduce_block(s.diagnostics_block())
    s.reset_diagnostics()
    ctx.sync_all()

    def timed_region(nsteps, instrument, split):
        """nsteps launches of the hot path, each bracketed by CUDA events, L2 flushed between them.  instrument: CUDA
        events around every launch of the dominant kernel as well (rmn_sampler_kernel_timing) -- those records sit
        between the kernels of a step, so the region that gives `value` runs WITHOUT them and a second region with them
        gives the roofline's kernel time and share.  Returns (ms summed over steps, first-half block, last block)."""
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(nsteps)]
        s.enable_kernel_timing(instrument)
        ctx.sync_all()
        half = nsteps // 2 if split and nsteps >= 2 and nsteps % 2 == 0 else 0
        first, b = None, None
        for i in range(nsteps):
            ctx.flush.fill_(i & 0xff)                  # L2 flush, outside the event pair
            if half and i == half:                     # second half-window of the split-chain diagnostics
                first = b.clone()
                s.reset_diagnostics()
            ev[i][0].record(stream)
            _lib.check(lib.rmn_sampler_run(s._handle, T, None, None, _lib.stream_ptr()))
            s.total_steps += T
            b = reduce_block(s.diagnostics_block())    # per-batch diagnostics all-reduce (NCCL)
            ev[i][1].record(stream)
        ctx.sync_all()
        return sum(x.elapsed_time(y) for x, y in ev), first, b

    launches0 = s.launch_count
    w0 = time.time()
    ms, blk_first, blk = timed_region(steps, False, True)
    w1 = time.time()
    launches = s.launch_count - launches0
    ms = ctx.max_over_ranks(ms)
    if dump_dir:
        dump_outputs(dump_dir, s, blk, ctx.rank, ctx.world)
    # roofline pass: the same launches with the dominant kernel's own CUDA events
    ms_roof, _, _ = timed_region(steps, True, False)
    kt = s.kernel_timing()                         # dominant kernel only: total ms / launches in the roofline pass
    s.enable_kernel_timing(False)
    ms_roof = ctx.max_over_ranks(ms_roof)
    diag, diag_kind = None, "whole window"
    if blk_first is not None:
        try:
            diag = summarize_split(blk_first.cpu().numpy(), blk.cpu().numpy())
            diag_kind = "split: %d half-chains of %d MH steps" % (diag["chains"], diag["steps"])
        except ValueError:
            diag = None
    if diag is None:
        diag = summarize_block(blk.cpu().numpy())
    nworld = 1 if scaling.startswith("none") else ctx.world      # K = 1 replicas: the value is a single chain's
    value = Kg * nworld * T * steps / (ms * 1e-3)
    e2e_d = run_e2e(ctx, s, T, Kg, nworld, steps) if e2e else None
    out = {"workload": wl, "precision": precision, "value": value, "unit": UNIT, "ms_per_step": ms / steps,
           "steps": steps, "warmup": max(warmup, 3), "scaling": scaling, "dtype": DTYPE_NOTE[precision],
           "chains_per_gpu": Kg, "chains_total": Kg * nworld, "iters_per_step": T, "burn_in_iters": burn,
           "desc": desc, "e2e": e2e_d, "gpu_launches": int(launches), "window": (w0, w1)}
    rhat = float(np.nanmax(diag["rhat"])) if np.any(np.isfinite(diag["rhat"])) else None
    ess_ok = rhat is not None and rhat < 1.05 and np.isfinite(diag["min_ess"])
    out["min_ess_per_sec"] = diag["min_ess"] / (ms * 1e-3) if ess_ok else None
    out["diagnostics"] = {"estimator": diag_kind + "; tau = n B / W over all chains", "accept_rate": diag["accept_rate"],
                          "max_rhat": rhat, "min_ess": diag["min_ess"] if np.isfinite(diag["min_ess"]) else None,
                          "overflows": diag["overflows"], "chains": diag["chains"], "steps_per_chain": diag["steps"]}
    if not ess_ok:
        out["diagnostics"]["min_ess_reason"] = ("split-R-hat %.3f >= 1.05 over the timed window (%d MH steps per half): "
                                               "the window is shorter than ~10 tau of the slowest functional"
                                               % (rhat, diag["steps"]) if rhat is not None else "no finite R-hat")
    if ctx.rank == 0:
        out["roofline"] = roofline_for(ctx, wl, precision, Kg, T, steps, kt, ms_roof)
        out["roofline"]["timed_in"] = ("a second pass of %d steps (%.3f ms/step) with CUDA events around every launch of the "
                                       "kernel on the launching stream; the `value` region runs without them"
                                       % (steps, ms_roof / steps))
    out["_sampler"] = s
    return out


def run_e2e(ctx, s, T, Kg, nworld, steps):
    """Same metric through the public API with HOST buffers (riemann_b200.pipeline.HostJobRunner): every step is one
    job -- the chains' start states are uploaded from pinned host memory, T iterations run, and states, log-posteriors
    and the diagnostics block come back to pinned host memory.  `value`: the jobs pipelined (copies of neighbouring
    jobs on side streams overlap the MH kernels; fill and drain inside the timed region); `serial_value`: every job
    upload -> run -> download -> synchronize, nothing overlapped."""
    torch = ctx.torch
    from riemann_b200.pipeline import HostJobRunner
    if s._is_cp:
        (k, cpx, cpv, sig), _ = s._download_state()
        job = tuple(torch.from_numpy(a).pin_memory() for a in (k, cpx, cpv, sig))
    else:
        th, _ = s._download_state()
        job = (torch.from_numpy(th).pin_memory(),)
    out = {}
    for key, overlap in (("serial_value", False), ("value", True)):
        runner = HostJobRunner(s, overlap=overlap)
        for _ in runner.run([job] * 2, T):              # warm-up (buffers, graph capture for this T)
            pass
        ctx.sync_all()
        t0 = time.perf_counter()
        n_out = 0
        for res in runner.run([job] * steps, T):
            n_out += 1
        ctx.sync_all()
        dt = ctx.max_over_ranks(time.perf_counter() - t0)
        assert n_out == steps and float(res["diagnostics"][0]) == Kg
        out[key] = Kg * nworld * T * steps / dt
        h2d, d2h = runner.h2d_bytes, runner.d2h_bytes
    return {"value": out["value"], "serial_value": out["serial_value"], "unit": UNIT, "h2d_bytes_per_step": int(h2d),
            "d2h_bytes_per_step": int(d2h), "steps": steps,
            "note": "host wall clock over `steps` jobs through riemann_b200.pipeline.HostJobRunner: pinned upload -> "
                    "set_state -> run -> get_state + diagnostics -> pinned download; `value` double-buffers the copies "
                    "on side streams (they overlap the kernels of the neighbouring jobs), `serial_value` does not"}


def ess_phase(ctx, s, T, half_launches, K_total):
    """min-ESS/sec of the changepoint workload as a measurement: two consecutive half-windows of half_launches x T
    MH steps each, device-timed like the bench steps (the diagnostics block is reduced once per half), evaluated
    split-chain over ALL chains.  Reported per functional with window_over_tau; min_ess_per_sec only when
    split-R-hat < 1.05, i.e. when each half-window holds >= ~10 tau of the slowest functional."""
    torch = ctx.torch
    from riemann_b200 import _lib
    from riemann_b200.distributed import reduce_block, summarize_split
    lib = _lib.load()
    stream = torch.cuda.current_stream()
    blks = []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ctx.sync_all()
    e0.record(stream)
    for h in range(2):
        s.reset_diagnostics()
        for _ in range(half_launches):
            _lib.check(lib.rmn_sampler_run(s._handle, T, None, None, _lib.stream_ptr()))
            s.total_steps += T
        blks.append(reduce_block(s.diagnostics_block()).clone())
    e1.record(stream)
    ctx.sync_all()
    ms = ctx.max_over_ranks(e0.elapsed_time(e1))
    d = summarize_split(blks[0].cpu().numpy(), blks[1].cpu().numpy())
    n_half = half_launches * T
    tau = np.asarray(d["tau"], dtype=np.float64)
    tmax = float(np.nanmax(tau))
    rhat = float(np.nanmax(d["rhat"]))
    ok = rhat < 1.05
    out = {"estimator": "split-chain moments over all %d chains: tau = n B / W, ESS = chains x n / tau; two half-windows "
                        "of %d MH steps, device-timed (CUDA events), diagnostics all-reduce included" % (K_total, n_half),
           "functionals": FUNC_NAMES["changepoint"], "tau_steps": [float(t) for t in tau],
           "ess": [float(e) for e in d["ess"]], "rhat": [float(r) for r in d["rhat"]],
           "window_steps": n_half, "window_over_tau": n_half / tmax, "max_rhat": rhat, "seconds": ms * 1e-3,
           "min_ess": d["min_ess"], "min_ess_per_sec": d["min_ess"] / (ms * 1e-3) if ok else None,
           "chain_steps_per_sec": K_total * 2 * n_half / (ms * 1e-3)}
    if not ok:
        out["reason"] = "split-R-hat %.3f >= 1.05: half-window = %.1f tau of the slowest functional" % (rhat, n_half / tmax)
        out["min_ess_per_sec_unconverged"] = d["min_ess"] / (ms * 1e-3)
    return out


def sokal_check(ctx, nchains=256, nsteps=120000, thin=8, burn=60000):
    """The reference's own estimator (emcee.autocorr.integrated_time, examples/test_randomwalk.py:42; restated in
    riemann_b200/diagnostics.py) on a traced subset of device chains -- the same estimator and functionals the CPU arm
    reports -- next to the moment-based tau of the full population."""
    from riemann_b200 import diagnostics as dgn, synthetic
    s2, _ = build_workload("changepoint", nchains, SEED + 1, 0, "f64")
    s2.run(burn, trace=False)
    t0 = time.perf_counter()
    s2.run(nsteps, thin, thin)
    dt = time.perf_counter() - t0
    tr = s2._chain_thetas
    c = synthetic.changepoint_problem()
    xq = c["xmin"] + (c["xmax"] - c["xmin"]) * (np.arange(6) + 0.5) / 6.0
    k = tr.k.astype(np.int64)                                              # [rec, K]
    # y_hat(x_q) = cpv[#{cpx < x_q}] with the padded layout (entries >= k are not changepoints)
    idx = np.arange(tr.cpx.shape[2])[None, None, :]
    cols = [tr.sig, k.astype(np.float64)]
    for q in range(6):
        cnt = np.sum((tr.cpx < xq[q]) & (idx < k[:, :, None]), axis=2)
        cols.append(np.take_along_axis(tr.cpv, cnt[:, :, None], axis=2)[:, :, 0])
    x = np.stack(cols, axis=2)
    tau = dgn.integrated_time_chains(x) * thin
    n = x.shape[0] * thin
    tmax = float(np.nanmax(tau))
    return {"estimator": "Sokal window (c = 5), ACF averaged over the chains; tau in MH steps",
            "functionals": FUNC_NAMES["changepoint"], "sokal_tau_steps": [float(t) for t in tau],
            "chains": nchains, "steps_per_chain": n, "thin": thin, "window_over_tau": n / tmax,
            "reliable": bool(n >= 50 * tmax), "trace_seconds": dt}


# ----------------------------------------------------------------------------
# multi-GPU self-checks (N >= 2, untimed)
# ----------------------------------------------------------------------------
def multi_gpu_checks(ctx):
    """(1) chain-shard invariance: the N ranks' shards of a Philox run equal, bit for bit, the same chains of the
    unsharded run (rank 0 runs all of them).  (2) row-sharded data mode: the rows of the reference-stream fixtures
    (tests/golden/{mala,hmc3,mmala}_logistic.npz, recorded through the reference's own Sampler) are split over the N
    ranks, the injected stream is replayed; chain within 1e-9 / 1e-8 of the recorded one, ranks bit-identical."""
    torch, dist = ctx.torch, ctx.dist
    from riemann_b200 import Sampler
    from riemann_b200.distributed import shard_chains, shard_rows
    res = {}
    # ---- (1)
    Ktot, Tn = 1024 * ctx.world, 300
    off, Kl = shard_chains(Ktot, ctx.rank, ctx.world)
    s, _ = build_workload("changepoint", Kl, SEED + 7, off, "f64")
    s.run(Tn, trace=False)
    (k, cpx, cpv, sig), lp = s._download_state()
    mine = torch.as_tensor(np.concatenate([k[:, None].astype(np.float64), cpx, cpv, sig[:, None], lp[:, None]], axis=1),
                           device="cuda")
    parts = [torch.empty_like(mine) for _ in range(ctx.world)]
    dist.all_gather(parts, mine)
    ok = True
    if ctx.rank == 0:
        sf, _ = build_workload("changepoint", Ktot, SEED + 7, 0, "f64")
        sf.run(Tn, trace=False)
        (k, cpx, cpv, sig), lp = sf._download_state()
        full = np.concatenate([k[:, None].astype(np.float64), cpx, cpv, sig[:, None], lp[:, None]], axis=1)
        ok = bool(np.array_equal(torch.cat(parts).cpu().numpy(), full, equal_nan=True))
        del sf
    res["chain_shard_invariance"] = {"ok": ok, "chains": Ktot, "steps": Tn, "ranks": ctx.world,
                                     "check": "gathered shards == unsharded run on rank 0, bitwise"}
    del s
    # ---- (2)
    from riemann_b200.models.logistic import LogisticRegression
    from riemann_b200.proposals.hamiltonian import MALA, SimplifiedMMALA, VanillaHMC
    rows = {}
    all_ok = True
    for name, tol in (("mala_logistic", 1e-9), ("hmc3_logistic", 1e-9), ("mmala_logistic", 1e-8)):
        path = os.path.join(ROOT, "tests", "golden", name + ".npz")
        if not os.path.exists(path):
            rows[name] = "fixture missing"
            all_ok = False
            continue
        g = np.load(path)
        offr, n = shard_rows(len(g["y"]), ctx.rank, ctx.world)
        dm = LogisticRegression(g["X"][offr:offr + n], g["y"][offr:offr + n], float(g["prior_var"]))
        if name == "mala_logistic":
            p = MALA(float(g["eps"]), dm.grad_log_posterior)
        elif name == "hmc3_logistic":
            p = VanillaHMC(float(g["eps"]), int(g["nsteps"]), dm.grad_log_posterior)
        else:
            p = SimplifiedMMALA(float(g["eps"]), dm)
        sr = Sampler(dm, p, g["thetas"][0], row_sharded=True)
        sr.run_injected(xi=g["xi"], u=g["u"])
        th = np.array(sr._chain_thetas)
        err = float(np.max(np.abs(th - g["thetas"]) / np.maximum(1.0, np.abs(g["thetas"]))))
        mine = torch.as_tensor(th, device="cuda")
        other = [torch.empty_like(mine) for _ in range(ctx.world)]
        dist.all_gather(other, mine)
        same = all(torch.equal(o, mine) for o in other)
        flag = torch.tensor([1.0 if (err < tol and same) else 0.0], device="cuda")
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        rows[name] = {"rel_err_vs_reference_chain": err, "tol": tol, "ranks_bit_identical": bool(same),
                      "ok": bool(flag.item() > 0.5)}
        all_ok = all_ok and rows[name]["ok"]
        del sr, dm
    res["row_sharded"] = {"ok": bool(all_ok), "ranks": ctx.world, "fixtures": rows}
    torch.cuda.empty_cache()
    return res


# ----------------------------------------------------------------------------
# engine arm
# ----------------------------------------------------------------------------
def shard_for(ctx, wl, sharding, chains_override=None):
    """-> (chains on this rank, global id of its first chain, total chains, `scaling` word)."""
    if sharding == "replica":
        return 1, 0, 1, "none (K = 1 latency; one replica per rank, the value is a single chain's)"
    if sharding == "strong":
        Kt = chains_override or CHAINS_TOTAL[wl]
        if Kt % ctx.world:
            raise SystemExit("%s: %d chains do not split over %d ranks" % (wl, Kt, ctx.world))
        Kg = Kt // ctx.world
        return Kg, ctx.rank * Kg, Kt, "strong"
    Kg = chains_override or CHAINS_PER_GPU[wl]
    return Kg, ctx.rank * Kg, Kg * ctx.world, "weak"


def public_entry(ctx, r, cpu=None):
    """Strip the private fields of a measure() result into the JSON entry of the `configs` array."""
    e = {k: v for k, v in r.items() if not k.startswith("_") and k not in ("window", "desc")}
    e["config"] = {"workload": "%s: %s; %d chains/GPU x %d MH iterations per step; Philox4x32-10 RNG; L2 flushed "
                               "(256 MiB write) between steps" % (r["workload"], r["desc"], r["chains_per_gpu"], r["iters_per_step"]),
                   "chains_per_gpu": r["chains_per_gpu"], "chains_total": r["chains_total"],
                   "iters_per_step": r["iters_per_step"]}
    if ctx.clocks:
        e["clocks"] = ctx.clocks.window(*r["window"])
    e["cpu_baseline"] = cpu
    return e


def run_engine(args):
    ctx = Ctx(args)
    torch = ctx.torch
    single = args.workload is not None
    wl = args.workload or "changepoint"
    T = args.iters or ITERS[wl]
    sharding = "weak"
    if single and args.strong:
        sharding = "strong"
    Kg, off, Ktot, scaling = shard_for(ctx, wl, sharding, args.chains)
    burn = args.burn if args.burn is not None else {"changepoint": 50000}.get(wl, 2 * T)
    head = measure(ctx, wl, args.precision, Kg, T, args.steps, args.warmup, burn, off, Ktot, scaling,
                   dump_dir=args.dump_outputs)
    s = head.pop("_sampler")

    ess = sokal = None
    if wl == "changepoint" and not args.no_ess:
        ess = ess_phase(ctx, s, T, args.ess_half_launches, Ktot)
        if ctx.rank == 0:
            sokal = sokal_check(ctx)
    del s
    torch.cuda.empty_cache()

    configs, pending_cpu = [], []
    if not single and not args.no_configs:
        only = set(args.only.split(",")) if args.only else None
        for key, w, prec, shd, Tn in SUBCONFIGS:
            if only and key not in only and w not in only:
                continue
            Kg2, off2, Kt2, sc2 = shard_for(ctx, w, shd)
            try:
                r = measure(ctx, w, prec, Kg2, Tn, args.steps, 3, 2 * Tn if shd != "replica" else 1000, off2, Kt2, sc2)
            except Exception as e:                       # a config that cannot run must not take the line down
                configs.append({"key": key, "workload": w, "precision": prec, "error": "%s: %s" % (type(e).__name__, e)})
                torch.cuda.empty_cache()
                continue
            r.pop("_sampler", None)
            r["key"] = key
            configs.append(r)
            torch.cuda.empty_cache()
        _DATA_CACHE.clear()
        torch.cuda.empty_cache()

    checks = None
    if ctx.world > 1 and not args.no_checks:
        checks = multi_gpu_checks(ctx)

    if ctx.clocks:
        ctx.clocks.stop()
    if ctx.rank != 0:
        ctx.close()
        return
    do_cpu = (not args.no_cpu) and ctx.world == 1            # contract: rank 0 at N = 1 only
    cpu_head = cpu_baseline(wl, args.cpu_seconds) if do_cpu else None
    entries = []
    cpu_cache = {}
    for r in configs:
        if "error" in r:
            entries.append(r)
            continue
        cpu = None
        if do_cpu and r["key"] != "gauss2d_rw_k1":
            if r["workload"] not in cpu_cache:
                cpu_cache[r["workload"]] = cpu_baseline(r["workload"], args.cpu_seconds_config)
            cpu = cpu_cache[r["workload"]]
        elif do_cpu:
            cpu = {"note": "K = 1: the CPU figure for one chain is cpu_baseline.value / cores of the gauss2d_rw entry"}
        entries.append(public_entry(ctx, r, cpu))

    line = {
        "metric": METRIC, "value": head["value"], "unit": UNIT, "n_gpus": ctx.world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": head["ms_per_step"], "higher_is_better": True,
        "scaling": scaling, "vs_baseline": None, "dtype": head["dtype"], "data": "synthetic",
        "config": {"workload": "%s: %s; %d chains/GPU x %d MH iterations per step; Philox4x32-10 RNG; "
                               "L2 flushed (256 MiB write) between steps, per-step CUDA events summed"
                               % (wl, head["desc"], Kg, T),
                   "chains_per_gpu": Kg, "chains_total": head["chains_total"], "iters_per_step": T,
                   "burn_in_iters": burn, "parallelism": "chains sharded, dp%d" % ctx.world},
        "min_ess_per_sec": (ess or {}).get("min_ess_per_sec") if ess is not None else head["min_ess_per_sec"],
        "diagnostics": head["diagnostics"],
        "ess": ess, "ess_sokal": sokal,
        "e2e": head["e2e"], "gpu_launches": head["gpu_launches"], "roofline": head["roofline"],
        "cpu_baseline": cpu_head,
        "clocks": ctx.clocks.window(*head["window"]) if ctx.clocks else None, "peaks_source": ctx.peak_src,
        "configs": entries, "multi_gpu_checks": checks,
    }
    if checks is not None:
        line["row_sharded_parity"] = checks["row_sharded"]["ok"]
        line["chain_shard_invariance"] = checks["chain_shard_invariance"]["ok"]
    print(json.dumps(line))
    ctx.close()


# ----------------------------------------------------------------------------
# reference arm
# ----------------------------------------------------------------------------
def run_reference(args):
    """--impl reference: the reference's own CPU sampler on this box's host cores, same metric / config.  The
    UNMODIFIED riemann package (staged under oracle/_ref/ by oracle/build_ref.py, imported through oracle/refshim.py)
    for the changepoint / Gaussian configs; the numpy port for the logistic models the reference does not contain."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = args.workload or "changepoint"
    W, K = max(args.warmup, 1), max(args.steps, 1)
    # a step = `per` seconds of every core's chain; the chains continue from step to step, so the tau / ESS window is
    # the whole timed region (args.cpu_seconds_reference of sampling per chain; the warm-up steps are the burn-in)
    per = max(1.0, min(30.0, args.cpu_seconds_reference / K))
    Wn = max(1, min(W, int(round(0.15 * args.cpu_seconds_reference / per))))
    vals, cb = cpu_reference_segments(wl, Wn, K, per)
    v = cb["value"]
    cb["per_step_values"] = [float(x) for x in vals]
    Kg = args.chains or CHAINS_PER_GPU[wl]
    entries = []
    if args.workload is None and not args.no_configs:
        for w in ("gauss2d_rw", "gauss1000_mala", "logistic_mala", "logistic_mmala"):
            c = cpu_baseline(w, args.cpu_seconds_config)
            entries.append({"key": w, "workload": w, "value": c["value"], "unit": UNIT, "dtype": "f64",
                            "min_ess_per_sec": c.get("min_ess_per_sec"), "cpu_baseline": c})
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus,
            "steps": K, "warmup": Wn, "ms_per_step": per * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "%s (CPU reference arm: one chain per host core, %.1f s per step, chains continue "
                                   "across steps)" % (wl, per),
                       "chains_per_gpu": Kg},
            "min_ess_per_sec": cb.get("min_ess_per_sec"),
            "cpu_baseline": cb,
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "configs": entries}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="engine", choices=["engine", "reference"])
    ap.add_argument("--workload", default=None, choices=sorted(CHAINS_PER_GPU),
                    help="single-workload line (profiling); default: changepoint headline + the `configs` array")
    ap.add_argument("--chains", type=int, default=None, help="chains per GPU (total chains with --strong)")
    ap.add_argument("--strong", action="store_true", help="single workload: --chains (or BASELINE's count) is the total")
    ap.add_argument("--iters", type=int, default=None, help="MH iterations per step")
    ap.add_argument("--burn", type=int, default=None)
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--cpu-seconds-config", type=float, default=3.0)
    ap.add_argument("--cpu-seconds-reference", type=float, default=80.0,
                    help="--impl reference: seconds of sampling per chain in the timed region (split over --steps)")
    ap.add_argument("--ess-half-launches", type=int, default=400,
                    help="changepoint ESS phase: launches (of --iters MH steps) per half-window")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-ess", action="store_true")
    ap.add_argument("--no-configs", action="store_true")
    ap.add_argument("--no-checks", action="store_true")
    ap.add_argument("--only", default=None, help="comma-separated keys / workloads of the configs array to run")
    ap.add_argument("--precision", default="f64", choices=["f64", "tf32x3", "tf32-metric"],
                    help="single workload: tf32x3 = tcgen05 tensor-core modes; tf32-metric = tcgen05 Fisher-metric GEMM")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write what the headline workload's last timed step computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the engine arm")
    # the tree may be read-only: no bytecode caches next to the sources, in this process or the spawned CPU-arm workers
    sys.dont_write_bytecode = True
    os.environ["PYTHONDONTWRITEBYTECODE"] = "1"
    if args.impl == "reference":
        run_reference(args)
    else:
        run_engine(args)


if __name__ == "__main__":
    main()
