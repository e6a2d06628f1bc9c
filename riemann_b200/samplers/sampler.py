"""
Sampler -- the many-chain, device-resident counterpart of riemann/samplers/sampler.py:28-90.

Same constructor and methods as the reference (``Sampler(model, proposal, theta0)``,
``run(Nsamples, Nburn=0, Nthin=1)``, ``sample()``, ``current_state()``, ``_add_state``)
and the same directly-read attributes ``_chain_thetas`` / ``_chain_logpost``.  Extra
keyword arguments select K chains, the Philox seed and the global chain offset (for
sharding over GPUs).  One ``run`` is one (or a few) kernel launches; the host never
sees an individual MH step.
"""
import ctypes as C

import numpy as np

from .. import _lib
from ..models.changepoint import (ChangepointParams, ChangepointRegression1D, pack_states,
                                  unpack_state)
from ..models.model import DeviceModel
from ..proposals.proposal import DeviceProposal
from ..sampling_errors import ParameterError

LANES = _lib.CP_LANES
TRACE_BYTES_LIMIT = 8 << 30


class ChangepointTrace(object):
    """History of K > 1 changepoint chains: arrays indexed [record, chain]."""

    def __init__(self, k, cpx, cpv, sig):
        self.k, self.cpx, self.cpv, self.sig = k, cpx, cpv, sig

    def __len__(self):
        return self.k.shape[0]

    def __getitem__(self, idx):
        if isinstance(idx, tuple):
            r, c = idx
            return unpack_state(self.k[r, c], self.cpx[r, c], self.cpv[r, c], self.sig[r, c])
        if isinstance(idx, slice):
            return ChangepointTrace(self.k[idx], self.cpx[idx], self.cpv[idx], self.sig[idx])
        return [self[idx, c] for c in range(self.k.shape[1])]


class Sampler(object):
    def __init__(self, model, proposal, theta0, K=None, seed=0, chain_offset=0, precision="f64", _tempering=None,
                 row_sharded=False, move_schedule=None):
        """
        :param theta0: starting point.  Fixed-d models: shape (d,) (shared by all K
            chains) or (K, d); a length-1 start is broadcast over the d coordinates, as numpy does inside
            the reference's model when examples/riemann_ex1.py:233 starts a d = 2 chain from a (1,) array.
            Changepoint model: a ChangepointParams or a list of K.
        :param K: number of independent chains on this device (default 1, the reference's case)
        :param seed, chain_offset: Philox key and the global id of chain 0 on this device
        :param precision: "f64" (default; fp64 like the reference) or "tf32x3" (dense Gaussian
            model: fp32 state, tcgen05 tensor-core product with a 3xTF32 split, fp64 accept test)
        :param move_schedule: changepoint model, Philox mode: "group" (default; aligned groups of 8 global chain ids
            share the move-type draws of a step, rmn_sampler_set_move_schedule) or "chain" (every chain draws its own).
        :param row_sharded: logistic model only.  Every rank of the torch.distributed group built its model from its
            own slice of the data rows (`distributed.shard_rows`) and runs the SAME K chains (same seed, chain_offset
            and start states); after every likelihood sweep the per-chain partial sums are all-reduced (NCCL, inside
            the library), so all ranks hold identical chains of the full-data posterior.
        """
        if not isinstance(model, DeviceModel):
            raise ParameterError("model has no device kernel: riemann_b200 samples only device "
                                 "models (there is no CPU fallback)")
        if not isinstance(proposal, DeviceProposal):
            raise ParameterError("proposal has no device kernel")
        if proposal._model is not None and proposal._model is not model:
            raise ParameterError("the proposal's gradient/metric belongs to a different model")
        if getattr(model, "_handle", None) is None:
            raise ParameterError("model has no data/device handle yet")
        torch = _lib.require_cuda()
        self._torch = torch
        self.model = model
        self.proposal = proposal
        self._is_cp = isinstance(model, ChangepointRegression1D)

        if self._is_cp:
            if isinstance(theta0, ChangepointParams):
                states = [theta0] * (K or 1)
            else:
                states = list(theta0)
                if K is not None and K != len(states):
                    raise ParameterError("K does not match the number of start states")
            self.K = len(states)
            self.d = model.Ndim
            self._squeeze = isinstance(theta0, ChangepointParams) and self.K == 1
        else:
            th = np.asarray(theta0, dtype=np.float64)
            self._scalar_theta0 = (th.ndim == 0)
            th = np.atleast_1d(th)
            if th.ndim == 1 and th.shape[0] == 1 and model.Ndim > 1:
                th = np.repeat(th, model.Ndim)
            if th.ndim == 1:
                th = np.tile(th[None, :], (K or 1, 1))
            elif K is not None and K != th.shape[0]:
                raise ParameterError("K does not match theta0.shape[0]")
            if th.ndim != 2 or th.shape[1] != model.Ndim:
                raise ParameterError("theta and model have incompatible shapes {} vs d={}"
                                     .format(th.shape, model.Ndim))
            self.K, self.d = th.shape
            self._squeeze = (self.K == 1 and np.ndim(theta0) <= 1)

        lib = _lib.load()
        ph = proposal._get_handle(self.d)
        if precision not in _lib.PRECISIONS:
            raise ParameterError("precision must be one of {}".format(sorted(_lib.PRECISIONS)))
        self.precision = precision
        prec = _lib.PRECISIONS[precision]
        nbytes = lib.rmn_sampler_workspace_bytes_ex(model._handle, ph, self.K, prec)
        if nbytes == 0:
            raise ParameterError(lib.rmn_last_error().decode() or
                                 "no device kernel for this model/proposal pair")
        self._ws = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
        h = C.c_void_p()
        _lib.check(lib.rmn_sampler_create_ex(C.byref(h), model._handle, ph, self.K, int(chain_offset),
                                             int(seed), _lib.ptr(self._ws), nbytes, prec))
        self._handle = h
        self.seed, self.chain_offset = int(seed), int(chain_offset)
        self.total_steps = 0
        self._tempered = _tempering is not None
        self._summary = None

        if move_schedule is not None:
            if move_schedule not in ("group", "chain"):
                raise ParameterError('move_schedule must be "group" or "chain"')
            _lib.check(lib.rmn_sampler_set_move_schedule(h, 1 if move_schedule == "group" else 0))
        self.row_sharded = bool(row_sharded)
        if self.row_sharded:                  # before the first evaluation: it already sums over the ranks' rows
            from ..distributed import exchange_unique_id, rank_world
            uid = exchange_unique_id(lambda buf, n: _lib.check(lib.rmn_nccl_unique_id(buf, n)))
            rank, world = rank_world()
            _lib.check(lib.rmn_sampler_set_row_comm(h, uid, len(uid), rank, world))
        if getattr(proposal, "_pooled_cov", False):      # the other ranks' chains join the covariance pool
            from ..distributed import exchange_unique_id, rank_world
            rank, world = rank_world()
            if world > 1:
                uid = exchange_unique_id(lambda buf, n: _lib.check(lib.rmn_nccl_unique_id(buf, n)))
                _lib.check(lib.rmn_sampler_set_row_comm(h, uid, len(uid), rank, world))
        if _tempering is not None:            # PTSampler: ladders along the chain axis, before the first evaluation
            betas, pswap = _tempering
            b = np.ascontiguousarray(betas, dtype=np.float64)
            _lib.check(lib.rmn_sampler_set_tempering(h, len(b), b.ctypes.data_as(C.c_void_p), float(pswap)))
        if self._is_cp:
            self._cp_upload(states)
        else:
            t = torch.as_tensor(np.ascontiguousarray(th), device="cuda")
            _lib.check(lib.rmn_sampler_set_state(h, _lib.ptr(t), _lib.stream_ptr()))
        th_now, lp_now = self._download_state()
        self._set_history([th_now], [lp_now])

    def __del__(self):
        try:
            if getattr(self, "_handle", None):
                _lib.load().rmn_sampler_destroy(self._handle)
                self._handle = None
        except Exception:
            pass

    # ------------------------------------------------------------------ state i/o
    def _cp_upload(self, states):
        torch = self._torch
        k, cpx, cpv, sig = pack_states(states)
        bufs = [torch.as_tensor(a, device="cuda") for a in (k, cpx, cpv, sig)]
        _lib.check(_lib.load().rmn_sampler_cp_set_state(
            self._handle, *[_lib.ptr(b) for b in bufs], _lib.stream_ptr()))
        torch.cuda.current_stream().synchronize()

    def _download_state(self):
        """Current state of all chains as host arrays (device -> host copy)."""
        torch, lib, K = self._torch, _lib.load(), self.K
        lp = torch.empty(K, dtype=torch.float64, device="cuda")
        if self._is_cp:
            k = torch.empty(K, dtype=torch.int32, device="cuda")
            cpx = torch.empty((K, LANES), dtype=torch.float64, device="cuda")
            cpv = torch.empty((K, LANES), dtype=torch.float64, device="cuda")
            sig = torch.empty(K, dtype=torch.float64, device="cuda")
            _lib.check(lib.rmn_sampler_cp_get_state(self._handle, _lib.ptr(k), _lib.ptr(cpx),
                                                    _lib.ptr(cpv), _lib.ptr(sig), _lib.ptr(lp),
                                                    _lib.stream_ptr()))
            return (k.cpu().numpy(), cpx.cpu().numpy(), cpv.cpu().numpy(), sig.cpu().numpy()), \
                lp.cpu().numpy()
        th = torch.empty((K, self.d), dtype=torch.float64, device="cuda")
        _lib.check(lib.rmn_sampler_get_state(self._handle, _lib.ptr(th), _lib.ptr(lp),
                                             _lib.stream_ptr()))
        return th.cpu().numpy(), lp.cpu().numpy()

    def state_tensors(self):
        """Current states as DEVICE tensors (theta[K,d], logpost[K]); fixed-d models only."""
        torch = self._torch
        th = torch.empty((self.K, self.d), dtype=torch.float64, device="cuda")
        lp = torch.empty(self.K, dtype=torch.float64, device="cuda")
        _lib.check(_lib.load().rmn_sampler_get_state(self._handle, _lib.ptr(th), _lib.ptr(lp),
                                                     _lib.stream_ptr()))
        return th, lp

    def set_state(self, theta):
        """Replace the states of all chains (re-evaluates log-posteriors on the device)."""
        if self._is_cp:
            self._cp_upload(list(theta))
        else:
            torch = self._torch
            t = torch.as_tensor(np.ascontiguousarray(np.asarray(theta, dtype=np.float64)
                                                     .reshape(self.K, self.d)), device="cuda")
            _lib.check(_lib.load().rmn_sampler_set_state(self._handle, _lib.ptr(t), _lib.stream_ptr()))
        th, lp = self._download_state()
        self._set_history([th], [lp])

    # ------------------------------------------------------------------ history
    def _set_history(self, thetas, logposts):
        """thetas/logposts: lists of per-record host arrays over all K chains."""
        if self._is_cp:
            k = np.stack([t[0] for t in thetas]); cpx = np.stack([t[1] for t in thetas])
            cpv = np.stack([t[2] for t in thetas]); sig = np.stack([t[3] for t in thetas])
            lp = np.stack(logposts)
            if self._squeeze:
                self._chain_thetas = [unpack_state(k[r, 0], cpx[r, 0], cpv[r, 0], sig[r, 0])
                                      for r in range(k.shape[0])]
                self._chain_logpost = [float(v) for v in lp[:, 0]]
            else:
                self._chain_thetas = ChangepointTrace(k, cpx, cpv, sig)
                self._chain_logpost = lp
        else:
            th = np.stack(thetas)
            lp = np.stack(logposts)
            if self._squeeze:
                self._chain_thetas = [th[r, 0].copy() for r in range(th.shape[0])]
                self._chain_logpost = [float(v) for v in lp[:, 0]]
            else:
                self._chain_thetas = th
                self._chain_logpost = lp

    def current_state(self):
        """(theta, log_posterior) of the current state (sampler.py:56-60)."""
        if self._squeeze:
            return self._chain_thetas[-1], self._chain_logpost[-1]
        if self._is_cp:
            return self._chain_thetas[len(self._chain_thetas) - 1], self._chain_logpost[-1]
        return self._chain_thetas[-1], self._chain_logpost[-1]

    def _add_state(self, theta, logpost):
        """sampler.py:62-70 hook: push an explicit state (it becomes the chain's state)."""
        self.set_state([theta] * self.K if self._is_cp else
                       np.tile(np.atleast_1d(theta)[None, :], (self.K, 1)) if np.ndim(theta) <= 1
                       else theta)

    # ------------------------------------------------------------------ running
    def _run_device(self, T, first_dev, thin, nrec, inject=None, extras=False):
        torch, K, d = self._torch, self.K, self.d
        tr = _lib.Trace()
        tr.first, tr.thin = int(first_dev), int(thin)
        bufs = {}
        if nrec > 0:
            bufs["lp"] = torch.empty((nrec, K), dtype=torch.float64, device="cuda")
            tr.d_logpost = bufs["lp"].data_ptr()
            if self._is_cp:
                bufs["k"] = torch.zeros((nrec, K), dtype=torch.int32, device="cuda")
                bufs["cpx"] = torch.empty((nrec, K, LANES), dtype=torch.float64, device="cuda")
                bufs["cpv"] = torch.empty((nrec, K, LANES), dtype=torch.float64, device="cuda")
                bufs["sig"] = torch.empty((nrec, K), dtype=torch.float64, device="cuda")
                tr.d_k, tr.d_cpx = bufs["k"].data_ptr(), bufs["cpx"].data_ptr()
                tr.d_cpv, tr.d_sig = bufs["cpv"].data_ptr(), bufs["sig"].data_ptr()
            else:
                bufs["theta"] = torch.empty((nrec, K, d), dtype=torch.float64, device="cuda")
                tr.d_theta = bufs["theta"].data_ptr()
        if extras:
            bufs["prop_lp"] = torch.empty((T, K), dtype=torch.float64, device="cuda")
            bufs["acc"] = torch.empty((T, K), dtype=torch.uint8, device="cuda")
            bufs["lqr"] = torch.empty((T, K), dtype=torch.float64, device="cuda")
            tr.d_prop_logpost, tr.d_accepted = bufs["prop_lp"].data_ptr(), bufs["acc"].data_ptr()
            tr.d_logqratio = bufs["lqr"].data_ptr()
            if self._is_cp:
                bufs["pk"] = torch.empty((T, K), dtype=torch.int32, device="cuda")
                bufs["pcpx"] = torch.empty((T, K, LANES), dtype=torch.float64, device="cuda")
                bufs["pcpv"] = torch.empty((T, K, LANES), dtype=torch.float64, device="cuda")
                bufs["psig"] = torch.empty((T, K), dtype=torch.float64, device="cuda")
                tr.d_prop_k, tr.d_prop_cpx = bufs["pk"].data_ptr(), bufs["pcpx"].data_ptr()
                tr.d_prop_cpv, tr.d_prop_sig = bufs["pcpv"].data_ptr(), bufs["psig"].data_ptr()
            else:
                bufs["pth"] = torch.empty((T, K, d), dtype=torch.float64, device="cuda")
                tr.d_prop_theta = bufs["pth"].data_ptr()
        inj = None
        if inject is not None:
            inj = _lib.Inject()
            keep = []
            for name in ("xi", "u", "tape", "usel"):
                if name in inject and inject[name] is not None:
                    t = torch.as_tensor(np.ascontiguousarray(inject[name], dtype=np.float64),
                                        device="cuda")
                    keep.append(t)
                    setattr(inj, "d_" + name, t.data_ptr())
            bufs["_inj"] = keep
        _lib.check(_lib.load().rmn_sampler_run(
            self._handle, int(T), C.byref(inj) if inj is not None else None, C.byref(tr),
            _lib.stream_ptr()))
        self.total_steps += int(T)
        return bufs

    def run(self, Nsamples, Nburn=0, Nthin=1, trace=True, inject=None, extras=False):
        """
        Run every chain for Nsamples MH iterations (sampler.py:44-54).  The history
        afterwards is ``[start state + Nsamples states][Nburn::Nthin]`` exactly as in the
        reference; with ``trace=False`` only the final state is kept (no trace memory).
        """
        T = int(Nsamples)
        if T < 0 or Nburn < 0 or Nthin < 1:
            raise ParameterError("need Nsamples >= 0, Nburn >= 0, Nthin >= 1")
        start_th, start_lp = self._last_record()
        if not trace:
            out = self._run_device(T, 0, 1, 0, inject, extras)
            th, lp = self._download_state()
            self._set_history([th], [lp])
            self._refresh_adapt()
            return self._extras(out) if extras else None
        first_dev = Nburn if Nburn >= 1 else Nthin
        nrec = 0 if first_dev > T else (T - first_dev) // Nthin + 1
        per_rec = self.K * ((2 * LANES + 3) if self._is_cp else (self.d + 1)) * 8
        if nrec * per_rec > TRACE_BYTES_LIMIT:
            raise ParameterError("trace of {} records x {} chains needs {:.1f} GB; raise Nthin/Nburn "
                                 "or pass trace=False".format(nrec, self.K, nrec * per_rec / 2**30))
        bufs = self._run_device(T, first_dev, Nthin, nrec, inject, extras)
        thetas, lps = [], []
        if Nburn == 0:
            thetas.append(start_th)
            lps.append(start_lp)
        if nrec > 0:
            lp = bufs["lp"].cpu().numpy()
            if self._is_cp:
                k, cpx, cpv, sig = (bufs[n].cpu().numpy() for n in ("k", "cpx", "cpv", "sig"))
                thetas += [(k[r], cpx[r], cpv[r], sig[r]) for r in range(nrec)]
            else:
                th = bufs["theta"].cpu().numpy()
                thetas += [th[r] for r in range(nrec)]
            lps += [lp[r] for r in range(nrec)]
        if not thetas:          # Nburn > Nsamples: empty history, like the reference's slice
            th, lp = self._download_state()
            self._set_history([th], [lp])
            if self._squeeze:
                self._chain_thetas, self._chain_logpost = [], []
        else:
            self._set_history(thetas, lps)
        self._final_state_cache = None
        self._refresh_adapt()
        if extras:
            return self._extras(bufs)
        return None

    def _extras(self, bufs):
        """Per-step proposal record: what Proposal.propose returned and what the sampler decided."""
        out = {"prop_logpost": bufs["prop_lp"].cpu().numpy(),
               "accepted": bufs["acc"].cpu().numpy().astype(bool),
               "logqratio": bufs["lqr"].cpu().numpy()}
        if self._is_cp:
            out.update(prop_k=bufs["pk"].cpu().numpy(), prop_cpx=bufs["pcpx"].cpu().numpy(),
                       prop_cpv=bufs["pcpv"].cpu().numpy(), prop_sig=bufs["psig"].cpu().numpy())
        else:
            out["prop_theta"] = bufs["pth"].cpu().numpy()
        return out

    def run_injected(self, xi=None, u=None, tape=None, Nburn=0, Nthin=1, usel=None):
        """
        Replay a given noise stream instead of Philox (parity mode):
        fixed-d: xi[T, K, d] (or [T, d] for K = 1) and u[T, K]; changepoint: tape[T, K, NSLOT].  Tempered samplers
        also take usel[T, K], the swap-selection uniforms.
        Returns the per-step proposal record: 'prop_theta' [T,K,d] (or prop_k/cpx/cpv/sig),
        'logqratio', 'prop_logpost', 'accepted' [T,K].
        """
        if self._is_cp:
            tape = np.asarray(tape, dtype=np.float64)
            if tape.ndim == 2:
                tape = tape[:, None, :]
            if tape.shape[1:] != (self.K, _lib.CP_NSLOT):
                raise ParameterError("tape must have shape [T, K, {}]".format(_lib.CP_NSLOT))
            T, inj = tape.shape[0], {"tape": tape}
            if usel is not None:                       # tempered samplers: swap-selection uniforms
                usel = np.asarray(usel, dtype=np.float64)
                if usel.ndim == 1:
                    usel = usel[:, None]
                if usel.shape != tape.shape[:2]:
                    raise ParameterError("usel must be [T, K] like the tape")
                inj["usel"] = usel
        else:
            xi = np.asarray(xi, dtype=np.float64)
            u = np.asarray(u, dtype=np.float64)
            if xi.ndim == 2:
                xi = xi[:, None, :]
            if u.ndim == 1:
                u = u[:, None]
            if xi.shape[1:] != (self.K, self.d) or u.shape != xi.shape[:2]:
                raise ParameterError("xi must be [T, K, d] and u [T, K]")
            T, inj = xi.shape[0], {"xi": xi, "u": u}
            if usel is not None:                       # tempered samplers: swap-selection uniforms
                usel = np.asarray(usel, dtype=np.float64)
                if usel.shape != u.shape:
                    raise ParameterError("usel must be [T, K] like u")
                inj["usel"] = usel
        return self.run(T, Nburn, Nthin, trace=True, inject=inj, extras=True)

    def _last_record(self):
        th, lp = self._download_state()
        return th, lp

    def sample(self):
        """One MH iteration for every chain (sampler.py:72-90); appends to the history."""
        prev_t, prev_l = self._chain_thetas, self._chain_logpost
        self.run(1, 1, 1)
        new_t, new_l = self._chain_thetas, self._chain_logpost
        if self._squeeze:
            self._chain_thetas = list(prev_t) + list(new_t)
            self._chain_logpost = list(prev_l) + list(new_l)
        elif self._is_cp:
            self._chain_thetas = ChangepointTrace(
                *[np.concatenate([getattr(prev_t, n), getattr(new_t, n)]) for n in ("k", "cpx", "cpv", "sig")])
            self._chain_logpost = np.concatenate([prev_l, new_l])
        else:
            self._chain_thetas = np.concatenate([prev_t, new_t])
            self._chain_logpost = np.concatenate([prev_l, new_l])
        return self.current_state()

    # ------------------------------------------------------------------ adaptation / diagnostics
    def _refresh_adapt(self):
        p = self.proposal
        if getattr(p, "_adapt_cov", False):            # AdaptCovProposal.L / .C (adaptive.py:61-63, 101-102)
            torch = self._torch
            L = torch.empty((self.K, self.d, self.d), dtype=torch.float64, device="cuda")
            _lib.check(_lib.load().rmn_sampler_get_adaptcov(self._handle, _lib.ptr(L), _lib.stream_ptr()))
            L = L.cpu().numpy()
            dd = float(self.d) ** 0.2 if self.total_steps >= 4 else 1.0   # before the first adaptation L = chol(C0)
            Cm = np.einsum("kij,klj->kil", L * dd, L * dd)          # L = chol(C) / d**0.2  (adaptive.py:101-102)
            p.L, p.C = (L[0], Cm[0]) if self.K == 1 else (L, Cm)
            if hasattr(p, "chM"):                                   # AdaptCovHMC: M = C, chM = L (hamiltonian.py:117)
                p.M, p.chM = p.C, p.L
        if getattr(p, "_pooled_cov", False):           # PooledAdaptCovRandomWalk: the population estimate
            torch = self._torch
            Cm = torch.empty((self.d, self.d), dtype=torch.float64, device="cuda")
            mean = torch.empty(self.d, dtype=torch.float64, device="cuda")
            cnt = torch.empty(1, dtype=torch.float64, device="cuda")
            _lib.check(_lib.load().rmn_sampler_get_pooled_cov(self._handle, _lib.ptr(Cm), _lib.ptr(mean), _lib.ptr(cnt),
                                                              _lib.stream_ptr()))
            p.pool_count = float(cnt.cpu().numpy()[0])
            if p.pool_count > 0:
                p.C, p.pool_mean = Cm.cpu().numpy(), mean.cpu().numpy()
        if not getattr(p, "_adaptive", False):
            return
        torch, K = self._torch, self.K
        sc = torch.empty(K, dtype=torch.float64, device="cuda")
        ns = torch.empty(K, dtype=torch.int64, device="cuda")
        na = torch.empty(K, dtype=torch.int64, device="cuda")
        _lib.check(_lib.load().rmn_sampler_get_adapt(self._handle, _lib.ptr(sc), _lib.ptr(ns),
                                                     _lib.ptr(na), _lib.stream_ptr()))
        sc, ns, na = sc.cpu().numpy(), ns.cpu().numpy(), na.cpu().numpy()
        rate = na / np.maximum(ns, 1)
        if K == 1:
            p.scale, p.Nsamples, p.Naccepts, p.accept_rate = float(sc[0]), int(ns[0]), int(na[0]), float(rate[0])
        else:
            p.scale, p.Nsamples, p.Naccepts, p.accept_rate = sc, ns, na, rate
        if hasattr(p, "eps0"):
            p.eps = p.scale * p.eps0                    # hamiltonian.py:102

    def set_adapt(self, scale=None, nsamples=None, naccepts=None):
        """Set the per-chain AdaptScale state (scalars broadcast over chains)."""
        torch, K = self._torch, self.K
        def dev(v, dt):
            if v is None:
                return None
            return torch.as_tensor(np.broadcast_to(np.asarray(v), (K,)).copy(), device="cuda").to(dt)
        sc, ns, na = dev(scale, torch.float64), dev(nsamples, torch.int64), dev(naccepts, torch.int64)
        _lib.check(_lib.load().rmn_sampler_set_adapt(self._handle, _lib.ptr(sc), _lib.ptr(ns),
                                                     _lib.ptr(na), _lib.stream_ptr()))
        torch.cuda.current_stream().synchronize()

    def get_checkpoint(self):
        """Everything needed to resume bit-for-bit: states, Philox step counter, AdaptScale state.
        Proposals that carry MORE per-chain state than that -- the Haario accumulators and Cholesky factor of the
        covariance-adapting proposals (adaptive.py:38-103), AdaptScalepCN's compounding rho (randomwalk.py:118) -- have no
        read/write ABI for it, so a checkpoint of them would resume silently different chains: refused."""
        p = self.proposal
        if getattr(p, "_adapt_cov", False) or getattr(p, "_pooled_cov", False) or type(p).__name__ == "AdaptScalepCN":
            raise ParameterError("get_checkpoint: {} keeps per-chain adaptation state (covariance accumulators / rho) "
                                 "that cannot be saved; checkpoint/resume covers fixed and AdaptScale proposals"
                                 .format(type(p).__name__))
        th, lp = self._download_state()
        ck = {"state": th, "step": int(_lib.load().rmn_sampler_get_step(self._handle)),
              "seed": self.seed, "chain_offset": self.chain_offset}
        if getattr(self.proposal, "_adaptive", False):
            self._refresh_adapt()
            p = self.proposal
            ck["adapt"] = (np.atleast_1d(p.scale).copy(), np.atleast_1d(p.Nsamples).copy(),
                           np.atleast_1d(p.Naccepts).copy())
        return ck

    def set_checkpoint(self, ck):
        if self._is_cp:
            k, cpx, cpv, sig = ck["state"]
            self.set_state([unpack_state(k[i], cpx[i], cpv[i], sig[i]) for i in range(self.K)])
        else:
            self.set_state(ck["state"])
        _lib.check(_lib.load().rmn_sampler_set_step(self._handle, int(ck["step"])))
        if "adapt" in ck:
            self.set_adapt(*ck["adapt"])
            self._refresh_adapt()

    def reset_diagnostics(self):
        _lib.check(_lib.load().rmn_sampler_reset_diagnostics(self._handle, _lib.stream_ptr()))

    def diagnostics_block(self):
        """Device tensor with the per-device diagnostics block (see riemann_b200.h)."""
        torch = self._torch
        nd = _lib.load().rmn_sampler_diag_dim(self._handle)
        blk = torch.zeros(_lib.DIAG_HDR + 3 * nd, dtype=torch.float64, device="cuda")
        _lib.check(_lib.load().rmn_sampler_reduce_diagnostics(self._handle, _lib.ptr(blk),
                                                              _lib.stream_ptr()))
        return blk

    def chain_moments(self):
        """Per-chain mean and (biased) variance of the tracked functionals since the last reset: two host arrays
        [nd, K] (rmn_sampler_chain_moments)."""
        torch = self._torch
        nd = _lib.load().rmn_sampler_diag_dim(self._handle)
        m = torch.empty((nd, self.K), dtype=torch.float64, device="cuda")
        v = torch.empty((nd, self.K), dtype=torch.float64, device="cuda")
        _lib.check(_lib.load().rmn_sampler_chain_moments(self._handle, _lib.ptr(m), _lib.ptr(v), _lib.stream_ptr()))
        return m.cpu().numpy(), v.cpu().numpy()

    def diagnostics(self, allreduce=True):
        """
        Acceptance rate, per-functional posterior mean/variance, split-free R-hat, tau and
        total ESS over ALL chains since the last reset.  With torch.distributed initialised
        the block is summed over ranks first (one small NCCL all-reduce per batch).
        """
        from ..distributed import reduce_block, summarize_block
        blk = self.diagnostics_block()
        if allreduce and not self.row_sharded:      # row-sharded: every rank holds the SAME K chains, nothing to add up
            blk = reduce_block(blk)
        return summarize_block(blk.cpu().numpy())

    # ------------------------------------------------------------------ posterior summaries (changepoint model)
    def set_posterior_summary(self, grid, value_range=None, value_bins=128, every=16):
        """
        Accumulate posterior summaries on the device from the next run on (rmn_sampler_cp_set_summary): after every MH
        step whose global index is a multiple of `every`, every chain's state adds to integer histograms of the number
        of changepoints, of the changepoint locations over the cells of `grid`, and of the posterior predictive
        ChangepointRegression1D.predict(theta, grid[g]) at every grid point over `value_bins` equal bins of
        `value_range` = (vlo, vhi) plus an under- and an overflow bin.  No trace is kept.  The counts are reset now and
        by reset_diagnostics, so they cover the same window as the diagnostics.  grid=None turns the summaries off.
        Untempered changepoint samplers only (PTSampler.set_posterior_summary serves one rung of a tempering ladder).
        """
        if not self._is_cp or self._tempered:
            raise ParameterError("posterior summaries are available for untempered changepoint samplers only")
        lib = _lib.load()
        if grid is None:
            _lib.check(lib.rmn_sampler_cp_set_summary(self._handle, 0, None, 0.0, 0.0, 0, 0))
            self._summary = None
            return
        from ..posterior_summary import check_summary_args
        g, vlo, vhi, H, every = check_summary_args(grid, value_range, value_bins, every)
        _lib.check(lib.rmn_sampler_cp_set_summary(self._handle, len(g), _lib.ptr(g), vlo, vhi, H, every))
        self._summary = (g, vlo, vhi, H)

    def posterior_summary(self, allreduce=True):
        """
        The summary counts since the last reset as a PosteriorSummary (riemann_b200/posterior_summary.py): grid,
        value_edges, khist, cpxhist, yhist, nsamples, and the binned estimates yhat_mean / yhat_quantiles(q).  With
        torch.distributed initialised the int64 counts are summed over the ranks (their chains are disjoint shards).
        """
        if self._summary is None:
            raise ParameterError("no posterior summary is set (set_posterior_summary)")
        return self._read_summary(self._summary, allreduce)

    def _read_summary(self, spec, allreduce):
        """The device counts (rmn_sampler_cp_get_summary) as a PosteriorSummary; spec = (grid, vlo, vhi, H) as set.
        Shared by posterior_summary and PTSampler.posterior_summary."""
        from ..distributed import reduce_counts
        from ..posterior_summary import PosteriorSummary
        torch, (g, vlo, vhi, H) = self._torch, spec
        G, L = len(g), _lib.CP_LANES
        buf = torch.zeros(1 + L + (G + 1) + G * (H + 2), dtype=torch.int64, device="cuda")
        ns = C.c_int64()
        _lib.check(_lib.load().rmn_sampler_cp_get_summary(
            self._handle, C.c_void_p(buf.data_ptr() + 8), C.c_void_p(buf.data_ptr() + 8 * (1 + L)),
            C.c_void_p(buf.data_ptr() + 8 * (2 + L + G)), C.byref(ns), _lib.stream_ptr()))
        buf[0] = ns.value
        if allreduce:
            buf = reduce_counts(buf)
        c = buf.cpu().numpy()
        return PosteriorSummary(g, vlo, vhi, c[1:1 + L], c[1 + L:2 + L + G], c[2 + L + G:].reshape(G, H + 2), c[0])

    # ------------------------------------------------------------------ trace wire format (SURVEY 8f N4)
    def save_trace(self, path):
        """Write the current history (`_chain_thetas` / `_chain_logpost`, i.e. the thinned device trace
        of the last run) to a compressed .npz: `theta[rec, K, d]` (or k / cpx / cpv / sig for the
        changepoint model), `logpost[rec, K]`, plus seed, chain offset, step counter and precision --
        enough to resume with `Sampler(..., theta0=last record)` + `rmn_sampler_set_step`."""
        meta = dict(seed=np.int64(self.seed), chain_offset=np.int64(self.chain_offset),
                    step=np.int64(_lib.load().rmn_sampler_get_step(self._handle)), K=np.int64(self.K),
                    precision=np.array(self.precision))
        lp = np.asarray(self._chain_logpost, dtype=np.float64)
        if self._is_cp:
            tr = self._chain_thetas
            if isinstance(tr, list):
                k, cpx, cpv, sig = pack_states(tr)
                k, cpx, cpv, sig = k[:, None], cpx[:, None], cpv[:, None], sig[:, None]
            else:
                k, cpx, cpv, sig = tr.k, tr.cpx, tr.cpv, tr.sig
            np.savez_compressed(path, k=k, cpx=cpx, cpv=cpv, sig=sig, logpost=lp.reshape(k.shape[0], -1), **meta)
        else:
            th = np.asarray(self._chain_thetas, dtype=np.float64)
            th = th.reshape(th.shape[0], self.K, self.d)
            np.savez_compressed(path, theta=th, logpost=lp.reshape(th.shape[0], self.K), **meta)

    @staticmethod
    def load_trace(path):
        """-> dict of the arrays `save_trace` wrote."""
        with np.load(path, allow_pickle=False) as z:
            return {k: z[k] for k in z.files}

    def enable_kernel_timing(self, enable=True):
        """CUDA-event timing of the dominant kernel's launches (measurement aid, see bench.py)."""
        _lib.check(_lib.load().rmn_sampler_enable_kernel_timing(self._handle, 1 if enable else 0))

    def kernel_timing(self):
        """-> dict(kernel, total_ms, launches, untimed) since the previous call; synchronizes."""
        ms, n, un, name = C.c_double(), C.c_int64(), C.c_int64(), C.c_char_p()
        _lib.check(_lib.load().rmn_sampler_kernel_timing(self._handle, C.byref(ms), C.byref(n), C.byref(un),
                                                         C.byref(name)))
        return {"kernel": (name.value or b"").decode(), "total_ms": ms.value, "launches": n.value,
                "untimed": un.value}

    @property
    def launch_count(self):
        return int(_lib.load().rmn_sampler_launch_count(self._handle))
