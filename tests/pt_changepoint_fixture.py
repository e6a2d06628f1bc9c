"""
PTSampler on the changepoint model: the replay draw source and the recorder of tests/golden/pt_changepoint.npz.

The port's PTSampler (oracle/riemann_port.py) runs on the reference's rules; `PTSlotTapeDraws` lets it replay a
recorded stream, and `pt_changepoint_arrays` records one, from the reference (R = oracle.refshim.load_reference())
or from the port (R = oracle.riemann_port: its module-level classes have the reference's names and signatures).

    python tests/pt_changepoint_fixture.py      # rewrites tests/golden/pt_changepoint.npz (from the port when the
                                                # reference tree is absent; the file records its `source`)
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import refshim                               # noqa: E402
from oracle import riemann_port as port                  # noqa: E402
from oracle.gen_golden import LANES, _cp_pack_state, _cp_tape_row   # noqa: E402


class PTSlotTapeDraws(port.PTTapeDraws):
    """Replay for the port's PTSampler on the changepoint proposal: usel[T, Nt] selection uniforms and a slot tape
    tape[T, Nt, NSLOT] (port.CP_SLOT_*), addressed by the chain the draw is made for.  The "acc" role is the accept
    uniform of a within-chain step or, for a swap initiator, the swap uniform (both in CP_SLOT_ACC)."""

    def __init__(self, usel, tape):
        self.usel, self.tape = (np.asarray(a, dtype=np.float64) for a in (usel, tape))
        self.t, self.i = 0, 0

    def normal(self, role, n):
        return self.tape[self.t, self.i, port.CP_SLOT_XI:port.CP_SLOT_XI + n].copy()

    def uniform(self, role, low=0.0, high=1.0):
        if role == "ptsel":
            return self.usel[self.t, self.i]
        return self.tape[self.t, self.i, port.SlotTapeDraws._slot[role]]      # stored already scaled

    def randint(self, role, n):
        return int(self.tape[self.t, self.i, port.CP_SLOT_N])


def step_draws(log, k):
    """Number of log entries one within-chain changepoint step takes (the control flow _cp_tape_row maps:
    examples/test_changepoint.py:44-73 + sampler.py:84), for a log that goes on with the ladder's other chains."""
    n = 1
    if float(log[0][1]) >= 0.20:
        n += 1
        if float(log[1][1]) >= 0.40:
            n += 1
            if float(log[2][1]) >= 0.60:
                birth = True
                if k > 0:
                    birth = float(log[n][1]) > 0.5
                    n += 1
                n += 2 if birth else 1                  # s, du or randint(k)
                return n + 1                            # accept uniform
    return n + 2                                        # normals, accept uniform


def pt_changepoint_arrays(R, T=1500, seed=605, betas=None, Pswap=0.1):
    """PTSampler on the changepoint model (default ladder 0.5**arange(5), the bench problem) with every draw recorded.
    Per PT step and chain i: one selection uniform; then, unless the chain was swapped by its upper neighbour, either a
    within-chain step (its draws mapped onto the slot tape by _cp_tape_row) or one swap uniform (the ACC slot).  An
    explicit ladder (`betas`) needs the port: the reference's `betas=` branch raises (ptsampler.py:62)."""
    pm, pprop, ptheta0, _ = port.make_changepoint_problem()
    model = R.ChangepointRegression1D(pm.x, pm.y, pm.xmin, pm.xmax, pm.lamb, pm.kmax, pm.alpha, pm.beta)
    prop = R.ChangepointRegression1DProp(model, pprop.hscale)
    np.random.seed(seed)
    with refshim.quiet():
        kw = {} if betas is None else {"betas": betas}
        pt = R.PTSampler(model, prop, R.ChangepointParams(ptheta0.cpx, ptheta0.cpv, ptheta0.sig), Pswap=Pswap, **kw)
    nt = len(pt.betas)
    usel, tape = np.zeros((T, nt)), np.zeros((T, nt, port.cp_nslot(LANES)))
    kind = np.zeros((T, nt), dtype=np.int8)            # 0 within-chain step, 1 swap initiator, 2 swapped partner
    with refshim.quiet(), np.errstate(all="ignore"), refshim.RecordingRNG() as rec:
        for t in range(T):
            a = rec.mark()
            pt.sample()
            log = rec.log[a:rec.mark()]
            k, i = 0, 0
            while i < nt:
                assert log[k][0] == "uniform"
                usel[t, i] = float(log[k][1]); k += 1
                if i > 0 and kind[t, i - 1] == 1:
                    kind[t, i] = 2
                elif usel[t, i] > pt.Pswap or i == nt - 1:
                    kc = len(pt.samplers[i]._chain_thetas[t].cpx)         # the chain's state before step t
                    n = step_draws(log[k:], kc)
                    tape[t, i] = _cp_tape_row(log[k:k + n], kc)
                    k += n
                else:
                    assert log[k][0] == "uniform"
                    kind[t, i] = 1; tape[t, i, port.CP_SLOT_ACC] = float(log[k][1]); k += 1
                i += 1
            assert k == len(log), (k, len(log))
    st = [[_cp_pack_state(th) for th in s._chain_thetas] for s in pt.samplers]        # [nt][T+1]
    assert max(x[0] for r in st for x in r) < LANES
    return dict(usel=usel, tape=tape, kind=kind, betas=np.asarray(pt.betas, dtype=np.float64),
                pswap=np.float64(pt.Pswap),
                k=np.array([[x[0] for x in r] for r in st], dtype=np.int32),
                cpx=np.array([[x[1] for x in r] for r in st]), cpv=np.array([[x[2] for x in r] for r in st]),
                sig=np.array([[x[3] for x in r] for r in st]),
                logpost=np.array([[float(np.squeeze(v)) for v in s._chain_logpost] for s in pt.samplers]),
                seed=np.int64(seed))


def main():
    if refshim.reference_available():
        R, source = refshim.load_reference(), "reference"
    else:
        R, source = port, "port"
    out = pt_changepoint_arrays(R)
    np.savez_compressed(os.path.join(ROOT, "tests", "golden", "pt_changepoint.npz"), source=np.array(source), **out)
    kind, k = out["kind"], out["k"]
    print("pt_changepoint: T=%d nt=%d swaps proposed=%d, k in [%d,%d] (source: %s)" % (
        kind.shape[0], kind.shape[1], int((kind == 1).sum()), k.min(), k.max(), source))


if __name__ == "__main__":
    main()
