// riemann_b200 -- fused T-step MH kernel for the changepoint regression model.
//
// GL lanes cooperate on one chain; the variable-dimension state (k <= LANES-1 changepoints)
// is held in shared-memory slots of the group's lanes, so insert/delete are loads of the
// neighbouring element's slot.  Per iteration the kernel replaces
//   Sampler.sample                                riemann/samplers/sampler.py:72-90
//   ChangepointRegression1DProp.propose           examples/test_changepoint.py:44-73
//   MetropolisRandomWalk.propose (3 block moves)  riemann/proposals/randomwalk.py:21-26
//   add_changepoint / subtract_changepoint        riemann/models/changepoint.py:193-240
//   ChangepointRegression1D.log_likelihood/log_prior/predict   changepoint.py:106-160,181
//   Model.log_posterior                           riemann/models/model.py:43-55
//
// Likelihood: x is sorted, so the prediction is constant on runs of data points; with
// prefix sums cy[i] = sum_{m<i} (y_m - c), cyy[i] = sum_{m<i} (y_m - c)^2 the residual
// sum of squares of segment j is  n_j (v_j-c)^2 - 2 (v_j-c) S1_j + S2_j,  where the run
// boundaries b_j = #{x_i <= cpx_j} come from a bucket table or a branch-free binary search
// (changepoint.cuh: run_boundary; equivalent to np.searchsorted(cpx, x), changepoint.py:181).
// O(k) or O(k log M) instead of O(M) per evaluation; all arithmetic fp64 like the reference.
// The data tables are staged in shared memory once per block and reused by all chains and
// all T iterations.
//
// Reference behaviours reproduced (SURVEY.md appendix A 10-12): k = number of STEPS in
// the three k-terms of the prior; constraints enforced only through nan/inf -> -inf;
// a fresh uniform per block-selection elif; trans-dimensional moves use log|J| alone
// as logqratio.
#include "changepoint.cuh"
#include <stdlib.h>
#include <algorithm>

#ifndef RMN_CP_DEFAULT_GL
#define RMN_CP_DEFAULT_GL 4
#endif


namespace {
using namespace cp;

// ---------------------------------------------------------------------------------------
// Group geometry.  GL lanes cooperate on one chain (32/GL chains per warp); lane l owns the
// EPL = LANES/GL elements e = l + GL*j, j = 0..EPL-1 ("row" j) of cpx, cpv and of the cached
// run boundaries (shared-memory slots for the state, registers for the proposal, statically
// indexed).  Rows beyond the warp's largest extent hold
// the canonical padding (cpx = 0, cpv = 0, boundary = M) and are skipped by a warp-uniform
// guard, so with the typical 3..8 changepoints a GL = 4 warp spends its instructions on 8
// chains and two rows instead of on 2 chains and ten idle lanes.
// ---------------------------------------------------------------------------------------
template <int GL> struct Geo {
    static_assert(GL == 4 || GL == 8 || GL == 16, "GL must be 4, 8 or 16");
    static constexpr int EPL = LANES / GL;
    static constexpr int LOG = (GL == 4) ? 2 : ((GL == 8) ? 3 : 4);
    static constexpr int NS = (RMN_CP_NDIAG + GL - 1) / GL;     // diagnostics slots per lane
    // rows below ALWAYS are processed unconditionally (straight-line code, the rows' dependent chains
    // interleave); only the rows above carry the warp-uniform guard.  12 elements cover k <= 10.
    static constexpr int ALWAYS = (GL == 4) ? 3 : EPL;
};

template <int GL>
__device__ __forceinline__ unsigned gballot(bool pred) {
    const unsigned full = __ballot_sync(0xffffffffu, pred);
    return (full >> (threadIdx.x & 31 & ~(GL - 1))) & ((1u << GL) - 1u);
}

template <int GL>
__device__ __forceinline__ double gsum(double v) {
#pragma unroll
    for (int o = GL / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o, GL);
    return v;
}

template <int GL>
__device__ __forceinline__ double gprod(double v) {
#pragma unroll
    for (int o = GL / 2; o > 0; o >>= 1) v *= __shfl_xor_sync(0xffffffffu, v, o, GL);
    return v;
}

// row j is live for this warp-step iff it can hold an element of any chain of the warp:
// elements 0..k+1 (k+1 after a birth), kw = warp maximum of k
#define ROW_ON(j) ((j) < Geo<GL>::ALWAYS || (j) * GL <= kw + 1)

// value of element e-1 for every row (element -1 = `first`)
template <int GL, typename T>
__device__ __forceinline__ void shift_prev(const T (&a)[Geo<GL>::EPL], T (&out)[Geo<GL>::EPL], T first,
                                           int lane, int kw) {
#pragma unroll
    for (int j = 0; j < Geo<GL>::EPL; ++j) {
        out[j] = a[j];
        if (ROW_ON(j)) {
            const T up = __shfl_up_sync(0xffffffffu, a[j], 1, GL);
            T w = first;
            if (j > 0) w = __shfl_sync(0xffffffffu, a[j > 0 ? j - 1 : 0], GL - 1, GL);
            out[j] = (lane == 0) ? w : up;
        }
    }
}

// value of element e+1 for every row (element LANES = `pad`)
template <int GL, typename T>
__device__ __forceinline__ void shift_next(const T (&a)[Geo<GL>::EPL], T (&out)[Geo<GL>::EPL], T pad,
                                           int lane, int kw) {
    constexpr int EPL = Geo<GL>::EPL;
#pragma unroll
    for (int j = 0; j < EPL; ++j) {
        out[j] = a[j];
        if (ROW_ON(j)) {
            const T dn = __shfl_down_sync(0xffffffffu, a[j], 1, GL);
            T w = pad;
            if (j + 1 < EPL) w = __shfl_sync(0xffffffffu, a[j + 1 < EPL ? j + 1 : j], 0, GL);
            out[j] = (lane == GL - 1) ? w : dn;
        }
    }
}

// The accepted state's rows live in shared memory for the duration of cp_block: slot [j][t] holds row j of thread t, so
// element e of the chain of the group whose first thread is gb sits in slot [e / GL][gb + e % GL], and every thread
// reads and writes its own slots in consecutive (conflict-free) words.  Reading another lane's slot needs a __syncwarp
// after that lane's last write (see cp_block).
template <int GL, typename T>
using Rows = T[Geo<GL>::EPL][128];

// element e of the chain, e in [0, LANES)
template <int GL, typename T>
__device__ __forceinline__ T elem_at(const Rows<GL, T>& a, int e) {
    return a[e >> Geo<GL>::LOG][(threadIdx.x & ~(GL - 1)) + (e & (GL - 1))];
}

// element e + off of the chain, off in {-1, 0, +1} chosen per chain (birth: -1 above the insertion point, death: +1
// from the removed element on, everything else 0); elements -1 and LANES read `pad`
template <int GL, typename T>
__device__ __forceinline__ T shifted(const Rows<GL, T>& a, int e, int off, T pad) {
    const int s = e + off;
    return ((unsigned)s < (unsigned)LANES) ? elem_at<GL, T>(a, s) : pad;
}

// #{e < k : cpx[e] < s}   (np.searchsorted(cpx, s), changepoint.py:206)
template <int GL>
__device__ __forceinline__ int count_below(const Rows<GL, double>& cx, int lane, int k, double s, int kw) {
    int n = 0;
#pragma unroll
    for (int j = 0; j < Geo<GL>::EPL; ++j)
        if (ROW_ON(j)) n += __popc(gballot<GL>(lane + GL * j < k && cx[j][threadIdx.x] < s));
    return n;
}

// ---------------------------------------------------------------------------------------
// Log-posterior of one state held across the GL lanes of a group, in three pieces, so that a move
// which leaves part of the state alone reuses the cached pieces of the current state:
//   cp_terms     per element: residual sum of squares of its run of data (prefix sums) -> ss,
//                height-prior term (changepoint.py:18-19,136) -> vt, gap to the previous changepoint
//                (:142-143) -> product gp.  The sum over changepoints of log(gap) is taken as ONE log of
//                the product of the gaps (a negative gap poisons the product with nan, exactly what a sum
//                containing log(negative) gives numpy; a zero gap gives -inf either way).
//   log4         the step's fp64 logarithms -- log gp, log sigma^2, log u (accept test), log|J| -- batched
//                on lanes 0..3 of the group: ONE `log` call per warp-step.
//   cp_assemble  the scalar arithmetic of changepoint.py:118-125,128-160 and model.py:50-54;
//                log(1/sigma^2) (:148) is -log(sigma^2) (+inf where 1/sigma^2 overflows, as in numpy).
// Every floating-point operation that is shared between the general path and the move-specific fast
// paths of the kernel is written with explicit round-to-nearest intrinsics, so all paths give the same
// bits (no context-dependent FMA contraction).  Differences from numpy's term-by-term sums are O(1e-15)
// relative (tests: 1e-9).
// ---------------------------------------------------------------------------------------
template <int GL>
__device__ __forceinline__ void cp_terms(const CPParams& P, const double2* __restrict__ cyc, int lane, int kw, int kk,
                                         const double (&nx)[Geo<GL>::EPL], const double (&nv)[Geo<GL>::EPL],
                                         const int (&nbu)[Geo<GL>::EPL], bool wss, bool wvt, bool wgp,
                                         double& ss, double& vt, double& gp) {
    // wss / wvt / wgp are WARP-UNIFORM: which of the three sums any chain of the warp needs recomputed.
    // Inside a live row every lane computes its element's term; elements beyond the chain's extent (e > kk, canonical
    // padding: cpx = 0, cpv = 0, boundary = M) contribute an exact identity instead of being branched around, so the
    // rows are straight-line code.  Each sum starts at +0.0 and a round-to-nearest sum that starts at +0.0 is never -0.0,
    // so adding +0.0 changes no bit of it; multiplying by 1.0 changes no bit of the product.
    constexpr int EPL = Geo<GL>::EPL;
    if (wss) {
        int pb[EPL];
        shift_prev<GL, int>(nbu, pb, 0, lane, kw);
        double a = 0.0;
#pragma unroll
        for (int j = 0; j < EPL; ++j) {
            if (ROW_ON(j)) {
                // taken as computed: a padding element has bu = bl = M (its predecessor is padding or the last step,
                // whose boundary is M too), so n = 0 and s1 = s2 = +0.0 exactly, and with cpv = 0 the finite vc gives
                // (-2 vc) s1 + s2 = +0.0 and (n vc) vc + 0.0 = +0.0.  This needs finite data: vc = -ycenter, cy[M] and
                // cyy[M] finite.  With non-finite data the term is NaN and can turn an infinite ss into NaN; the
                // log-likelihood is -inf either way (cp_assemble maps NaN to -inf), so no chain changes.
                const int bu = nbu[j], bl = pb[j];
                const double n = (double)(bu - bl);
                const double2 pu = cyc[bu], pl = cyc[bl];                                 // {cy, cyy}: one load each
                const double s1 = __dsub_rn(pu.x, pl.x);
                const double s2 = __dsub_rn(pu.y, pl.y);
                const double vc = __dsub_rn(nv[j], P.ycenter);
                a = __dadd_rn(a, __fma_rn(__dmul_rn(n, vc), vc, __fma_rn(-2.0 * vc, s1, s2)));   // n vc^2 - 2 vc s1 + s2
            }
        }
        ss = gsum<GL>(a);
    }
    if (wgp) {
        double px[EPL];
        shift_prev<GL, double>(nx, px, P.xmin, lane, kw);
        double g = 1.0;
#pragma unroll
        for (int j = 0; j < EPL; ++j) {
            const int e = lane + GL * j;
            if (ROW_ON(j)) {
                // a padding gap is 0 - 0 = 0, which would zero the product: it takes the factor 1.0 instead
                const double gap = __dsub_rn((e < kk) ? nx[j] : P.xmax, px[j]);           // changepoint.py:142-143
                g = __dmul_rn(g, (e > kk) ? 1.0 : ((gap < 0.0) ? NAN : gap));
            }
        }
        gp = gprod<GL>(g);
    }
    if (wvt) {
        double b = 0.0;
#pragma unroll
        for (int j = 0; j < EPL; ++j) {
            if (ROW_ON(j)) {
                // a padding height is 0 and log(0) = -inf: the term is selected to 0.0 before it is added (and the log
                // takes 1.0 there, so that it stays on its fast path)
                const bool on = lane + GL * j <= kk;
                double t = __fma_rn(-P.beta, nv[j], P.cv);                                // changepoint.py:18-19,136
                if (!P.alpha_is_one) t = __fma_rn(P.alpha - 1.0, log(on ? nv[j] : 1.0), t);
                else if (!(nv[j] > 0.0)) t = NAN;                                         // 0 * log(v<=0) is nan in numpy
                b = __dadd_rn(b, on ? t : 0.0);
            }
        }
        vt = gsum<GL>(b);
    }
}

// log of four per-chain arguments with one call: lane (l & 3) of the group takes argument l & 3
template <int GL>
__device__ __forceinline__ void log4(int lane, double a0, double a1, double a2, double a3, double& l0, double& l1,
                                     double& l2, double& l3) {
    const int sl = lane & 3;
    const double larg = (sl == 0) ? a0 : ((sl == 1) ? a1 : ((sl == 2) ? a2 : a3));
    const double lres = log(larg);
    l0 = __shfl_sync(0xffffffffu, lres, 0, GL);
    l1 = __shfl_sync(0xffffffffu, lres, 1, GL);
    l2 = __shfl_sync(0xffffffffu, lres, 2, GL);
    l3 = __shfl_sync(0xffffffffu, lres, 3, GL);
}

// ss / sigma^2, the residual term of the likelihood (changepoint.py:118-120); taken before the logarithms of the step
// so that their results are not live across the division
__device__ __forceinline__ double cp_ss_over_s2(double ss, double nsig) { return __ddiv_rn(ss, __dmul_rn(nsig, nsig)); }

// which: 0 = log posterior (model.py:43-55), 1 = log likelihood, 2 = log prior; sss = cp_ss_over_s2(ss, nsig)
__device__ __forceinline__ double cp_assemble(const CPParams& P, int kk, double sss, double vt, double lg, double nsig,
                                              double log_s2, int which) {
    const double s2v = __dmul_rn(nsig, nsig);
    const int ks = kk + 1;                                     // number of steps
    double logl = -0.5 * __dadd_rn(__fma_rn((double)P.M, log_s2, sss), P.Mlog2pi);   // :118-120
    if (isnan(logl)) logl = -INFINITY;                         // :124-125
    double lsig = (s2v < 5.562684646268003e-309) ? INFINITY : -log_s2;      // log(1/sigma^2), :148
    if (nsig < 0.0) lsig = NAN;                                // :146-147
    const double lps = __fma_rn(-(double)ks, P.logL, __dadd_rn(P.tab2[ks], lg));
    double logp = __dadd_rn(__dadd_rn(__dadd_rn(P.tab1[ks], vt), lps), lsig);              // :156
    if (isnan(logp)) logp = -INFINITY;                         // :158-159
    if (which == 1) return logl;
    if (which == 2) return logp;
    return combine_logpost(logp, logl);
}

// full evaluation (pointwise entry, state caches at kernel entry)
template <int GL>
__device__ __forceinline__ double cp_logpost_rows(const CPParams& P, const double2* __restrict__ cyc, int lane,
                                                  int kw, int kk,
                                                  const double (&nx)[Geo<GL>::EPL], const double (&nv)[Geo<GL>::EPL],
                                                  const int (&nbu)[Geo<GL>::EPL], double nsig, int which,
                                                  double& ss, double& vt, double& lg, double& log_s2) {
    double gp, d2, d3;
    cp_terms<GL>(P, cyc, lane, kw, kk, nx, nv, nbu, true, true, true, ss, vt, gp);
    const double sss = cp_ss_over_s2(ss, nsig);
    log4<GL>(lane, gp, __dmul_rn(nsig, nsig), 1.0, 1.0, lg, log_s2, d2, d3);
    return cp_assemble(P, kk, sss, vt, lg, nsig, log_s2, which);
}

// resident blocks of 128 threads per SM the register allocation targets (GL = 4 and 8), DESIGN.md 4.1
#ifndef RMN_CP_MINBLOCKS
#define RMN_CP_MINBLOCKS 4          /* one-slice kernel (traced, injected, short or whole-wave runs) */
#endif
#ifndef RMN_CP_MINBLOCKS_SLICED
#define RMN_CP_MINBLOCKS_SLICED 6   /* time-sliced kernel: 80 registers, 24 warps/SM */
#endif
#ifndef RMN_CP_MINBLOCKS_SUMMARY
#define RMN_CP_MINBLOCKS_SUMMARY 5  /* time-sliced summary kernel: 96 registers (at 80 the sampling spills in the T loop) */
#endif
#ifndef RMN_CP_FASTPATHS
#define RMN_CP_FASTPATHS 1   /* move-specific paths for warps whose chains all drew the same move type */
#endif

// ---------------------------------------------------------------------------------------
// The T-step kernel.
//
// Move schedule (Philox mode).  Which of the four moves a chain attempts at step t is drawn
// independently of its state (three fresh uniforms, test_changepoint.py:48-54).  shared_mv = 1: the
// 32/GL chains of a warp -- global chain ids aligned to 32/GL, so the grouping does not depend on how the
// chains are sharded -- take the three selection words from the group's first chain.  Each chain still
// sees an i.i.d. sequence of move types with the reference's probabilities, independent of its state,
// so each is an exact replica of the reference sampler; given the schedule the chains of a group are
// independent, and in stationarity their ergodic averages are uncorrelated (every schedule's kernel
// preserves the target).  The warp then executes ONE move type per step: a real branch to a
// move-specific path instead of the union of all four by selection.  shared_mv = 0: per-chain move
// types (the general path every step).  Injected mode replays per-chain move types from the tape and
// takes a fast path whenever the warp happens to be uniform (always for K = 1), so the fast paths are
// covered by the reference-stream parity tests.
//
// Fast paths (cached per chain: ss, vt, lg = log gap product, ls2 = log sigma^2 of the CURRENT state):
//   sigma move  test_changepoint.py:54-56   likelihood and prior from the cached sums, no search
//   cpv move    :51-53                      residual / height-prior sums; gaps and run boundaries cached
//   cpx move    :48-50                      searches, residual sums, gap product; height-prior sum cached
//   birth/death :57-71                      the general path
// ---------------------------------------------------------------------------------------
// Parallel tempering (rmn_sampler_set_tempering, ptsampler.py:41-127): chains c = l*nt + i form ladder l, rung i samples
// log_prior + betas[i] * log_likelihood.  Given only to cp_tempered_kernel; see there for the layout.
struct CPTemper {
    double betas[8];
    double pswap;
    int nt;                     // temperatures, 2..8
    int S;                      // groups a ladder occupies: the power of two >= nt
    uint8_t* dir;               // [K] direction label of the replica each chain holds (CP_DIR_*), in the workspace
    unsigned long long* swaps;  // [CP_SWAP_COUNTERS] swap statistics since the last reset (rmn_sampler_cp_get_swap_stats)
};
// Swap statistics, pooled over the ladders.  A replica's label is UP once it last touched rung 0 and DOWN once it last
// touched rung nt-1 (NONE before either); it travels with the state on every swap, and a DOWN replica that arrives at
// rung 0 completes a round trip.  Counters: proposed [7] | accepted [7] (pair i, i+1, i = the initiator's rung) |
// up [8] | down [8] (chains at rung i by label, every RMN_CP_DIAG_EVERY-th step after its swaps) | round trips [1].
enum : uint8_t { CP_DIR_NONE = 0, CP_DIR_UP = 1, CP_DIR_DOWN = 2 };
// in the kernel's shared slot of a group the label sits beside two flags of the group itself, which stay when the label moves
constexpr int CP_DIR_MASK = 3, CP_RUNG_FIRST = 4, CP_RUNG_LAST = 8;
constexpr int CP_SW_PROP = 0, CP_SW_ACC = 7, CP_SW_UP = 14, CP_SW_DOWN = 22, CP_SW_RT = 30, CP_SWAP_COUNTERS = 31;
// the per-group counters of the kernel: swaps it initiated / took as initiator, round trips completed at it (rung 0),
// samples of its label
constexpr int CP_G_PROP = 0, CP_G_ACC = 1, CP_G_RT = 2, CP_G_UP = 3, CP_G_DOWN = 4, CP_G_COUNTERS = 5;

// Posterior summaries (rmn_sampler_cp_set_summary), given only to the cp_summary kernels.  After every step s with
// s % every == 0 each live chain's state adds, with i_j = #{g : xg[g] <= cpx[j]} and the prediction on the grid
// yhat(xg[g]) = cpv[#{j < k : cpx[j] < xg[g]}] (ChangepointRegression1D.predict, changepoint.py:181):
//   khist[k] += 1;  cpxhist[i_j] += 1 for j < k;  yhist[g][bin(yhat(xg[g]))] += 1 for every g,
// the last one as a difference array over g: segment s = 0..k covers the grid indices [i_{s-1}, i_s) (i_{-1} = 0,
// i_k = G) at the one bin b_s = bin(cpv[s]), so it adds +1 at D[i_{s-1}][b_s] and -1 at D[i_s][b_s] (nothing for an
// empty segment or at row G); the prefix sum over g of D is yhist (cp_summary_readout_kernel).  Every counter is a 64-bit
// integer (the -1 in two's complement), so the counts do not depend on the order of the atomics.  Row 0 of D (every
// chain's first segment starts there), khist and cpxhist are counted per block in shared memory and flushed at the end of
// cp_block; the rest of D goes to global memory directly.
struct CPSummary {
    const double* xg;            // grid, NaN-padded to 2 * GP2 entries (padded_upper_bound)
    int G, GP2, H;
    double vlo, inv;             // inv = H / (vhi - vlo), on the host in fp64
    long long every;
    unsigned long long* khist;   // [LANES]
    unsigned long long* cpxhist; // [G + 1]
    unsigned long long* D;       // [G][H + 2]
};
// the block's shared counters: khist [LANES] | cpxhist [G + 1] | D row 0 [H + 2]
__host__ __device__ __forceinline__ int summary_counters(int G, int H) { return LANES + (G + 1) + (H + 2); }

// value bin of y: 1 + floor((y - vlo) * inv) clamped to [0, H + 1]; NaN counts in bin 0
__device__ __forceinline__ int summary_bin(const CPSummary& S, double y) {
    const double t = __dmul_rn(__dsub_rn(y, S.vlo), S.inv);
    return (t >= 0.0) ? ((t < (double)S.H) ? 1 + (int)t : S.H + 1) : 0;
}

// one chain's sampled state (rows as accepted; the caller brackets this with __syncwarp): O(k) searches and atomics
template <int GL>
__device__ __forceinline__ void summary_sample(const CPSummary& S, unsigned long long* ssum,
                                               const Rows<GL, double>& cx, const Rows<GL, double>& cv, int lane, int k,
                                               bool live) {
    constexpr int EPL = Geo<GL>::EPL;
    const int kw = __reduce_max_sync(0xffffffffu, k);
    unsigned long long* s_khist = ssum;
    unsigned long long* s_cpxhist = ssum + LANES;
    unsigned long long* s_d0 = s_cpxhist + S.G + 1;
    if (live && lane == 0) atomicAdd(s_khist + k, 1ull);
    double q[EPL];
    int i[EPL], ip[EPL];
#pragma unroll
    for (int j = 0; j < EPL; ++j) q[j] = cx[j][threadIdx.x];
    padded_upper_bound<EPL>(S.xg, S.GP2, q, i);
#pragma unroll
    for (int j = 0; j < EPL; ++j) if (lane + GL * j >= k) i[j] = S.G;      // i_k = G (and the padding beyond)
    shift_prev<GL, int>(i, ip, 0, lane, kw);                                // i_{e-1}, i_{-1} = 0
    const int W = S.H + 2;
#pragma unroll
    for (int j = 0; j < EPL; ++j) {
        const int e = lane + GL * j;
        if (ROW_ON(j) && live && e <= k) {
            if (e < k) atomicAdd(s_cpxhist + i[j], 1ull);
            if (ip[j] < i[j]) {                                             // segment e is not empty
                const int b = summary_bin(S, cv[j][threadIdx.x]);
                if (ip[j] == 0) atomicAdd(s_d0 + b, 1ull);
                else atomicAdd(S.D + (size_t)ip[j] * W + b, 1ull);
                if (i[j] < S.G) atomicAdd(S.D + (size_t)i[j] * W + b, ~0ull);
            }
        }
    }
}

// GUARD = false: the instantiation for per-chain move schedules in Philox mode -- the warp executes the union of the
// moves every step, so the votes and the guards that a uniform warp would use are compiled out (same arithmetic, same bits).
// TEMPER: the ladder layout and the swap moves of cp_tempered_kernel (tp, usel_tape); every addition sits under
// `if constexpr`, so the untempered instantiations are unchanged.
// SUMMARY: the posterior summaries of the cp_summary kernels (sp, and ssum = the block's shared counters, see CPSummary),
// likewise under `if constexpr`.  TEMPER and SUMMARY together (cp_tempered_summary_kernel): only the chains of rung
// `rung` are sampled.
template <bool INJ, int DATA, int GL, bool GUARD, bool TEMPER = false, typename IT = int64_t, bool SUMMARY = false>
__device__ __forceinline__ void cp_block(const CPParams& P, const double* __restrict__ xs, CPState st,
                                         int64_t K, int64_t t_begin, IT nt, int64_t step0, uint64_t seed,
                                         int64_t chain_offset, const double* __restrict__ tape, const rmn_trace_t& tr,
                                         int shared_mv, int64_t blk, const CPTemper* tp = nullptr,
                                         const double* __restrict__ usel_tape = nullptr, const CPSummary* sp = nullptr,
                                         unsigned long long* ssum = nullptr, int rung = 0) {
    // iterations [t_begin, t_begin + nt) of the launch for the 128 / GL chains of block `blk`; the chain state is read from and
    // written back to global memory (L2-coherent loads: in the time-sliced kernel another SM wrote it)
    constexpr int EPL = Geo<GL>::EPL;
    constexpr int NS = Geo<GL>::NS;
    constexpr int CPW = 32 / GL;                  // chains per warp = chains per schedule group
    constexpr unsigned FULL = 0xffffffffu;
    constexpr bool BUCKETS = (DATA == 2);
    const double2* cyc = (const double2*)(xs + P.XP);
    const double2* bx = cyc + P.M + 1;                // bucket table (P.G > 0)

    const int lane = threadIdx.x & (GL - 1);
    int64_t c_raw, c;
    bool live;
    int ti = 0;                                       // tempered: this group's rung
    if constexpr (TEMPER) {
        // ladder slot q of the grid = S consecutive groups of one warp, rung ti = group index within the slot; with a
        // shared move schedule the warp's CPW / S ladders are aligned to GLOBAL ladder ids (`head` dead leading slots)
        const int64_t L = K / tp->nt;
        const int head = shared_mv ? (int)((chain_offset / tp->nt) & (CPW / tp->S - 1)) : 0;
        const int64_t grp = (blk * (int64_t)blockDim.x + threadIdx.x) / GL;
        const int64_t lad = grp / tp->S - head;
        ti = (int)(grp & (tp->S - 1));
        live = lad >= 0 && lad < L && ti < tp->nt;
        c_raw = lad * tp->nt + ti;                    // global id chain_offset + c_raw keys Philox
        // dead slots and idle rungs (ti >= nt) shadow a live chain for the shuffles and never store
        c = (lad < 0 ? 0 : (lad < L ? lad : L - 1)) * tp->nt + min(ti, tp->nt - 1);
    } else {
        // schedule groups are aligned to GLOBAL chain ids: `head` leading groups of the grid are dead
        const int head = shared_mv ? (int)(chain_offset & (CPW - 1)) : 0;
        c_raw = (blk * (int64_t)blockDim.x + threadIdx.x) / GL - head;
        live = c_raw >= 0 && c_raw < K;
        c = c_raw < 0 ? 0 : (c_raw < K ? c_raw : K - 1);   // dead groups shadow a live chain, never store
    }

    int k = __ldcg(st.k + c);
    // the state's rows: cpx, cpv and the cached run boundaries (see Rows).  They take no registers across the T loop;
    // rows above the warp's extent (ROW_ON) keep the canonical padding they were loaded with.
    __shared__ double s_cx[EPL][128], s_cv[EPL][128];
    __shared__ int s_bu[EPL][128];
    double sig = __ldcg(st.sig + c);
    double lp = __ldcg(st.lp + c);
    // pieces of lp (see cp_terms / cp_assemble), one slot per chain of the block in shared memory: only the moves that
    // leave a piece alone read them, so they take no registers across the T loop.  Every lane of a group writes the
    // same values and reads back its own writes.
    __shared__ double s_ss[128 / GL], s_vt[128 / GL], s_lg[128 / GL];
    // tempered: the untempered log-likelihood and log-prior of the state, which the swap test reads for both partners
    __shared__ double s_ll[TEMPER ? 128 / GL : 1], s_lpr[TEMPER ? 128 / GL : 1];
    const int g = threadIdx.x / GL;
    __shared__ int64_t s_chain[128 / GL];             // the chain the group writes back at the end, -1: none
    s_chain[g] = live ? c : -1;
    // tempered: the label of the replica the group holds (dead slots and idle rungs: NONE, so they never count) and the
    // group's swap counters (CP_G_*).  A group keeps its rung for the launch, so lane 0 counts in its own slots with plain
    // adds -- no atomics in the T loop (a 64-bit shared atomic is a compare-and-swap loop) -- and the block adds them up
    // by rung at the end.
    __shared__ uint8_t s_dir[TEMPER ? 128 / GL : 1];
    __shared__ unsigned long long s_sw[TEMPER ? CP_G_COUNTERS : 1][TEMPER ? 128 / GL : 1];
    if constexpr (TEMPER) {
        s_dir[g] = live ? (__ldcg(tp->dir + c) | ((ti == 0) ? CP_RUNG_FIRST : 0) | ((ti == tp->nt - 1) ? CP_RUNG_LAST : 0))
                        : CP_DIR_NONE;
#pragma unroll
        for (int q = 0; q < CP_G_COUNTERS; ++q) s_sw[q][g] = 0;
    }
    {
        double cx[EPL], cv[EPL];
        int bu[EPL];
#pragma unroll
        for (int j = 0; j < EPL; ++j) {
            const int e = lane + GL * j;
            cx[j] = __ldcg(st.cpx + c * LANES + e);
            cv[j] = __ldcg(st.cpv + c * LANES + e);
            bu[j] = (e < k) ? run_boundary<BUCKETS>(P, xs, bx, cx[j]) : P.M;
            s_cx[j][threadIdx.x] = cx[j]; s_cv[j][threadIdx.x] = cv[j]; s_bu[j][threadIdx.x] = bu[j];
        }
        double ss0, vt0, lg0, ls20;
        const double v0 = cp_logpost_rows<GL>(P, cyc, lane, __reduce_max_sync(FULL, k), k, cx, cv, bu, sig, TEMPER ? 1 : 0,
                                              ss0, vt0, lg0, ls20);
        s_ss[g] = ss0; s_vt[g] = vt0; s_lg[g] = lg0;
        if constexpr (TEMPER) {
            s_ll[g] = v0;
            s_lpr[g] = cp_assemble(P, k, cp_ss_over_s2(ss0, sig), vt0, lg0, sig, ls20, 2);
        }
    }
    double beta = 1.0;                                // this rung's inverse temperature
    if constexpr (TEMPER) beta = tp->betas[min(ti, tp->nt - 1)];
    // the tempered summary kernel reads it and the rung from slots of the group in shared memory: at 128 registers the
    // three they take across the T loop are what the summary sampling would spill
    __shared__ double s_beta[(TEMPER && SUMMARY) ? 128 / GL : 1];
    __shared__ int s_ti[(TEMPER && SUMMARY) ? 128 / GL : 1];
    if constexpr (TEMPER && SUMMARY) { s_beta[g] = beta; s_ti[g] = ti; }
    // diagnostics sums: lane l, slot s holds functional l + GL*s of the chain.  They stay in shared memory for the
    // launch (no registers across the T loop) and every sample is added to the running sum in time order, so the sums
    // do not depend on how the launch is sliced.
    __shared__ double s_S1[NS][128], s_S2[NS][128];
#pragma unroll
    for (int s = 0; s < NS; ++s) {
        const int64_t i = (int64_t)(lane + GL * s) * K + c;
        const bool on = lane + GL * s < RMN_CP_NDIAG;
        s_S1[s][threadIdx.x] = on ? __ldcg(st.S1 + i) : 0.0;
        s_S2[s][threadIdx.x] = on ? __ldcg(st.S2 + i) : 0.0;
    }
    __shared__ int s_nacc[128], s_novf[128];        // accept / overflow counts of the launch, one per thread
    s_nacc[threadIdx.x] = 0; s_novf[threadIdx.x] = 0;
    // summaries: the next sampled step, one slot per thread (every thread of the block walks the same steps)
    __shared__ long long s_snext[SUMMARY ? 128 : 1];
    if constexpr (SUMMARY) {
        const long long s0 = step0 + t_begin, r = s0 % sp->every;
        s_snext[threadIdx.x] = (r == 0) ? s0 : s0 - r + sp->every;
        for (int i = threadIdx.x; i < summary_counters(sp->G, sp->H); i += blockDim.x) ssum[i] = 0;
        __syncthreads();
    }
    const RngKey rk(seed, (uint64_t)(chain_offset + c_raw));
    const TraceSel ts{tr.first, tr.thin > 0 ? tr.thin : 1};
    const bool tracing = tr.d_k || tr.d_cpx || tr.d_cpv || tr.d_sig || tr.d_logpost;
    const bool tracing_prop = tr.d_prop_logpost || tr.d_accepted || tr.d_logqratio || tr.d_prop_k ||
                              tr.d_prop_sig || tr.d_prop_cpx || tr.d_prop_cpv;

    // per-step proposal record (parity harness): what Proposal.propose returned, what the sampler decided
    auto trace_prop = [&](int64_t t, double lpn, bool acc, double lqr, int kk, double nsig,
                          const double (&nx)[EPL], const double (&nv)[EPL]) {
        if (!(live && tracing_prop)) return;
        if (lane == 0) {
            if (tr.d_prop_logpost) tr.d_prop_logpost[t * K + c] = lpn;
            if (tr.d_accepted) tr.d_accepted[t * K + c] = acc ? 1 : 0;
            if (tr.d_logqratio) tr.d_logqratio[t * K + c] = lqr;
            if (tr.d_prop_k) tr.d_prop_k[t * K + c] = kk;
            if (tr.d_prop_sig) tr.d_prop_sig[t * K + c] = nsig;
        }
#pragma unroll
        for (int j = 0; j < EPL; ++j) {
            const int e = lane + GL * j;
            if (tr.d_prop_cpx) tr.d_prop_cpx[(t * K + c) * LANES + e] = nx[j];
            if (tr.d_prop_cpv) tr.d_prop_cpv[(t * K + c) * LANES + e] = nv[j];
        }
    };

    // the Philox block of step t+1 is issued during step t (it depends on nothing but the counter), so its
    // integer multiplies fill the fp64 / LDS latency of the evaluation
    uint4 rA = make_uint4(0, 0, 0, 0);
    if (!INJ) rA = rk.block((uint64_t)(step0 + t_begin), (uint32_t)lane);

    // IT = int (a time slice): the loop carries a 32-bit count instead of a 64-bit bound
    int64_t t = t_begin;
    for (IT n = nt; n > 0; --n, ++t) {
        const uint64_t step = (uint64_t)(step0 + t);
        const int kw = __reduce_max_sync(FULL, k);
        double snew, du, uacc;
        int nrand, mv;
        bool birth;
        const double* row = nullptr;
        const uint4 r = rA;
        if (INJ) {
            row = tape + (t * K + c) * RMN_CP_NSLOT;
            const double u1 = row[RMN_CP_SLOT_SEL1], u2 = row[RMN_CP_SLOT_SEL2], u3 = row[RMN_CP_SLOT_SEL3];
            const double ubd = row[RMN_CP_SLOT_BD];
            snew = row[RMN_CP_SLOT_S]; du = row[RMN_CP_SLOT_DU];
            nrand = (int)row[RMN_CP_SLOT_N]; uacc = row[RMN_CP_SLOT_ACC];
            // which block moves (fresh uniform per elif, test_changepoint.py:48-54); birth/death :59
            mv = (u1 < P.p1) ? 0 : ((u2 < P.p2) ? 1 : ((u3 < P.p3) ? 2 : 3));
            birth = (k == 0) || (ubd > 0.5);
        } else {
            // ONE Philox block per lane and step: words x,y -> Box-Muller pair = the normals of this lane's
            // rows 0 and 1; the spare words z,w of lanes 0..3 carry the chain-level uniforms (the three
            // move-selection words come from the schedule group's first chain when shared_mv).
            const int mvw = shared_mv ? 32 : GL;
            const uint32_t z0 = __shfl_sync(FULL, r.z, 0, mvw), w0 = __shfl_sync(FULL, r.w, 0, mvw);
            const uint32_t z1 = __shfl_sync(FULL, r.z, 1, mvw), w1 = __shfl_sync(FULL, r.w, 1, GL);
            const uint32_t z2 = __shfl_sync(FULL, r.z, 2, GL), w2 = __shfl_sync(FULL, r.w, 2, GL);
            const uint32_t z3 = __shfl_sync(FULL, r.z, 3, GL), w3 = __shfl_sync(FULL, r.w, 3, GL);
            mv = (z0 < P.t1) ? 0 : ((w0 < P.t2) ? 1 : ((z1 < P.t3) ? 2 : 3));   // same tests on raw words
            birth = (k == 0) || (w1 >= 0x80000000u);                            // u > 0.5
            snew = P.xmin + (P.xmax - P.xmin) * u01_fast(z2);
            du = -0.1 + 0.2 * u01_fast(w2);
            nrand = (int)(u01_fast(z3) * (double)k);
            uacc = u01_fast(w3);
        }
        nrand = max(0, min(nrand, k - 1));
        // Tempered: swap roles (ptsampler.py:102-112).  Rung i initiates a swap with i+1 iff it was not itself swapped by
        // i-1, !(usel > pswap) and i < nt-1 -- sequential along the ladder: a ballot of lane 0 of every group, then at most
        // nt-1 iterations.  Every decision reads start-of-step states (participants make no within-chain move), so all
        // swaps of the step are decided at once.  Philox: usel from block (step, 2 GL + lane), read by lane 0.
        bool is_init = false, is_part = false, regular = true;
        if constexpr (TEMPER) {
            const double usel = INJ ? usel_tape[t * K + c] : u01_fast(rk.block(step, (uint32_t)(2 * GL + lane)).x);
            const int ri = SUMMARY ? s_ti[g] : ti;      // this group's rung
            const bool want = live && lane == 0 && ri < tp->nt - 1 && !(usel > tp->pswap);
            // the ladder's first group in the warp (the summary kernel: the group's index in the warp minus its rung,
            // from the shared slot, so that the shift below is not held across the T loop)
            const int base = SUMMARY ? ((threadIdx.x & 31) / GL) - ri : ((threadIdx.x & 31) / GL) & ~(tp->S - 1);
            const unsigned wb = __ballot_sync(FULL, want) >> (base * GL);
            unsigned init = 0;
            for (int b = 0; b < tp->nt - 1; ++b)
                if (((wb >> (b * GL)) & 1u) && !(b > 0 && ((init >> (b - 1)) & 1u))) init |= 1u << b;
            is_init = live && ((init >> ri) & 1u);
            is_part = live && ri > 0 && ((init >> (ri - 1)) & 1u);
            regular = !is_init && !is_part;
        }
        // What the warp as a whole needs this step (warp-uniform).  With a shared move schedule all chains of the
        // warp drew the same move, so most of the step's blocks are skipped by real branches; with per-chain move types
        // the guards are almost always taken and the warp executes the union, selecting per chain.
        const bool any0 = __any_sync(FULL, mv == 0), any1 = __any_sync(FULL, mv == 1);
        const bool any3 = __any_sync(FULL, mv == 3);
        const bool skip = RMN_CP_FASTPATHS && GUARD && (INJ || shared_mv);   // per-chain Philox mode keeps ONE instruction stream
        const bool need_xi = !skip || __any_sync(FULL, mv != 3);

        // ---- birth / death: the chain-level numbers (position, heights, |J|) first, while the proposal's rows are not
        //      yet live -- the divisions and the square root are the step's widest point
        int kk = k, nb = 0;
        double jarg = 1.0, hnew = 0.0;
        bool ovf = false, td = false;
        if (any3) {                                                     // warp-uniform
            __syncwarp();                                               // the other lanes' last writes to their slots
            nb = count_below<GL>(s_cx, lane, k, snew, kw);              // searchsorted(cpx, s), :206
            const double hb = elem_at<GL, double>(s_cv, nb);            // nb, nrand + 1 <= k: a live row
            const double h1d = elem_at<GL, double>(s_cv, nrand);
            const double h2d = elem_at<GL, double>(s_cv, nrand + 1);
            // birth (changepoint.py:57,61,72-74) and death (:67-68,76-78) share one instruction
            // stream: the operands of each division / square root are selected per chain
            const double q1 = birth ? du / P.sqrtM : h2d / h1d;
            const double ub = 0.5 + q1;                                 // birth: u, :61
            const double q2 = birth ? (1.0 - ub) / ub : 1.0 / (1.0 + q1);       // birth: f^2; death: u, :68
            const double u = birth ? ub : q2;
            const double rr = sqrt(birth ? q2 : h1d * h2d);             // birth: f, :57; death: h, :67
            jarg = fabs((birth ? hb : rr) / (u * (1.0 - u)));           // |J| resp. 1/|J^-1|
            // the new height this lane holds: birth, element nb: hb / f, element nb + 1: hb f (the two are on
            // neighbouring lanes); death, element nrand: h
            hnew = birth ? ((lane == (nb & (GL - 1))) ? hb / rr : hb * rr) : rr;
            ovf = (mv == 3) && birth && (k + 1 > LANES - 1);
            td = (mv == 3) && !ovf;
            if (!(mv == 3)) jarg = 1.0;
            if (td) kk = birth ? k + 1 : k - 1;
        }

        // normals of the block moves: rows 0,1 from this step's block, rows 2,3 (only when some chain of the
        // warp has an element there and a location / height move is being made) from a second block
        double xi[EPL];
#pragma unroll
        for (int j = 0; j < EPL; ++j) xi[j] = 0.0;
        if (INJ) {
#pragma unroll
            for (int j = 0; j < EPL; ++j) xi[j] = row[RMN_CP_SLOT_XI + lane + GL * j];
        } else if (need_xi) {
            float n0, n1;
            box_muller(r.x, r.y, n0, n1);
            xi[0] = (double)n0;
            if (EPL > 1) xi[1 % EPL] = (double)n1;
            if (EPL > 2 && kw >= 2 * GL && (!skip || any0 || any1)) {
                const uint4 q = rk.block(step, (uint32_t)(GL + lane));
                box_muller(q.x, q.y, n0, n1);
                xi[2 % EPL] = (double)n0; xi[3 % EPL] = (double)n1;
            }
        }

        // ---- build the proposal by selection (the chains of a warp never diverge on mv).  Only live rows (ROW_ON) are
        //      touched: a row above holds the canonical padding in the state and in the proposal alike (every element
        //      of it is beyond k + 1), so its proposal IS the padding and needs no load.  Inside a row, per-lane
        //      predicates select between values that are all computed (no divergent branches).
        int nbu[EPL];
        double nx[EPL], nv[EPL], nsig = sig;
#pragma unroll
        for (int j = 0; j < EPL; ++j) {
            nx[j] = 0.0; nv[j] = 0.0; nbu[j] = P.M;
            if (ROW_ON(j)) { nx[j] = s_cx[j][threadIdx.x]; nv[j] = s_cv[j][threadIdx.x]; nbu[j] = s_bu[j][threadIdx.x]; }
        }
        if (!skip || any0) {
            const double sxk = P.sx[k];
#pragma unroll
            for (int j = 0; j < EPL; ++j) {
                const int e = lane + GL * j;
                if (ROW_ON(j)) {
                    const double x1 = __dadd_rn(nx[j], __dmul_rn(sxk, xi[j]));           // randomwalk.py:26, scale = 1
                    nx[j] = (mv == 0 && e < k) ? x1 : nx[j];
                }
            }
        }
        if (!skip || any1) {
#pragma unroll
            for (int j = 0; j < EPL; ++j) {
                const int e = lane + GL * j;
                if (ROW_ON(j)) {
                    const double v1 = __dadd_rn(nv[j], __dmul_rn(P.sv, xi[j]));
                    nv[j] = (mv == 1 && e <= k) ? v1 : nv[j];
                }
            }
        }
        const double xi0 = __shfl_sync(FULL, xi[0], 0, GL);
        if (mv == 2) nsig = __dadd_rn(sig, __dmul_rn(P.ss, xi0));
        if (any3) {
            // insert / delete = every element reads its neighbour below (birth, above the insertion
            // point) or above (death, from the removed element on); other chains read themselves
            const int dir = birth ? -1 : 1;
            const int pivot = birth ? nb : nrand - 1;                   // elements <= pivot stay
#pragma unroll
            for (int j = 0; j < EPL; ++j) {
                const int e = lane + GL * j;
                if (ROW_ON(j) && td) {                                  // rows above hold the padding: nothing moves
                    const int off = (e > pivot) ? dir : 0;
                    nx[j] = shifted<GL, double>(s_cx, e, off, 0.0);
                    nv[j] = shifted<GL, double>(s_cv, e, off, 0.0);
                    nbu[j] = shifted<GL, int>(s_bu, e, off, P.M);
                }
                if (td) {
                    if (birth) {
                        if (e == nb) { nx[j] = snew; nv[j] = hnew; }   // its boundary is searched below
                        if (e == nb + 1) nv[j] = hnew;
                    } else if (e == nrand) {
                        nv[j] = hnew;
                    }
                }
                // elements beyond the new extent hold zeros (canonical padding)
                if (e >= kk) { nx[j] = 0.0; nbu[j] = P.M; }
                if (e > kk) nv[j] = 0.0;
            }
        }
        // run boundaries only move when a location moves: a cpx block move (every element) or a
        // birth (the new element).
        const bool moved_x = (mv == 0) || (mv == 3 && birth && !ovf);
        if (!skip || any0 || any3) {
            constexpr int NA = Geo<GL>::ALWAYS;
            double qa[NA];
            int sa[NA];
#pragma unroll
            for (int j = 0; j < NA; ++j) qa[j] = nx[j];
            run_boundary<BUCKETS, NA>(P, xs, bx, qa, sa);
#pragma unroll
            for (int j = 0; j < EPL; ++j) {
                const int e = lane + GL * j;
                if (ROW_ON(j)) {                                        // no element of a row above moves
                    const int sb = (j < NA) ? sa[j < NA ? j : 0] : run_boundary<BUCKETS>(P, xs, bx, nx[j]);
                    nbu[j] = (moved_x && e < kk && (mv == 0 || e == nb)) ? sb : nbu[j];
                }
            }
        }
        if (!INJ) rA = rk.block(step + 1, (uint32_t)lane);
        // ---- log-posterior of the proposal from the pieces that changed (a sigma move: none of the three sums;
        //      a height move: ss, vt; a location move: ss, gp; birth / death: all), every fp64 log of the step in
        //      one call.  A chain whose move leaves a piece alone recomputes the cached value bit for bit.
        double nss = 0.0, nvt = 0.0, gp = 1.0, nlg, nls2, logu, ljac;
        const bool wss = !skip || any0 || any1 || any3, wvt = !skip || any1 || any3, wgp = !skip || any0 || any3;
        cp_terms<GL>(P, cyc, lane, kw, kk, nx, nv, nbu, wss, wvt, wgp, nss, nvt, gp);
        if (!wss) nss = s_ss[g];
        if (!wvt) nvt = s_vt[g];
        const double sss = cp_ss_over_s2(nss, nsig);
        log4<GL>(lane, gp, __dmul_rn(nsig, nsig), uacc, jarg, nlg, nls2, logu, ljac);
        if (!wgp) nlg = s_lg[g];
        double lpn, nll = 0.0, nlpr = 0.0;
        if constexpr (TEMPER) {
            // TemperedModel (ptsampler.py:33-37): combine(log_prior, beta * log_likelihood); beta = 0 times -inf is nan -> -inf
            nll = cp_assemble(P, kk, sss, nvt, nlg, nsig, nls2, 1);
            nlpr = cp_assemble(P, kk, sss, nvt, nlg, nsig, nls2, 2);
            lpn = combine_logpost(nlpr, __dmul_rn((TEMPER && SUMMARY) ? s_beta[g] : beta, nll));
        } else {
            lpn = cp_assemble(P, kk, sss, nvt, nlg, nsig, nls2, 0);
        }
        const double lqr = (mv == 3) ? (birth ? ljac : -ljac) : 0.0;

        // sampler.py:83-84 with Python's min(0, nan) == 0
        const double delta = lpn - lp - lqr;
        const double mh = (delta < 0.0) ? delta : 0.0;
        const bool acc = regular && !ovf && (logu < mh);
        trace_prop(t, lpn, acc, lqr, kk, nsig, nx, nv);
        if (any3) __syncwarp();                           // every lane has read the birth / death rows
        if (acc) {
            k = kk; sig = nsig; lp = lpn;
            s_ss[g] = nss; s_vt[g] = nvt; s_lg[g] = nlg;
            if constexpr (TEMPER) { s_ll[g] = nll; s_lpr[g] = nlpr; }
#pragma unroll
            for (int j = 0; j < EPL; ++j) {
                if (ROW_ON(j)) { s_cx[j][threadIdx.x] = nx[j]; s_cv[j][threadIdx.x] = nv[j]; s_bu[j][threadIdx.x] = nbu[j]; }
            }
        }
        if (acc) s_nacc[threadIdx.x] += 1;
        if (ovf && regular) s_novf[threadIdx.x] += 1;

        if constexpr (TEMPER) {
            // ---- swaps (ptsampler.py:113-125), only in warps where one is proposed.  The initiator (group g) sees its
            //      partner in group g+1, GL lanes up; the state rows, k, sig, lp and the shared-memory slots of both move.
            if (__any_sync(FULL, is_init)) {
                __syncwarp();                                 // the partner's slots as its lanes last wrote them
                const int go = is_init ? g + 1 : (is_part ? g - 1 : g);         // the partner's slot
                const double ll_i = s_ll[g], lpr_i = s_lpr[g];
                const double ll_o = s_ll[go], lpr_o = s_lpr[go], ss_o = s_ss[go], vt_o = s_vt[go], lg_o = s_lg[go];
                const int ri = SUMMARY ? s_ti[g] : ti;
                const double beta_o = tp->betas[min(ri + 1, tp->nt - 1)];
                const double lp_jj = __shfl_down_sync(FULL, lp, GL);
                const double lp_ij = combine_logpost(lpr_o, __dmul_rn((TEMPER && SUMMARY) ? s_beta[g] : beta, ll_o));   // model_i at theta_j
                const double lp_ji = combine_logpost(lpr_i, __dmul_rn(beta_o, ll_i));    // model_j at theta_i
                const double x = exp((lp_ji + lp_ij) - (lp + lp_jj));
                const double mhr = (x < 1.0) ? x : 1.0;                                  // Python min(1, x): nan -> 1
                const bool sw = is_init && (uacc < mhr);                                 // :121
                const bool sw_prev = __shfl_up_sync(FULL, (int)sw, GL) != 0;
                const double lp_ji_prev = __shfl_up_sync(FULL, lp_ji, GL);
                const bool take = is_init ? sw : (is_part && sw_prev);
                const double lp_o = is_init ? lp_ij : lp_ji_prev;
                // swap statistics.  The labels move by shuffle: every lane has read its own group's label before any
                // lane leaves the shuffle, so the new one can be written at once, and nothing of this stays live across
                // the exchange of the rows below
                {
                    const int dl = s_dir[g];
                    const int dd = __shfl_down_sync(FULL, dl, GL), du = __shfl_up_sync(FULL, dl, GL);
                    const int din = (is_init ? dd : du) & CP_DIR_MASK;    // the partner's replica, as it arrives here
                    if (lane == 0) {
                        if (is_init) s_sw[CP_G_PROP][g] += 1;
                        if (sw) s_sw[CP_G_ACC][g] += 1;
                        if (take && (dl & CP_RUNG_FIRST) && din == CP_DIR_DOWN) s_sw[CP_G_RT][g] += 1;   // back at rung 0
                    }
                    if (take)
                        s_dir[g] = (dl & ~CP_DIR_MASK) |
                                   ((dl & CP_RUNG_FIRST) ? CP_DIR_UP : ((dl & CP_RUNG_LAST) ? CP_DIR_DOWN : din));
                }
                const int tq = go * GL + lane;                // the partner's slots (its own for a non-participant)
                double ox[EPL], ov[EPL];
                int ob[EPL];
#pragma unroll
                for (int j = 0; j < EPL; ++j) { ox[j] = s_cx[j][tq]; ov[j] = s_cv[j][tq]; ob[j] = s_bu[j][tq]; }
                const int kd = __shfl_down_sync(FULL, k, GL), ku = __shfl_up_sync(FULL, k, GL);
                const double sd = __shfl_down_sync(FULL, sig, GL), su = __shfl_up_sync(FULL, sig, GL);
                const int ko = is_init ? kd : ku;
                const double so = is_init ? sd : su;
                // a participant's proposal record is its partner's state, with logqratio = 0
                if (is_init || is_part) trace_prop(t, lp_o, take, 0.0, ko, so, ox, ov);
                __syncwarp();                                 // every lane has read its partner's slots
                if (take) {
                    k = ko; sig = so; lp = lp_o;
                    s_ss[g] = ss_o; s_vt[g] = vt_o; s_lg[g] = lg_o; s_ll[g] = ll_o; s_lpr[g] = lpr_o;
#pragma unroll
                    for (int j = 0; j < EPL; ++j) {
                        // rows above hold the padding in both partners
                        if (ROW_ON(j)) { s_cx[j][threadIdx.x] = ox[j]; s_cv[j][threadIdx.x] = ov[j]; s_bu[j][threadIdx.x] = ob[j]; }
                    }
                }
            }
        }

        if ((step % RMN_CP_DIAG_EVERY) == 0) {              // thinned accumulation (warp-uniform)
            __syncwarp();                                   // the rows as the other lanes accepted them
            if constexpr (TEMPER) {                         // the flow histogram, after this step's swaps
                const int d = s_dir[g] & CP_DIR_MASK;
                if (lane == 0 && d != CP_DIR_NONE) s_sw[(d == CP_DIR_UP) ? CP_G_UP : CP_G_DOWN][g] += 1;
            }
            const int kd = __reduce_max_sync(FULL, k);      // (an accepted birth may have raised the extent)
            double f[NS];
#pragma unroll
            for (int s = 0; s < NS; ++s) f[s] = 0.0;
            if (lane == 0) f[0] = sig;
            if (lane == 1 % GL) f[1 / GL] = (double)k;
#pragma unroll
            for (int q = 0; q < NQ; ++q) {
                const int cnt = count_below<GL>(s_cx, lane, k, P.xq[q], kd);
                const double yq = elem_at<GL, double>(s_cv, cnt);        // cnt <= k
                if (lane == (2 + q) % GL) f[(2 + q) / GL] = yq;
            }
#pragma unroll
            for (int s = 0; s < NS; ++s) {
                s_S1[s][threadIdx.x] = __dadd_rn(s_S1[s][threadIdx.x], f[s]);
                s_S2[s][threadIdx.x] = __fma_rn(f[s], f[s], s_S2[s][threadIdx.x]);
            }
            __syncwarp();                                   // every lane has read the rows before the next step writes
        }
        if constexpr (SUMMARY) {
            if ((long long)step == s_snext[threadIdx.x]) {  // warp-uniform
                s_snext[threadIdx.x] += sp->every;
                __syncwarp();                               // the rows as the other lanes accepted them
                // tempered: the group's rung is its index in the ladder slot (a block holds whole slots); the state is
                // the one after this step's swaps
                const bool sampled = s_chain[g] >= 0 && (!TEMPER || (g & (tp->S - 1)) == rung);
                summary_sample<GL>(*sp, ssum, s_cx, s_cv, lane, k, sampled);
                __syncwarp();                               // every lane has read the rows before the next step writes
            }
        }

        if (live && tracing) {
            const long long rrec = ts.slot(t + 1);
            if (rrec >= 0) {
#pragma unroll
                for (int j = 0; j < EPL; ++j) {
                    const int e = lane + GL * j;
                    if (tr.d_cpx) tr.d_cpx[(rrec * K + c) * LANES + e] = s_cx[j][threadIdx.x];
                    if (tr.d_cpv) tr.d_cpv[(rrec * K + c) * LANES + e] = s_cv[j][threadIdx.x];
                }
                if (lane == 0) {
                    if (tr.d_k) tr.d_k[rrec * K + c] = k;
                    if (tr.d_sig) tr.d_sig[rrec * K + c] = sig;
                    if (tr.d_logpost) tr.d_logpost[rrec * K + c] = lp;
                }
            }
        }
    }

    // the chain is read back from its slot: keeping c and `live` in registers across the T loop would cost registers the
    // loop needs
    const int64_t cw = s_chain[g];
    if (cw >= 0) {
        const int64_t c = cw;
#pragma unroll
        for (int j = 0; j < EPL; ++j) {
            const int e = lane + GL * j;
            st.cpx[c * LANES + e] = s_cx[j][threadIdx.x];
            st.cpv[c * LANES + e] = s_cv[j][threadIdx.x];
        }
        if (lane == 0) {
            st.k[c] = k;
            st.sig[c] = sig;
            st.lp[c] = lp;
            st.dacc[c] = __ldcg(st.dacc + c) + s_nacc[threadIdx.x];
            st.dovf[c] = __ldcg(st.dovf + c) + s_novf[threadIdx.x];
            if constexpr (TEMPER) tp->dir[c] = s_dir[g] & CP_DIR_MASK;
        }
#pragma unroll
        for (int s = 0; s < NS; ++s) {
            const int64_t i = (int64_t)(lane + GL * s) * K + c;
            if (lane + GL * s < RMN_CP_NDIAG) {
                st.S1[i] = s_S1[s][threadIdx.x];
                st.S2[i] = s_S2[s][threadIdx.x];
            }
        }
    }
    if constexpr (SUMMARY) {
        __syncthreads();                                // every warp's last sample is in the shared counters
        const int n1 = LANES, n2 = LANES + sp->G + 1;
        // tempered: the block size as the literal it always is (the slots above are sized for 128 threads), so that
        // blockDim.x is not held across the T loop -- at 128 registers the summary kernel would spill it
        for (int i = threadIdx.x; i < summary_counters(sp->G, sp->H); i += (TEMPER ? 128u : blockDim.x)) {
            const unsigned long long v = ssum[i];
            if (v) atomicAdd((i < n1) ? sp->khist + i : ((i < n2) ? sp->cpxhist + (i - n1) : sp->D + (i - n2)), v);
        }
    }
    if constexpr (TEMPER) {
        __syncthreads();                                // every group's last count is in its slots
        // thread j adds up counter j of CPTemper::swaps over the block's groups of its rung (group g is rung g & (S-1):
        // a block holds whole ladder slots)
        const int j = threadIdx.x;
        if (j < CP_SWAP_COUNTERS) {
            const int q = (j < CP_SW_ACC) ? CP_G_PROP : (j < CP_SW_UP) ? CP_G_ACC : (j < CP_SW_DOWN) ? CP_G_UP
                        : (j < CP_SW_RT) ? CP_G_DOWN : CP_G_RT;
            const int r = (j < CP_SW_ACC) ? j : (j < CP_SW_UP) ? j - CP_SW_ACC : (j < CP_SW_DOWN) ? j - CP_SW_UP
                        : (j < CP_SW_RT) ? j - CP_SW_DOWN : 0;
            unsigned long long v = 0;
            if (r < tp->nt)
                for (int gg = r; gg < 128 / GL; gg += tp->S) v += s_sw[q][gg];
            if (v) atomicAdd(tp->swaps + j, v);
        }
    }
}

// DATA: 0 = data tables read from global memory (too large for shared memory), 1 = staged in shared
// memory, 2 = staged with the bucket table (P.G > 0: run_boundary's lookup; the bench data).  The table exists only for
// M <= BUCKET_GMAX, so its data is always staged.
template <bool INJ, int DATA, int GL, bool GUARD = true>
__global__ void __launch_bounds__(128, (GL == 16) ? 8 : RMN_CP_MINBLOCKS)
changepoint_kernel(const __grid_constant__ CPParams P, const double* __restrict__ gdata, CPState st,
                   int64_t K, int64_t T, int64_t step0, uint64_t seed, int64_t chain_offset,
                   const double* __restrict__ tape, rmn_trace_t tr, int shared_mv) {
    extern __shared__ double smem[];
    const double* xs = gdata;
    if (DATA != 0) {
        const int n = P.XP + 2 * P.M + 2 + ((DATA == 2) ? P.G * 5 / 2 : 0);
        for (int i = threadIdx.x; i < n; i += blockDim.x) smem[i] = gdata[i];
        __syncthreads();
        xs = smem;
    }
    cp_block<INJ, DATA, GL, GUARD>(P, xs, st, K, 0, T, step0, seed, chain_offset, tape, tr, shared_mv, blockIdx.x);
}

// Time-sliced form of the same run (plain Philox runs without traces).  A launch of B blocks that do not fit the SMs'
// resident-block slots S in a whole number of waves ends with a partly filled wave (2,048 blocks on 740 slots = 2.77 waves
// at the bench shape).  Here S persistent blocks take the items (time slice j, block b), index
// j B + b, from an atomic counter in increasing order: every persistent block gets the same amount of work to within one
// item, the state of a slice's chains travels through global memory, and a flag per chain block orders the slices of the
// same chains (the predecessor is B >> S items earlier, so the wait is almost never taken).  Philox is keyed by
// (step, chain), so the chains are bit-identical to the one-slice launch.
// The body is shared with cp_summary_sliced_kernel (SUMMARY: sp and the block's shared counters ssum, see CPSummary).
template <int DATA, int GL, bool GUARD, bool SUMMARY>
__device__ __forceinline__ void cp_sliced_body(const CPParams& P, const double* __restrict__ xs, CPState st, int64_t K,
                                               int64_t T, int64_t step0, uint64_t seed, int64_t chain_offset,
                                               int shared_mv, int nblk, int slice, int nslice, int* __restrict__ done,
                                               const CPSummary* sp, unsigned long long* ssum) {
    rmn_trace_t tr{};
    __shared__ int s_item;
    const int items = nblk * nslice;
    for (;;) {
        // items are handed out in increasing order to blocks that are RUNNING: the predecessor of an item was taken
        // earlier, so its owner is resident whatever else shares the device -- the wait below cannot deadlock
        if (threadIdx.x == 0) {
            const int it = atomicAdd(done + nblk, 1);
            const int j = it / nblk, b = it % nblk;
            if (it < items && j > 0) {
                while (*reinterpret_cast<volatile int*>(done + b) < j) __nanosleep(64);
                __threadfence();
            }
            s_item = it;
        }
        __syncthreads();
        const int it = s_item;
        __syncthreads();
        if (it >= items) break;
        const int j = it / nblk, b = it % nblk;
        const int64_t t0 = (int64_t)j * slice, t1 = (t0 + slice < T) ? t0 + slice : T;
        if constexpr (SUMMARY)
            cp_block<false, DATA, GL, GUARD, false, int, true>(P, xs, st, K, t0, (int)(t1 - t0), step0, seed, chain_offset,
                                                               nullptr, tr, shared_mv, b, nullptr, nullptr, sp, ssum);
        else
            cp_block<false, DATA, GL, GUARD>(P, xs, st, K, t0, (int)(t1 - t0), step0, seed, chain_offset, nullptr, tr, shared_mv, b);
        __threadfence();
        __syncthreads();
        // the item is read again (s_item is not written before the next __syncthreads): keeping it live across the T
        // loop would cost a register the loop needs
        if (threadIdx.x == 0) *reinterpret_cast<volatile int*>(done + s_item % nblk) = s_item / nblk + 1;
    }
}

template <int DATA, int GL, bool GUARD = true>
__global__ void __launch_bounds__(128, (GL == 16) ? 8 : RMN_CP_MINBLOCKS_SLICED)
changepoint_sliced_kernel(const __grid_constant__ CPParams P, const double* __restrict__ gdata, CPState st,
                          int64_t K, int64_t T, int64_t step0, uint64_t seed, int64_t chain_offset, int shared_mv,
                          int nblk, int slice, int nslice, int* __restrict__ done) {
    extern __shared__ double smem[];
    const double* xs = gdata;
    if (DATA != 0) {
        const int n = P.XP + 2 * P.M + 2 + ((DATA == 2) ? P.G * 5 / 2 : 0);
        for (int i = threadIdx.x; i < n; i += blockDim.x) smem[i] = gdata[i];
        __syncthreads();
        xs = smem;
    }
    cp_sliced_body<DATA, GL, GUARD, false>(P, xs, st, K, T, step0, seed, chain_offset, shared_mv, nblk, slice, nslice, done,
                                           nullptr, nullptr);
}

// Posterior summaries (rmn_sampler_cp_set_summary, GL = 4): the one-slice and the time-sliced launch of the same run with
// the summary sampling compiled in (cp_block<..., SUMMARY = true>).  Dynamic shared memory: the staged data tables (DATA
// > 0), then the block's summary counters.  The chains are those of changepoint_kernel / changepoint_sliced_kernel bit
// for bit: the sampling only reads the accepted rows.
template <bool INJ, int DATA, bool GUARD>
__global__ void __launch_bounds__(128, RMN_CP_MINBLOCKS)
cp_summary_kernel(const __grid_constant__ CPParams P, const __grid_constant__ CPSummary SP,
                  const double* __restrict__ gdata, CPState st, int64_t K, int64_t T, int64_t step0, uint64_t seed,
                  int64_t chain_offset, const double* __restrict__ tape, rmn_trace_t tr, int shared_mv) {
    extern __shared__ double smem[];
    const double* xs = gdata;
    const int n = (DATA != 0) ? P.XP + 2 * P.M + 2 + ((DATA == 2) ? P.G * 5 / 2 : 0) : 0;
    if (DATA != 0) {
        for (int i = threadIdx.x; i < n; i += blockDim.x) smem[i] = gdata[i];
        __syncthreads();
        xs = smem;
    }
    cp_block<INJ, DATA, 4, GUARD, false, int64_t, true>(P, xs, st, K, 0, T, step0, seed, chain_offset, tape, tr, shared_mv,
                                                         blockIdx.x, nullptr, nullptr, &SP,
                                                         reinterpret_cast<unsigned long long*>(smem + n));
}

template <int DATA, bool GUARD>
__global__ void __launch_bounds__(128, RMN_CP_MINBLOCKS_SUMMARY)
cp_summary_sliced_kernel(const __grid_constant__ CPParams P, const __grid_constant__ CPSummary SP,
                         const double* __restrict__ gdata, CPState st, int64_t K, int64_t T, int64_t step0,
                         uint64_t seed, int64_t chain_offset, int shared_mv, int nblk, int slice, int nslice,
                         int* __restrict__ done) {
    extern __shared__ double smem[];
    const int n = P.XP + 2 * P.M + 2 + ((DATA == 2) ? P.G * 5 / 2 : 0);
    for (int i = threadIdx.x; i < n; i += blockDim.x) smem[i] = gdata[i];
    __syncthreads();
    cp_sliced_body<DATA, 4, GUARD, true>(P, smem, st, K, T, step0, seed, chain_offset, shared_mv, nblk, slice, nslice, done,
                                         &SP, reinterpret_cast<unsigned long long*>(smem + n));
}

// D [G][W] -> yhist [G][W] by a prefix sum over g, one thread per bin column (int64, exact); khist and cpxhist copied
__global__ void cp_summary_readout_kernel(const unsigned long long* __restrict__ khist,
                                          const unsigned long long* __restrict__ cpxhist,
                                          const unsigned long long* __restrict__ D, int G, int W, int64_t* d_khist,
                                          int64_t* d_cpxhist, int64_t* d_yhist) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (d_khist && i < LANES) d_khist[i] = (int64_t)khist[i];
    if (d_cpxhist && i <= G) d_cpxhist[i] = (int64_t)cpxhist[i];
    if (d_yhist && i < W) {
        unsigned long long acc = 0;
        for (int g = 0; g < G; ++g) {
            acc += D[(size_t)g * W + i];
            d_yhist[(size_t)g * W + i] = (int64_t)acc;
        }
    }
}

// Tempered form of changepoint_kernel's one-slice launch (rmn_sampler_set_tempering, GL = 4).
//
// Layout.  Ladder l occupies S = next_pow2(nt) consecutive 4-lane groups of one warp, rung i in group i of the slot, so
// a warp holds 8 / S ladders and a ladder never straddles a warp; the S - nt idle groups shadow a live chain for the
// shuffles and never store.  nt <= 8 (a larger ladder would need a cross-warp exchange through shared memory).
// Swap exchange.  Partners are adjacent groups, GL lanes apart: each lane reads its partner's state slots (rows of cpx, cpv
// and the cached run boundaries) between two __syncwarp, k, sig and lp come by shuffles, and the per-chain shared-memory
// slots (ss, vt, lg and the untempered log-likelihood / log-prior the swap test needs) move with the state.
// The exchange sits under a warp-uniform __any_sync: a warp without a swap this step pays only the ballot.
// Random numbers.  The untempered counters: block (step, lane) for the main words, (step, GL + lane) for rows 2-3; plus
// (step, 2 GL + lane) for the swap-selection uniform, read by lane 0 of the group.  A swap initiator's swap uniform is
// its accept word (w3), which its within-chain test does not use that step.  Philox stays keyed by the global chain id,
// and with the "group" move schedule the schedule group is the warp's ladders aligned to global ladder ids, so a shard
// reproduces its slice of the full run bit for bit.  Injected mode: usel[t*K + c] and the tape's ACC slot.
template <bool INJ, int DATA>
__global__ void __launch_bounds__(128, RMN_CP_MINBLOCKS)
cp_tempered_kernel(const __grid_constant__ CPParams P, const __grid_constant__ CPTemper TP,
                   const double* __restrict__ gdata, CPState st, int64_t K, int64_t T, int64_t step0, uint64_t seed,
                   int64_t chain_offset, const double* __restrict__ tape, const double* __restrict__ usel,
                   rmn_trace_t tr, int shared_mv) {
    extern __shared__ double smem[];
    const double* xs = gdata;
    if (DATA != 0) {
        const int n = P.XP + 2 * P.M + 2 + ((DATA == 2) ? P.G * 5 / 2 : 0);
        for (int i = threadIdx.x; i < n; i += blockDim.x) smem[i] = gdata[i];
        __syncthreads();
        xs = smem;
    }
    cp_block<INJ, DATA, 4, true, true>(P, xs, st, K, 0, T, step0, seed, chain_offset, tape, tr, shared_mv, blockIdx.x,
                                       &TP, usel);
}

// cp_tempered_kernel with the posterior summaries of rung `rung` of every ladder compiled in (rmn_sampler_cp_set_rung_summary):
// the groups of that rung are sampled after the step's swaps, the others pass `live` = false to summary_sample (the
// sampled-step test stays warp-uniform).  `rung` is an argument of its own, so CPTemper and CPSummary, and with them the
// parameter layout of the other kernels, stay as they are.  Dynamic shared memory as in cp_summary_kernel.  The chains
// are those of cp_tempered_kernel bit for bit.
template <bool INJ, int DATA>
__global__ void __launch_bounds__(128, RMN_CP_MINBLOCKS)
cp_tempered_summary_kernel(const __grid_constant__ CPParams P, const __grid_constant__ CPTemper TP,
                           const __grid_constant__ CPSummary SP, int rung, const double* __restrict__ gdata, CPState st,
                           int64_t K, int64_t T, int64_t step0, uint64_t seed, int64_t chain_offset,
                           const double* __restrict__ tape, const double* __restrict__ usel, rmn_trace_t tr,
                           int shared_mv) {
    extern __shared__ double smem[];
    const double* xs = gdata;
    const int n = (DATA != 0) ? P.XP + 2 * P.M + 2 + ((DATA == 2) ? P.G * 5 / 2 : 0) : 0;
    if (DATA != 0) {
        for (int i = threadIdx.x; i < n; i += blockDim.x) smem[i] = gdata[i];
        __syncthreads();
        xs = smem;
    }
    cp_block<INJ, DATA, 4, true, true, int64_t, true>(P, xs, st, K, 0, T, step0, seed, chain_offset, tape, tr, shared_mv,
                                                       blockIdx.x, &TP, usel, &SP,
                                                       reinterpret_cast<unsigned long long*>(smem + n), rung);
}

// evaluate n states given in the canonical layout (pointwise parity entry + set_state); tempered (tp != nullptr): the
// carried log-posterior combine(log_prior, betas[c % nt] * log_likelihood), and the replica labels are initialised
template <bool TEMPER>
__device__ __forceinline__ void cp_eval_body(const CPParams& P, const double* __restrict__ gdata, int which,
                                             int64_t n, const int32_t* __restrict__ kin, const double* __restrict__ cpx,
                                             const double* __restrict__ cpv, const double* __restrict__ sig,
                                             double* __restrict__ out, const CPTemper* tp) {
    constexpr int GL = 16;
    const int lane = threadIdx.x & (GL - 1);
    const int64_t c_raw = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) / GL;
    const bool live = c_raw < n;
    const int64_t c = live ? c_raw : n - 1;
    const double* xs = gdata;
    const double2* cyc = (const double2*)(xs + P.XP);
    const double2* bx = cyc + P.M + 1;                // bucket table (P.G > 0)
    const int k = kin[c];
    const int kw = LANES;                                        // every row on
    double x1[1] = {cpx[c * LANES + lane]}, v1[1] = {cpv[c * LANES + lane]};
    int b1[1] = {P.M};
    if (lane < k) b1[0] = P.G ? run_boundary<true>(P, xs, bx, x1[0]) : run_boundary<false>(P, xs, bx, x1[0]);
    if (lane >= k) x1[0] = 0.0;
    if (lane > k) v1[0] = 0.0;
    double ss, vt, lg, ls2;
    double v = cp_logpost_rows<GL>(P, cyc, lane, kw, k, x1, v1, b1, sig[c], TEMPER ? 1 : which, ss, vt, lg, ls2);
    if constexpr (TEMPER) {
        const double lpr = cp_assemble(P, k, cp_ss_over_s2(ss, sig[c]), vt, lg, sig[c], ls2, 2);
        v = combine_logpost(lpr, __dmul_rn(tp->betas[c % tp->nt], v));
    }
    if (live && lane == 0) {
        out[c] = v;
        // set_state starts the replica walk: the replica at rung 0 moves up, the one at rung nt-1 down
        if constexpr (TEMPER) {
            const int i = (int)(c % tp->nt);
            tp->dir[c] = (i == 0) ? CP_DIR_UP : ((i == tp->nt - 1) ? CP_DIR_DOWN : CP_DIR_NONE);
        }
    }
}

__global__ void __launch_bounds__(128)
cp_eval_kernel(const __grid_constant__ CPParams P, const double* __restrict__ gdata, int which,
               int64_t n, const int32_t* __restrict__ kin, const double* __restrict__ cpx,
               const double* __restrict__ cpv, const double* __restrict__ sig,
               double* __restrict__ out) {
    cp_eval_body<false>(P, gdata, which, n, kin, cpx, cpv, sig, out, nullptr);
}

// the chains' carried log-posterior on a ladder (chain_offset is a multiple of nt, so chain c is rung c % nt)
__global__ void __launch_bounds__(128)
cp_eval_tempered_kernel(const __grid_constant__ CPParams P, const __grid_constant__ CPTemper TP,
                        const double* __restrict__ gdata, int64_t n, const int32_t* __restrict__ kin,
                        const double* __restrict__ cpx, const double* __restrict__ cpv,
                        const double* __restrict__ sig, double* __restrict__ out) {
    cp_eval_body<true>(P, gdata, 0, n, kin, cpx, cpv, sig, out, &TP);
}

__global__ void cp_copy_state_kernel(int64_t K, const int32_t* k_in, const double* cpx_in,
                                     const double* cpv_in, const double* sig_in, int32_t* k_out,
                                     double* cpx_out, double* cpv_out, double* sig_out,
                                     const double* lp_in, double* lp_out) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= K * LANES) return;
    const int64_t c = i / LANES;
    const int lane = (int)(i % LANES);
    const int k = k_in[c];
    if (cpx_out) cpx_out[i] = (lane < k) ? cpx_in[i] : 0.0;
    if (cpv_out) cpv_out[i] = (lane <= k) ? cpv_in[i] : 0.0;
    if (lane == 0) {
        if (k_out) k_out[c] = k;
        if (sig_out) sig_out[c] = sig_in[c];
        if (lp_out && lp_in) lp_out[c] = lp_in[c];
    }
}

static CPParams make_params(const rmn_model* m, const rmn_proposal* p) {
    CPParams P{};
    P.M = m->M;
    int p2 = 1;
    while (p2 * 2 <= m->M) p2 *= 2;
    P.P2 = (m->M >= 1) ? p2 : 0;
    P.XP = 2 * P.P2;
    P.G = m->cp_G; P.bscale = m->cp_bscale; P.boff = m->cp_boff;
    P.alpha_is_one = (m->alpha == 1.0);
    P.xmin = m->xmin; P.xmax = m->xmax; P.alpha = m->alpha; P.beta = m->beta;
    P.cv = m->cv;
    P.logL = log(m->xmax - m->xmin);
    P.ycenter = m->ycenter;
    P.Mlog2pi = (double)m->M * log(2.0 * M_PI);
    P.sqrtM = sqrt((double)m->M);
    for (int ks = 0; ks <= LANES; ++ks) {
        P.tab1[ks] = (ks >= 1) ? (double)ks * log(m->lamb) - lgamma((double)ks) - m->lamb : 0.0;
        P.tab2[ks] = lgamma(2.0 * ks + 1.0);
    }
    const double hs = p ? p->hscale : 1.0;
    for (int k = 0; k <= LANES; ++k) P.sx[k] = sqrt(0.01 * (m->xmax - m->xmin) / (double)(k + 1));
    P.sv = sqrt(0.01 * (hs * hs) / (double)m->M);
    P.ss = sqrt(0.01 * hs);
    P.p1 = p ? p->p_cum[0] : 0.2; P.p2 = p ? p->p_cum[1] : 0.4; P.p3 = p ? p->p_cum[2] : 0.6;
    // (x + 0.5) 2^-32 < p  <=>  x < ceil(p 2^32 - 0.5)
    auto thr = [](double pc) {
        const double v = ceil(pc * 4294967296.0 - 0.5);
        return (uint32_t)(v <= 0.0 ? 0.0 : (v >= 4294967295.0 ? 4294967295.0 : v));
    };
    P.t1 = thr(P.p1); P.t2 = thr(P.p2); P.t3 = thr(P.p3); P.tpad = 0;
    for (int q = 0; q < NQ; ++q)
        P.xq[q] = m->xmin + (m->xmax - m->xmin) * (q + 0.5) / (double)NQ;
    return P;
}

struct ChangepointSampler : SamplerImpl {
    rmn_sampler* s;
    CPState st{};
    CPParams P;
    bool use_smem;
    size_t smem_bytes;
    int gl = RMN_CP_DEFAULT_GL;     // lanes per chain (4, 8 or 16); RMN_CP_GL overrides (A/B measurements)
    int shared_mv = 1;              // Philox mode: move types shared by aligned groups of 32/gl chains (see the kernel);
                                    // rmn_sampler_set_move_schedule / RMN_CP_SCHEDULE=chain select per-chain move types
    explicit ChangepointSampler(rmn_sampler* s_) : s(s_) {
        P = make_params(s->model, s->prop);
        if (const char* e = getenv("RMN_CP_GL")) {
            const int v = atoi(e);
            if (v == 4 || v == 8 || v == 16) gl = v;
        }
        if (const char* e = getenv("RMN_CP_SCHEDULE")) shared_mv = (e[0] == 'c' || e[0] == '0') ? 0 : 1;
        if (const char* e = getenv("RMN_CP_SLICED")) sliced = (e[0] == '0') ? 0 : 1;
        if (const char* e = getenv("RMN_CP_GUARD")) force_guard = (e[0] == '1') ? 1 : 0;
        const size_t tables = (size_t)(P.XP + 2 * P.M + 2) * 8;
        smem_bytes = tables + (size_t)P.G * 20;     // the bucket table is staged with the data
        use_smem = tables <= 96 * 1024;
    }
    size_t workspace_bytes() const override {
        const size_t K = (size_t)s->K;
        // the replica labels of tempering (one byte per chain) for every sampler: the size is asked before
        // rmn_sampler_set_tempering
        return align256(K * 4) + 2 * align256(K * LANES * 8) + 4 * align256(K * 8) +
               2 * align256(RMN_CP_NDIAG * K * 8) + align256(K) + 256;
    }
    uint8_t* d_dir = nullptr;       // [K] replica labels (CPTemper::dir), in the workspace
    int bind(void* ws) override {
        const size_t K = (size_t)s->K;
        char* p = (char*)ws;
        st.k = (int32_t*)p; p += align256(K * 4);
        st.cpx = (double*)p; p += align256(K * LANES * 8);
        st.cpv = (double*)p; p += align256(K * LANES * 8);
        st.sig = (double*)p; p += align256(K * 8);
        st.lp = (double*)p; p += align256(K * 8);
        st.dacc = (long long*)p; p += align256(K * 8);
        st.dovf = (long long*)p; p += align256(K * 8);
        st.S1 = (double*)p; p += align256(RMN_CP_NDIAG * K * 8);
        st.S2 = (double*)p; p += align256(RMN_CP_NDIAG * K * 8);
        d_dir = (uint8_t*)p; p += align256(K);
        RMN_CUDA(cudaMemset(ws, 0, workspace_bytes()));
        if (use_smem) {
            RMN_CUDA(set_smem_attr<4>());
            RMN_CUDA(set_smem_attr<8>());
            RMN_CUDA(set_smem_attr<16>());
        }
        return RMN_OK;
    }
    // without the attribute a kernel may take 48 KB minus its STATIC shared memory (the diagnostics sums, counts and
    // cached pieces and state rows of cp_block: 6-17 KB) as dynamic shared memory
    cudaError_t raise_smem(const void* kernel, size_t bytes) const {
        cudaFuncAttributes a{};
        cudaError_t e = cudaFuncGetAttributes(&a, kernel);
        if (e != cudaSuccess) return e;
        return (bytes + a.sharedSizeBytes > 48 * 1024) ? rmn_raise_dyn_smem(kernel, bytes) : cudaSuccess;
    }
    cudaError_t raise_smem(const void* kernel) const { return raise_smem(kernel, smem_bytes); }
    // the staged kernels this data launches: DATA = 2 with the bucket table, 1 without
    template <int GL> cudaError_t set_smem_attr() { return (P.G > 0) ? set_smem_attr<2, GL>() : set_smem_attr<1, GL>(); }
    template <int DATA, int GL> cudaError_t set_smem_attr() {
        cudaError_t e = raise_smem((const void*)changepoint_kernel<false, DATA, GL>);
        if (e != cudaSuccess) return e;
        e = raise_smem((const void*)changepoint_kernel<true, DATA, GL>);
        if (e != cudaSuccess || GL != 4) return e;
        e = raise_smem((const void*)changepoint_kernel<false, DATA, 4, false>);
        if (e != cudaSuccess) return e;
        e = raise_smem((const void*)changepoint_sliced_kernel<DATA, 4, false>);
        if (e != cudaSuccess) return e;
        e = raise_smem((const void*)cp_tempered_kernel<false, DATA>);
        if (e != cudaSuccess) return e;
        e = raise_smem((const void*)cp_tempered_kernel<true, DATA>);
        if (e != cudaSuccess) return e;
        return raise_smem((const void*)changepoint_sliced_kernel<DATA, 4>);
    }
    unsigned grid(int gl = LANES) const { return (unsigned)((s->K * gl + 127) / 128); }
    // grid of the T-step kernel: schedule groups are aligned to global chain ids, so up to 32/gl - 1 leading
    // groups of the grid are dead when the shard does not start on a group boundary
    unsigned run_grid(int gl, int shared) const {
        const int64_t head = shared ? (s->chain_offset & (int64_t)(32 / gl - 1)) : 0;
        return (unsigned)(((s->K + head) * gl + 127) / 128);
    }
    int set_move_schedule(int mode) override {
        RMN_REQUIRE(mode == 0 || mode == 1, "move schedule: 0 = per chain, 1 = shared by aligned groups of chains");
        shared_mv = mode;
        return RMN_OK;
    }

    // parallel tempering (PTSampler, ptsampler.py:41-81): chains c = l*nt + i form ladder l with betas[i]; call before
    // set_state.  A ladder lives inside one warp (cp_tempered_kernel), hence nt <= 8.
    CPTemper tp{};
    bool tempered = false;
    int set_tempering(int nt, const double* betas, double pswap) override {
        RMN_REQUIRE(nt >= 2 && nt <= 8 && betas,
                    "set_tempering: the changepoint model takes ladders of 2 <= nt <= 8 temperatures (got %d)", nt);
        RMN_REQUIRE(pswap > 0.0 && pswap < 1.0, "Pswap must be a number between 0 and 1");
        RMN_REQUIRE(s->K % nt == 0, "set_tempering: the number of chains (%lld) must be a multiple of nt = %d", (long long)s->K, nt);
        RMN_REQUIRE(s->chain_offset % nt == 0, "set_tempering: chain_offset must be a multiple of nt");
        CPTemper t{};
        for (int i = 0; i < nt; ++i) {
            RMN_REQUIRE(betas[i] >= 0.0 && betas[i] <= 1.0, "beta = %g must be a number between 0 and 1", betas[i]);
            t.betas[i] = betas[i];
        }
        t.nt = nt; t.pswap = pswap; t.S = 1;
        while (t.S < nt) t.S *= 2;
        if (!d_swaps && cudaMalloc(&d_swaps, CP_SWAP_COUNTERS * 8) != cudaSuccess) {
            d_swaps = nullptr;
            rmn_set_error("set_tempering: device allocation failed");
            return RMN_ERR_CUDA;
        }
        RMN_CUDA(cudaMemset(d_swaps, 0, CP_SWAP_COUNTERS * 8));
        // the replica walk starts here (rung 0 UP, rung nt-1 DOWN), and again at every set_state (cp_eval_tempered_kernel)
        std::vector<uint8_t> lab((size_t)s->K);
        for (int64_t c = 0; c < s->K; ++c)
            lab[c] = (c % nt == 0) ? CP_DIR_UP : ((c % nt == nt - 1) ? CP_DIR_DOWN : CP_DIR_NONE);
        RMN_CUDA(cudaMemcpy(d_dir, lab.data(), lab.size(), cudaMemcpyHostToDevice));
        t.dir = d_dir; t.swaps = d_swaps;
        tp = t; tempered = true;
        return RMN_OK;
    }
    unsigned long long* d_swaps = nullptr;      // the swap statistics (CPTemper::swaps), owned by the handle
    int cp_get_swap_stats(int64_t* d_proposed, int64_t* d_accepted, int64_t* d_up, int64_t* d_down,
                          int64_t* d_round_trips, cudaStream_t stream) override {
        if (!tempered) {
            rmn_set_error("swap statistics are counted for tempered changepoint samplers only (rmn_sampler_set_tempering)");
            return RMN_ERR_UNSUPPORTED;
        }
        const int nt = tp.nt;
        auto copy = [&](int64_t* dst, int at, int n) {
            return dst ? cudaMemcpyAsync(dst, d_swaps + at, (size_t)n * 8, cudaMemcpyDeviceToDevice, stream) : cudaSuccess;
        };
        RMN_CUDA(copy(d_proposed, CP_SW_PROP, nt - 1));
        RMN_CUDA(copy(d_accepted, CP_SW_ACC, nt - 1));
        RMN_CUDA(copy(d_up, CP_SW_UP, nt));
        RMN_CUDA(copy(d_down, CP_SW_DOWN, nt));
        RMN_CUDA(copy(d_round_trips, CP_SW_RT, 1));
        return RMN_OK;
    }

    int cp_set_state(const int32_t* d_k, const double* d_cpx, const double* d_cpv,
                     const double* d_sig, cudaStream_t stream) override {
        const int64_t n = s->K * LANES;
        cp_copy_state_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(
            s->K, d_k, d_cpx, d_cpv, d_sig, st.k, st.cpx, st.cpv, st.sig, nullptr, nullptr);
        RMN_KERNEL_CHECK();
        if (tempered)
            cp_eval_tempered_kernel<<<grid(), 128, 0, stream>>>(P, tp, s->model->d_cpdata, s->K, st.k, st.cpx,
                                                                st.cpv, st.sig, st.lp);
        else
            cp_eval_kernel<<<grid(), 128, 0, stream>>>(P, s->model->d_cpdata, 0, s->K, st.k, st.cpx,
                                                       st.cpv, st.sig, st.lp);
        RMN_KERNEL_CHECK();
        launches += 2;
        return RMN_OK;
    }
    int cp_get_state(int32_t* d_k, double* d_cpx, double* d_cpv, double* d_sig, double* d_lp,
                     cudaStream_t stream) override {
        const int64_t n = s->K * LANES;
        cp_copy_state_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(
            s->K, st.k, st.cpx, st.cpv, st.sig, d_k, d_cpx, d_cpv, d_sig, st.lp, d_lp);
        RMN_KERNEL_CHECK();
        launches++;
        return RMN_OK;
    }
    template <bool INJ>
    void launch(int64_t T, const double* tape, const rmn_trace_t& t0, cudaStream_t stream) {
        switch (gl) {
            case 16: launch_gl<INJ, 16>(T, tape, t0, stream); break;
            case 8: launch_gl<INJ, 8>(T, tape, t0, stream); break;
            default: launch_gl<INJ, 4>(T, tape, t0, stream); break;
        }
    }
    // time-sliced launch (changepoint_sliced_kernel): plain Philox runs whose blocks do not fill a whole number of waves
    int* d_done = nullptr;
    int done_cap = 0;
    int sliced = 1;                 // RMN_CP_SLICED=0 switches it off (A/B)
    int force_guard = 0;            // RMN_CP_GUARD=1: per-chain schedules through the guarded instantiation (A/B)
    ~ChangepointSampler() override {
        if (d_done) cudaFree(d_done);
        if (d_swaps) cudaFree(d_swaps);
        free_summary();
    }
    bool last_sliced = false;       // which kernel the last plain launch used (the timer label is corrected after the launch)
    template <int DATA, int GL, bool GUARD, bool SUM = false>
    bool launch_sliced(int64_t T, unsigned nblk, int sh, size_t smem, cudaStream_t stream) {
        constexpr int SLICE_MIN = 100;          // iterations: the state round trip and the entry evaluation cost about one
        last_sliced = false;
        if (!sliced || T < 2 * SLICE_MIN) return false;
        int dev = 0, sms = 0, per_sm = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        const void* kfn = SUM ? (const void*)cp_summary_sliced_kernel<DATA, GUARD> : (const void*)changepoint_sliced_kernel<DATA, GL, GUARD>;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kfn, 128, smem) != cudaSuccess || per_sm < 1)
            return false;
        const unsigned slots = (unsigned)(per_sm * sms);
        if (nblk <= slots || nblk % slots == 0) return false;       // one wave, or whole waves: nothing to gain
        // slices: the count with the least modelled time = rounds of the striped walk per item, times the slice overhead
        // (state round trip + entry evaluation, about 2.5 iterations' worth)
        int nslice = 2;
        double best = 0.0;
        for (int v = 2; v <= 16 && (int64_t)v * SLICE_MIN <= T; ++v) {
            const double items = (double)nblk * v;
            const double cost = ceil(items / slots) / (items / slots) * (1.0 + 2.5 * v / (double)T);
            if (best == 0.0 || cost < best - 1e-9) { best = cost; nslice = v; }
        }
        if (best >= ceil((double)nblk / slots) / ((double)nblk / slots)) return false;     // the plain launch is as good
        const int slice = (int)((T + nslice - 1) / nslice);
        nslice = (int)((T + slice - 1) / slice);
        if ((int)nblk > done_cap) {
            if (d_done) cudaFree(d_done);
            d_done = nullptr; done_cap = 0;
            if (cudaMalloc(&d_done, ((size_t)nblk + 1) * sizeof(int)) != cudaSuccess) return false;     // flags + item counter
            done_cap = (int)nblk;
        }
        if (cudaMemsetAsync(d_done, 0, ((size_t)nblk + 1) * sizeof(int), stream) != cudaSuccess) return false;
        if constexpr (SUM)
            cp_summary_sliced_kernel<DATA, GUARD><<<slots, 128, smem, stream>>>(
                P, sum, s->model->d_cpdata, st, s->K, T, step0, s->seed, s->chain_offset, sh, (int)nblk, slice, nslice, d_done);
        else
            changepoint_sliced_kernel<DATA, GL, GUARD><<<slots, 128, smem, stream>>>(
                P, s->model->d_cpdata, st, s->K, T, step0, s->seed, s->chain_offset, sh, (int)nblk, slice, nslice, d_done);
        last_sliced = true;
        return true;
    }
    template <bool INJ, int GL>
    void launch_gl(int64_t T, const double* tape, const rmn_trace_t& t0, cudaStream_t stream) {
        if constexpr (!INJ && GL == 4) {
            // per-chain move schedules: the instantiation without the warp-uniform guards (RMN_CP_GUARD=1 keeps them: A/B
            // and the bit-identity test)
            if (!shared_mv && !force_guard) { launch_gl_g<INJ, GL, false>(T, tape, t0, stream); return; }
        }
        launch_gl_g<INJ, GL, true>(T, tape, t0, stream);
    }
    static bool is_traced(const rmn_trace_t& t0) {
        return t0.d_k || t0.d_cpx || t0.d_cpv || t0.d_sig || t0.d_logpost || t0.d_prop_logpost || t0.d_accepted ||
               t0.d_logqratio || t0.d_prop_k || t0.d_prop_sig || t0.d_prop_cpx || t0.d_prop_cpv;
    }
    template <bool INJ, int GL, bool GUARD>
    void launch_gl_g(int64_t T, const double* tape, const rmn_trace_t& t0, cudaStream_t stream) {
        const int sh = INJ ? 0 : shared_mv;
        const unsigned g = run_grid(GL, sh);
        last_sliced = false;
        const bool traced = is_traced(t0);
        if constexpr (!INJ && GL == 4) {
            if (!traced && use_smem && P.G > 0) { if (launch_sliced<2, GL, GUARD>(T, g, sh, smem_bytes, stream)) return; }
            else if (!traced && use_smem) { if (launch_sliced<1, GL, GUARD>(T, g, sh, smem_bytes, stream)) return; }
        }
        if (use_smem && P.G > 0)
            changepoint_kernel<INJ, 2, GL, GUARD><<<g, 128, smem_bytes, stream>>>(
                P, s->model->d_cpdata, st, s->K, T, step0, s->seed, s->chain_offset, tape, t0, sh);
        else if (use_smem)
            changepoint_kernel<INJ, 1, GL, GUARD><<<g, 128, smem_bytes, stream>>>(
                P, s->model->d_cpdata, st, s->K, T, step0, s->seed, s->chain_offset, tape, t0, sh);
        else
            changepoint_kernel<INJ, 0, GL, GUARD><<<g, 128, 0, stream>>>(
                P, s->model->d_cpdata, st, s->K, T, step0, s->seed, s->chain_offset, tape, t0, sh);
    }
    // ---- posterior summaries (CPSummary; rmn_sampler_cp_set_summary / rmn_sampler_cp_get_summary)
    CPSummary sum{};
    bool summary = false;
    int64_t sum_samples = 0;        // sampled chain-steps since the last reset
    int sum_rung = -1;              // tempered: the rung whose chains are sampled (rmn_sampler_cp_set_rung_summary)
    size_t sum_smem() const { return (size_t)summary_counters(sum.G, sum.H) * 8; }
    void free_summary() {
        if (sum.xg) cudaFree((void*)sum.xg);
        if (sum.khist) cudaFree(sum.khist);
        sum = CPSummary{}; summary = false; sum_samples = 0; sum_rung = -1;
    }
    size_t sum_count_bytes() const { return ((size_t)LANES + sum.G + 1 + (size_t)sum.G * (sum.H + 2)) * 8; }
    int cp_set_summary(int G, const double* grid, double vlo, double vhi, int H, int64_t every) override {
        if (G == 0) { free_summary(); return RMN_OK; }
        if (tempered || gl != 4) {
            rmn_set_error("posterior summaries run on the untempered changepoint sampler at 4 lanes per chain only%s",
                          tempered ? " (this sampler is tempered)" : " (RMN_CP_GL selects another width)");
            return RMN_ERR_UNSUPPORTED;
        }
        const int e = alloc_summary("rmn_sampler_cp_set_summary", G, grid, vlo, vhi, H, every);
        if (e != RMN_OK) return e;
        if (use_smem) {
            const size_t b = smem_bytes + sum_smem();
            const void* kf[] = {(const void*)cp_summary_kernel<false, 1, true>, (const void*)cp_summary_kernel<false, 1, false>,
                                (const void*)cp_summary_kernel<true, 1, true>, (const void*)cp_summary_kernel<false, 2, true>,
                                (const void*)cp_summary_kernel<false, 2, false>, (const void*)cp_summary_kernel<true, 2, true>,
                                (const void*)cp_summary_sliced_kernel<1, true>, (const void*)cp_summary_sliced_kernel<1, false>,
                                (const void*)cp_summary_sliced_kernel<2, true>, (const void*)cp_summary_sliced_kernel<2, false>};
            for (const void* f : kf) RMN_CUDA(raise_smem(f, b));
        }
        return RMN_OK;
    }
    // tempered samplers: the summaries of the chains of one rung of every ladder (cp_tempered_summary_kernel)
    int cp_set_rung_summary(int rung, int G, const double* grid, double vlo, double vhi, int H, int64_t every) override {
        if (!tempered) {
            rmn_set_error("rung summaries run on tempered changepoint samplers only (rmn_sampler_cp_set_summary serves "
                          "untempered ones)");
            return RMN_ERR_UNSUPPORTED;
        }
        if (G == 0) { free_summary(); return RMN_OK; }
        RMN_REQUIRE(rung >= 0 && rung < tp.nt, "rmn_sampler_cp_set_rung_summary: need 0 <= rung < %d (got %d)", tp.nt, rung);
        const int e = alloc_summary("rmn_sampler_cp_set_rung_summary", G, grid, vlo, vhi, H, every);
        if (e != RMN_OK) return e;
        sum_rung = rung;
        if (use_smem) {
            const size_t b = smem_bytes + sum_smem();
            const void* kf[] = {(const void*)cp_tempered_summary_kernel<false, 1>, (const void*)cp_tempered_summary_kernel<true, 1>,
                                (const void*)cp_tempered_summary_kernel<false, 2>, (const void*)cp_tempered_summary_kernel<true, 2>};
            for (const void* f : kf) RMN_CUDA(raise_smem(f, b));
        }
        return RMN_OK;
    }
    // the checks and buffers common to both entries (fn: the entry's name in the error messages); resets the counts
    int alloc_summary(const char* fn, int G, const double* grid, double vlo, double vhi, int H, int64_t every) {
        RMN_REQUIRE(G >= 1 && G <= 1024 && grid, "%s: need 1 <= G <= 1024 grid points (got %d)", fn, G);
        for (int i = 0; i < G; ++i) {
            RMN_REQUIRE(isfinite(grid[i]), "%s: grid point %d is not finite", fn, i);
            RMN_REQUIRE(i == 0 || grid[i] > grid[i - 1], "%s: the grid must be strictly increasing", fn);
        }
        RMN_REQUIRE(H >= 1 && H <= 1024, "%s: need 1 <= H <= 1024 value bins (got %d)", fn, H);
        const double inv = (double)H / (vhi - vlo);
        RMN_REQUIRE(isfinite(vlo) && isfinite(vhi) && vlo < vhi && isfinite(inv) && inv > 0.0,
                    "%s: need a finite value range vlo < vhi", fn);
        RMN_REQUIRE(every >= 1 && every <= ((int64_t)1 << 62), "%s: need 1 <= every <= 2^62", fn);
        free_summary();
        CPSummary q{};
        q.G = G; q.H = H; q.vlo = vlo; q.inv = inv; q.every = every;
        q.GP2 = 1;
        while (q.GP2 * 2 <= G) q.GP2 *= 2;
        std::vector<double> tab(2 * (size_t)q.GP2, NAN);             // padded_upper_bound's table
        std::copy(grid, grid + G, tab.begin());
        sum = q;
        double* d_xg = nullptr;
        unsigned long long* d_cnt = nullptr;
        if (cudaMalloc(&d_xg, tab.size() * 8) != cudaSuccess || cudaMalloc(&d_cnt, sum_count_bytes()) != cudaSuccess) {
            if (d_xg) cudaFree(d_xg);
            sum = CPSummary{};
            rmn_set_error("%s: device allocation failed", fn);
            return RMN_ERR_CUDA;
        }
        sum.xg = d_xg;
        sum.khist = d_cnt; sum.cpxhist = d_cnt + LANES; sum.D = sum.cpxhist + G + 1;
        summary = true;
        RMN_CUDA(cudaMemcpy(d_xg, tab.data(), tab.size() * 8, cudaMemcpyHostToDevice));
        RMN_CUDA(cudaMemset(d_cnt, 0, sum_count_bytes()));
        return RMN_OK;
    }
    int cp_get_summary(int64_t* d_khist, int64_t* d_cpxhist, int64_t* d_yhist, int64_t* h_nsamples,
                       cudaStream_t stream) override {
        RMN_REQUIRE(summary, "rmn_sampler_cp_get_summary: no summary is set (rmn_sampler_cp_set_summary)");
        const int W = sum.H + 2, n = std::max(W, sum.G + 1);
        cp_summary_readout_kernel<<<(unsigned)((n + 127) / 128), 128, 0, stream>>>(sum.khist, sum.cpxhist, sum.D, sum.G, W,
                                                                                  d_khist, d_cpxhist, d_yhist);
        RMN_KERNEL_CHECK();
        launches++;
        if (h_nsamples) *h_nsamples = sum_samples;
        return RMN_OK;
    }
    template <bool INJ, bool GUARD>
    void launch_summary(int64_t T, const double* tape, const rmn_trace_t& t0, cudaStream_t stream) {
        const int sh = INJ ? 0 : shared_mv;
        const unsigned g = run_grid(4, sh);
        const size_t ss = sum_smem();
        last_sliced = false;
        if constexpr (!INJ) {
            if (!is_traced(t0) && use_smem && P.G > 0) { if (launch_sliced<2, 4, GUARD, true>(T, g, sh, smem_bytes + ss, stream)) return; }
            else if (!is_traced(t0) && use_smem) { if (launch_sliced<1, 4, GUARD, true>(T, g, sh, smem_bytes + ss, stream)) return; }
        }
        if (use_smem && P.G > 0)
            cp_summary_kernel<INJ, 2, GUARD><<<g, 128, smem_bytes + ss, stream>>>(
                P, sum, s->model->d_cpdata, st, s->K, T, step0, s->seed, s->chain_offset, tape, t0, sh);
        else if (use_smem)
            cp_summary_kernel<INJ, 1, GUARD><<<g, 128, smem_bytes + ss, stream>>>(
                P, sum, s->model->d_cpdata, st, s->K, T, step0, s->seed, s->chain_offset, tape, t0, sh);
        else
            cp_summary_kernel<INJ, 0, GUARD><<<g, 128, ss, stream>>>(
                P, sum, s->model->d_cpdata, st, s->K, T, step0, s->seed, s->chain_offset, tape, t0, sh);
    }

    // tempered runs: the one-slice launch at GL = 4 (RMN_CP_GL does not apply); one ladder slot of S groups per ladder
    template <bool INJ>
    void launch_tempered(int64_t T, const rmn_inject_t* inj, const rmn_trace_t& t0, cudaStream_t stream) {
        const int sh = INJ ? 0 : shared_mv;
        const int64_t L = s->K / tp.nt;
        const int64_t head = sh ? ((s->chain_offset / tp.nt) & (int64_t)(8 / tp.S - 1)) : 0;
        const unsigned g = (unsigned)(((L + head) * tp.S * 4 + 127) / 128);
        const double* tape = INJ ? inj->d_tape : nullptr;
        const double* usel = INJ ? inj->d_usel : nullptr;
        if (summary) {
            const size_t ss = sum_smem();
            if (use_smem && P.G > 0)
                cp_tempered_summary_kernel<INJ, 2><<<g, 128, smem_bytes + ss, stream>>>(
                    P, tp, sum, sum_rung, s->model->d_cpdata, st, s->K, T, step0, s->seed, s->chain_offset, tape, usel, t0, sh);
            else if (use_smem)
                cp_tempered_summary_kernel<INJ, 1><<<g, 128, smem_bytes + ss, stream>>>(
                    P, tp, sum, sum_rung, s->model->d_cpdata, st, s->K, T, step0, s->seed, s->chain_offset, tape, usel, t0, sh);
            else
                cp_tempered_summary_kernel<INJ, 0><<<g, 128, ss, stream>>>(
                    P, tp, sum, sum_rung, s->model->d_cpdata, st, s->K, T, step0, s->seed, s->chain_offset, tape, usel, t0, sh);
            return;
        }
        if (use_smem && P.G > 0)
            cp_tempered_kernel<INJ, 2><<<g, 128, smem_bytes, stream>>>(
                P, tp, s->model->d_cpdata, st, s->K, T, step0, s->seed, s->chain_offset, tape, usel, t0, sh);
        else if (use_smem)
            cp_tempered_kernel<INJ, 1><<<g, 128, smem_bytes, stream>>>(
                P, tp, s->model->d_cpdata, st, s->K, T, step0, s->seed, s->chain_offset, tape, usel, t0, sh);
        else
            cp_tempered_kernel<INJ, 0><<<g, 128, 0, stream>>>(
                P, tp, s->model->d_cpdata, st, s->K, T, step0, s->seed, s->chain_offset, tape, usel, t0, sh);
    }
    int run(int64_t T, const rmn_inject_t* inj, const rmn_trace_t* tr, cudaStream_t stream) override {
        rmn_trace_t t0{};
        if (tr) t0 = *tr;
        if (t0.thin <= 0) t0.thin = 1;
        if (inj) RMN_REQUIRE(inj->d_tape, "injected changepoint run needs d_tape");
        if (inj && tempered) RMN_REQUIRE(inj->d_usel, "injected tempered run needs d_usel (selection uniforms)");
        if (summary && tempered && sum_rung < 0) {
            rmn_set_error("posterior summaries of a tempered sampler are those of one rung (rmn_sampler_cp_set_rung_summary)");
            return RMN_ERR_UNSUPPORTED;
        }
        ktimer.begin(tempered ? (summary ? "cp_tempered_summary_kernel" : "cp_tempered_kernel")
                              : (summary ? "cp_summary_kernel" : "changepoint_kernel"), stream);
        if (tempered) {
            if (inj) launch_tempered<true>(T, inj, t0, stream);
            else launch_tempered<false>(T, nullptr, t0, stream);
        } else if (summary) {
            // GL = 4 (cp_set_summary refuses other widths); per-chain move schedules without the guards as in launch_gl
            if (inj) launch_summary<true, true>(T, inj->d_tape, t0, stream);
            else if (!shared_mv && !force_guard) launch_summary<false, false>(T, nullptr, t0, stream);
            else launch_summary<false, true>(T, nullptr, t0, stream);
            if (last_sliced) ktimer.name = "cp_summary_sliced_kernel";
        } else if (inj) {
            launch<true>(T, inj->d_tape, t0, stream);
        } else {
            launch<false>(T, nullptr, t0, stream);
            if (last_sliced) ktimer.name = "changepoint_sliced_kernel";
        }
        ktimer.end(stream);
        RMN_KERNEL_CHECK();
        launches++;
        // samples = #{ s in [step0, step0+T) : s % EVERY == 0 }
        const int64_t E = RMN_CP_DIAG_EVERY;
        diag_samples += (step0 + T + E - 1) / E - (step0 + E - 1) / E;
        if (summary) {
            // every live chain (tempered: one per ladder, the chain of rung sum_rung) at each sampled step;
            // ceil(n / every) = #{s in [0, n) : s % every == 0} without overflow
            auto upto = [&](int64_t n) { return n / sum.every + (n % sum.every != 0); };
            sum_samples += (tempered ? s->K / tp.nt : s->K) * (upto(step0 + T) - upto(step0));
        }
        step0 += T; diag_steps += T;
        return RMN_OK;
    }
    int diag_dim() const override { return RMN_CP_NDIAG; }
    int reset_diag(cudaStream_t stream) override {
        RMN_CUDA(cudaMemsetAsync(st.S1, 0, (size_t)RMN_CP_NDIAG * s->K * 8, stream));
        RMN_CUDA(cudaMemsetAsync(st.S2, 0, (size_t)RMN_CP_NDIAG * s->K * 8, stream));
        RMN_CUDA(cudaMemsetAsync(st.dacc, 0, (size_t)s->K * 8, stream));
        RMN_CUDA(cudaMemsetAsync(st.dovf, 0, (size_t)s->K * 8, stream));
        diag_steps = 0; diag_samples = 0;
        if (summary) {                  // the summaries cover the same window as the diagnostics
            RMN_CUDA(cudaMemsetAsync(sum.khist, 0, sum_count_bytes(), stream));
            sum_samples = 0;
        }
        // the swap counts too; the replica labels are state of the walk and stay, so a trip in progress still completes
        if (tempered) RMN_CUDA(cudaMemsetAsync(d_swaps, 0, CP_SWAP_COUNTERS * 8, stream));
        return RMN_OK;
    }
    int chain_sums(const double** S1, const double** S2, int64_t* n) override {
        *S1 = st.S1; *S2 = st.S2; *n = diag_samples;
        return RMN_OK;
    }
    int reduce_diag(double* d_block, cudaStream_t stream) override {
        launches++;
        return rmn_reduce_diag_block(s->K, RMN_CP_NDIAG, diag_samples, diag_steps, st.S1, st.S2, st.dacc, st.dovf,
                                     d_block, stream);
    }
};

}  // namespace

SamplerImpl* make_changepoint_sampler(rmn_sampler* s) { return new ChangepointSampler(s); }

int cp_pointwise(rmn_model* m, int which, int64_t n, const int32_t* d_k, const double* d_cpx,
                 const double* d_cpv, const double* d_sig, double* d_out, cudaStream_t st) {
    if (n <= 0) return RMN_OK;
    const CPParams P = make_params(m, nullptr);
    cp_eval_kernel<<<(unsigned)((n * LANES + 127) / 128), 128, 0, st>>>(P, m->d_cpdata, which, n, d_k,
                                                                        d_cpx, d_cpv, d_sig, d_out);
    RMN_KERNEL_CHECK();
    return RMN_OK;
}

