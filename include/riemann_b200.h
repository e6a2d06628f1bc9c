/*
 * riemann_b200 -- C ABI of the B200-native many-chain Metropolis-Hastings engine.
 *
 * The reference (rscalzo/riemann) has no FFI layer: its boundary is the duck-typed
 * Python protocol  Model.log_posterior / Proposal.propose+adapt / Sampler.run+sample
 * (riemann/models/model.py:27-64, riemann/proposals/proposal.py:10-26,
 * riemann/samplers/sampler.py:34-90).  The Python host classes in riemann_b200/
 * keep those signatures and bind the entry points below through ctypes
 * (riemann_b200/_lib.py); INTEGRATION.md shows the binding a maintainer would add.
 *
 * Conventions
 *   - every function returns int: RMN_OK or a negative RMN_ERR_*; nothing throws.
 *     rmn_last_error() returns a thread-local message for the last failure.
 *   - "d_" pointers are DEVICE pointers owned by the caller (e.g. tensor.data_ptr());
 *     "h_" pointers are HOST pointers, copied during the call.
 *   - all per-chain state of a sampler lives in ONE caller-provided device workspace
 *     (size from rmn_sampler_workspace_bytes); the library never allocates chain
 *     state.  Handles own only small hyper-parameter tables.
 *   - every call that touches the device takes a cudaStream_t (as void*) and only
 *     enqueues work on it; no hidden synchronisation.
 *   - canonical external layouts: fixed-d states  theta[K][d] (row-major fp64);
 *     changepoint states  k[K] (int32), cpx[K][RMN_CP_LANES], cpv[K][RMN_CP_LANES],
 *     sig[K].  Internal layouts differ (see DESIGN.md) and are converted by
 *     set_state/get_state.
 *   - a handle is bound to the device current at creation and is not thread-safe.
 */
#ifndef RIEMANN_B200_H
#define RIEMANN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RMN_VERSION 100

#define RMN_OK 0
#define RMN_ERR_PARAM (-1)        /* bad argument      -> riemann ParameterError   */
#define RMN_ERR_CUDA (-2)         /* CUDA failure      -> RuntimeError             */
#define RMN_ERR_UNSUPPORTED (-3)  /* no device kernel for this model/proposal pair */

typedef struct rmn_model rmn_model_t;
typedef struct rmn_proposal rmn_proposal_t;
typedef struct rmn_sampler rmn_sampler_t;

int rmn_version(void);
const char* rmn_last_error(void);

/* ---------------------------------------------------------------- models ---- */

/* MultiGaussianDist (riemann/models/gaussian.py:27-58).  h_prec = C^{-1} (d x d,
 * row-major), h_linv = L^{-1} with C = L L^T (d x d row-major, lower; may be NULL
 * for d > RMN_SMALL_D_MAX), logdetC = 2 sum log diag L (gaussian.py:43). */
int rmn_model_gaussian_create(rmn_model_t** out, int d, const double* h_mu,
                              const double* h_prec, const double* h_linv, double logdetC);

/* ChangepointRegression1D (riemann/models/changepoint.py:81-181).  x must be sorted
 * ascending (generate_synthetic_data, :170).  kmax is stored and, as in the
 * reference (:100), never enforced. */
int rmn_model_changepoint_create(rmn_model_t** out, int M, const double* h_x,
                                 const double* h_y, double xmin, double xmax,
                                 double lamb, int kmax, double alpha, double beta);

/* Bayesian logistic regression, prior N(0, prior_var I) -- not in the reference;
 * follows the Model protocol (model.py:27-55).  d_X is [N][d] row-major fp64,
 * d_y is [N] fp64 in {0,1}; both stay owned by the caller and must outlive the
 * model. */
int rmn_model_logistic_create(rmn_model_t** out, int64_t N, int d, const double* d_X,
                              const double* d_y, double prior_var);

int rmn_model_destroy(rmn_model_t* m);
int rmn_model_dim(const rmn_model_t* m);

/* Pointwise evaluation for n arbitrary points (parity harness; also backs the
 * scalar-theta Model.log_posterior / log_likelihood / log_prior of the host
 * classes).  which: 0 = log_posterior (model.py:43-55 inf/nan rule applied),
 * 1 = log_likelihood, 2 = log_prior. */
int rmn_model_logpost(rmn_model_t* m, int which, int64_t n, const double* d_theta,
                      double* d_out, void* stream);
int rmn_model_grad(rmn_model_t* m, int64_t n, const double* d_theta, double* d_grad,
                   void* stream);
/* Fisher metric G[n][d][d] (logistic model only). */
int rmn_model_metric(rmn_model_t* m, int64_t n, const double* d_theta, double* d_G,
                     void* stream);
int rmn_model_cp_logpost(rmn_model_t* m, int which, int64_t n, const int32_t* d_k,
                         const double* d_cpx, const double* d_cpv, const double* d_sig,
                         double* d_out, void* stream);

/* -------------------------------------------------------------- proposals ---- */

#define RMN_SMALL_D_MAX 8 /* fully fused register-resident kernels up to this d */

/* MetropolisRandomWalk / AdaptScaleRandomWalk (riemann/proposals/randomwalk.py:12-37):
 * theta' = theta + scale * L xi.  h_L = chol(C) (d x d row-major, lower).
 * adapt != 0 enables AdaptScaleProposal (adaptive.py:11-35) PER CHAIN with the
 * given target acceptance rate (0.25 in the reference). */
int rmn_proposal_rw_create(rmn_proposal_t** out, int d, const double* h_L, int adapt,
                           double target);

/* AdaptCovRandomWalk = AdaptiveMetropolisRandomWalk = HaarioRandomWalk (riemann/proposals/randomwalk.py:40-59,
 * adaptive.py:38-103): per chain, the proposal covariance follows the sample covariance of the chain's history,
 * recomputed (and refactored in-kernel) whenever the number of states is a perfect square > 2; options t_adapt,
 * marginalize, smooth_adapt as in the reference.  h_C0 is the initial covariance, h_L0 = chol(C0), both d x d
 * row-major.  Small-d path only (d <= 8). */
int rmn_proposal_adaptcov_create(rmn_proposal_t** out, int d, const double* h_C0, const double* h_L0,
                                 double t_adapt, int marginalize, int smooth_adapt);

/* AdaptCovHMC (hamiltonian.py:106-119): the mass matrix of an HMC proposal created WITHOUT one becomes the chain's adapted
 * covariance (M = C, chM = L of adaptive.py:101-102), starting from M0 / chol(M0).  Small-d path only. */
int rmn_proposal_hmc_set_cov_adapt(rmn_proposal_t* p, const double* h_M0, const double* h_L0, double t_adapt,
                                   int marginalize, int smooth_adapt);

/* AdaptScaleProposal mix-in (adaptive.py:11-35) on an already created proposal: AdaptScaleCovRandomWalk
 * (randomwalk.py:62-75: scale then covariance adaptation every step) = adaptcov_create + this; AdaptScalepCN
 * (randomwalk.py:103-119, reproduced as written: rho <- tanh(rho / scale) compounding, rho_c fixed) = pcn_create +
 * this (small-d path only).  Call before rmn_sampler_create. */
int rmn_proposal_set_scale_adapt(rmn_proposal_t* p, int adapt, double target);

/* VanillaHMC / AdaptScaleHMC (riemann/proposals/hamiltonian.py:13-103); nsteps = 1
 * is MALA.  The gradient is the model's own grad log posterior.  Mass matrix
 * optional: pass h_chM = chol(M), h_Minv = M^{-1}, h_chMinv = chol(M)^{-1}
 * (each d x d row-major) or all NULL.  adapt != 0: eps = scale * eps0, per chain. */
int rmn_proposal_hmc_create(rmn_proposal_t** out, int d, double eps, int nsteps,
                            const double* h_chM, const double* h_Minv,
                            const double* h_chMinv, int adapt, double target);

/* pCN (riemann/proposals/randomwalk.py:78-100). h_L = chol(C); h_Linv its inverse. */
int rmn_proposal_pcn_create(rmn_proposal_t** out, int d, const double* h_L,
                            const double* h_Linv, double rho);

/* Simplified manifold MALA with the model's Fisher metric (not in the reference;
 * Proposal protocol proposal.py:10-17). */
int rmn_proposal_mmala_create(rmn_proposal_t** out, int d, double eps);

/* ChangepointRegression1DProp (examples/test_changepoint.py:18-73).  p_cum[3] are the
 * sequential thresholds (.20, .40, .60 there). */
int rmn_proposal_changepoint_create(rmn_proposal_t** out, double hscale,
                                    const double* h_p_cum);

int rmn_proposal_destroy(rmn_proposal_t* p);

/* --------------------------------------------------------------- samplers ---- */

#define RMN_CP_LANES 16                  /* lanes per chain; at most LANES-1 changepoints */
#define RMN_CP_SLOT_SEL1 0               /* injected-tape slots, one row per MH step:   */
#define RMN_CP_SLOT_SEL2 1               /*   block-selection uniforms (test_changepoint.py:48,51,54) */
#define RMN_CP_SLOT_SEL3 2
#define RMN_CP_SLOT_BD 3                 /*   birth/death coin (:59)                    */
#define RMN_CP_SLOT_S 4                  /*   U(xmin,xmax) (:60), already scaled        */
#define RMN_CP_SLOT_DU 5                 /*   U(-0.1,0.1) (:61), already scaled         */
#define RMN_CP_SLOT_N 6                  /*   randint(k) (:67) as a double              */
#define RMN_CP_SLOT_ACC 7                /*   accept uniform (sampler.py:84)            */
#define RMN_CP_SLOT_XI 8                 /*   normals xi_0..xi_{LANES-1}                */
#define RMN_CP_NSLOT (RMN_CP_SLOT_XI + RMN_CP_LANES)

#define RMN_CP_NDIAG 8                   /* tracked functionals: sig, k, yhat(6 query points) */

/* Injected randomness (the reference's own numpy stream, replayed):
 *   fixed-d samplers: xi[(t*K + c)*d + j], u[t*K + c]
 *   changepoint:      tape[(t*K + c)*RMN_CP_NSLOT + slot]  (xi unused) */
typedef struct {
    const double* d_xi;
    const double* d_u;
    const double* d_tape;
    const double* d_usel;   /* tempered samplers: swap-selection uniforms usel[t*K + c] (ptsampler.py:104);
                             * d_u then holds the accept uniform of a within-chain step or the swap uniform (:121);
                             * on the changepoint model the tape's RMN_CP_SLOT_ACC slot does, for a swap initiator the
                             * swap uniform (the other slots of a swap participant's row are not read) */
} rmn_inject_t;

/* Optional trace.  History index i = 0 is the state at entry, i = t+1 the state after
 * step t of this call (sampler.py:49-54).  States with i >= first and
 * (i - first) % thin == 0, i >= 1, are written to record r = (i - first) / thin.
 *   fixed-d:      d_theta[r][K][d], d_logpost[r][K]
 *   changepoint:  d_k[r][K], d_cpx[r][K][LANES], d_cpv[r][K][LANES], d_sig[r][K]
 * d_prop_logpost[t][K] / d_accepted[t][K] / d_logqratio[t][K] (every step, unthinned)
 * expose the proposed log-posterior, the decision and log q(theta'|theta)/q(theta|theta')
 * (proposal.py:15); d_prop_theta[t][K][d] (fixed-d) or d_prop_k/cpx/cpv/sig (changepoint,
 * canonical layout per step) expose the proposed state itself = what Proposal.propose
 * returns.  Any pointer may be NULL. */
typedef struct {
    int64_t first;
    int64_t thin;
    double* d_theta;
    double* d_logpost;
    int32_t* d_k;
    double* d_cpx;
    double* d_cpv;
    double* d_sig;
    double* d_prop_logpost;
    uint8_t* d_accepted;
    double* d_logqratio;
    double* d_prop_theta;
    int32_t* d_prop_k;
    double* d_prop_cpx;
    double* d_prop_cpv;
    double* d_prop_sig;
} rmn_trace_t;

size_t rmn_sampler_workspace_bytes(const rmn_model_t* m, const rmn_proposal_t* p, int64_t K);

/* K chains on this device; chain c has global id chain_offset + c, which keys its
 * Philox substream (results do not depend on how chains are sharded over GPUs). */
int rmn_sampler_create(rmn_sampler_t** out, rmn_model_t* m, rmn_proposal_t* p, int64_t K,
                       int64_t chain_offset, uint64_t seed, void* d_workspace,
                       size_t workspace_bytes);
/* Precision modes.  RMN_PREC_F64 (default): fp64 state and arithmetic like the reference's numpy (DMMA / DFMA).
 * RMN_PREC_TF32X3: the path's dense contraction on the tcgen05 tensor cores, fp32-accurate (a TF32 MMA for the leading
 * term plus two correction MMAs per product: TF32 in the dense Gaussian GEMM, scaled fp16 at twice the depth in the logistic sweep),
 * everything that enters the accept test reduced in fp64.  ONE stated budget per mode (riemann_b200/budgets.py, asserted by
 * the tests together with an accept-decision gate) on the log-posterior DIFFERENCE proposal - state of sampler.py:83:
 *   dense Gaussian model (fp32 chain state, the K x d by d x d product of the INCREMENT):  5e-7 d   (5e-4 at d = 1000)
 *   logistic model, MALA / HMC / RW / pCN / mMALA (ONE fused kernel per likelihood sweep, logistic_fused.cu: logits into
 *   tensor memory, sigmoid / softplus out of it, R = y - p back into tensor memory as the fp16 operand of the gradient
 *   product -- the gradient only shapes the proposal):  1e-3 sqrt(N / 1e6)   (1e-3 at N = 1e6, SURVEY 8d's gate).  A state's log-posterior also carries a constant offset (<= 5e-8 N,
 *   the fp32 softplus) that is the same for every state and cancels in every Metropolis-Hastings ratio.
 *   With simplified mMALA the Fisher metric of the proposal is one GEMM with bf16 operands (round to nearest, fp32
 *   accumulate; see RMN_PREC_TF32_METRIC for why any deterministic metric keeps the sampler exact). */
#define RMN_PREC_F64 0
#define RMN_PREC_TF32X3 1
/* RMN_PREC_TF32_METRIC: logistic model + simplified mMALA only -- the Fisher metric of the proposal,
 * X^T diag(p(1-p)) X per chain, as ONE single-pass TF32 GEMM on tcgen05 (weights x Khatri-Rao table);
 * log-posterior, gradient, Cholesky and the accept test stay fp64.  The metric only shapes the proposal
 * and the same function theta -> G(theta) enters both proposal densities, so the sampler stays exact. */
#define RMN_PREC_TF32_METRIC 2
size_t rmn_sampler_workspace_bytes_ex(const rmn_model_t* m, const rmn_proposal_t* p, int64_t K, int precision);
int rmn_sampler_create_ex(rmn_sampler_t** out, rmn_model_t* m, rmn_proposal_t* p, int64_t K,
                          int64_t chain_offset, uint64_t seed, void* d_workspace,
                          size_t workspace_bytes, int precision);
int rmn_sampler_destroy(rmn_sampler_t* s);

/* AdaptCovProposal.L of every chain: d_L[K][d][d] (lower triangular). */
int rmn_sampler_get_adaptcov(rmn_sampler_t* s, double* d_L, void* stream);

/* PTSampler (riemann/samplers/ptsampler.py:41-127) on the Gaussian models (small-d and dense path, f64), the logistic
 * model (any precision; the prior is not tempered) and the changepoint model (ChangepointRegression1DProp; a ladder
 * lives inside one warp, so nt <= 8 there; the prior is not tempered): chains c = l*nt + i form ladder l,
 * chain i of a ladder samples TemperedModel(model, h_betas[i]) (likelihood * beta, :33-34); every step each chain either
 * takes a within-chain MH step or, with probability pswap and sequentially along the ladder exactly as :102-125,
 * proposes a swap with its lower neighbour.  K and chain_offset must be multiples of nt (2..32, 2..8 on the changepoint
 * model); non-adaptive RW / pCN proposals, or the changepoint proposal.
 * Call before rmn_sampler_set_state.  On the changepoint model the kernel also counts swap acceptance per pair and the
 * replicas' round trips along the ladder: rmn_sampler_cp_get_swap_stats. */
int rmn_sampler_set_tempering(rmn_sampler_t* s, int nt, const double* h_betas, double pswap);

/* = emcee.autocorr.integrated_time(chain) as called at examples/test_randomwalk.py:42 ("steps per independent sample"),
 * on the device: d_x is a thinned trace x[n][nchains][nfunc] exactly as rmn_trace_t.d_theta holds it.  Per functional:
 * FFT autocorrelation function of every chain (centred, zero-padded to 2 * next_pow2(n); batched cuFFT, resolved at
 * run time), normalised per chain and averaged over the chains ("walkers"), tau(W) = 2 sum_{t<=W} rho(t) - 1, Sokal's
 * automatic window = first W >= c * tau(W) (emcee's default c = 5; the last lag if none).  h_tau[nfunc] (host) receives
 * tau in units of trace rows, h_window[nfunc] (host, may be NULL) the window.  Synchronous; allocates its own scratch
 * (2 * 8 * nchains * nfunc * 2 * next_pow2(n) bytes).  emcee is not vendored by the reference: parity unpinned, the
 * algorithm is restated from its publication (host twin: riemann_b200/diagnostics.py; the tests compare the two). */
int rmn_autocorr_tau(const double* d_x, int64_t n, int64_t nchains, int64_t nfunc, double c, double* h_tau,
                     int64_t* h_window, void* stream);

/* Row-sharded data mode (absent in the reference, whose models hold all their data in one numpy array; SURVEY.md 8f N4:
 * "data-parallel over N when X does not fit").  Every rank creates the logistic model from ITS slice of the rows and a
 * sampler over the SAME K chains (same seed and chain_offset); after every likelihood sweep the per-chain partial
 * log-likelihoods, gradients and (mMALA) metrics are summed over the ranks with one grouped NCCL all-reduce on the
 * sampler's stream, so every rank takes the same accept decisions and the chains stay bit-identical across ranks.
 * rmn_nccl_unique_id: rank 0 fills `out` (>= 128 bytes) with an ncclUniqueId and sends it to the other ranks (any
 * transport; the Python host uses torch.distributed).  rmn_sampler_set_row_comm: collective over the `world` ranks
 * (ncclCommInitRank); call before rmn_sampler_set_state.  f64 precision.  world = 1 is allowed (no-op exchange). */
int rmn_nccl_unique_id(void* out, size_t nbytes);
int rmn_sampler_set_row_comm(rmn_sampler_t* s, const void* unique_id, size_t nbytes, int rank, int world);

/* = Sampler.__init__ (sampler.py:34-42): store the states and evaluate their
 * log-posterior (and gradient / metric caches) on the device. */
int rmn_sampler_set_state(rmn_sampler_t* s, const double* d_theta, void* stream);
int rmn_sampler_get_state(rmn_sampler_t* s, double* d_theta, double* d_logpost, void* stream);
int rmn_sampler_cp_set_state(rmn_sampler_t* s, const int32_t* d_k, const double* d_cpx,
                             const double* d_cpv, const double* d_sig, void* stream);
int rmn_sampler_cp_get_state(rmn_sampler_t* s, int32_t* d_k, double* d_cpx, double* d_cpv,
                             double* d_sig, double* d_logpost, void* stream);

/* T iterations of Sampler.sample (sampler.py:72-90) for every chain.
 * inj == NULL: Philox4x32-10 randomness; else the injected stream is replayed. */
int rmn_sampler_run(rmn_sampler_t* s, int64_t T, const rmn_inject_t* inj,
                    const rmn_trace_t* trace, void* stream);

/* AdaptScaleProposal state per chain (adaptive.py:19-24): scale, Nsamples, Naccepts. */
int rmn_sampler_get_adapt(rmn_sampler_t* s, double* d_scale, int64_t* d_nsamples,
                          int64_t* d_naccepts, void* stream);
int rmn_sampler_set_adapt(rmn_sampler_t* s, const double* d_scale, const int64_t* d_nsamples,
                          const int64_t* d_naccepts, void* stream);
/* Global index of the next MH step = the Philox counter; with get/set_state and get/set_adapt
 * this is the complete resumable state of a sampler (checkpoint / resume). */
int64_t rmn_sampler_get_step(const rmn_sampler_t* s);
int rmn_sampler_set_step(rmn_sampler_t* s, int64_t step);

/* Diagnostics since the last reset.  nd = rmn_sampler_diag_dim(), H = RMN_DIAG_HDR.  The block is
 *   [0] K   [1] functional samples per chain (the changepoint kernel accumulates every
 *   RMN_CP_DIAG_EVERY-th step, the others every step)   [2] total accepts
 *   [3] KCAP overflow events   [4] MH steps per chain   [5] reserved
 *   [H..H+nd)        sum_c m_c[j]          (m_c = per-chain mean of functional j)
 *   [H+nd..H+2nd)    sum_c m_c[j]^2
 *   [H+2nd..H+3nd)   sum_c v_c[j]          (v_c = per-chain biased variance)
 * entries [0],[2],[3] and the sums are additive over chains, so blocks from several GPUs
 * combine with one all-reduce(sum); split-R-hat and ESS follow on the host. */
#define RMN_DIAG_HDR 6
int rmn_sampler_diag_dim(const rmn_sampler_t* s);
int rmn_sampler_reset_diagnostics(rmn_sampler_t* s, void* stream);
int rmn_sampler_reduce_diagnostics(rmn_sampler_t* s, double* d_block, void* stream);

/* Covariance adaptation POOLED over the chains (SURVEY.md section 8f, N5; Haario's adaptive Metropolis, which the
 * reference runs per chain in AdaptCovProposal.adapt, riemann/proposals/adaptive.py:38-103, on one chain's history).
 * With K chains the history of one chain is replaced by the population: every t_adapt MH steps the states of ALL chains
 * (of all ranks when a communicator is set, rmn_sampler_set_row_comm) are added to running sums
 * S1 = sum theta, S2 = sum theta theta^T, n; the random-walk covariance becomes sd * (S2 / n - m m^T) + jitter * I, its
 * Cholesky factor is recomputed on the device and used by every chain from the next step on (randomwalk.py:25-26 with the
 * new L).  stop_after > 0: no adaptation after that many steps (the chain is a plain MH chain from then on, as a
 * burn-in-only adaptation should be); 0 = adapt forever (diminishing: the sums keep growing).
 * Dense Gaussian path (d > 8), f64 precision.  rmn_sampler_get_pooled_cov copies the current estimate out:
 * d_cov[d][d] = S2 / n - m m^T, d_mean[d], d_count[1] = n (device pointers). */
int rmn_proposal_rw_set_pooled_cov_adapt(rmn_proposal_t* p, int64_t t_adapt, double sd, double jitter, int64_t stop_after);
int rmn_sampler_get_pooled_cov(rmn_sampler_t* s, double* d_cov, double* d_mean, double* d_count, void* stream);

/* Per-chain mean and biased variance of the tracked functionals since the last reset: d_mean[nd][K], d_var[nd][K]
 * (chain fastest; either may be NULL).  What `Sampler._chain_thetas` gives the reference's scripts for one chain
 * (examples/test_randomwalk.py:41-46 computes its statistics from the trace) without keeping a trace of K chains;
 * used for per-chain R-hat and for the independence checks of the shared move schedule. */
int rmn_sampler_chain_moments(rmn_sampler_t* s, double* d_mean, double* d_var, void* stream);

/* Changepoint samplers, Philox mode: how the move type of a step (ChangepointRegression1DProp.propose draws it
 * independently of the state, examples/test_changepoint.py:48-54) is assigned to chains.
 *   1 (default)  the chains of an aligned group of 8 consecutive GLOBAL chain ids (one warp) share the three
 *                selection draws of a step, so a warp executes one move-specific code path per step.  Every chain
 *                still sees an i.i.d. move sequence with the reference's probabilities, independent of its state:
 *                each chain is an exact replica of the reference sampler; chains of a group are conditionally
 *                independent given the schedule and uncorrelated in stationarity.  Independent of the sharding.
 *   0            every chain draws its own move types.
 * Injected runs always replay the per-chain move types of the tape.  Call before rmn_sampler_run. */
int rmn_sampler_set_move_schedule(rmn_sampler_t* s, int mode);

/* Posterior summaries of an untempered changepoint sampler, accumulated on the device as 64-bit integer histograms (no
 * trace needed).  After every MH step whose global index s (rmn_sampler_get_step counts them) satisfies s % every == 0,
 * the state of every chain adds
 *   khist[k] += 1                         k = number of changepoints, 0..RMN_CP_LANES-1;
 *   cpxhist[i] += 1 per changepoint x     i = #{g : h_grid[g] <= x} in 0..G (numpy searchsorted(grid, x, 'right'));
 *   yhist[g][b] += 1 per grid point g     b = value bin of the prediction y = cpv[searchsorted(cpx[:k], grid[g])]
 *                                         (ChangepointRegression1D.predict, changepoint.py:181): 1 + floor((y - vlo) * inv)
 *                                         with inv = H / (vhi - vlo) in fp64 and round-to-nearest products, clamped to
 *                                         bin 0 (below vlo, and NaN) and bin H + 1 (at or above vhi);
 * and the count of sampled chain-steps grows by one.  Integer sums do not depend on the order of the additions, so the
 * counts are identical for any split of a run into calls, time slices or chain shards.  rmn_sampler_reset_diagnostics
 * also zeroes them.  The chains themselves are unchanged bit for bit.
 * rmn_sampler_cp_set_summary: 1 <= G <= 1024 strictly increasing finite grid points h_grid (host), finite vlo < vhi,
 * 1 <= H <= 1024 value bins, 1 <= every <= 2^62; resets the counts.  G = 0 turns the summaries off and frees their
 * buffers.  Changepoint samplers at 4 lanes per chain only (RMN_CP_GL unset or 4), not tempered: RMN_ERR_UNSUPPORTED.
 * rmn_sampler_cp_get_summary: d_khist[RMN_CP_LANES], d_cpxhist[G + 1], d_yhist[G][H + 2] (device, int64, any may be
 * NULL) and *h_nsamples (host, may be NULL), the counts since the last reset; enqueued on `stream`. */
int rmn_sampler_cp_set_summary(rmn_sampler_t* s, int G, const double* h_grid, double vlo, double vhi, int H,
                               int64_t every);
int rmn_sampler_cp_get_summary(rmn_sampler_t* s, int64_t* d_khist, int64_t* d_cpxhist, int64_t* d_yhist,
                               int64_t* h_nsamples, void* stream);

/* The same summaries for a tempered changepoint sampler (rmn_sampler_set_tempering): only the chain of rung `rung`
 * (inverse temperature h_betas[rung]) of every ladder is sampled, in its state after the step's swaps, so the count of
 * sampled chain-steps grows by K / nt per sampled step.  Same arguments and checks as rmn_sampler_cp_set_summary plus
 * 0 <= rung < nt; G = 0 turns the summaries off.  The counts are read with rmn_sampler_cp_get_summary and zeroed by
 * rmn_sampler_reset_diagnostics; the chains are unchanged bit for bit.  Untempered samplers and other model families:
 * RMN_ERR_UNSUPPORTED (rmn_sampler_cp_set_summary serves the untempered changepoint sampler, and refuses tempered ones). */
int rmn_sampler_cp_set_rung_summary(rmn_sampler_t* s, int rung, int G, const double* h_grid, double vlo, double vhi,
                                    int H, int64_t every);

/* Swap statistics of a tempered changepoint sampler (rmn_sampler_set_tempering) since the last
 * rmn_sampler_reset_diagnostics, pooled over its ladders, int64 device arrays (any may be NULL):
 *   d_proposed[nt-1], d_accepted[nt-1]  swaps initiated by rung i with rung i+1 / taken;
 *   d_up[nt], d_down[nt]                at every step s with s % RMN_CP_DIAG_EVERY == 0, chains at rung i whose
 *                                       replica last touched rung 0 / rung nt-1;
 *   d_round_trips[1]                    replicas that went from rung 0 to rung nt-1 and back to rung 0.
 * A replica's direction travels with its state; rmn_sampler_cp_set_state starts the walk (rung 0 up, rung nt-1 down,
 * the others neither), and rmn_sampler_reset_diagnostics zeroes the counts but keeps the directions, so a trip in
 * progress still completes.  Integer counts: identical for any split of a run into calls and any sharding of the
 * ladders.  Enqueued on `stream`.  The chains are unchanged by the counting.  Untempered samplers and other model
 * families: RMN_ERR_UNSUPPORTED. */
int rmn_sampler_cp_get_swap_stats(rmn_sampler_t* s, int64_t* d_proposed, int64_t* d_accepted, int64_t* d_up,
                                  int64_t* d_down, int64_t* d_round_trips, void* stream);

/* Number of kernel launches this handle has enqueued so far. */
int64_t rmn_sampler_launch_count(const rmn_sampler_t* s);

/* Measurement aid: CUDA-event timing of the sampler's DOMINANT kernel (changepoint_kernel,
 * small_gauss_kernel, gemm_abt_kernel, tf32x3_gemm_kernel, lg_eval_kernel / lg_metric_kernel), one event
 * pair per launch on the launching stream.  rmn_sampler_kernel_timing waits for the last recorded
 * event, returns the summed duration and the number of timed launches since the previous call (at most
 * 8192 per window; `untimed` counts the rest) and the kernel's name, and starts a new window. */
int rmn_sampler_enable_kernel_timing(rmn_sampler_t* s, int enable);
int rmn_sampler_kernel_timing(rmn_sampler_t* s, double* total_ms, int64_t* launches, int64_t* untimed,
                              const char** kernel_name);

/* Raw device RNG, for known-answer tests: out[n][4] = Philox4x32-10(ctr[n][4], key[n][2]). */
int rmn_philox_raw(int64_t n, const uint32_t* d_ctr, const uint32_t* d_key, uint32_t* d_out,
                   void* stream);
/* The engine's N(0,1)/U(0,1) for (seed, chain, step): normals[n][nn] and uniform[n]. */
int rmn_rng_draws(uint64_t seed, int64_t chain0, int64_t step, int64_t n, int nn,
                  double* d_normals, double* d_uniform, void* stream);

/* fp32-accurate tensor-core product (tcgen05.mma.kind::tf32, TMA, TMEM), validation entry:
 * C[M][N] (fp32, row-major) ~= (Ah + Al)(Bh + Bl)^T  with Ah Bh^T + Ah Bl^T + Al Bh^T accumulated
 * in fp32; A* are [M][K], B* are [N][K] fp32 with the "hi" parts TF32-exact; K % 16 == 0, N % 4 == 0.
 * It is the GEMM behind the tf32x3 precision mode of the dense Gaussian sampler. */
int rmn_tf32x3_gemm(int64_t M, int N, int K, const float* d_Ah, const float* d_Al, const float* d_Bh,
                    const float* d_Bl, float* d_C, void* stream);
/* Split-K mode of the same kernel (few output tiles, long contraction): C[s][M][N], s < *used_splits <= ksplit,
 * are partial products over contiguous ranges of K; their sum is the product. */
int rmn_tf32x3_gemm_splitk(int64_t M, int N, int K, int ksplit, const float* d_Ah, const float* d_Al,
                           const float* d_Bh, const float* d_Bl, float* d_C, int* used_splits, void* stream);
/* Single-pass TF32 product on the same kernel, validation entry: C[M][N] (fp32) ~= A B^T, A [M][K],
 * B [N][K] fp32 (the tensor core drops the low 13 mantissa bits of each operand); K % 32 == 0, N % 4 == 0.
 * It is the GEMM behind RMN_PREC_TF32_METRIC. */
int rmn_tf32_gemm(int64_t M, int N, int K, const float* d_A, const float* d_B, float* d_C, void* stream);
/* The same kernel with bf16 operands (tcgen05.mma.kind::f16, fp32 accumulate): C[M][N] (fp32) = A B^T, A [M][K] and
 * B [N][K] bf16 row-major; K % 64 == 0, N % 4 == 0.  Used for the Fisher metric of the mMALA proposal in the tf32x3
 * precision mode (a product that only shapes a proposal; the reference has no counterpart). */
int rmn_bf16_gemm(int64_t M, int N, int K, const void* d_A, const void* d_B, float* d_C, void* stream);

/* The logistic likelihood's pointwise stage (riemann_b200/csrc/logistic_math.cuh), validation entry:
 * p[i] = sigmoid(z[i]), sp[i] = softplus(z[i]), pq[i] = p (1 - p), fp64, |error| <~ 2e-16 absolute. */
int rmn_logistic_math(int64_t n, const double* d_z, double* d_p, double* d_sp, double* d_pq, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* RIEMANN_B200_H */
