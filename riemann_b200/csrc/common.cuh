// riemann_b200 -- shared device utilities and host-side handle definitions.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>
#include <string>
#include <vector>

#include "../../include/riemann_b200.h"

// ----------------------------------------------------------------------------
// error plumbing (host)
// ----------------------------------------------------------------------------
void rmn_set_error(const char* fmt, ...);

#define RMN_CUDA(call)                                                             \
    do {                                                                           \
        cudaError_t e__ = (call);                                                  \
        if (e__ != cudaSuccess) {                                                  \
            rmn_set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call,            \
                          cudaGetErrorString(e__));                                \
            return RMN_ERR_CUDA;                                                   \
        }                                                                          \
    } while (0)

#define RMN_REQUIRE(cond, ...)                                                     \
    do {                                                                           \
        if (!(cond)) {                                                             \
            rmn_set_error(__VA_ARGS__);                                            \
            return RMN_ERR_PARAM;                                                  \
        }                                                                          \
    } while (0)

#define RMN_KERNEL_CHECK() RMN_CUDA(cudaGetLastError())

// ----------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al. SC'11).  Replaces numpy's global MT19937 stream
// (randomwalk.py:25, sampler.py:84).  key = (seed_lo, seed_hi),
// counter = (block, step_lo, step_hi, global chain id).
// ----------------------------------------------------------------------------
#define RMN_PHILOX_M0 0xD2511F53u
#define RMN_PHILOX_M1 0xCD9E8D57u
#define RMN_PHILOX_W0 0x9E3779B9u
#define RMN_PHILOX_W1 0xBB67AE85u
#define RMN_BLOCK_ACCEPT 0xFFFFFFFFu /* block index reserved for the accept uniform */
#define RMN_BLOCK_AUX 0xFFFFFFFEu    /* selection / auxiliary uniforms               */
#define RMN_BLOCK_AUX2 0xFFFFFFFDu

__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(RMN_PHILOX_M0, c.x), lo0 = RMN_PHILOX_M0 * c.x;
        const uint32_t hi1 = __umulhi(RMN_PHILOX_M1, c.z), lo1 = RMN_PHILOX_M1 * c.z;
        c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
        k.x += RMN_PHILOX_W0;
        k.y += RMN_PHILOX_W1;
    }
    return c;
}

struct RngKey {
    uint2 key;
    uint32_t chain;
    __device__ __forceinline__ RngKey(uint64_t seed, uint64_t chain_id)
        : key(make_uint2((uint32_t)seed, (uint32_t)(seed >> 32))), chain((uint32_t)chain_id) {}
    __device__ __forceinline__ uint4 block(uint64_t step, uint32_t blk) const {
        return philox4x32_10(make_uint4(blk, (uint32_t)step, (uint32_t)(step >> 32), chain), key);
    }
};

// uniform on (0,1): (x + 0.5) * 2^-32, exact in fp64
__device__ __forceinline__ double u01(uint32_t x) {
    return ((double)x + 0.5) * (1.0 / 4294967296.0);
}

// Box-Muller in fp32 (cuRAND-style 32-bit uniforms), widened to fp64 afterwards.
// The randomness is not parity-bound (parity runs inject the reference's stream).
__device__ __forceinline__ void box_muller(uint32_t a, uint32_t b, float& n0, float& n1) {
    const float u1 = fmaf((float)a, 2.3283064365386963e-10f, 1.1641532182693481e-10f);
    const float ang = fmaf((float)b, 2.3283064365386963e-10f * 6.283185307179586f,
                           1.1641532182693481e-10f * 6.283185307179586f - 3.14159265358979f);
    const float r = sqrtf(-2.0f * __logf(u1));
    float s, c;
    __sincosf(ang, &s, &c);
    n0 = r * c;
    n1 = r * s;
}

// nanosecond wall clock common to all SMs (timeline aids)
__device__ __forceinline__ long long rmn_globaltimer() {
    long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// four N(0,1) from one Philox block
__device__ __forceinline__ void normal4(const uint4 r, double out[4]) {
    float a, b, c, d;
    box_muller(r.x, r.y, a, b);
    box_muller(r.z, r.w, c, d);
    out[0] = a; out[1] = b; out[2] = c; out[3] = d;
}

// ----------------------------------------------------------------------------
// Metropolis-Hastings accept rule, sampler.py:83-84.
//   mhratio = min(0, lp' - lp - logqratio)  with PYTHON's min: nan -> 0
//   accept iff log(u) < mhratio (strict)
// ----------------------------------------------------------------------------
__device__ __forceinline__ bool mh_accept(double lp_new, double lp_old, double lqr, double u) {
    const double delta = lp_new - lp_old - lqr;
    const double mh = (delta < 0.0) ? delta : 0.0;   // false for nan -> 0
    return log(u) < mh;
}

// model.py:50-54: any inf (either sign) or nan in prior or likelihood -> -inf
__device__ __forceinline__ double combine_logpost(double logp, double logl) {
    return (isfinite(logp) && isfinite(logl)) ? (logp + logl) : -INFINITY;
}

// AdaptScaleProposal.adapt (adaptive.py:26-35), one chain
struct AdaptState {
    double scale;
    long long nsamples;
    long long naccepts;
    __device__ __forceinline__ void update(bool moved, double target) {
        const bool first = (nsamples == 0);          // last_theta is None -> counts as accept
        nsamples += 1;
        naccepts += (moved || first) ? 1 : 0;
        const double rate = (double)naccepts / (double)nsamples;
        const double r = exp(1.0 / (double)nsamples);
        if (rate > target) scale = __dmul_rn(scale, r);
        else scale = __ddiv_rn(scale, r);
    }
};

template <int W>
__device__ __forceinline__ double group_sum(double v) {
#pragma unroll
    for (int o = W / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o, W);
    return v;
}

// trace bookkeeping: history index i (>=1) -> record slot or -1
struct TraceSel {
    long long first, thin;
    __device__ __forceinline__ long long slot(long long i) const {
        if (i < first) return -1;
        const long long r = i - first;
        return (r % thin == 0) ? r / thin : -1;
    }
};

// ----------------------------------------------------------------------------
// host-side handles
// ----------------------------------------------------------------------------
enum { RMN_MODEL_GAUSS = 1, RMN_MODEL_CP = 2, RMN_MODEL_LOGISTIC = 3 };
enum { RMN_PROP_RW = 1, RMN_PROP_HMC = 2, RMN_PROP_PCN = 3, RMN_PROP_MMALA = 4, RMN_PROP_CP = 5 };

struct rmn_model {
    int kind = 0;
    int d = 0;
    int device = 0;
    // gaussian
    std::vector<double> h_mu, h_linv;    // linv: packed lower triangle, row-major
    double logdetC = 0.0;
    double* d_mu = nullptr;              // [d]
    double* d_prec = nullptr;            // [d][d]
    // changepoint
    int M = 0, kmax = 0;
    double xmin = 0, xmax = 0, lamb = 0, alpha = 0, beta = 0, ycenter = 0;
    double* d_cpdata = nullptr;          // x[XP] | {cy, cyy}[M+1] | bucket table int32[cp_G] (changepoint.cuh: CPParams)
    int cp_G = 0;                        // buckets of the run-boundary table, 0 = none
    double cp_bscale = 0, cp_boff = 0;
    double tabA[RMN_CP_LANES + 1];       // k log lam - gammaln(k) - lam + gammaln(2k+1), k = #steps
    double cv = 0.0;                     // alpha log beta - gammaln(alpha)
    // logistic
    int64_t N = 0;
    const double* d_X = nullptr;
    const double* d_y = nullptr;
    double prior_var = 1.0;
};

struct rmn_proposal {
    int kind = 0;
    int d = 0;
    int adapt = 0;
    double target = 0.0;
    // rw / pcn
    std::vector<double> h_L, h_Linv;     // full d x d row-major
    double rho = 0.0;
    // hmc
    double eps = 0.0;
    int nsteps = 1;
    bool has_mass = false;
    std::vector<double> h_chM, h_Minv, h_chMinv;
    // device copies for the large-d path
    double* d_L = nullptr;
    // covariance adaptation (AdaptCovRandomWalk, adaptive.py:38-103)
    int acov = 0, ac_marginalize = 0, ac_smooth = 0;
    double ac_t_adapt = 1.0;
    std::vector<double> h_C0;            // full d x d
    // pooled covariance adaptation (SURVEY 8f N5 "pooled across chains"; dense Gaussian path): every pool_t_adapt steps the
    // proposal covariance becomes pool_sd * (covariance of ALL chains' states accumulated so far) + pool_jitter * I
    int pool_cov = 0;
    int64_t pool_t_adapt = 0, pool_stop = 0;
    double pool_sd = 0.0, pool_jitter = 0.0;
    // changepoint mix
    double hscale = 0.0;
    double p_cum[3] = {0.20, 0.40, 0.60};
};

// Optional CUDA-event timing of a sampler's dominant kernel (rmn_sampler_enable_kernel_timing): one event
// pair around each launch on the launching stream, resolved by rmn_sampler_kernel_timing.  bench.py uses
// it for `roofline.achieved` (algorithmic work / the kernel's own average launch duration).
struct KernelTimer {
    bool on = false;
    const char* name = "";
    std::vector<cudaEvent_t> ev;
    size_t used = 0;
    static constexpr size_t CAP = 16384;       // events; later launches of a window are not timed
    int64_t untimed = 0;
    bool armed = false;
    void begin(const char* kname, cudaStream_t st) {
        armed = false;
        if (!on) return;
        name = kname;
        if (used + 2 > CAP) { ++untimed; return; }
        while (ev.size() < used + 2) {
            cudaEvent_t e;
            if (cudaEventCreate(&e) != cudaSuccess) { ++untimed; return; }
            ev.push_back(e);
        }
        cudaEventRecord(ev[used], st);
        armed = true;
    }
    void end(cudaStream_t st) {
        if (!armed) return;
        cudaEventRecord(ev[used + 1], st);
        used += 2;
        armed = false;
    }
    // total ms and number of timed launches since the last collect; synchronizes on the last event
    int collect(double* ms, int64_t* n) {
        double tot = 0.0;
        if (used) cudaEventSynchronize(ev[used - 1]);
        for (size_t i = 0; i + 1 < used; i += 2) {
            float t = 0.f;
            if (cudaEventElapsedTime(&t, ev[i], ev[i + 1]) == cudaSuccess) tot += t;
        }
        if (ms) *ms = tot;
        if (n) *n = (int64_t)(used / 2);
        used = 0; untimed = 0;
        return 0;
    }
    ~KernelTimer() { for (cudaEvent_t e : ev) cudaEventDestroy(e); }
};

struct rmn_sampler;
// integrated autocorrelation time of a device trace (acf.cu)
int rmn_autocorr_tau_impl(const double* d_x, int64_t n, int64_t K, int64_t nd, double c, double* h_tau,
                          int64_t* h_window, cudaStream_t stream);

// Row-sharded likelihood (comm.cu): an NCCL communicator over the ranks that each hold a slice of the data rows.
struct RowComm { void* comm = nullptr; int rank = 0, world = 1; };
int rmn_rowcomm_unique_id(void* out, size_t nbytes);
int rmn_rowcomm_init(RowComm* rc, const void* unique_id, size_t nbytes, int rank, int world);
int rmn_rowcomm_allreduce_f64(RowComm* rc, double* const* bufs, const size_t* counts, int nbuf, cudaStream_t stream);
void rmn_rowcomm_destroy(RowComm* rc);

struct SamplerImpl {
    virtual ~SamplerImpl() {}
    KernelTimer ktimer;
    virtual size_t workspace_bytes() const = 0;
    virtual int bind(void* ws) = 0;
    virtual int set_state(const double* d_theta, cudaStream_t st) { return unsupported("set_state"); }
    virtual int get_state(double* d_theta, double* d_lp, cudaStream_t st) { return unsupported("get_state"); }
    virtual int cp_set_state(const int32_t*, const double*, const double*, const double*, cudaStream_t) { return unsupported("cp_set_state"); }
    virtual int cp_get_state(int32_t*, double*, double*, double*, double*, cudaStream_t) { return unsupported("cp_get_state"); }
    virtual int run(int64_t T, const rmn_inject_t* inj, const rmn_trace_t* tr, cudaStream_t st) = 0;
    virtual int get_adaptcov(double*, cudaStream_t) { return unsupported("get_adaptcov (small-d AdaptCovRandomWalk samplers only)"); }
    virtual int get_pooled_cov(double*, double*, double*, cudaStream_t) { return unsupported("get_pooled_cov (dense Gaussian samplers with PooledAdaptCovRandomWalk only)"); }
    virtual int set_row_comm(const void*, size_t, int, int) { return unsupported("row-sharded data mode (logistic samplers in f64 precision only)"); }
    virtual int set_tempering(int, const double*, double) { return unsupported("parallel tempering (Gaussian and logistic samplers with RW / pCN proposals, changepoint samplers)"); }
    virtual int get_adapt(double*, int64_t*, int64_t*, cudaStream_t) { return unsupported("get_adapt"); }
    virtual int set_adapt(const double*, const int64_t*, const int64_t*, cudaStream_t) { return unsupported("set_adapt"); }
    virtual int set_move_schedule(int) { return unsupported("move schedule (changepoint samplers only)"); }
    virtual int cp_set_summary(int, const double*, double, double, int, int64_t) { return unsupported("posterior summaries (changepoint samplers only)"); }
    virtual int cp_set_rung_summary(int, int, const double*, double, double, int, int64_t) { return unsupported("rung posterior summaries (tempered changepoint samplers only)"); }
    virtual int cp_get_summary(int64_t*, int64_t*, int64_t*, int64_t*, cudaStream_t) { return unsupported("posterior summaries (changepoint samplers only)"); }
    virtual int cp_get_swap_stats(int64_t*, int64_t*, int64_t*, int64_t*, int64_t*, cudaStream_t) { return unsupported("swap statistics (tempered changepoint samplers only)"); }
    // raw per-chain diagnostics sums S1, S2 [nd][K] (chain fastest) and the number of samples behind them
    virtual int chain_sums(const double** S1, const double** S2, int64_t* nsamples) { return unsupported("per-chain moments"); }
    virtual int diag_dim() const = 0;
    virtual int reset_diag(cudaStream_t st) = 0;
    virtual int reduce_diag(double* d_block, cudaStream_t st) = 0;
    int unsupported(const char* what) {
        rmn_set_error("%s is not available for this sampler family", what);
        return RMN_ERR_UNSUPPORTED;
    }
    int64_t launches = 0;
    int64_t step0 = 0;        // global MH step index of the next iteration (Philox counter)
    int64_t diag_steps = 0;   // steps since the last diagnostics reset
    int64_t diag_samples = 0; // functional samples accumulated since the reset (families that thin)
};

struct rmn_sampler {
    rmn_model* model = nullptr;
    rmn_proposal* prop = nullptr;
    int64_t K = 0, chain_offset = 0;
    uint64_t seed = 0;
    int precision = 0;
    SamplerImpl* impl = nullptr;
};

// factories implemented per family
SamplerImpl* make_small_gauss_sampler(rmn_sampler* s);
SamplerImpl* make_changepoint_sampler(rmn_sampler* s);
SamplerImpl* make_dense_gauss_sampler(rmn_sampler* s);
SamplerImpl* make_logistic_sampler(rmn_sampler* s);
SamplerImpl* make_dense_tf32_sampler(rmn_sampler* s);

// pointwise evaluators implemented per family
int gauss_pointwise(rmn_model* m, int which, int64_t n, const double* d_theta, double* d_out,
                    double* d_grad, cudaStream_t st);
int cp_pointwise(rmn_model* m, int which, int64_t n, const int32_t* d_k, const double* d_cpx,
                 const double* d_cpv, const double* d_sig, double* d_out, cudaStream_t st);
int logistic_pointwise(rmn_model* m, int which, int64_t n, const double* d_theta, double* d_out,
                       double* d_grad, double* d_metric, cudaStream_t st);

// generic helper kernels (util.cu)
int rmn_fill_f64(double* p, int64_t n, double v, cudaStream_t st);
int rmn_fill_i64(long long* p, int64_t n, long long v, cudaStream_t st);
int rmn_copy_adapt(int64_t K, const double* sc_in, const int64_t* ns_in, const int64_t* na_in, double* sc,
                   long long* ns, long long* na, cudaStream_t st);
// per-chain sums -> diagnostics block; S1/S2 are [nd][K] (chain fastest)
int rmn_reduce_diag_block(int64_t K, int nd, int64_t nsamples, int64_t nsteps, const double* S1, const double* S2,
                          const long long* acc, const long long* ovf, double* d_block,
                          cudaStream_t st);

// per-chain mean / biased variance of the tracked functionals from the raw sums (util.cu)
int rmn_chain_moments(int64_t K, int nd, int64_t nsamples, const double* S1, const double* S2, double* d_mean,
                      double* d_var, cudaStream_t st);

// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-device property of the KERNEL, shared by every sampler in the
// process: only ever raise it, so a sampler created later with a smaller shape cannot lower the limit under one
// that is still alive (util.cu keeps the largest value requested per (device, kernel)).
cudaError_t rmn_raise_dyn_smem(const void* kernel, size_t bytes);
#define RMN_RAISE_SMEM(kernel, bytes) RMN_CUDA(rmn_raise_dyn_smem((const void*)(kernel), (size_t)(bytes)))

static inline size_t align256(size_t x) { return (x + 255) & ~size_t(255); }
