// riemann_b200 -- C ABI entry points (see include/riemann_b200.h).
#include <stdarg.h>
#include <stdio.h>
#include <string.h>
#include <algorithm>

#include "common.cuh"
#include "changepoint.cuh"
#include <nvtx3/nvToolsExt.h>      // header-only; a no-op unless a profiler injects itself (NVTX_INJECTION64_PATH)

static thread_local char g_err[1024] = "";

// NVTX range around the calls of the per-iteration path, so a timeline shows set_state / run / get_state per job
struct NvtxRange {
    explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
};

void rmn_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

extern "C" int rmn_version(void) { return RMN_VERSION; }
extern "C" const char* rmn_last_error(void) { return g_err; }

static bool finite_all(const double* p, size_t n) {
    for (size_t i = 0; i < n; ++i)
        if (!isfinite(p[i])) return false;
    return true;
}

// ---------------------------------------------------------------- models ----
extern "C" int rmn_model_gaussian_create(rmn_model_t** out, int d, const double* h_mu,
                                         const double* h_prec, const double* h_linv,
                                         double logdetC) {
    RMN_REQUIRE(out && h_mu && h_prec, "rmn_model_gaussian_create: null argument");
    RMN_REQUIRE(d >= 1, "rmn_model_gaussian_create: d must be >= 1 (got %d)", d);
    RMN_REQUIRE(d > RMN_SMALL_D_MAX || h_linv, "rmn_model_gaussian_create: h_linv required for d <= %d",
                RMN_SMALL_D_MAX);
    RMN_REQUIRE(finite_all(h_prec, (size_t)d * d) && finite_all(h_mu, d) && isfinite(logdetC),
                "rmn_model_gaussian_create: non-finite hyper-parameter");
    rmn_model* m = new rmn_model();
    m->kind = RMN_MODEL_GAUSS;
    m->d = d;
    m->logdetC = logdetC;
    m->h_mu.assign(h_mu, h_mu + d);
    if (h_linv && d <= RMN_SMALL_D_MAX) {
        m->h_linv.resize((size_t)d * (d + 1) / 2);
        for (int i = 0; i < d; ++i)
            for (int j = 0; j <= i; ++j) m->h_linv[i * (i + 1) / 2 + j] = h_linv[(size_t)i * d + j];
    }
    cudaGetDevice(&m->device);
    if (cudaMalloc(&m->d_mu, (size_t)d * 8) != cudaSuccess ||
        cudaMalloc(&m->d_prec, (size_t)d * d * 8) != cudaSuccess ||
        cudaMemcpy(m->d_mu, h_mu, (size_t)d * 8, cudaMemcpyHostToDevice) != cudaSuccess ||
        cudaMemcpy(m->d_prec, h_prec, (size_t)d * d * 8, cudaMemcpyHostToDevice) != cudaSuccess) {
        rmn_set_error("rmn_model_gaussian_create: device allocation/upload failed: %s",
                      cudaGetErrorString(cudaGetLastError()));
        rmn_model_destroy(m);
        return RMN_ERR_CUDA;
    }
    *out = m;
    return RMN_OK;
}

extern "C" int rmn_model_changepoint_create(rmn_model_t** out, int M, const double* h_x,
                                            const double* h_y, double xmin, double xmax,
                                            double lamb, int kmax, double alpha, double beta) {
    RMN_REQUIRE(out && (M == 0 || (h_x && h_y)), "rmn_model_changepoint_create: null argument");
    RMN_REQUIRE(M >= 1, "rmn_model_changepoint_create: need at least one data point (M=%d)", M);
    RMN_REQUIRE(xmax > xmin, "rmn_model_changepoint_create: require xmax > xmin");
    RMN_REQUIRE(lamb > 0 && alpha > 0 && beta > 0,
                "rmn_model_changepoint_create: lamb, alpha, beta must be positive");
    for (int i = 1; i < M; ++i)
        RMN_REQUIRE(h_x[i] >= h_x[i - 1], "rmn_model_changepoint_create: x must be sorted ascending");
    rmn_model* m = new rmn_model();
    m->kind = RMN_MODEL_CP;
    m->d = 2 * RMN_CP_LANES + 1;
    m->M = M; m->kmax = kmax;
    m->xmin = xmin; m->xmax = xmax; m->lamb = lamb; m->alpha = alpha; m->beta = beta;
    m->cv = alpha * log(beta) - lgamma(alpha);
    double mean = 0.0;
    for (int i = 0; i < M; ++i) mean += h_y[i];
    mean /= (double)M;
    m->ycenter = mean;
    // run-boundary bucket table (changepoint.cuh: run_boundary): the fewest buckets, a power of two from M up to
    // BUCKET_GMAX, in which no bucket holds more than BUCKET_W points.  Other data keeps the binary search (G = 0).
    bool finite = true;
    for (int i = 0; i < M; ++i) finite = finite && isfinite(h_x[i]);
    int G = 2;
    while (G < M) G *= 2;
    for (std::vector<int> cnt; finite && G <= cp::BUCKET_GMAX; G *= 2) {
        const double scale = G / (xmax - xmin), off = -xmin * scale;
        if (!(isfinite(scale) && isfinite(off))) break;
        cnt.assign(G, 0);
        int C = 0;
        for (int i = 0; i < M; ++i) C = std::max(C, ++cnt[cp::bucket_of(h_x[i], scale, off, G)]);
        if (C <= cp::BUCKET_W) {
            m->cp_G = G; m->cp_bscale = scale; m->cp_boff = off;
            break;
        }
    }
    int p2 = 1;
    while (p2 * 2 <= M) p2 *= 2;
    const int XP = 2 * p2;                         // x table padded with NaN (changepoint.cuh: run_boundary)
    std::vector<double> buf((size_t)XP + 2 * (size_t)M + 2 + (size_t)m->cp_G * 5 / 2, NAN);
    double* x = buf.data();
    double* cyc = x + XP;                          // {cy, cyy} pairs
    cyc[0] = 0.0; cyc[1] = 0.0;
    for (int i = 0; i < M; ++i) {
        x[i] = h_x[i];
        const double r = h_y[i] - mean;
        cyc[2 * i + 2] = cyc[2 * i] + r;
        cyc[2 * i + 3] = cyc[2 * i + 1] + r * r;
    }
    if (m->cp_G > 0) {
        // bx[b] = {x[s], x[s + 1]}, bstart[b] = s = min(#{i : bucket(x_i) < b}, XP - 2)
        double* bx = cyc + 2 * (size_t)M + 2;
        std::vector<int> bstart(m->cp_G);
        for (int b = 0, i = 0; b < m->cp_G; ++b) {
            while (i < M && cp::bucket_of(h_x[i], m->cp_bscale, m->cp_boff, m->cp_G) < b) ++i;
            bstart[b] = std::min(i, XP - 2);
            bx[2 * b] = x[bstart[b]];
            bx[2 * b + 1] = x[bstart[b] + 1];
        }
        memcpy(bx + 2 * (size_t)m->cp_G, bstart.data(), bstart.size() * sizeof(int));
    }
    cudaGetDevice(&m->device);
    if (cudaMalloc(&m->d_cpdata, buf.size() * 8) != cudaSuccess ||
        cudaMemcpy(m->d_cpdata, buf.data(), buf.size() * 8, cudaMemcpyHostToDevice) != cudaSuccess) {
        rmn_set_error("rmn_model_changepoint_create: device allocation/upload failed");
        rmn_model_destroy(m);
        return RMN_ERR_CUDA;
    }
    *out = m;
    return RMN_OK;
}

extern "C" int rmn_model_logistic_create(rmn_model_t** out, int64_t N, int d, const double* d_X,
                                         const double* d_y, double prior_var) {
    RMN_REQUIRE(out && d_X && d_y, "rmn_model_logistic_create: null argument");
    RMN_REQUIRE(N >= 1 && d >= 1, "rmn_model_logistic_create: need N >= 1 and d >= 1");
    RMN_REQUIRE(prior_var > 0, "rmn_model_logistic_create: prior_var must be positive");
    rmn_model* m = new rmn_model();
    m->kind = RMN_MODEL_LOGISTIC;
    m->d = d; m->N = N; m->d_X = d_X; m->d_y = d_y; m->prior_var = prior_var;
    cudaGetDevice(&m->device);
    *out = m;
    return RMN_OK;
}

extern "C" int rmn_model_destroy(rmn_model_t* m) {
    if (!m) return RMN_OK;
    if (m->d_mu) cudaFree(m->d_mu);
    if (m->d_prec) cudaFree(m->d_prec);
    if (m->d_cpdata) cudaFree(m->d_cpdata);
    delete m;
    return RMN_OK;
}

extern "C" int rmn_model_dim(const rmn_model_t* m) { return m ? m->d : 0; }

extern "C" int rmn_model_logpost(rmn_model_t* m, int which, int64_t n, const double* d_theta,
                                 double* d_out, void* stream) {
    RMN_REQUIRE(m && d_theta && d_out && n >= 0, "rmn_model_logpost: bad argument");
    RMN_REQUIRE(which >= 0 && which <= 2, "rmn_model_logpost: which must be 0, 1 or 2");
    if (m->kind == RMN_MODEL_GAUSS) return gauss_pointwise(m, which, n, d_theta, d_out, nullptr, (cudaStream_t)stream);
    if (m->kind == RMN_MODEL_LOGISTIC)
        return logistic_pointwise(m, which, n, d_theta, d_out, nullptr, nullptr, (cudaStream_t)stream);
    rmn_set_error("rmn_model_logpost: use rmn_model_cp_logpost for the changepoint model");
    return RMN_ERR_UNSUPPORTED;
}

extern "C" int rmn_model_grad(rmn_model_t* m, int64_t n, const double* d_theta, double* d_grad,
                              void* stream) {
    RMN_REQUIRE(m && d_theta && d_grad && n >= 0, "rmn_model_grad: bad argument");
    if (m->kind == RMN_MODEL_GAUSS) return gauss_pointwise(m, 0, n, d_theta, nullptr, d_grad, (cudaStream_t)stream);
    if (m->kind == RMN_MODEL_LOGISTIC)
        return logistic_pointwise(m, 0, n, d_theta, nullptr, d_grad, nullptr, (cudaStream_t)stream);
    rmn_set_error("rmn_model_grad: the changepoint model has no gradient (changepoint.py:110-115)");
    return RMN_ERR_UNSUPPORTED;
}

extern "C" int rmn_model_metric(rmn_model_t* m, int64_t n, const double* d_theta, double* d_G,
                                void* stream) {
    RMN_REQUIRE(m && d_theta && d_G && n >= 0, "rmn_model_metric: bad argument");
    if (m->kind == RMN_MODEL_LOGISTIC)
        return logistic_pointwise(m, 0, n, d_theta, nullptr, nullptr, d_G, (cudaStream_t)stream);
    rmn_set_error("rmn_model_metric: only the logistic model defines a Fisher metric");
    return RMN_ERR_UNSUPPORTED;
}

extern "C" int rmn_model_cp_logpost(rmn_model_t* m, int which, int64_t n, const int32_t* d_k,
                                    const double* d_cpx, const double* d_cpv, const double* d_sig,
                                    double* d_out, void* stream) {
    RMN_REQUIRE(m && d_k && d_cpx && d_cpv && d_sig && d_out && n >= 0, "rmn_model_cp_logpost: bad argument");
    RMN_REQUIRE(m->kind == RMN_MODEL_CP, "rmn_model_cp_logpost: not a changepoint model");
    RMN_REQUIRE(which >= 0 && which <= 2, "rmn_model_cp_logpost: which must be 0, 1 or 2");
    return cp_pointwise(m, which, n, d_k, d_cpx, d_cpv, d_sig, d_out, (cudaStream_t)stream);
}

// -------------------------------------------------------------- proposals ----
static int lower_ok(const double* L, int d, const char* what) {
    for (int i = 0; i < d; ++i) {
        RMN_REQUIRE(isfinite(L[(size_t)i * d + i]) && L[(size_t)i * d + i] > 0,
                    "%s: Cholesky factor must have a positive diagonal", what);
    }
    return RMN_OK;
}

extern "C" int rmn_proposal_rw_create(rmn_proposal_t** out, int d, const double* h_L, int adapt,
                                      double target) {
    RMN_REQUIRE(out && h_L && d >= 1, "rmn_proposal_rw_create: bad argument");
    if (int rc = lower_ok(h_L, d, "rmn_proposal_rw_create")) return rc;
    RMN_REQUIRE(!adapt || (target > 0 && target < 1), "rmn_proposal_rw_create: target must be in (0,1)");
    rmn_proposal* p = new rmn_proposal();
    p->kind = RMN_PROP_RW; p->d = d; p->adapt = adapt; p->target = target;
    p->h_L.assign(h_L, h_L + (size_t)d * d);
    *out = p;
    return RMN_OK;
}

extern "C" int rmn_proposal_adaptcov_create(rmn_proposal_t** out, int d, const double* h_C0, const double* h_L0,
                                            double t_adapt, int marginalize, int smooth_adapt) {
    RMN_REQUIRE(out && h_C0 && h_L0 && d >= 1, "rmn_proposal_adaptcov_create: bad argument");
    RMN_REQUIRE(d <= RMN_SMALL_D_MAX, "AdaptCovRandomWalk runs on the small-d path only (d <= %d, got %d)", RMN_SMALL_D_MAX, d);
    if (int rc = lower_ok(h_L0, d, "rmn_proposal_adaptcov_create")) return rc;
    RMN_REQUIRE(t_adapt >= 0 && isfinite(t_adapt), "rmn_proposal_adaptcov_create: t_adapt must be >= 0");
    RMN_REQUIRE(smooth_adapt || t_adapt <= 4.0,
                "AdaptCovRandomWalk: strict Haario mode with t_adapt > 4 is not reproduced (the reference rescales its "
                "current C in place there, adaptive.py:89-101); use smooth_adapt or t_adapt <= 4");
    rmn_proposal* p = new rmn_proposal();
    p->kind = RMN_PROP_RW; p->d = d; p->adapt = 0; p->target = 0.25;
    p->h_L.assign(h_L0, h_L0 + (size_t)d * d);
    p->h_C0.assign(h_C0, h_C0 + (size_t)d * d);
    p->acov = 1; p->ac_marginalize = marginalize ? 1 : 0; p->ac_smooth = smooth_adapt ? 1 : 0; p->ac_t_adapt = t_adapt;
    *out = p;
    return RMN_OK;
}

extern "C" int rmn_proposal_hmc_set_cov_adapt(rmn_proposal_t* p, const double* h_M0, const double* h_L0, double t_adapt,
                                              int marginalize, int smooth_adapt) {
    RMN_REQUIRE(p && h_M0 && h_L0, "rmn_proposal_hmc_set_cov_adapt: bad argument");
    RMN_REQUIRE(p->kind == RMN_PROP_HMC && !p->has_mass, "rmn_proposal_hmc_set_cov_adapt: an HMC proposal created without a mass matrix");
    RMN_REQUIRE(p->d <= RMN_SMALL_D_MAX, "AdaptCovHMC runs on the small-d path only (d <= %d, got %d)", RMN_SMALL_D_MAX, p->d);
    if (int rc = lower_ok(h_L0, p->d, "rmn_proposal_hmc_set_cov_adapt")) return rc;
    RMN_REQUIRE(t_adapt >= 0 && isfinite(t_adapt), "rmn_proposal_hmc_set_cov_adapt: t_adapt must be >= 0");
    RMN_REQUIRE(smooth_adapt || t_adapt <= 4.0,
                "AdaptCovHMC: strict Haario mode with t_adapt > 4 is not reproduced (adaptive.py:89-101); use smooth_adapt "
                "or t_adapt <= 4");
    const size_t n = (size_t)p->d * p->d;
    p->h_L.assign(h_L0, h_L0 + n);
    p->h_C0.assign(h_M0, h_M0 + n);
    p->acov = 1; p->ac_marginalize = marginalize ? 1 : 0; p->ac_smooth = smooth_adapt ? 1 : 0; p->ac_t_adapt = t_adapt;
    return RMN_OK;
}

extern "C" int rmn_proposal_set_scale_adapt(rmn_proposal_t* p, int adapt, double target) {
    RMN_REQUIRE(p, "rmn_proposal_set_scale_adapt: null proposal");
    RMN_REQUIRE(p->kind == RMN_PROP_RW || p->kind == RMN_PROP_HMC || p->kind == RMN_PROP_PCN,
                "rmn_proposal_set_scale_adapt: random-walk, pCN and HMC proposals only");
    RMN_REQUIRE(!adapt || (target > 0 && target < 1), "rmn_proposal_set_scale_adapt: target must be in (0,1)");
    RMN_REQUIRE(!(adapt && p->kind == RMN_PROP_PCN && p->d > RMN_SMALL_D_MAX),
                "AdaptScalepCN runs on the small-d path only (d <= %d)", RMN_SMALL_D_MAX);
    p->adapt = adapt ? 1 : 0; p->target = target;
    return RMN_OK;
}

extern "C" int rmn_proposal_hmc_create(rmn_proposal_t** out, int d, double eps, int nsteps,
                                       const double* h_chM, const double* h_Minv,
                                       const double* h_chMinv, int adapt, double target) {
    RMN_REQUIRE(out && d >= 1, "rmn_proposal_hmc_create: bad argument");
    RMN_REQUIRE(eps > 0 && isfinite(eps), "rmn_proposal_hmc_create: eps must be positive");
    RMN_REQUIRE(nsteps >= 1, "rmn_proposal_hmc_create: Nsteps must be >= 1");
    const bool any = h_chM || h_Minv || h_chMinv, all = h_chM && h_Minv && h_chMinv;
    RMN_REQUIRE(any == all, "rmn_proposal_hmc_create: pass all of chM, Minv, chMinv or none");
    RMN_REQUIRE(!adapt || (target > 0 && target < 1), "rmn_proposal_hmc_create: target must be in (0,1)");
    rmn_proposal* p = new rmn_proposal();
    p->kind = RMN_PROP_HMC; p->d = d; p->eps = eps; p->nsteps = nsteps;
    p->adapt = adapt; p->target = target; p->has_mass = all;
    if (all) {
        p->h_chM.assign(h_chM, h_chM + (size_t)d * d);
        p->h_Minv.assign(h_Minv, h_Minv + (size_t)d * d);
        p->h_chMinv.assign(h_chMinv, h_chMinv + (size_t)d * d);
    }
    *out = p;
    return RMN_OK;
}

extern "C" int rmn_proposal_pcn_create(rmn_proposal_t** out, int d, const double* h_L,
                                       const double* h_Linv, double rho) {
    RMN_REQUIRE(out && h_L && h_Linv && d >= 1, "rmn_proposal_pcn_create: bad argument");
    RMN_REQUIRE(rho > -1 && rho < 1, "rmn_proposal_pcn_create: need |rho| < 1");
    if (int rc = lower_ok(h_L, d, "rmn_proposal_pcn_create")) return rc;
    rmn_proposal* p = new rmn_proposal();
    p->kind = RMN_PROP_PCN; p->d = d; p->rho = rho;
    p->h_L.assign(h_L, h_L + (size_t)d * d);
    p->h_Linv.assign(h_Linv, h_Linv + (size_t)d * d);
    *out = p;
    return RMN_OK;
}

extern "C" int rmn_proposal_mmala_create(rmn_proposal_t** out, int d, double eps) {
    RMN_REQUIRE(out && d >= 1, "rmn_proposal_mmala_create: bad argument");
    RMN_REQUIRE(eps > 0 && isfinite(eps), "rmn_proposal_mmala_create: eps must be positive");
    rmn_proposal* p = new rmn_proposal();
    p->kind = RMN_PROP_MMALA; p->d = d; p->eps = eps;
    *out = p;
    return RMN_OK;
}

extern "C" int rmn_proposal_changepoint_create(rmn_proposal_t** out, double hscale,
                                               const double* h_p_cum) {
    RMN_REQUIRE(out, "rmn_proposal_changepoint_create: bad argument");
    RMN_REQUIRE(hscale > 0 && isfinite(hscale), "rmn_proposal_changepoint_create: hscale must be positive");
    rmn_proposal* p = new rmn_proposal();
    p->kind = RMN_PROP_CP; p->hscale = hscale;
    if (h_p_cum) for (int i = 0; i < 3; ++i) p->p_cum[i] = h_p_cum[i];
    *out = p;
    return RMN_OK;
}

extern "C" int rmn_proposal_destroy(rmn_proposal_t* p) {
    if (!p) return RMN_OK;
    if (p->d_L) cudaFree(p->d_L);
    delete p;
    return RMN_OK;
}

// --------------------------------------------------------------- samplers ----
static SamplerImpl* make_impl(rmn_sampler* s, int* rc) {
    const rmn_model* m = s->model;
    const rmn_proposal* p = s->prop;
    *rc = RMN_ERR_UNSUPPORTED;
    if (m->kind == RMN_MODEL_CP) {
        if (p->kind != RMN_PROP_CP) {
            rmn_set_error("the changepoint model needs the changepoint mixture proposal");
            return nullptr;
        }
        return make_changepoint_sampler(s);
    }
    if (p->kind == RMN_PROP_CP) {
        rmn_set_error("the changepoint mixture proposal needs the changepoint model");
        return nullptr;
    }
    if (p->d != m->d) {
        rmn_set_error("theta and proposal have incompatible shapes (model d=%d, proposal d=%d)", m->d, p->d);
        *rc = RMN_ERR_PARAM;
        return nullptr;
    }
    if (p->pool_cov && !(m->kind == RMN_MODEL_GAUSS && m->d > RMN_SMALL_D_MAX && s->precision == RMN_PREC_F64)) {
        rmn_set_error("pooled covariance adaptation: dense Gaussian model (d > %d) in f64 precision", RMN_SMALL_D_MAX);
        return nullptr;
    }
    if (p->acov && !(m->kind == RMN_MODEL_GAUSS && m->d <= RMN_SMALL_D_MAX && s->precision == RMN_PREC_F64)) {
        rmn_set_error("covariance-adapting proposals (AdaptCov*) run on the small-d Gaussian path only (d <= %d, fp64)",
                      RMN_SMALL_D_MAX);
        return nullptr;
    }
    if (s->precision == RMN_PREC_TF32X3)
        return (m->kind == RMN_MODEL_LOGISTIC) ? make_logistic_sampler(s) : make_dense_tf32_sampler(s);
    if (s->precision == RMN_PREC_TF32_METRIC) {
        if (m->kind != RMN_MODEL_LOGISTIC || p->kind != RMN_PROP_MMALA) {
            rmn_set_error("precision tf32-metric needs the logistic model with the simplified mMALA proposal");
            return nullptr;
        }
        return make_logistic_sampler(s);
    }
    if (s->precision != RMN_PREC_F64) {
        rmn_set_error("unknown precision mode %d", s->precision);
        *rc = RMN_ERR_PARAM;
        return nullptr;
    }
    if (m->kind == RMN_MODEL_GAUSS) {
        if (p->kind == RMN_PROP_MMALA) {
            rmn_set_error("mMALA needs a model with a Fisher metric (logistic)");
            return nullptr;
        }
        if (m->d <= RMN_SMALL_D_MAX) return make_small_gauss_sampler(s);
        return make_dense_gauss_sampler(s);
    }
    if (m->kind == RMN_MODEL_LOGISTIC) return make_logistic_sampler(s);
    rmn_set_error("no device kernel for this model");
    return nullptr;
}

extern "C" size_t rmn_sampler_workspace_bytes(const rmn_model_t* m, const rmn_proposal_t* p, int64_t K) {
    return rmn_sampler_workspace_bytes_ex(m, p, K, RMN_PREC_F64);
}

extern "C" size_t rmn_sampler_workspace_bytes_ex(const rmn_model_t* m, const rmn_proposal_t* p, int64_t K,
                                                 int precision) {
    if (!m || !p || K < 1) return 0;
    rmn_sampler tmp;
    tmp.model = const_cast<rmn_model*>(m);
    tmp.prop = const_cast<rmn_proposal*>(p);
    tmp.K = K;
    tmp.precision = precision;
    int rc;
    SamplerImpl* impl = make_impl(&tmp, &rc);
    if (!impl) return 0;
    const size_t n = impl->workspace_bytes();
    delete impl;
    return n;
}

extern "C" int rmn_sampler_create(rmn_sampler_t** out, rmn_model_t* m, rmn_proposal_t* p, int64_t K,
                                  int64_t chain_offset, uint64_t seed, void* d_workspace,
                                  size_t workspace_bytes) {
    return rmn_sampler_create_ex(out, m, p, K, chain_offset, seed, d_workspace, workspace_bytes, RMN_PREC_F64);
}

extern "C" int rmn_sampler_create_ex(rmn_sampler_t** out, rmn_model_t* m, rmn_proposal_t* p, int64_t K,
                                     int64_t chain_offset, uint64_t seed, void* d_workspace,
                                     size_t workspace_bytes, int precision) {
    RMN_REQUIRE(out && m && p && d_workspace, "rmn_sampler_create: null argument");
    RMN_REQUIRE(K >= 1, "rmn_sampler_create: need K >= 1 chains");
    RMN_REQUIRE(chain_offset >= 0, "rmn_sampler_create: chain_offset must be >= 0");
    rmn_sampler* s = new rmn_sampler();
    s->model = m; s->prop = p; s->K = K; s->chain_offset = chain_offset; s->seed = seed;
    s->precision = precision;
    int rc;
    s->impl = make_impl(s, &rc);
    if (!s->impl) { delete s; return rc; }
    if (workspace_bytes < s->impl->workspace_bytes()) {
        rmn_set_error("rmn_sampler_create: workspace too small (%zu < %zu bytes)", workspace_bytes,
                      s->impl->workspace_bytes());
        delete s->impl; delete s;
        return RMN_ERR_PARAM;
    }
    rc = s->impl->bind(d_workspace);
    if (rc != RMN_OK) { delete s->impl; delete s; return rc; }
    *out = s;
    return RMN_OK;
}

extern "C" int rmn_sampler_destroy(rmn_sampler_t* s) {
    if (!s) return RMN_OK;
    delete s->impl;
    delete s;
    return RMN_OK;
}

#define RMN_S(s) RMN_REQUIRE((s) && (s)->impl, "null sampler handle")

extern "C" int rmn_sampler_set_state(rmn_sampler_t* s, const double* d_theta, void* stream) {
    NvtxRange nvtx_("rmn_sampler_set_state");
    RMN_S(s); RMN_REQUIRE(d_theta, "rmn_sampler_set_state: null theta");
    return s->impl->set_state(d_theta, (cudaStream_t)stream);
}
extern "C" int rmn_sampler_get_state(rmn_sampler_t* s, double* d_theta, double* d_logpost, void* stream) {
    NvtxRange nvtx_("rmn_sampler_get_state");
    RMN_S(s);
    return s->impl->get_state(d_theta, d_logpost, (cudaStream_t)stream);
}
extern "C" int rmn_sampler_cp_set_state(rmn_sampler_t* s, const int32_t* d_k, const double* d_cpx,
                                        const double* d_cpv, const double* d_sig, void* stream) {
    NvtxRange nvtx_("rmn_sampler_cp_set_state");
    RMN_S(s); RMN_REQUIRE(d_k && d_cpx && d_cpv && d_sig, "rmn_sampler_cp_set_state: null argument");
    return s->impl->cp_set_state(d_k, d_cpx, d_cpv, d_sig, (cudaStream_t)stream);
}
extern "C" int rmn_sampler_cp_get_state(rmn_sampler_t* s, int32_t* d_k, double* d_cpx, double* d_cpv,
                                        double* d_sig, double* d_logpost, void* stream) {
    NvtxRange nvtx_("rmn_sampler_cp_get_state");
    RMN_S(s);
    return s->impl->cp_get_state(d_k, d_cpx, d_cpv, d_sig, d_logpost, (cudaStream_t)stream);
}
extern "C" int rmn_sampler_run(rmn_sampler_t* s, int64_t T, const rmn_inject_t* inj,
                               const rmn_trace_t* trace, void* stream) {
    NvtxRange nvtx_("rmn_sampler_run");
    RMN_S(s); RMN_REQUIRE(T >= 0, "rmn_sampler_run: T must be >= 0");
    if (trace) RMN_REQUIRE(trace->thin >= 1 && trace->first >= 0, "rmn_sampler_run: need thin >= 1, first >= 0");
    if (T == 0) return RMN_OK;
    return s->impl->run(T, inj, trace, (cudaStream_t)stream);
}
extern "C" int rmn_sampler_get_adapt(rmn_sampler_t* s, double* d_scale, int64_t* d_nsamples,
                                     int64_t* d_naccepts, void* stream) {
    RMN_S(s);
    return s->impl->get_adapt(d_scale, d_nsamples, d_naccepts, (cudaStream_t)stream);
}
extern "C" int rmn_sampler_set_adapt(rmn_sampler_t* s, const double* d_scale, const int64_t* d_nsamples,
                                     const int64_t* d_naccepts, void* stream) {
    RMN_S(s);
    return s->impl->set_adapt(d_scale, d_nsamples, d_naccepts, (cudaStream_t)stream);
}
extern "C" int64_t rmn_sampler_get_step(const rmn_sampler_t* s) { return (s && s->impl) ? s->impl->step0 : -1; }
extern "C" int rmn_sampler_set_step(rmn_sampler_t* s, int64_t step) {
    RMN_S(s); RMN_REQUIRE(step >= 0, "rmn_sampler_set_step: step must be >= 0");
    s->impl->step0 = step;
    return RMN_OK;
}
extern "C" int rmn_sampler_diag_dim(const rmn_sampler_t* s) { return (s && s->impl) ? s->impl->diag_dim() : 0; }
extern "C" int rmn_sampler_reset_diagnostics(rmn_sampler_t* s, void* stream) {
    RMN_S(s);
    return s->impl->reset_diag((cudaStream_t)stream);
}
extern "C" int rmn_sampler_reduce_diagnostics(rmn_sampler_t* s, double* d_block, void* stream) {
    NvtxRange nvtx_("rmn_sampler_reduce_diagnostics");
    RMN_S(s); RMN_REQUIRE(d_block, "rmn_sampler_reduce_diagnostics: null block");
    return s->impl->reduce_diag(d_block, (cudaStream_t)stream);
}
extern "C" int rmn_proposal_rw_set_pooled_cov_adapt(rmn_proposal_t* p, int64_t t_adapt, double sd, double jitter,
                                                    int64_t stop_after) {
    RMN_REQUIRE(p, "rmn_proposal_rw_set_pooled_cov_adapt: null proposal");
    RMN_REQUIRE(p->kind == RMN_PROP_RW && !p->acov, "rmn_proposal_rw_set_pooled_cov_adapt: a random-walk proposal without per-chain covariance adaptation");
    RMN_REQUIRE(p->d > RMN_SMALL_D_MAX, "pooled covariance adaptation runs on the dense path (d > %d); d <= %d has the per-chain AdaptCovRandomWalk",
                RMN_SMALL_D_MAX, RMN_SMALL_D_MAX);
    RMN_REQUIRE(t_adapt >= 1 && sd > 0 && isfinite(sd) && jitter >= 0 && isfinite(jitter) && stop_after >= 0,
                "rmn_proposal_rw_set_pooled_cov_adapt: need t_adapt >= 1, sd > 0, jitter >= 0, stop_after >= 0");
    p->pool_cov = 1; p->pool_t_adapt = t_adapt; p->pool_sd = sd; p->pool_jitter = jitter; p->pool_stop = stop_after;
    return RMN_OK;
}
extern "C" int rmn_sampler_get_pooled_cov(rmn_sampler_t* s, double* d_cov, double* d_mean, double* d_count, void* stream) {
    RMN_REQUIRE(s && s->impl && d_cov && d_mean && d_count, "rmn_sampler_get_pooled_cov: bad argument");
    return s->impl->get_pooled_cov(d_cov, d_mean, d_count, (cudaStream_t)stream);
}
extern "C" int rmn_sampler_get_adaptcov(rmn_sampler_t* s, double* d_L, void* stream) {
    RMN_REQUIRE(s && s->impl && d_L, "rmn_sampler_get_adaptcov: bad argument");
    return s->impl->get_adaptcov(d_L, (cudaStream_t)stream);
}

extern "C" int rmn_sampler_set_tempering(rmn_sampler_t* s, int nt, const double* h_betas, double pswap) {
    RMN_REQUIRE(s && s->impl, "rmn_sampler_set_tempering: null sampler");
    return s->impl->set_tempering(nt, h_betas, pswap);
}

extern "C" int rmn_sampler_set_move_schedule(rmn_sampler_t* s, int mode) {
    RMN_REQUIRE(s && s->impl, "rmn_sampler_set_move_schedule: null sampler");
    return s->impl->set_move_schedule(mode);
}

extern "C" int rmn_sampler_cp_set_summary(rmn_sampler_t* s, int G, const double* h_grid, double vlo, double vhi, int H,
                                          int64_t every) {
    RMN_REQUIRE(s && s->impl, "rmn_sampler_cp_set_summary: null sampler");
    return s->impl->cp_set_summary(G, h_grid, vlo, vhi, H, every);
}

extern "C" int rmn_sampler_cp_set_rung_summary(rmn_sampler_t* s, int rung, int G, const double* h_grid, double vlo,
                                               double vhi, int H, int64_t every) {
    RMN_REQUIRE(s && s->impl, "rmn_sampler_cp_set_rung_summary: null sampler");
    return s->impl->cp_set_rung_summary(rung, G, h_grid, vlo, vhi, H, every);
}

extern "C" int rmn_sampler_cp_get_summary(rmn_sampler_t* s, int64_t* d_khist, int64_t* d_cpxhist, int64_t* d_yhist,
                                          int64_t* h_nsamples, void* stream) {
    NvtxRange nvtx_("rmn_sampler_cp_get_summary");
    RMN_REQUIRE(s && s->impl, "rmn_sampler_cp_get_summary: null sampler");
    return s->impl->cp_get_summary(d_khist, d_cpxhist, d_yhist, h_nsamples, (cudaStream_t)stream);
}

extern "C" int rmn_sampler_cp_get_swap_stats(rmn_sampler_t* s, int64_t* d_proposed, int64_t* d_accepted, int64_t* d_up,
                                             int64_t* d_down, int64_t* d_round_trips, void* stream) {
    RMN_REQUIRE(s && s->impl, "rmn_sampler_cp_get_swap_stats: null sampler");
    return s->impl->cp_get_swap_stats(d_proposed, d_accepted, d_up, d_down, d_round_trips, (cudaStream_t)stream);
}

extern "C" int rmn_sampler_chain_moments(rmn_sampler_t* s, double* d_mean, double* d_var, void* stream) {
    RMN_REQUIRE(s && s->impl, "rmn_sampler_chain_moments: null sampler");
    const double *S1 = nullptr, *S2 = nullptr;
    int64_t n = 0;
    const int rc = s->impl->chain_sums(&S1, &S2, &n);
    if (rc != RMN_OK) return rc;
    return rmn_chain_moments(s->K, s->impl->diag_dim(), n, S1, S2, d_mean, d_var, (cudaStream_t)stream);
}

extern "C" int rmn_autocorr_tau(const double* d_x, int64_t n, int64_t nchains, int64_t nfunc, double c, double* h_tau,
                                int64_t* h_window, void* stream) {
    return rmn_autocorr_tau_impl(d_x, n, nchains, nfunc, c, h_tau, h_window, (cudaStream_t)stream);
}

extern "C" int rmn_nccl_unique_id(void* out, size_t nbytes) { return rmn_rowcomm_unique_id(out, nbytes); }

extern "C" int rmn_sampler_set_row_comm(rmn_sampler_t* s, const void* unique_id, size_t nbytes, int rank, int world) {
    RMN_REQUIRE(s && s->impl, "rmn_sampler_set_row_comm: null sampler");
    return s->impl->set_row_comm(unique_id, nbytes, rank, world);
}

extern "C" int64_t rmn_sampler_launch_count(const rmn_sampler_t* s) { return (s && s->impl) ? s->impl->launches : 0; }

extern "C" int rmn_sampler_enable_kernel_timing(rmn_sampler_t* s, int enable) {
    RMN_REQUIRE(s && s->impl, "rmn_sampler_enable_kernel_timing: null sampler");
    s->impl->ktimer.on = enable != 0;
    s->impl->ktimer.used = 0; s->impl->ktimer.untimed = 0;
    return RMN_OK;
}
extern "C" int rmn_sampler_kernel_timing(rmn_sampler_t* s, double* total_ms, int64_t* launches, int64_t* untimed,
                                         const char** kernel_name) {
    RMN_REQUIRE(s && s->impl, "rmn_sampler_kernel_timing: null sampler");
    if (untimed) *untimed = s->impl->ktimer.untimed;
    if (kernel_name) *kernel_name = s->impl->ktimer.name;
    s->impl->ktimer.collect(total_ms, launches);
    return RMN_OK;
}
