// riemann_b200 -- definitions of the changepoint kernels (changepoint.cu).
#pragma once
#include "common.cuh"

namespace cp {

constexpr int LANES = RMN_CP_LANES;
constexpr int NQ = 6;   // prediction query points tracked by the diagnostics
#ifndef RMN_CP_DIAG_EVERY
#define RMN_CP_DIAG_EVERY 16  // diagnostics functionals are accumulated every 16th MH step (tau of every tracked
                              // functional is > 100 steps on this posterior; 4 -> 16 is +13 % throughput, gpurun r2e)
#endif

struct CPParams {
    // device data (rmn_model_changepoint_create): x[XP] | {cy, cyy}[M+1] | bx[G] (double2) | bstart[G] (int32), the
    // last two only when G > 0.  XP = 2*P2 (P2 = largest power of two <= M) is even, so the 16-byte pairs are 16-byte
    // aligned.
    int M, P2, alpha_is_one, XP;
    int G;                      // buckets of the run-boundary table, 0 = none (binary search); see run_boundary
    double bscale, boff;        // bucket of c = bucket_of(c, bscale, boff, G)
    double xmin, xmax, alpha, beta, cv, logL, ycenter, Mlog2pi, sqrtM;
    double tab1[LANES + 1];     // k log(lam) - gammaln(k) - lam        changepoint.py:134
    double tab2[LANES + 1];     // gammaln(2k+1)                        changepoint.py:143
    double sx[LANES + 1];       // sqrt(0.01 (xmax-xmin)/(k+1))         test_changepoint.py:36
    double sv, ss;              // sqrt(0.01 hscale^2/M), sqrt(0.01 hscale)   :37-38
    double p1, p2, p3;          // sequential selection thresholds      :28-30
    uint32_t t1, t2, t3, tpad;  // the same thresholds on the raw 32-bit Philox words
    double xq[NQ];
};

struct CPState {
    int32_t* k;          // [K]
    double* cpx;         // [K][LANES]
    double* cpv;         // [K][LANES]
    double* sig;         // [K]
    double* lp;          // [K]
    long long* dacc;     // [K]
    long long* dovf;     // [K]
    double* S1;          // [NDIAG][K]
    double* S2;          // [NDIAG][K]
};

__device__ __forceinline__ unsigned group_ballot(bool pred) {
    const unsigned full = __ballot_sync(0xffffffffu, pred);
    return (full >> (threadIdx.x & 16)) & 0xffffu;
}

// #{i : x_i <= c}  (upper bound, np.searchsorted(x, c, 'right')) for R queries, always in [0, M].
//
// Binary search (G = 0): the x table is padded with NaN up to XP = 2*P2 entries: a NaN never compares <= c, so the
// search needs no bound check and stops at M by itself; a NaN / +inf query gives 0 / M like the unpadded search.  One
// LDS + one compare + one predicated add per level; the R searches' levels are interleaved, so their dependent LDS
// chains overlap.
//
// Bucket table (G > 0, built by rmn_model_changepoint_create): the query's bucket b = bucket_of(c) is a monotone
// function of c (NaN -> 0).  The host evaluates the same function on every x_i and stores
// s = bstart[b] = min(#{i : bucket(x_i) < b}, XP - 2) and bx[b] = {x[s], x[s + 1]}, and it builds the table only when
// no bucket holds more than BUCKET_W = 2 points (the lookup makes two compares).  For a query c in bucket b, every x_i
// of a lower bucket is < c and every x_i of a higher bucket is > c, so the answer lies in [s, s + 2] and is s plus the
// two compares x[s + m] <= c, m = 0, 1.  bstart[b] and bx[b] are two independent loads (the clamp to XP - 2 keeps
// s + 1 inside the x table, whose NaN padding compares false).  NaN and -inf queries land in bucket 0, where bstart = 0
// and every compare is false (x is finite).  The result is an integer, the same one the binary search finds.
constexpr int BUCKET_W = 2;
constexpr int BUCKET_GMAX = 1024;   // largest table: 20 KB

// the bucket of c, on the host (building the table) and on the device (looking it up) alike: trunc(fma(c, bscale,
// boff)) clamped to [0, G-1], NaN -> 0
__host__ __device__ __forceinline__ int bucket_of(double c, double bscale, double boff, int G) {
    const double t = fma(c, bscale, boff);
#ifdef __CUDA_ARCH__
    return (t > 0.0) ? (int)min(__double2uint_rz(t), (unsigned)(G - 1)) : 0;   // the conversion saturates: +inf -> UINT_MAX
#else
    return (t > 0.0) ? ((t < (double)(G - 1)) ? (int)t : G - 1) : 0;
#endif
}

// The binary search of run_boundary over any sorted table t of n entries padded with NaN up to 2 * P2 (P2 = the largest
// power of two <= n): #{i : t_i <= c} for R queries, in [0, n].  The posterior summaries search their grid with it.
template <int R>
__device__ __forceinline__ void padded_upper_bound(const double* __restrict__ t, int P2, const double (&c)[R],
                                                   int (&pos)[R]) {
    const char* base = (const char*)t;
    unsigned off[R];
#pragma unroll
    for (int r = 0; r < R; ++r) off[r] = 0;
    for (int step = P2; step > 0; step >>= 1) {
        double v[R];
#pragma unroll
        for (int r = 0; r < R; ++r) v[r] = *(const double*)(base + off[r] + (step - 1) * 8);
#pragma unroll
        for (int r = 0; r < R; ++r) if (v[r] <= c[r]) off[r] += 8u * step;
    }
#pragma unroll
    for (int r = 0; r < R; ++r) pos[r] = (int)(off[r] >> 3);
}

template <bool BUCKETS, int R>
__device__ __forceinline__ void run_boundary(const CPParams& P, const double* __restrict__ xs,
                                             const double2* __restrict__ bx, const double (&c)[R], int (&pos)[R]) {
    if (BUCKETS) {
        const int* bstart = (const int*)(bx + P.G);
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const int b = bucket_of(c[r], P.bscale, P.boff, P.G);
            const double2 w = bx[b];
            pos[r] = bstart[b] + (w.x <= c[r]) + (w.y <= c[r]);
        }
    } else {
        padded_upper_bound<R>(xs, P.P2, c, pos);
    }
}

template <bool BUCKETS>
__device__ __forceinline__ int run_boundary(const CPParams& P, const double* __restrict__ xs,
                                            const double2* __restrict__ bx, double c) {
    const double q[1] = {c};
    int pos[1];
    run_boundary<BUCKETS, 1>(P, xs, bx, q, pos);
    return pos[0];
}

// uniform on (0,1) from 32 random bits with 2 fp64 instructions: [1,2) mantissa trick + 2^-33
__device__ __forceinline__ double u01_fast(uint32_t x) {
    return __hiloint2double(0x3ff00000 | (x >> 12), x << 20) - (1.0 - 1.1641532182693481e-10);
}


}  // namespace cp
