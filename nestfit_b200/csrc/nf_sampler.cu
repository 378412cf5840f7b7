// Batched nested-sampling driver: many pixels ("runs") advance in lock-step and
// every iteration's constrained-prior proposals of all in-flight pixels are
// scored by ONE launch of the fused likelihood kernel.
//
// It replaces the reference's per-pixel, serial MultiNest callback loop
//   run_multinest -> MultiNest `run` -> mn_loglikelihood -> Runner.c_loglikelihood
//   (nestfit/core/core.pyx:622-624,727-823; nestfit/core/cmultinest.pxd:5-33)
// and produces what `mn_dump` (core.pyx:627-687) persists: ln Z, its error,
// max log-likelihood, the weighted posterior sample, best-fit and MAP vectors.
// MultiNest itself (Feroz & Hobson 2008; Feroz, Hobson & Bridges 2009) is an
// external, un-vendored Fortran library: this is an algorithmic replacement with
// the same published scheme, not a port -- ln Z / posterior parity is
// statistical ("parity unpinned", SURVEY.md 8c).
//
// Algorithm per run (all in the unit cube, FP64):
//   live set of `nlive` points; per lock-step iteration K candidates are drawn
//   uniformly from a bounding ellipsoid of the live set (enlarged to the larger
//   of 1.2 x the bounding volume and X_i / efr, MultiNest's `efr`; the unit cube
//   itself while that volume is >= 1/2), transformed to physical parameters,
//   scored, and then consumed *in order*: candidate k replaces the current worst
//   live point iff lnL_k > lnL_worst, which records the worst point as a dead
//   point with prior-mass weight X_{i-1} - X_i, X_i = exp(-i / nlive).  A
//   candidate tested against the then-current threshold is an exact rejection
//   sample of the constrained prior, so no proposal is wasted by the batching.
//   Termination (MultiNest `tol`): ln(Z + L_max X_i) - ln Z < tol; the remaining
//   live points are then added with weight X_i / nlive.

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <algorithm>
#include <cstring>
#include <new>
#include <vector>

#include "nf_internal.cuh"

#define NS_MAX_DIM 32
#define NS_FULL 0xffffffffu

struct nf_sampler {
    const nf_pixels *px;
    const nf_priors *pr;
    int device, ncomp, flags, ndim;
    nf_ns_config cfg;
    int64_t n_run;
    int K;                             // proposals per run per lock-step while the block is full (cfg.n_prop)
    int Kmax;                          // ... and the most a run may get once few runs remain (cfg.n_prop_max)
    int64_t cand_cap;                  // capacity of the candidate buffers (vectors)
    int32_t *krun, *cand_off;          // [n_run] proposals of run r this cohort; [n_run] first candidate of active slot a
    // device state
    int32_t *pix_ids, *nlive;          // [n_run]
    double *live_u, *live_th, *live_l; // [n_run][nlive_max][ndim], .., [n_run][nlive_max]
    double *cand_u, *cand_th, *cand_l; // [n_run][K][ndim], .., [n_run][K]
    int32_t *cand_pix;                 // [n_run][K]
    double *bound;                     // [n_run][ndim + ndim*ndim + 2]: mean, scaled L, {use_cube, -}
    // dead points (then the final live points) of all runs in one pool: run r owns rows
    // [dead_off[r], dead_off[r] + dead_cap[r]), dead_cap[r] = min(max_samples, (max_samples / nlive_max) nlive[r])
    float *dead_th;                    // [dead_rows][ndim]
    double *dead_l, *dead_lw;          // [dead_rows]
    int64_t *dead_off;                 // [n_run + 1] (device)
    int32_t *dead_cap;                 // [n_run] (device)
    int64_t dead_rows;
    std::vector<int64_t> *h_dead_off;  // host copy
    // products (nf_ns_products_*): rows kept per run and their offsets in the packed posterior pool
    int32_t *keep_n;                   // [n_run] (device)
    int64_t *post_off;                 // [n_run + 1] (device)
    std::vector<int64_t> *h_post_off;
    bool post_ready;                   // nf_ns_products_rows has set post_off
    double *lnZ, *H, *lmax;            // [n_run]
    int32_t *n_dead, *it, *done, *n_it_lock;
    int64_t *n_eval;
    double *bestfit, *mapfit, *lnZ_err; // [n_run][ndim] x2, [n_run]
    int32_t *act;                      // [n_run] active run list
    int32_t *n_act_dev;
    // constrained random walk (used when ellipsoidal rejection sampling stalls)
    int32_t *mode, *coh_step, *coh_acc, *eff_acc, *eff_prop, *chain_moved;
    double *lstar, *scale, *chain_u, *chain_th, *chain_l;
    int walks;
    int update_every;                  // lock-steps between rebuilds of a run's ellipsoid decomposition (mmodal)
    int da;                            // dimensions the likelihood depends on (the others are constant / duplicated)
    signed char adim[NS_MAX_DIM];      // their indices in the unit-cube vector
    int32_t *n_act_host;               // pinned: {n_act, n_cand}
    cudaStream_t stream;
    int lock_iters;
    int64_t launches;
};

namespace {

// ---- Philox4x32-10 counter-based RNG ---------------------------------------
__device__ __forceinline__ void philox_round(uint32_t &c0, uint32_t &c1, uint32_t &c2, uint32_t &c3, uint32_t k0,
                                             uint32_t k1)
{
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
}

struct Philox {
    uint32_t c[4], k[2], out[4];
    int have;
    __device__ Philox(uint64_t seed, uint32_t a, uint32_t b, uint32_t cidx)
    {
        k[0] = (uint32_t)seed; k[1] = (uint32_t)(seed >> 32);
        c[0] = 0; c[1] = a; c[2] = b; c[3] = cidx;
        have = 0;
    }
    __device__ void refill()
    {
        uint32_t x0 = c[0], x1 = c[1], x2 = c[2], x3 = c[3], k0 = k[0], k1 = k[1];
#pragma unroll
        for (int r = 0; r < 10; ++r) {
            philox_round(x0, x1, x2, x3, k0, k1);
            k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
        }
        out[0] = x0; out[1] = x1; out[2] = x2; out[3] = x3;
        c[0]++;
        have = 4;
    }
    __device__ uint32_t next()
    {
        if (!have) refill();
        return out[--have];
    }
    // uniform in (0,1), 53 bits
    __device__ double uniform()
    {
        const uint64_t a = next(), b = next();
        const uint64_t v = ((a << 32) | b) >> 11;
        return ((double)v + 0.5) * (1.0 / 9007199254740992.0);
    }
    // two standard normals (Box-Muller in FP32: proposal directions do not need more)
    __device__ void normal2(double &z0, double &z1)
    {
        const float u1 = ((float)(next() >> 8) + 0.5f) * (1.0f / 16777216.0f);
        const float u2 = ((float)(next() >> 8) + 0.5f) * (1.0f / 16777216.0f);
        const float r = sqrtf(-2.0f * __logf(u1));
        float s, c2;
        sincospif(2.0f * u2, &s, &c2);
        z0 = (double)(r * c2); z1 = (double)(r * s);
    }
};

__device__ __forceinline__ double logaddexp(double a, double b)
{
    if (a == -INFINITY) return b;
    if (b == -INFINITY) return a;
    const double m = fmax(a, b);
    return m + log1p(exp(-fabs(a - b)));
}

// ---- initial live points: uniform in the unit cube -------------------------
__global__ void ns_init_live_kernel(double *live_u, double *live_th, int64_t n_run, int nlive_max, int ndim,
                                    uint64_t seed)
{
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;   // (run, point)
    if (idx >= n_run * nlive_max) return;
    const int64_t r = idx / nlive_max;
    const int p = (int)(idx - r * nlive_max);
    Philox rng(seed, (uint32_t)r, 0xFFFFFFFFu, (uint32_t)p);
    double *u = live_u + idx * ndim, *th = live_th + idx * ndim;
    for (int k = 0; k < ndim; ++k) { const double v = rng.uniform(); u[k] = v; th[k] = v; }
}

// pixel of every initial live point (run r, point p)
__global__ void ns_live_map_kernel(const int32_t *pix_ids, int32_t *map, int64_t n_run, int nlive_max)
{
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx < n_run * nlive_max) map[idx] = pix_ids[idx / nlive_max];
}

__global__ void ns_init_state_kernel(double *lnZ, double *H, double *lmax, int32_t *n_dead, int32_t *it,
                                     int32_t *done, int64_t *n_eval, int32_t *act, const int32_t *nlive,
                                     double *live_l, int64_t n_run, int nlive_max, int32_t *mode,
                                     int32_t *coh_step, int32_t *coh_acc, int32_t *eff_acc, int32_t *eff_prop,
                                     double *scale, int start_mode)
{
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_run) return;
    mode[r] = start_mode; coh_step[r] = 0; coh_acc[r] = 0; eff_acc[r] = 0; eff_prop[r] = 0; scale[r] = 0.3;
    lnZ[r] = -INFINITY; H[r] = 0.0; n_dead[r] = 0; it[r] = 0; done[r] = 0; n_eval[r] = nlive[r];
    act[r] = (int32_t)r;
    double m = -INFINITY;
    for (int p = 0; p < nlive[r]; ++p) {
        double l = live_l[r * nlive_max + p];
        // a draw the priors map to NaN scores NaN: treat it as MultiNest's logZero (it dies first, weight 0)
        if (!(l == l)) { l = -INFINITY; live_l[r * nlive_max + p] = l; }
        if (l > m) m = l;
    }
    lmax[r] = m;
}

// The unit-cube dimensions a run's likelihood depends on.  A ConstantPrior row and the second row of a
// DuplicatePrior (core.pyx:200-238) are overwritten by the prior transform whatever the cube value is, so the
// constrained prior is uniform and independent in those dimensions: they are drawn uniformly on their own
// and kept out of the bounding ellipsoid and of the random-walk metric (an ellipsoid has to span the full
// [0, 1] of such a dimension, which costs volume -- rejection efficiency -- for nothing).
struct NsDims {
    int da, nfree;
    signed char adim[NS_MAX_DIM];      // dimensions inside the ellipsoid / walk metric
    signed char fdim[NS_MAX_DIM];      // the others: uniform on their own
};

// ---- bound of the live set: up to NS_MAX_ELL ellipsoids (one CTA per active run) ------------
// Layout of a run's bound: {n_ell, use_cube, -, -} then NS_MAX_ELL records {mean[d], L[d][d], ln V} in the
// active dimensions (d = dims.da; the stride is computed with the full ndim).
#define NS_MAX_ELL 8
#define NS_KMEANS_ITERS 8
#define NS_BOUND_HDR 4
__host__ __device__ inline int64_t ns_ell_stride(int ndim) { return (int64_t)ndim + (int64_t)ndim * ndim + 1; }
__host__ __device__ inline int64_t ns_bound_stride(int ndim) { return NS_BOUND_HDR + NS_MAX_ELL * ns_ell_stride(ndim); }

// ---- ONE bounding ellipsoid of the live set (one CTA per active run): the light kernel behind mmodal = False,
// rebuilt every lock-step; same record layout as the decomposition kernel below, n_ell = 1 ----
__global__ void __launch_bounds__(128)
ns_bounds_single_kernel(const int32_t *act, const int32_t *n_act_dev, const int32_t *nlive_arr, const int32_t *it_arr,
                 const double *live_u, double *bound, int nlive_max, int ndim, double efr, const int32_t *mode,
                 const int32_t *coh_step, const NsDims dims)
{
    __shared__ double s_mean[NS_MAX_DIM];
    __shared__ double s_c[NS_MAX_DIM][NS_MAX_DIM + 1];
    __shared__ double s_red[128];
    if ((int)blockIdx.x >= *n_act_dev) return;
    const int r = act[blockIdx.x];
    // a random-walk cohort keeps the metric it started with: rebuild only at cohort start
    if (mode[r] == 1 && coh_step[r] != 0) return;
    const int nl = nlive_arr[r];
    const int tid = threadIdx.x, d = dims.da, ds = ndim;      // d: active dimensions; ds: row stride of the live set
    const double *U = live_u + (int64_t)r * nlive_max * ds;
    if (tid < d) {
        double s = 0.0;
        const int ja = dims.adim[tid];
        for (int p = 0; p < nl; ++p) s += U[p * ds + ja];
        s_mean[tid] = s / (double)nl;
    }
    __syncthreads();
    const int npair = d * (d + 1) / 2;
    for (int e = tid; e < npair; e += blockDim.x) {
        // unpack (a >= b) from the triangular index
        int a = (int)((sqrt(8.0 * (double)e + 1.0) - 1.0) * 0.5);
        while ((a + 1) * (a + 2) / 2 <= e) ++a;
        while (a * (a + 1) / 2 > e) --a;
        const int b = e - a * (a + 1) / 2;
        double s = 0.0;
        const double ma = s_mean[a], mb = s_mean[b];
        const int ja = dims.adim[a], jb = dims.adim[b];
        for (int p = 0; p < nl; ++p) s += (U[p * ds + ja] - ma) * (U[p * ds + jb] - mb);
        s /= (double)(nl > 1 ? nl - 1 : 1);
        if (a == b) s += 1e-12;
        s_c[a][b] = s;
        s_c[b][a] = s;
    }
    __syncthreads();
    // Cholesky (lower) in place by warp 0: lane <-> row
    if (tid < 32) {
        for (int j = 0; j < d; ++j) {
            double djj = s_c[j][j];
            for (int k = 0; k < j; ++k) djj -= s_c[j][k] * s_c[j][k];
            djj = sqrt(fmax(djj, 1e-300));
            __syncwarp();
            if (tid == 0) s_c[j][j] = djj;
            if (tid > j && tid < d) {
                double v = s_c[tid][j];
                for (int k = 0; k < j; ++k) v -= s_c[tid][k] * s_c[j][k];
                s_c[tid][j] = v / djj;
            }
            __syncwarp();
        }
    }
    __syncthreads();
    // largest Mahalanobis radius over the live points
    double fmx = 0.0;
    for (int p = tid; p < nl; p += blockDim.x) {
        double y[NS_MAX_DIM];
        double r2 = 0.0;
        for (int a = 0; a < d; ++a) {
            double v = U[p * ds + dims.adim[a]] - s_mean[a];
            for (int k = 0; k < a; ++k) v -= s_c[a][k] * y[k];
            v /= s_c[a][a];
            y[a] = v;
            r2 += v * v;
        }
        fmx = fmax(fmx, r2);
    }
    s_red[tid] = fmx;
    __syncthreads();
    for (int o = 64; o > 0; o >>= 1) {
        if (tid < o) s_red[tid] = fmax(s_red[tid], s_red[tid + o]);
        __syncthreads();
    }
    const double f = s_red[0];
    // volumes: ln V = ln V_d + (d/2) ln f + sum ln L_jj
    double lndet = 0.0;
    for (int j = 0; j < d; ++j) lndet += log(s_c[j][j]);
    const double lnVd = 0.5 * d * log(M_PI) - lgamma(0.5 * d + 1.0);
    const double lnV_bound = lnVd + 0.5 * d * log(f) + lndet + log(1.2);
    const double lnX = -(double)it_arr[r] / (double)nl;
    const double lnV_target = lnX - log(efr);
    const double lnV = fmax(lnV_bound, lnV_target);
    // linear scale applied to L so that the ellipsoid has volume V
    const double scale = exp((lnV - lnVd - lndet) / (double)d);
    double *B = bound + (int64_t)r * ns_bound_stride(ds);      // {n_ell, use_cube, -, -} {mean[d], L[d][d], ln V}
    double *E = B + NS_BOUND_HDR;
    if (tid < d) E[tid] = s_mean[tid];
    for (int e = tid; e < d * d; e += blockDim.x) {
        const int a = e / d, b = e - a * d;
        E[d + e] = b <= a ? scale * s_c[a][b] : 0.0;
    }
    if (tid == 0) {
        const bool degenerate = !(f > 0.0) || !isfinite(scale);
        B[0] = 1.0;
        B[1] = (lnV > log(0.5) || degenerate) ? 1.0 : 0.0;   // sample the unit cube itself
        E[d + d * d] = lnV;
    }
}


struct BoundsSmem {
    double mean[NS_MAX_DIM];
    double c[NS_MAX_DIM][NS_MAX_DIM + 1];
    double var[NS_MAX_DIM];            // diagonal of the covariance before the factorisation
    double red[128];
    int redi[128];
    double c0[NS_MAX_DIM], c1[NS_MAX_DIM];
    int cnt[2];
    int todo[2 * NS_MAX_ELL];          // cluster labels waiting to be examined
    int flag;
};

// Covariance ellipsoid through the farthest of the live points carrying label `want` (any label if lab == nullptr):
// mean and lower Cholesky factor in S.mean / S.c, the index of the point of largest Mahalanobis radius, the number
// of points; ln V = max(1.2 x the bounding volume, lnV_min) and the linear scale that gives the factor that volume.
__device__ void ns_ell_fit(BoundsSmem &S, const double *U, int ds, const NsDims &dims, const short *lab, int want,
                           int nl, double lnV_base, double &lnV, double &scale, int &far, int &count)
{
    const int tid = threadIdx.x, d = dims.da;
    __syncthreads();
    if (tid < d) {
        double sum = 0.0;
        int n = 0;
        const int ja = dims.adim[tid];
        for (int p = 0; p < nl; ++p)
            if (!lab || lab[p] == want) { sum += U[p * ds + ja]; ++n; }
        S.mean[tid] = sum / (double)(n > 0 ? n : 1);
        if (tid == 0) S.cnt[0] = n;
    }
    __syncthreads();
    const int n = S.cnt[0];
    const int npair = d * (d + 1) / 2;
    for (int e = tid; e < npair; e += blockDim.x) {
        int a = (int)((sqrt(8.0 * (double)e + 1.0) - 1.0) * 0.5);      // (a >= b) from the triangular index
        while ((a + 1) * (a + 2) / 2 <= e) ++a;
        while (a * (a + 1) / 2 > e) --a;
        const int b = e - a * (a + 1) / 2;
        double sum = 0.0;
        const double ma = S.mean[a], mb = S.mean[b];
        const int ja = dims.adim[a], jb = dims.adim[b];
        for (int p = 0; p < nl; ++p)
            if (!lab || lab[p] == want) sum += (U[p * ds + ja] - ma) * (U[p * ds + jb] - mb);
        sum /= (double)(n > 1 ? n - 1 : 1);
        if (a == b) { S.var[a] = sum; sum += 1e-12; }
        S.c[a][b] = sum;
        S.c[b][a] = sum;
    }
    __syncthreads();
    if (tid < 32) {          // Cholesky (lower) in place by warp 0: lane <-> row
        for (int j = 0; j < d; ++j) {
            double djj = S.c[j][j];
            for (int k = 0; k < j; ++k) djj -= S.c[j][k] * S.c[j][k];
            djj = sqrt(fmax(djj, 1e-300));
            __syncwarp();
            if (tid == 0) S.c[j][j] = djj;
            if (tid > j && tid < d) {
                double v = S.c[tid][j];
                for (int k = 0; k < j; ++k) v -= S.c[tid][k] * S.c[j][k];
                S.c[tid][j] = v / djj;
            }
            __syncwarp();
        }
    }
    __syncthreads();
    double fmx = -1.0;       // largest Mahalanobis radius over the cluster and where it is
    int imx = 0;
    for (int p = tid; p < nl; p += blockDim.x) {
        if (lab && lab[p] != want) continue;
        double y[NS_MAX_DIM];
        double r2 = 0.0;
        for (int a = 0; a < d; ++a) {
            double v = U[p * ds + dims.adim[a]] - S.mean[a];
            for (int k = 0; k < a; ++k) v -= S.c[a][k] * y[k];
            v /= S.c[a][a];
            y[a] = v;
            r2 += v * v;
        }
        if (r2 > fmx) { fmx = r2; imx = p; }
    }
    S.red[tid] = fmx;
    S.redi[tid] = imx;
    __syncthreads();
    for (int o = 64; o > 0; o >>= 1) {
        if (tid < o && (S.red[tid + o] > S.red[tid] || (S.red[tid + o] == S.red[tid] && S.redi[tid + o] < S.redi[tid]))) {
            S.red[tid] = S.red[tid + o];
            S.redi[tid] = S.redi[tid + o];
        }
        __syncthreads();
    }
    const double f = fmax(S.red[0], 1e-300);
    far = S.redi[0];
    count = n;
    double lndet = 0.0;
    for (int j = 0; j < d; ++j) lndet += log(S.c[j][j]);
    const double lnVd = 0.5 * d * log(M_PI) - lgamma(0.5 * d + 1.0);
    lnV = fmax(lnVd + 0.5 * d * log(f) + lndet + log(1.2), lnV_base + log((double)(n > 0 ? n : 1)));
    scale = exp((lnV - lnVd - lndet) / (double)d);
    __syncthreads();
}

// MultiNest-style decomposition (Feroz, Hobson & Bridges 2009, sect. 5.1-5.2, as configured by the reference with
// mmodal = True, efr = 0.3: core.pyx:727-732): breadth-first 2-means splits of the live set -- seeded at the point of
// largest Mahalanobis radius and the point farthest from it, distances scaled by the parent's per-dimension spread --
// kept when the children's volumes add up to less than half the parent's, or when the parent exceeds twice its share
// X n_c / (efr nlive) of the prior volume and the children are smaller at all.  Every ellipsoid is enlarged to
// 1.2 x its bounding volume and to at least its share of X / efr.  (oracle/ns_port.py:multi_ellipsoid_bound is the
// numpy restatement.)  A run in random-walk mode keeps ONE ellipsoid, the metric of its walk, rebuilt at cohort start.
__global__ void __launch_bounds__(128)
ns_bounds_kernel(const int32_t *act, const int32_t *n_act_dev, const int32_t *nlive_arr, const int32_t *it_arr,
                 const double *live_u, double *bound, int nlive_max, int ndim, double efr, const int32_t *mode,
                 const int32_t *coh_step, const NsDims dims, int lock, int update_every, int multi)
{
    __shared__ BoundsSmem S;
    extern __shared__ short s_lab[];                 // [nlive_max] cluster label of every live point
    if ((int)blockIdx.x >= *n_act_dev) return;
    const int r = act[blockIdx.x];
    const bool walk = mode[r] == 1;
    if (walk && coh_step[r] != 0) return;            // a cohort keeps the metric it started with
    double *B = bound + (int64_t)r * ns_bound_stride(ndim);
    const int nl = nlive_arr[r];
    const int tid = threadIdx.x, d = dims.da, ds = ndim;
    const double lnX = -(double)it_arr[r] / (double)nl;
    const bool use_cube = !walk && lnX - log(efr) > log(0.5);
    if (use_cube) {
        if (tid == 0) { B[0] = 0.0; B[1] = 1.0; B[2] = -1.0e30; }
        return;
    }
    // the decomposition is rebuilt every `update_every` lock-steps; in between the ellipsoids stay valid supersets
    // (the constrained region only shrinks)
    const int it_now = it_arr[r];
    if (!walk && B[1] < 0.5 && B[0] >= 1.0 && (lock % update_every) != 0) return;
    const double *U = live_u + (int64_t)r * nlive_max * ds;
    const double lnpv = walk ? -INFINITY : lnX - log(efr) - log((double)nl);
    const int64_t es = ns_ell_stride(ndim);
    const int minpts = d + 1;
    for (int p = tid; p < nl; p += blockDim.x) s_lab[p] = 0;
    int n_todo = 1, n_done = 0, next_label = 1;
    if (tid == 0) S.todo[0] = 0;
    __syncthreads();
    while (n_todo > 0) {
        const int label = S.todo[0];
        __syncthreads();
        if (tid == 0) for (int k = 1; k < n_todo; ++k) S.todo[k - 1] = S.todo[k];
        --n_todo;
        double lnV, scale;
        int far, cnt;
        ns_ell_fit(S, U, ds, dims, s_lab, label, nl, lnpv, lnV, scale, far, cnt);
        bool split = false;
        int la = 0, lb = 0;
        if (multi && !walk && cnt >= 2 * minpts && n_todo + n_done + 2 <= NS_MAX_ELL) {
            // ---- 2-means on the cluster ----
            if (tid < d) {
                S.c0[tid] = U[far * ds + dims.adim[tid]];
                S.mean[tid] = 1.0 / fmax(sqrt(fmax(S.var[tid], 0.0)), 1e-300);      // per-dimension scale (mean is free now)
            }
            __syncthreads();
            double best = -1.0;
            int ibest = far;
            for (int p = tid; p < nl; p += blockDim.x) {
                if (s_lab[p] != label) continue;
                double d2 = 0.0;
                for (int a = 0; a < d; ++a) { const double t = (U[p * ds + dims.adim[a]] - S.c0[a]) * S.mean[a]; d2 += t * t; }
                if (d2 > best) { best = d2; ibest = p; }
            }
            S.red[tid] = best; S.redi[tid] = ibest;
            __syncthreads();
            for (int o = 64; o > 0; o >>= 1) {
                if (tid < o && (S.red[tid + o] > S.red[tid] || (S.red[tid + o] == S.red[tid] && S.redi[tid + o] < S.redi[tid]))) {
                    S.red[tid] = S.red[tid + o]; S.redi[tid] = S.redi[tid + o];
                }
                __syncthreads();
            }
            if (tid < d) S.c1[tid] = U[S.redi[0] * ds + dims.adim[tid]];
            la = next_label; lb = next_label + 1;
            __syncthreads();
            for (int iter = 0; iter < NS_KMEANS_ITERS; ++iter) {
                for (int p = tid; p < nl; p += blockDim.x) {
                    const short cur = s_lab[p];
                    if (cur != label && cur != la && cur != lb) continue;
                    double d0 = 0.0, d1 = 0.0;
                    for (int a = 0; a < d; ++a) {
                        const double u = U[p * ds + dims.adim[a]], w = S.mean[a];
                        const double t0 = (u - S.c0[a]) * w, t1 = (u - S.c1[a]) * w;
                        d0 += t0 * t0; d1 += t1 * t1;
                    }
                    s_lab[p] = (short)(d1 < d0 ? lb : la);
                }
                __syncthreads();
                if (tid < d) {
                    double s0 = 0.0, s1 = 0.0;
                    int n0 = 0, n1 = 0;
                    const int ja = dims.adim[tid];
                    for (int p = 0; p < nl; ++p) {
                        const short cur = s_lab[p];
                        if (cur == la) { s0 += U[p * ds + ja]; ++n0; }
                        else if (cur == lb) { s1 += U[p * ds + ja]; ++n1; }
                    }
                    if (tid == 0) { S.cnt[0] = n0; S.cnt[1] = n1; }
                    if (n0 > 0 && n1 > 0) { S.c0[tid] = s0 / n0; S.c1[tid] = s1 / n1; }
                }
                __syncthreads();
                if (S.cnt[0] == 0 || S.cnt[1] == 0) break;
            }
            const int na = S.cnt[0], nb = S.cnt[1];
            if (na >= minpts && nb >= minpts) {
                double va, vb, sc2;
                int f2, c2;
                ns_ell_fit(S, U, ds, dims, s_lab, la, nl, lnpv, va, sc2, f2, c2);
                ns_ell_fit(S, U, ds, dims, s_lab, lb, nl, lnpv, vb, sc2, f2, c2);
                const double m = fmax(va, vb), lnsum = m + log(exp(va - m) + exp(vb - m));
                split = lnsum < lnV + log(0.5) || (lnV > log(2.0) + log((double)cnt) + lnpv && lnsum < lnV);
            }
            if (!split) {          // undo the labels; the parent's factor is recomputed below
                for (int p = tid; p < nl; p += blockDim.x)
                    if (s_lab[p] == la || s_lab[p] == lb) s_lab[p] = (short)label;
                __syncthreads();
                ns_ell_fit(S, U, ds, dims, s_lab, label, nl, lnpv, lnV, scale, far, cnt);
            }
        }
        if (split) {
            if (tid == 0) { S.todo[n_todo] = la; S.todo[n_todo + 1] = lb; }
            n_todo += 2;
            next_label += 2;
        } else {
            double *E = B + NS_BOUND_HDR + (int64_t)n_done * es;
            if (tid < d) E[tid] = S.mean[tid];
            for (int e = tid; e < d * d; e += blockDim.x) {
                const int a = e / d, b = e - a * d;
                E[d + e] = b <= a ? scale * S.c[a][b] : 0.0;
            }
            if (tid == 0) E[d + d * d] = lnV;
            ++n_done;
        }
        __syncthreads();
    }
    if (tid == 0) { B[0] = (double)n_done; B[1] = 0.0; B[2] = (double)it_now; }
}

// Device-side view of the sampler state handed to the kernels by value.
struct NsDev {
    const int32_t *act;
    const int32_t *n_act_dev;          // {n_act, n_cand}: grids are sized from a host-side upper bound
    const int32_t *pix_ids, *nlive;
    double *live_u, *live_th, *live_l;
    double *cand_u, *cand_th, *cand_l;
    int32_t *cand_pix;
    double *bound;
    float *dead_th;
    double *dead_l, *dead_lw;
    const int64_t *dead_off;
    const int32_t *dead_cap;
    double *lnZ, *H, *lmax;
    int32_t *n_dead, *it, *done;
    int64_t *n_eval;
    // constrained random-walk state
    int32_t *mode, *coh_step, *coh_acc, *eff_acc, *eff_prop, *chain_moved;
    double *lstar, *scale, *chain_u, *chain_th, *chain_l;
    const int32_t *krun, *cand_off;
    NsDims dims;
    int K, Kmax, d, nlive_max, max_samples, max_iter, walks, flags;
    double tol, efr;
    uint64_t seed;
    int lock;
};

// uniform point in the unit d-ball
__device__ void unit_ball(Philox &rng, int d, double *y)
{
    double n2 = 0.0;
    for (int j = 0; j < d; j += 2) {
        double z0, z1;
        rng.normal2(z0, z1);
        y[j] = z0; n2 += z0 * z0;
        if (j + 1 < d) { y[j + 1] = z1; n2 += z1 * z1; }
    }
    const double rad = (double)exp2f(__log2f((float)rng.uniform()) / (float)d) / sqrt(n2);
    for (int j = 0; j < d; ++j) y[j] *= rad;
}

// ---- proposals: K candidates (or K random-walk steps) per active run ---------
template <bool MULTI>
__global__ void ns_propose_kernel(const NsDev D)
{
    const int kblocks = (D.Kmax + (int)blockDim.x - 1) / (int)blockDim.x;
    const int a = blockIdx.x / kblocks, k = (blockIdx.x - a * kblocks) * blockDim.x + threadIdx.x;    // (active slot, candidate / chain)
    if (a >= *D.n_act_dev) return;
    const int r = D.act[a];
    if (k >= D.krun[r]) return;
    const int64_t idx = (int64_t)D.cand_off[a] + k;
    const int d = D.d, da = D.dims.da;
    const double *B = D.bound + (int64_t)r * ns_bound_stride(d);
    const int64_t es = ns_ell_stride(d);
    const double *E0 = B + NS_BOUND_HDR;                  // first ellipsoid {mean, L, ln V}
    Philox rng(D.seed, (uint32_t)r, (uint32_t)D.lock, (uint32_t)k);
    double u[NS_MAX_DIM], y[NS_MAX_DIM];
    bool ok = false;
    // the dimensions the likelihood does not see: uniform, whatever the method
    for (int j = 0; j < D.dims.nfree; ++j) u[D.dims.fdim[j]] = rng.uniform();
    if (D.mode[r] != 1) {
        // rejection sampling from the union of the bounding ellipsoids (or the unit cube itself)
        if (B[1] > 0.5) {
            for (int j = 0; j < da; ++j) u[D.dims.adim[j]] = rng.uniform();
            ok = true;
        } else if (!MULTI) {
            for (int tries = 0; tries < 64 && !ok; ++tries) {
                unit_ball(rng, da, y);
                ok = true;
                for (int i = 0; i < da; ++i) {
                    double v = E0[i];
                    for (int j = 0; j <= i; ++j) v += E0[da + i * da + j] * y[j];
                    u[D.dims.adim[i]] = v;
                    if (!(v > 0.0 && v < 1.0)) ok = false;
                }
            }
        } else {
            const int n_ell = (int)B[0];
            double lnVmax = -INFINITY, wsum = 0.0, wts[NS_MAX_ELL];
            for (int e = 0; e < n_ell; ++e) lnVmax = fmax(lnVmax, E0[e * es + da + da * da]);
            for (int e = 0; e < n_ell; ++e) { wts[e] = exp(E0[e * es + da + da * da] - lnVmax); wsum += wts[e]; }
            for (int tries = 0; tries < 64 && !ok; ++tries) {
                // pick an ellipsoid by volume, draw a point in it, keep it with probability 1 / (number of
                // ellipsoids that contain it): uniform over the union
                int pick = 0;
                if (n_ell > 1) {
                    double t = rng.uniform() * wsum;
                    while (pick < n_ell - 1 && t >= wts[pick]) { t -= wts[pick]; ++pick; }
                }
                const double *E = E0 + pick * es;
                unit_ball(rng, da, y);
                ok = true;
                double x[NS_MAX_DIM];
                for (int i = 0; i < da; ++i) {
                    double v = E[i];
                    for (int j = 0; j <= i; ++j) v += E[da + i * da + j] * y[j];
                    x[i] = v;
                    if (!(v > 0.0 && v < 1.0)) ok = false;
                }
                if (ok && n_ell > 1) {
                    int q = 1;
                    for (int e = 0; e < n_ell; ++e) {
                        if (e == pick) continue;
                        const double *F = E0 + e * es;
                        double r2 = 0.0;
                        for (int i = 0; i < da && r2 <= 1.0; ++i) {        // forward substitution L z = x - mean
                            double v = x[i] - F[i];
                            for (int j = 0; j < i; ++j) v -= F[da + i * da + j] * y[j];
                            v /= F[da + i * da + i];
                            y[i] = v;
                            r2 += v * v;
                        }
                        q += r2 <= 1.0;
                    }
                    if (q > 1 && rng.uniform() * (double)q >= 1.0) ok = false;
                }
                if (ok) for (int i = 0; i < da; ++i) u[D.dims.adim[i]] = x[i];
            }
        }
    } else {
        // constrained random walk: chain k takes one step of size `scale` in the metric of the
        // live set's bounding ellipsoid; a cohort of K chains starts from random live points
        double *cu = D.chain_u + ((int64_t)r * D.Kmax + k) * d;
        if (D.coh_step[r] == 0) {
            const int nl = D.nlive[r];
            int j = (int)(rng.uniform() * (double)nl);
            j = min(j, nl - 1);
            const double *lu = D.live_u + ((int64_t)r * D.nlive_max + j) * d;
            const double *lt = D.live_th + ((int64_t)r * D.nlive_max + j) * d;
            double *ct = D.chain_th + ((int64_t)r * D.Kmax + k) * d;
            for (int i = 0; i < d; ++i) { cu[i] = lu[i]; ct[i] = lt[i]; }
            D.chain_l[(int64_t)r * D.Kmax + k] = D.live_l[(int64_t)r * D.nlive_max + j];
            D.chain_moved[(int64_t)r * D.Kmax + k] = 0;
        }
        ok = true;
        unit_ball(rng, da, y);
        const double sc = D.scale[r];
        for (int i = 0; i < da; ++i) {
            double v = 0.0;
            for (int j = 0; j <= i; ++j) v += E0[da + i * da + j] * y[j];
            v = cu[D.dims.adim[i]] + sc * v;
            u[D.dims.adim[i]] = v;
            if (!(v > 0.0 && v < 1.0)) ok = false;
        }
    }
    double *ou = D.cand_u + idx * d, *ot = D.cand_th + idx * d;
    for (int j = 0; j < d; ++j) {
        const double v = ok ? u[j] : nan("");    // NaN -> NaN lnL -> never accepted
        ou[j] = v;
        ot[j] = v;
    }
    D.cand_pix[idx] = D.pix_ids[r];
}

// Running state of one run held in registers by every lane of its warp.
struct RunState {
    double lnZ, H, lmax;
    double mn;          // current worst live log-likelihood and its slot (recomputed after every insertion)
    int im;
    int it, nd;
    int cap;            // rows this run owns in the dead pool, and its first row
    int64_t off;
    bool done;
};

__device__ __forceinline__ void warp_argmin(const double *LL, int nl, int lane, double &mn, int &im)
{
    mn = INFINITY;
    im = 0;
    for (int p = lane; p < nl; p += 32) {
        const double v = LL[p];
        if (v < mn) { mn = v; im = p; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double v2 = __shfl_xor_sync(NS_FULL, mn, o);
        const int i2 = __shfl_xor_sync(NS_FULL, im, o);
        if (v2 < mn || (v2 == mn && i2 < im)) { mn = v2; im = i2; }
    }
}

// Nested-sampling step with candidate (cu, ct, lc): if it beats the current worst live
// point, that point dies with prior-mass weight X_{i-1} - X_i and the candidate takes
// its slot.  Warp-cooperative; returns true when the candidate was inserted.
__device__ bool try_insert(const NsDev &D, int r, int nl, int lane, double lnshell, const double *cu,
                           const double *ct, double lc, RunState &S, double *LL)
{
    const int d = D.d;
    const double mn = S.mn;
    const int im = S.im;
    if (!(lc > mn)) return false;          // rejected (also NaN)
    const double lnw = -(double)S.it / (double)nl + lnshell;
    const double lw = mn + lnw;
    const double lnZ_new = logaddexp(S.lnZ, lw);
    if (lnZ_new > -INFINITY) {
        const double t1 = exp(lw - lnZ_new) * mn;
        const double t2 = (S.lnZ > -INFINITY) ? exp(S.lnZ - lnZ_new) * (S.H + S.lnZ) : 0.0;
        S.H = t1 + t2 - lnZ_new;
    }
    S.lnZ = lnZ_new;
    if (S.nd < S.cap) {
        const double *th = D.live_th + ((int64_t)r * D.nlive_max + im) * d;
        const int64_t row = S.off + S.nd;
        float *dt = D.dead_th + row * d;
        for (int j = lane; j < d; j += 32) dt[j] = (float)th[j];
        if (lane == 0) {
            D.dead_l[row] = mn;
            D.dead_lw[row] = lnw;
        }
        ++S.nd;
    }
    double *lu = D.live_u + ((int64_t)r * D.nlive_max + im) * d, *lt = D.live_th + ((int64_t)r * D.nlive_max + im) * d;
    for (int j = lane; j < d; j += 32) { lu[j] = cu[j]; lt[j] = ct[j]; }
    if (lane == 0) { LL[im] = lc; D.live_l[(int64_t)r * D.nlive_max + im] = lc; }
    __syncwarp();
    warp_argmin(LL, nl, lane, S.mn, S.im);
    ++S.it;
    S.lmax = fmax(S.lmax, lc);
    // MultiNest `tol`: largest possible remaining contribution L_max X_i
    const double lnX = -(double)S.it / (double)nl;
    if (logaddexp(S.lnZ, S.lmax + lnX) - S.lnZ < D.tol) S.done = true;
    if (S.it >= D.max_iter || S.nd + nl >= S.cap) S.done = true;
    return true;
}

// ---- consume the scored proposals (one warp per active run) ------------------
__global__ void __launch_bounds__(128) ns_update_kernel(const NsDev D)
{
    extern __shared__ double s_live_l[];     // [warps per CTA][nlive_max]: this run's live log-likelihoods
    const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (w >= *D.n_act_dev) return;
    const int r = D.act[w];
    const int nl = D.nlive[r], d = D.d, K = D.krun[r], KS = D.Kmax;
    double *LL = s_live_l + (size_t)(threadIdx.x >> 5) * D.nlive_max;
    for (int p = lane; p < nl; p += 32) LL[p] = D.live_l[(int64_t)r * D.nlive_max + p];
    __syncwarp();
    RunState S;
    warp_argmin(LL, nl, lane, S.mn, S.im);
    S.lnZ = D.lnZ[r]; S.H = D.H[r]; S.lmax = D.lmax[r]; S.it = D.it[r]; S.nd = D.n_dead[r]; S.done = false;
    S.cap = D.dead_cap[r]; S.off = D.dead_off[r];
    int64_t nev = D.n_eval[r];
    // ln(1 - exp(-1/nlive)): ln of the prior-mass shell X_{i-1} - X_i relative to X_{i-1}
    const double lnshell = log(-expm1(-1.0 / (double)nl));
    const int64_t c0 = (int64_t)D.cand_off[w];  // candidate slots of this run in this iteration
    int mode = D.mode[r];
    if (mode != 1) {
        int n_ok = 0, n_acc = 0;
        for (int k = 0; k < K && !S.done; ++k) {
            const double *cu = D.cand_u + (c0 + k) * d;
            if (!(cu[0] == cu[0])) continue;      // no valid draw inside the unit cube: not a candidate
            ++nev; ++n_ok;
            if (try_insert(D, r, nl, lane, lnshell, cu, D.cand_th + (c0 + k) * d, D.cand_l[c0 + k], S, LL)) ++n_acc;
        }
        // windowed acceptance rate; fall back to the random walk when rejection sampling stalls
        int ea = D.eff_acc[r] + n_acc, ep = D.eff_prop[r] + n_ok;
        if (ep >= 512) {
            if ((D.flags & 3) != 2 && mode == 0 && (double)ea < (double)ep / (1.2 * (double)D.walks)) {
                mode = 2;                      // hand over to the random walk at the next aligned lock-step
                if (lane == 0) D.mode[r] = 2;
            }
            ea = 0; ep = 0;
        }
        if (lane == 0) { D.eff_acc[r] = ea; D.eff_prop[r] = ep; }
        // Random-walk cohorts of all runs start on the same lock-steps (multiples of `walks`), so that
        // the serial insertion work at a cohort's end falls on one lock-step in `walks` for every run.
        // This step's candidates were rejection-sampling proposals and have been consumed as such;
        // the next lock-step opens the first cohort (coh_step = 0 makes the proposal kernel start chains).
        if (mode == 2 && (D.lock + 1) % D.walks == 0 && lane == 0) {
            D.mode[r] = 1; D.coh_step[r] = 0; D.scale[r] = 0.3;
        }
    } else {
        int step = D.coh_step[r];
        double lstar;
        if (step == 0) {                        // a new cohort: threshold = current worst live point
            lstar = S.mn;
            if (lane == 0) { D.lstar[r] = lstar; D.coh_acc[r] = 0; }
        } else {
            lstar = D.lstar[r];
        }
        int acc = 0, nok = 0;
        for (int k = lane; k < K; k += 32) {
            const double *cu = D.cand_u + (c0 + k) * d;
            const double lc = D.cand_l[c0 + k];
            const bool ok = cu[0] == cu[0];
            if (ok) ++nok;
            if (ok && lc > lstar) {
                double *hu = D.chain_u + ((int64_t)r * KS + k) * d, *ht = D.chain_th + ((int64_t)r * KS + k) * d;
                const double *ct = D.cand_th + (c0 + k) * d;
                for (int j = 0; j < d; ++j) { hu[j] = cu[j]; ht[j] = ct[j]; }
                D.chain_l[(int64_t)r * KS + k] = lc;
                D.chain_moved[(int64_t)r * KS + k] = 1;
                ++acc;
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            acc += __shfl_xor_sync(NS_FULL, acc, o);
            nok += __shfl_xor_sync(NS_FULL, nok, o);
        }
        nev += nok;
        const int cacc = (step == 0 ? 0 : D.coh_acc[r]) + acc;
        ++step;
        __syncwarp();
        if (step >= D.walks) {
            // the cohort's end points are candidates for the then-current threshold, in order
            for (int k = 0; k < K && !S.done; ++k) {
                if (!D.chain_moved[(int64_t)r * KS + k]) continue;      // never moved: still a live point
                try_insert(D, r, nl, lane, lnshell, D.chain_u + ((int64_t)r * KS + k) * d,
                           D.chain_th + ((int64_t)r * KS + k) * d, D.chain_l[(int64_t)r * KS + k], S, LL);
            }
            // step size follows the acceptance fraction (target 1/2)
            const double facc = (double)cacc / (double)(K * D.walks);
            double sc = D.scale[r] * exp((facc - 0.5) / (0.5 * (double)d));
            sc = fmin(fmax(sc, 1e-5), 2.0);
            if (lane == 0) D.scale[r] = sc;
            step = 0;
        }
        if (lane == 0) { D.coh_step[r] = step; D.coh_acc[r] = cacc; }
    }
    if (lane == 0) {
        D.lnZ[r] = S.lnZ; D.H[r] = S.H; D.lmax[r] = S.lmax; D.it[r] = S.it; D.n_dead[r] = S.nd; D.n_eval[r] = nev;
        if (S.done) D.done[r] = 1;
    }
}

// ---- active-list compaction + proposal plan of the next lock-step (single CTA) -------
// Runs that finished leave the active list.  While the block is full every run proposes K
// candidates per lock-step; once few runs remain each gets more (a multiple of K up to Kmax,
// aiming at `target` vectors per launch) so that the tail of a wave still fills the GPU.  A
// random-walk cohort keeps the size it started with.
__global__ void __launch_bounds__(1024)
ns_compact_kernel(const int32_t *done, int32_t *act, int32_t *n_act_dev, int32_t *n_act_host, int64_t n_run,
                  const int32_t *mode, const int32_t *coh_step, int32_t *krun, int32_t *cand_off, int K, int Kmax,
                  int64_t target)
{
    __shared__ int s_cnt[1024];
    __shared__ int s_base;
    const int tid = threadIdx.x;
    if (tid == 0) s_base = 0;
    __syncthreads();
    for (int64_t base = 0; base < n_run; base += 1024) {
        const int64_t r = base + tid;
        const int keep = (r < n_run && !done[r]) ? 1 : 0;
        s_cnt[tid] = keep;
        __syncthreads();
        for (int o = 1; o < 1024; o <<= 1) {      // inclusive scan
            const int v = tid >= o ? s_cnt[tid - o] : 0;
            __syncthreads();
            s_cnt[tid] += v;
            __syncthreads();
        }
        if (keep) act[s_base + s_cnt[tid] - 1] = (int32_t)r;
        __syncthreads();
        if (tid == 1023) s_base += s_cnt[1023];
        __syncthreads();
    }
    const int n_act = s_base;
    __syncthreads();
    int knew = K;
    if (n_act > 0 && Kmax > K) {
        const int64_t want = (target + n_act - 1) / n_act;
        int64_t m = (want + K - 1) / K;
        if (m < 1) m = 1;
        if (m * K > Kmax) m = Kmax / K;
        knew = (int)m * K;
    }
    if (tid == 0) s_base = 0;
    __syncthreads();
    for (int base = 0; base < n_act; base += 1024) {
        const int a = base + tid;
        int k = 0;
        if (a < n_act) {
            const int r = act[a];
            if (mode[r] != 1 || coh_step[r] == 0) krun[r] = knew;
            k = krun[r];
        }
        s_cnt[tid] = k;
        __syncthreads();
        for (int o = 1; o < 1024; o <<= 1) {
            const int v = tid >= o ? s_cnt[tid - o] : 0;
            __syncthreads();
            s_cnt[tid] += v;
            __syncthreads();
        }
        if (a < n_act) cand_off[a] = s_base + s_cnt[tid] - k;
        __syncthreads();
        if (tid == 1023) s_base += s_cnt[1023];
        __syncthreads();
    }
    if (tid == 0) { n_act_dev[0] = n_act; n_act_dev[1] = s_base; n_act_host[0] = n_act; n_act_host[1] = s_base; }
}

// ---- finalisation: add the live points, normalise, pick best-fit / MAP ------
__global__ void __launch_bounds__(128)
ns_finalize_kernel(const int32_t *nlive_arr, const double *live_th, const double *live_l, float *dead_th_pool,
                   double *dead_l_pool, double *dead_lw_pool, double *lnZ_a, double *H_a, int32_t *n_dead_a,
                   const int32_t *it_a, double *lnZ_err, double *bestfit, double *mapfit, int64_t n_run, int ndim,
                   int nlive_max, const int64_t *dead_off, const int32_t *dead_cap)
{
    const int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (r >= n_run) return;
    const int nl = nlive_arr[r], d = ndim;
    const int max_samples = dead_cap[r];
    // this run's rows of the pool
    float *dead_th = dead_th_pool + dead_off[r] * d;
    double *dead_l = dead_l_pool + dead_off[r], *dead_lw = dead_lw_pool + dead_off[r];
    int nd = n_dead_a[r];
    double lnZ = lnZ_a[r], H = H_a[r];
    const double lnw_live = -(double)it_a[r] / (double)nl - log((double)nl);   // X_i / nlive
    for (int p = 0; p < nl && nd < max_samples; ++p) {
        const double l = live_l[r * nlive_max + p];
        const double lw = l + lnw_live;
        const double lnZ_new = logaddexp(lnZ, lw);
        if (lnZ_new > -INFINITY) {
            const double t1 = exp(lw - lnZ_new) * l;
            const double t2 = (lnZ > -INFINITY) ? exp(lnZ - lnZ_new) * (H + lnZ) : 0.0;
            H = t1 + t2 - lnZ_new;
        }
        lnZ = lnZ_new;
        const double *th = live_th + (r * nlive_max + p) * d;
        float *dt = dead_th + (int64_t)nd * d;
        for (int j = lane; j < d; j += 32) dt[j] = (float)th[j];
        if (lane == 0) { dead_l[nd] = l; dead_lw[nd] = lnw_live; }
        ++nd;
    }
    __syncwarp();
    // best fit = max likelihood sample; MAP = sample of largest posterior weight L_i w_i
    double bl = -INFINITY, bw = -INFINITY;
    int bi = 0, wi = 0;
    for (int p = lane; p < nd; p += 32) {
        const double l = dead_l[p], lw = l + dead_lw[p];
        if (l > bl) { bl = l; bi = p; }
        if (lw > bw) { bw = lw; wi = p; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double l2 = __shfl_xor_sync(NS_FULL, bl, o);
        const int i2 = __shfl_xor_sync(NS_FULL, bi, o);
        if (l2 > bl || (l2 == bl && i2 < bi)) { bl = l2; bi = i2; }
        const double w2 = __shfl_xor_sync(NS_FULL, bw, o);
        const int j2 = __shfl_xor_sync(NS_FULL, wi, o);
        if (w2 > bw || (w2 == bw && j2 < wi)) { bw = w2; wi = j2; }
    }
    for (int j = lane; j < d; j += 32) {
        bestfit[r * d + j] = (double)dead_th[(int64_t)bi * d + j];
        mapfit[r * d + j] = (double)dead_th[(int64_t)wi * d + j];
    }
    if (lane == 0) {
        lnZ_a[r] = lnZ;
        H_a[r] = H;
        n_dead_a[r] = nd;
        lnZ_err[r] = sqrt(fmax(H, 0.0) / (double)nl);
    }
}


// ---- posterior products of all runs (what the reference's dumper writes per run) ----------
// Rows a run keeps: its dead points and final live points without the logZero ones (NaN prior
// draws among the first live set, lnL = -inf, weight 0).  One warp per run.
__global__ void __launch_bounds__(128)
ns_keep_count_kernel(const double *dead_l, const int64_t *dead_off, const int32_t *n_dead, int32_t *keep_n,
                     int64_t n_run)
{
    const int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (r >= n_run) return;
    const double *L = dead_l + dead_off[r];
    const int nd = n_dead[r];
    int cnt = 0;
    for (int p = lane; p < nd; p += 32) cnt += L[p] > -INFINITY;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(NS_FULL, cnt, o);
    if (lane == 0) keep_n[r] = cnt;
}

// float32 rows {theta[d], lnL, posterior weight exp(lnL + ln w - ln Z)} in death order: the layout of the
// reference's `posteriors` dataset (core.pyx:680).  One warp per run, ordered compaction.
__global__ void __launch_bounds__(128)
ns_pack_post_kernel(const float *dead_th, const double *dead_l, const double *dead_lw, const int64_t *dead_off,
                    const int32_t *n_dead, const double *lnZ, const int64_t *post_off, float *post, int64_t n_run,
                    int d)
{
    const int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (r >= n_run) return;
    const int64_t off = dead_off[r];
    const int nd = n_dead[r], w = d + 2;
    const double z = lnZ[r];
    float *out = post + post_off[r] * w;
    int at = 0;
    for (int base = 0; base < nd; base += 32) {
        const int p = base + lane;
        const double l = p < nd ? dead_l[off + p] : -INFINITY;
        const bool keep = l > -INFINITY;
        const unsigned m = __ballot_sync(NS_FULL, keep);
        if (keep) {
            float *row = out + (int64_t)(at + __popc(m & ((1u << lane) - 1u))) * w;
            const float *th = dead_th + (off + p) * d;
            for (int j = 0; j < d; ++j) row[j] = th[j];
            row[d] = (float)l;
            row[d + 1] = (float)exp(l + dead_lw[off + p] - z);
        }
        at += __popc(m);
    }
}

// numpy.quantile(theta[:, j], q) -- linear interpolation between order statistics, unweighted like the
// reference's Dumper.calc_marginals (core.pyx:596-598) -- for one (run, parameter) per CTA: the column
// is sorted by a bitonic network in shared memory (or in `scratch` for runs with more rows than fit).
__global__ void __launch_bounds__(512)
ns_marginals_kernel(const float *post, const int64_t *post_off, const int32_t *run_list, int n_list, int d,
                    const double *quant, int n_q, double *marg, float *scratch, int scratch_stride)
{
    extern __shared__ float s_key[];
    const int item = blockIdx.x;                  // (entry of run_list, parameter)
    const int e = item / d, j = item - e * d;
    if (e >= n_list) return;
    const int r = run_list[e];
    const int64_t o = post_off[r];
    const int n = (int)(post_off[r + 1] - o), w = d + 2;
    int np2 = 1;
    while (np2 < n) np2 <<= 1;
    float *key = scratch ? scratch + (int64_t)item * scratch_stride : s_key;
    for (int i = threadIdx.x; i < np2; i += blockDim.x) key[i] = i < n ? post[(o + i) * w + j] : INFINITY;
    __syncthreads();
    for (int k = 2; k <= np2; k <<= 1)
        for (int st = k >> 1; st > 0; st >>= 1) {
            for (int t = threadIdx.x; t < (np2 >> 1); t += blockDim.x) {
                const int lo = ((t & ~(st - 1)) << 1) | (t & (st - 1)), hi = lo | st;
                const float a = key[lo], b = key[hi];
                const bool up = (lo & k) == 0;
                if ((a > b) == up) { key[lo] = b; key[hi] = a; }
            }
            __syncthreads();
        }
    if ((int)threadIdx.x < n_q) {
        double v = nan("");
        if (n > 0) {
            const double h = quant[threadIdx.x] * (double)(n - 1);
            int lo = (int)floor(h);
            lo = min(max(lo, 0), n - 1);
            const int hi = min(lo + 1, n - 1);
            const double a = (double)key[lo], b = (double)key[hi], t = h - (double)lo;
            v = a + (b - a) * t;                  // numpy's 'linear' method
        }
        marg[((int64_t)r * n_q + threadIdx.x) * d + j] = v;
    }
}

// ---- intensity credible intervals (nf_ns_intensity) ------------------------------------------------
// The kept rows of runs [r0, r0 + n_r) (the rows ns_pack_post_kernel writes, in the same order), each split into
// its ncomp single-component vectors on the run's pixel: vec [(row * ncomp + c)][n_model] FP32, vpix likewise, and
// the row's float32 posterior weight, computed as ns_pack_post_kernel does.  Rows are counted from the group's
// first row.  One warp per run, ordered compaction.
__global__ void __launch_bounds__(128)
ns_int_gather_kernel(const float *dead_th, const double *dead_l, const double *dead_lw, const int64_t *dead_off,
                     const int32_t *n_dead, const double *lnZ, const int64_t *post_off, const int32_t *pix_ids,
                     int64_t r0, int64_t n_r, int d, int ncomp, float *vec, int32_t *vpix, float *wt)
{
    const int64_t e = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (e >= n_r) return;
    const int64_t r = r0 + e;
    const int64_t off = dead_off[r], row0 = post_off[r] - post_off[r0];
    const int nd = n_dead[r], nm = d / ncomp;
    const double z = lnZ[r];
    const int32_t pix = pix_ids[r];
    int at = 0;
    for (int base = 0; base < nd; base += 32) {
        const int p = base + lane;
        const double l = p < nd ? dead_l[off + p] : -INFINITY;
        const bool keep = l > -INFINITY;
        const unsigned m = __ballot_sync(NS_FULL, keep);
        if (keep) {
            const int64_t row = row0 + at + __popc(m & ((1u << lane) - 1u));
            const float *th = dead_th + (off + p) * d;
            for (int c = 0; c < ncomp; ++c) {             // parameter-major, component-minor rows
                float *v = vec + (row * ncomp + c) * nm;
                for (int j = 0; j < nm; ++j) v[j] = th[j * ncomp + c];
                vpix[row * ncomp + c] = pix;
            }
            wt[row] = (float)exp(l + dead_lw[off + p] - z);
        }
        at += __popc(m);
    }
}

// Posterior-weighted quantiles of one (entry of run_list, spectrum, component, quantity) per CTA, quantity 0 the
// peak and 1 the channel sum of the component's model.  The (value, row) keys of the run's rows are sorted by a
// bitonic network in shared memory (or in `scratch` for runs with more rows than fit): equal values keep their row
// order, as numpy.argsort(kind='stable') -- duplicate rows (a final live point equal to a dead one) make the
// interpolation depend on it.  The weights then become their running FP64 sum in row order of the sorted list, summed
// one after the other like numpy.cumsum, and every quantile q is numpy.interp(q, cw / cw[-1], x_sorted), branch for
// branch.  Each entry is a double value and an 8-byte slot holding {float weight, int row} while sorting and the
// running sum after.
struct NsWRow {
    float w;
    int row;
};
__global__ void __launch_bounds__(512)
ns_wquant_kernel(const float *peak, const double *sum, const float *wt, const int64_t *post_off, int64_t row_base,
                 const int32_t *run_list, int n_list, int n_spec, int ncomp, const double *quant, int n_q,
                 double *peak_q, double *integ_q, double *scratch, int scratch_stride)
{
    extern __shared__ double s_kw[];
    const int item = blockIdx.x;
    const int per = n_spec * ncomp * 2;
    const int e = item / per, rest = item - e * per;
    if (e >= n_list) return;
    const int qty = rest & 1, sc = rest >> 1, s = sc / ncomp, c = sc - s * ncomp;
    const int r = run_list[e];
    const int64_t o = post_off[r] - row_base;
    const int n = (int)(post_off[r + 1] - post_off[r]);
    const int tid = threadIdx.x, nt = blockDim.x;
    int np2 = 1;
    while (np2 < n) np2 <<= 1;
    double *key = scratch ? scratch + (int64_t)item * 2 * scratch_stride : s_kw;
    double *cw = key + (scratch ? scratch_stride : np2);
    NsWRow *slot = reinterpret_cast<NsWRow *>(cw);
    for (int i = tid; i < np2; i += nt) {
        const int64_t v = ((o + i) * ncomp + c) * n_spec + s;
        key[i] = i < n ? (qty ? sum[v] : (double)peak[v]) : INFINITY;
        slot[i] = NsWRow{i < n ? wt[o + i] : 0.0f, i};
    }
    __syncthreads();
    for (int k = 2; k <= np2; k <<= 1)
        for (int st = k >> 1; st > 0; st >>= 1) {
            for (int t = tid; t < (np2 >> 1); t += nt) {
                const int lo = ((t & ~(st - 1)) << 1) | (t & (st - 1)), hi = lo | st;
                const double a = key[lo], b = key[hi];
                const NsWRow sa = slot[lo], sb = slot[hi];
                const bool up = (lo & k) == 0;
                if ((a > b || (a == b && sa.row > sb.row)) == up) {
                    key[lo] = b; key[hi] = a;
                    slot[lo] = sb; slot[hi] = sa;
                }
            }
            __syncthreads();
        }
    if (tid == 0) {             // numpy.cumsum: one addition after the other
        double run = 0.0;
        for (int i = 0; i < n; ++i) {
            run += (double)slot[i].w;
            cw[i] = run;
        }
    }
    __syncthreads();
    if (tid < n_q) {
        double v = nan("");
        if (n > 0) {
            const double q = quant[tid], tot = cw[n - 1];
            int lo = 0, hi = n;              // j = (number of i with cw_i / tot <= q) - 1
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if (q >= cw[mid] / tot) lo = mid + 1;
                else hi = mid;
            }
            const int j = lo - 1;
            if (j < 0) v = key[0];
            else if (j >= n - 1) v = key[n - 1];
            else {
                const double xj = cw[j] / tot, xj1 = cw[j + 1] / tot;
                if (xj == q) v = key[j];
                else {
                    const double slope = (key[j + 1] - key[j]) / (xj1 - xj);
                    v = slope * (q - xj) + key[j];
                    if (isnan(v)) {
                        v = slope * (q - xj1) + key[j + 1];
                        if (isnan(v) && key[j] == key[j + 1]) v = key[j];
                    }
                }
            }
        }
        (qty ? integ_q : peak_q)[(((int64_t)r * n_q + tid) * n_spec + s) * ncomp + c] = v;
    }
}

#define NS_CUDA(expr) do { cudaError_t e__ = (expr); if (e__ != cudaSuccess) return (int)e__; } while (0)

int score(nf_sampler *s, double *params, const int32_t *pix, int64_t vpp, int64_t B, double *lnl,
          const int32_t *B_dev = nullptr)
{
    NS_CUDA(nf_launch_prior_transform(s->pr, params, B, s->ncomp, s->stream, B_dev));
    NfLikeArgs a;
    std::memset(&a, 0, sizeof(a));
    const nf_pixels *px = s->px;
    a.data = px->data; a.inv2s2 = px->inv2s2; a.d2chunk = px->d2chunk; a.params = params; a.pix_of_vec = pix; a.vecs_per_pix = 1;
    a.B = B; a.B_dev = B_dev; a.pix_stride = (int64_t)px->n_spec * px->n_pad; a.lnL = lnl; a.pred = nullptr; a.param_f64 = 1;
    a.ncomp = s->ncomp; a.n_spec = px->n_spec; a.n_chan = px->n_chan; a.n_pad = px->n_pad;
    a.cold = (s->flags & NF_FLAG_COLD) != 0; a.lte = (s->flags & NF_FLAG_LTE) != 0;
    a.tile_vecs = (int)(vpp > 0 ? vpp : 0);     // a CTA tile never straddles the proposals of two runs (pixels)
    for (int k = 0; k < px->n_spec; ++k) a.spec[k] = px->spec[k];
    a.pixmeta = px->pixmeta;
    NS_CUDA(px->model == NF_MODEL_NH3 ? nf_launch_nh3(a, s->stream)
            : px->model == NF_MODEL_N2HP ? nf_launch_n2hp(a, s->stream) : nf_launch_gauss(a, s->stream));
    s->launches += 2;
    return NF_OK;
}

template <typename T>
cudaError_t dalloc(T **p, size_t n) { return cudaMalloc((void **)p, n * sizeof(T)); }

// Scratch that lives for part of one call: stream-ordered allocation (NF_SYNC_ALLOC=1 falls back to cudaMalloc /
// cudaFree, a debugging aid).
bool ns_sync_alloc()
{
    static const bool on = getenv("NF_SYNC_ALLOC") != nullptr;
    return on;
}
cudaError_t ns_scratch_alloc(void **p, size_t bytes, cudaStream_t st)
{
    return ns_sync_alloc() ? cudaMalloc(p, bytes) : cudaMallocAsync(p, bytes, st);
}
void ns_scratch_free(void *p, cudaStream_t st)
{
    if (!p) return;
    if (ns_sync_alloc()) { cudaStreamSynchronize(st); cudaFree(p); }
    else cudaFreeAsync(p, st);
}

}  // namespace

extern "C" {

int nf_ns_create(const nf_pixels *px, const nf_priors *pr, int ncomp, int model_flags, const nf_ns_config *cfg,
                 int64_t n_run, const int32_t *pix_ids, const int32_t *nlive, nf_sampler **out)
{
    if (!out) return NF_EINVAL;
    *out = nullptr;
    if (!px || !pr || !cfg || !pix_ids || !nlive || n_run < 1 || ncomp < 1) return NF_EINVAL;
    if (px->device != pr->device) return NF_EINVAL;
    const int n_model = px->model == NF_MODEL_NH3 ? 6 : (px->model == NF_MODEL_N2HP ? 4 : 3);
    if (pr->n_model != n_model) return NF_EINVAL;
    const int ndim = n_model * ncomp;
    if (ndim > NS_MAX_DIM) return NF_EINVAL;
    if (px->model != NF_MODEL_GAUSS && ncomp > NF_MAX_NCOMP_NH3) return NF_EINVAL;
    if (cfg->nlive_max < 8 || cfg->n_prop < 1 || cfg->max_samples < 2 * cfg->nlive_max || !(cfg->tol > 0.0) ||
        !(cfg->efr > 0.0 && cfg->efr <= 1.0) || cfg->max_iter < 1)
        return NF_EINVAL;
    for (int64_t r = 0; r < n_run; ++r) {
        if (pix_ids[r] < 0 || pix_ids[r] >= px->n_pix) return NF_EINVAL;
        if (nlive[r] < 8 || nlive[r] > cfg->nlive_max) return NF_EINVAL;
    }
    int prev = -1;
    cudaGetDevice(&prev);
    if (cudaSetDevice(px->device) != cudaSuccess) return NF_ENODEV;
    nf_sampler *s = new (std::nothrow) nf_sampler();
    if (!s) { if (prev >= 0) cudaSetDevice(prev); return NF_ENOMEM; }
    std::memset(s, 0, sizeof(*s));
    s->px = px; s->pr = pr; s->device = px->device; s->ncomp = ncomp; s->flags = model_flags; s->ndim = ndim;
    s->cfg = *cfg; s->n_run = n_run; s->K = cfg->n_prop;
    s->Kmax = cfg->n_prop_max > cfg->n_prop ? (cfg->n_prop_max / cfg->n_prop) * cfg->n_prop : cfg->n_prop;
    if (s->cfg.target_batch < 1) s->cfg.target_batch = 65536;
    // sum_a k_a <= max(n_act K, target + n_act K) over a shrinking active list
    s->cand_cap = n_run * (int64_t)s->K + (s->Kmax > s->K ? (int64_t)s->cfg.target_batch : 0);
    const size_t R = (size_t)n_run, NL = (size_t)cfg->nlive_max, D = (size_t)ndim, K = (size_t)s->Kmax,
                 CC = (size_t)s->cand_cap;
    // dead-point pool: every run gets rows in proportion to its own live set (not the wave's largest)
    s->h_dead_off = new (std::nothrow) std::vector<int64_t>((size_t)n_run + 1, 0);
    s->h_post_off = new (std::nothrow) std::vector<int64_t>((size_t)n_run + 1, 0);
    std::vector<int32_t> h_cap((size_t)n_run);
    if (!s->h_dead_off || !s->h_post_off) { delete s->h_dead_off; delete s->h_post_off; delete s; return NF_ENOMEM; }
    {
        const int64_t per_live = cfg->max_samples / cfg->nlive_max;       // >= 2 (checked above)
        for (int64_t r = 0; r < n_run; ++r) {
            int64_t c = per_live * nlive[r];
            if (c > cfg->max_samples) c = cfg->max_samples;
            h_cap[(size_t)r] = (int32_t)c;
            (*s->h_dead_off)[(size_t)r + 1] = (*s->h_dead_off)[(size_t)r] + c;
        }
        s->dead_rows = (*s->h_dead_off)[(size_t)n_run];
    }
    const size_t MS = (size_t)s->dead_rows;
    cudaError_t e = cudaSuccess;
    auto A = [&](cudaError_t x) { if (e == cudaSuccess) e = x; };
    A(dalloc(&s->pix_ids, R)); A(dalloc(&s->nlive, R));
    A(dalloc(&s->live_u, R * NL * D)); A(dalloc(&s->live_th, R * NL * D)); A(dalloc(&s->live_l, R * NL));
    A(dalloc(&s->cand_u, CC * D)); A(dalloc(&s->cand_th, CC * D)); A(dalloc(&s->cand_l, CC));
    A(dalloc(&s->cand_pix, CC)); A(dalloc(&s->krun, R)); A(dalloc(&s->cand_off, R));
    A(dalloc(&s->bound, R * (size_t)ns_bound_stride(ndim)));

    A(dalloc(&s->dead_th, MS * D)); A(dalloc(&s->dead_l, MS)); A(dalloc(&s->dead_lw, MS));
    A(dalloc(&s->dead_off, R + 1)); A(dalloc(&s->dead_cap, R)); A(dalloc(&s->keep_n, R)); A(dalloc(&s->post_off, R + 1));
    A(dalloc(&s->lnZ, R)); A(dalloc(&s->H, R)); A(dalloc(&s->lmax, R)); A(dalloc(&s->lnZ_err, R));
    A(dalloc(&s->n_dead, R)); A(dalloc(&s->it, R)); A(dalloc(&s->done, R)); A(dalloc(&s->n_eval, R));
    A(dalloc(&s->bestfit, R * D)); A(dalloc(&s->mapfit, R * D));
    A(dalloc(&s->act, R)); A(dalloc(&s->n_act_dev, 2));
    A(dalloc(&s->mode, R)); A(dalloc(&s->coh_step, R)); A(dalloc(&s->coh_acc, R)); A(dalloc(&s->eff_acc, R));
    A(dalloc(&s->eff_prop, R)); A(dalloc(&s->chain_moved, R * K)); A(dalloc(&s->lstar, R)); A(dalloc(&s->scale, R));
    A(dalloc(&s->chain_u, R * K * D)); A(dalloc(&s->chain_th, R * K * D)); A(dalloc(&s->chain_l, R * K));
    // active dimensions from the prior plan (host copy): rows written by a ConstantPrior and the duplicate
    // row of a DuplicatePrior do not depend on the cube value
    {
        bool dummy[NS_MAX_DIM] = {false};
        for (int k = 0; k < pr->n_prior && pr->h_priors; ++k) {
            const nf_prior_desc &p = pr->h_priors[k];
            const int row = p.kind == NF_PRIOR_CONSTANT ? p.p_ix : (p.kind == NF_PRIOR_DUPLICATE ? p.p_ix2 : -1);
            if (row >= 0 && row < n_model)
                for (int c = 0; c < ncomp; ++c) dummy[row * ncomp + c] = true;
        }
        // a row another prior writes as well stays active (DuplicatePrior's source row, nested sigma rows)
        for (int k = 0; k < pr->n_prior && pr->h_priors; ++k) {
            const nf_prior_desc &p = pr->h_priors[k];
            if (p.kind != NF_PRIOR_CONSTANT)
                for (int c = 0; c < ncomp; ++c) dummy[p.p_ix * ncomp + c] = false;
            if (p.kind == NF_PRIOR_RESOLVED_CENSEP || p.kind == NF_PRIOR_RESOLVED_PLACEMENT) {
                const nf_prior_desc &q = pr->h_priors[p.nested];
                if (q.kind != NF_PRIOR_CONSTANT)
                    for (int c = 0; c < ncomp; ++c) dummy[q.p_ix * ncomp + c] = false;
            }
        }
        s->da = 0;
        for (int j = 0; j < ndim; ++j)
            if (!dummy[j] || (cfg->flags & 4)) s->adim[s->da++] = (signed char)j;
        if (s->da == 0)
            for (int j = 0; j < ndim; ++j) s->adim[s->da++] = (signed char)j;
    }
    s->walks = cfg->bound_update_interval > 1 ? cfg->bound_update_interval : 20 + s->da;
    s->update_every = 8;            // lock-steps between rebuilds of the decomposition (mmodal)
    if (const char *ue = getenv("NF_NS_UPDATE_EVERY")) s->update_every = atoi(ue) > 0 ? atoi(ue) : 8;
    A(cudaMallocHost((void **)&s->n_act_host, 2 * sizeof(int32_t)));
    A(cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking));
    // Everything the sampler's kernels read is uploaded ON THE SAMPLER'S STREAM.  A plain cudaMemcpy from pageable
    // memory returns once the data are staged; the DMA then runs in the legacy stream, which does not order with a
    // non-blocking stream: under load (several samplers from several host threads) the first kernels would read
    // pixel indices that have not arrived yet.
    if (e == cudaSuccess)
        e = cudaMemsetAsync(s->bound, 0, R * (size_t)ns_bound_stride(ndim) * sizeof(double), s->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(s->pix_ids, pix_ids, R * sizeof(int32_t), cudaMemcpyHostToDevice, s->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(s->nlive, nlive, R * sizeof(int32_t), cudaMemcpyHostToDevice, s->stream);
    if (e == cudaSuccess)
        e = cudaMemcpyAsync(s->dead_off, s->h_dead_off->data(), (R + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, s->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(s->dead_cap, h_cap.data(), R * sizeof(int32_t), cudaMemcpyHostToDevice, s->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s->stream);      // the host arrays may go away after the call
    if (prev >= 0) cudaSetDevice(prev);
    if (e != cudaSuccess) { nf_ns_free(s); return (int)e; }
    *out = s;
    return NF_OK;
}

int nf_ns_free(nf_sampler *s)
{
    if (!s) return NF_OK;
    int prev = -1;
    cudaGetDevice(&prev);
    cudaSetDevice(s->device);
    void *ptrs[] = {s->pix_ids, s->nlive, s->live_u, s->live_th, s->live_l, s->cand_u, s->cand_th, s->cand_l,
                    s->cand_pix, s->krun, s->cand_off, s->bound, s->dead_th, s->dead_l, s->dead_lw, s->lnZ, s->H, s->lmax, s->lnZ_err,
                    s->n_dead, s->it, s->done, s->n_eval, s->bestfit, s->mapfit, s->act, s->n_act_dev,
                    s->mode, s->coh_step, s->coh_acc, s->eff_acc, s->eff_prop, s->chain_moved, s->lstar, s->scale,
                    s->chain_u, s->chain_th, s->chain_l, s->dead_off, s->dead_cap, s->keep_n, s->post_off};
    for (void *p : ptrs) if (p) cudaFree(p);
    delete s->h_dead_off;
    delete s->h_post_off;
    if (s->n_act_host) cudaFreeHost(s->n_act_host);
    if (s->stream) cudaStreamDestroy(s->stream);
    if (prev >= 0) cudaSetDevice(prev);
    delete s;
    return NF_OK;
}

int nf_ns_run(nf_sampler *s)
{
    if (!s) return NF_EINVAL;
    int prev = -1;
    cudaGetDevice(&prev);
    if (cudaSetDevice(s->device) != cudaSuccess) return NF_ENODEV;
    s->post_ready = false;             // the row offsets of nf_ns_products_rows describe the previous run
    const int d = s->ndim, NL = s->cfg.nlive_max, K = s->K;
    const int64_t R = s->n_run;
    cudaStream_t st = s->stream;
    int rc = NF_OK;
    // initial live points: uniform cube draws, scored in one batch
    {
        const int64_t n = R * NL;
        ns_init_live_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(s->live_u, s->live_th, R, NL, d, s->cfg.seed);
        // pixel of every (run, point): reuse cand_pix-like map built on the fly via vecs_per_pix is not
        // possible (runs index arbitrary pixels), so score run by run blocks through an explicit map
        int32_t *map = nullptr;
        if (ns_scratch_alloc((void **)&map, (size_t)n * sizeof(int32_t), st) != cudaSuccess) { rc = NF_ENOMEM; }
        if (rc == NF_OK) {
            ns_live_map_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(s->pix_ids, map, R, NL);
            rc = score(s, s->live_th, map, NL, n, s->live_l);
            ns_scratch_free(map, st);
        }
        if (rc == NF_OK) {
            ns_init_state_kernel<<<(unsigned)((R + 127) / 128), 128, 0, st>>>(s->lnZ, s->H, s->lmax, s->n_dead, s->it,
                                                                            s->done, s->n_eval, s->act, s->nlive,
                                                                            s->live_l, R, NL, s->mode, s->coh_step,
                                                                            s->coh_acc, s->eff_acc, s->eff_prop,
                                                                            s->scale, ((s->cfg.flags & 3) == 1) ? 1 : 0);
            s->launches += 2;
        }
    }
    // the first proposal plan
    if (rc == NF_OK) {
        ns_compact_kernel<<<1, 1024, 0, st>>>(s->done, s->act, s->n_act_dev, s->n_act_host, R, s->mode, s->coh_step,
                                              s->krun, s->cand_off, K, s->Kmax, (int64_t)s->cfg.target_batch);
        cudaError_t e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) rc = (int)e;
    }
    if (rc == NF_OK && getenv("NF_NS_DEBUG")) {
        std::vector<double> ll((size_t)R * NL);
        cudaMemcpy(ll.data(), s->live_l, ll.size() * 8, cudaMemcpyDeviceToHost);
        double mn = 1e300, mx = -1e300; size_t nz = 0, nn = 0;
        for (double v : ll) { if (v != v) { ++nn; continue; } mn = v < mn ? v : mn; mx = v > mx ? v : mx; if (v == 0.0) ++nz; }
        fprintf(stderr, "[ns] initial live lnL: min %.6g max %.6g zeros %zu nans %zu of %zu\n", mn, mx, nz, nn, ll.size());
    }
    int n_act = rc == NF_OK ? s->n_act_host[0] : 0;
    int lock = 0;
    // The counts of the next lock-step (active runs, candidates) stay on the device; the host
    // sizes grids from upper bounds -- the active list only shrinks and the candidate total is
    // at most n_act K + target -- and reads the counts back every `sync_every` lock-steps.
    const size_t upd_smem = (size_t)4 * NL * sizeof(double);
    if (nf_ensure_dyn_smem((const void *)ns_update_kernel, upd_smem) != cudaSuccess)
        rc = NF_EINVAL;
    const bool debug = getenv("NF_NS_DEBUG") != nullptr;
    // NF_NS_PROFILE=1: per-kernel device time of every lock-step (CUDA events, synchronous)
    const bool prof = getenv("NF_NS_PROFILE") != nullptr;
    cudaEvent_t pev[6];
    double pms[5] = {0, 0, 0, 0, 0}, ptail[5] = {0, 0, 0, 0, 0};
    int ntail = 0;
    double pwall = 0.0;
    if (prof) for (int i = 0; i < 6; ++i) cudaEventCreate(&pev[i]);
    const int sync_every = (debug || prof) ? 1 : 8;
    // lock-step iterations are bounded: a run needs at most max_iter * walks of them
    const int64_t lock_cap = (int64_t)s->cfg.max_iter * (int64_t)(s->walks + 1);
    while (rc == NF_OK && n_act > 0 && (int64_t)lock < lock_cap && lock < 2000000000) {
        NsDev D;
        D.act = s->act; D.n_act_dev = s->n_act_dev; D.pix_ids = s->pix_ids; D.nlive = s->nlive;
        D.live_u = s->live_u; D.live_th = s->live_th; D.live_l = s->live_l;
        D.cand_u = s->cand_u; D.cand_th = s->cand_th; D.cand_l = s->cand_l; D.cand_pix = s->cand_pix;
        D.bound = s->bound; D.dead_th = s->dead_th; D.dead_l = s->dead_l; D.dead_lw = s->dead_lw;
        D.dead_off = s->dead_off; D.dead_cap = s->dead_cap;
        D.lnZ = s->lnZ; D.H = s->H; D.lmax = s->lmax; D.n_dead = s->n_dead; D.it = s->it; D.done = s->done;
        D.n_eval = s->n_eval; D.mode = s->mode; D.coh_step = s->coh_step; D.coh_acc = s->coh_acc;
        D.eff_acc = s->eff_acc; D.eff_prop = s->eff_prop; D.chain_moved = s->chain_moved; D.lstar = s->lstar;
        D.scale = s->scale; D.chain_u = s->chain_u; D.chain_th = s->chain_th; D.chain_l = s->chain_l;
        D.krun = s->krun; D.cand_off = s->cand_off;
        D.dims.da = s->da;
        std::memcpy(D.dims.adim, s->adim, sizeof(D.dims.adim));
        D.dims.nfree = 0;
        for (int j = 0; j < d; ++j) {
            bool active = false;
            for (int i = 0; i < s->da; ++i) active |= s->adim[i] == j;
            if (!active) D.dims.fdim[D.dims.nfree++] = (signed char)j;
        }
        D.K = K; D.Kmax = s->Kmax; D.d = d; D.nlive_max = NL; D.max_samples = s->cfg.max_samples; D.max_iter = s->cfg.max_iter;
        D.walks = s->walks; D.flags = s->cfg.flags; D.tol = s->cfg.tol; D.efr = s->cfg.efr; D.seed = s->cfg.seed;
        D.lock = lock;
        int64_t cand_ub = (int64_t)n_act * K + (s->Kmax > K ? (int64_t)s->cfg.target_batch : 0);
        if (cand_ub > s->cand_cap) cand_ub = s->cand_cap;
        if (prof) cudaEventRecord(pev[0], st);
        if (s->cfg.flags & 8)
            ns_bounds_single_kernel<<<n_act, 128, 0, st>>>(s->act, s->n_act_dev, s->nlive, s->it, s->live_u, s->bound, NL, d,
                                                           s->cfg.efr, s->mode, s->coh_step, D.dims);
        else
            ns_bounds_kernel<<<n_act, 128, (size_t)NL * sizeof(short), st>>>(s->act, s->n_act_dev, s->nlive, s->it, s->live_u,
                                                                             s->bound, NL, d, s->cfg.efr, s->mode,
                                                                             s->coh_step, D.dims, lock, s->update_every, 1);
        if (prof) cudaEventRecord(pev[1], st);
        if (s->cfg.flags & 8)
            ns_propose_kernel<false><<<(unsigned)((s->Kmax + 127) / 128) * (unsigned)n_act, 128, 0, st>>>(D);
        else
            ns_propose_kernel<true><<<(unsigned)((s->Kmax + 127) / 128) * (unsigned)n_act, 128, 0, st>>>(D);
        if (prof) cudaEventRecord(pev[2], st);
        // few vectors in flight (tail of a wave): smaller CTA tiles, so that the launch spreads over
        // more SMs and a lock-step's latency drops
        const int tile = ((int64_t)n_act * K >= 32768 || K % 8 != 0) ? K : 8;
        rc = score(s, s->cand_th, s->cand_pix, tile, cand_ub, s->cand_l, s->n_act_dev + 1);
        if (rc != NF_OK) break;
        if (prof) cudaEventRecord(pev[3], st);
        ns_update_kernel<<<(n_act * 32 + 127) / 128, 128, upd_smem, st>>>(D);
        if (prof) cudaEventRecord(pev[4], st);
        ns_compact_kernel<<<1, 1024, 0, st>>>(s->done, s->act, s->n_act_dev, s->n_act_host, R, s->mode, s->coh_step,
                                              s->krun, s->cand_off, K, s->Kmax, (int64_t)s->cfg.target_batch);
        if (prof) {
            cudaEventRecord(pev[5], st);
            cudaEventSynchronize(pev[5]);
            const bool tail = s->n_act_host[0] * K < 8192;
            if (tail) ++ntail;
            for (int i = 0; i < 5; ++i) {
                float ms = 0.f;
                cudaEventElapsedTime(&ms, pev[i], pev[i + 1]);
                pms[i] += ms;
                if (tail) ptail[i] += ms;
            }
            float ms = 0.f; cudaEventElapsedTime(&ms, pev[0], pev[5]); pwall += ms;
            if (lock % 500 == 0)
                fprintf(stderr, "[ns-prof] lock %d n_act %d n_cand %d\n", lock, s->n_act_host[0], s->n_act_host[1]);
        }
        s->launches += 4;
        ++lock;
        if (lock % sync_every == 0) {
            cudaError_t e = cudaStreamSynchronize(st);
            if (e != cudaSuccess) { rc = (int)e; break; }
            n_act = s->n_act_host[0];
        }
        if (getenv("NF_NS_DEBUG") && (lock % atoi(getenv("NF_NS_DEBUG"))) == 0 && n_act > 0) {
            // diagnostics of the first still-active run
            int32_t r0 = 0, it0 = 0; int64_t ne = 0; double z0 = 0, lm = 0;
            cudaMemcpy(&r0, s->act, 4, cudaMemcpyDeviceToHost);
            cudaMemcpy(&it0, s->it + r0, 4, cudaMemcpyDeviceToHost);
            cudaMemcpy(&ne, s->n_eval + r0, 8, cudaMemcpyDeviceToHost);
            cudaMemcpy(&z0, s->lnZ + r0, 8, cudaMemcpyDeviceToHost);
            cudaMemcpy(&lm, s->lmax + r0, 8, cudaMemcpyDeviceToHost);
            std::vector<double> B((size_t)ns_bound_stride(d));
            cudaMemcpy(B.data(), s->bound + (size_t)r0 * ns_bound_stride(d), B.size() * 8, cudaMemcpyDeviceToHost);
            std::vector<double> cu((size_t)K * d);
            cudaMemcpy(cu.data(), s->cand_u, cu.size() * 8, cudaMemcpyDeviceToHost);   // slot 0 = first active run
            int valid = 0;
            for (int k = 0; k < K; ++k) if (cu[(size_t)k * d] == cu[(size_t)k * d]) ++valid;
            int32_t md = 0; double sc = 0;
            cudaMemcpy(&md, s->mode + r0, 4, cudaMemcpyDeviceToHost);
            cudaMemcpy(&sc, s->scale + r0, 8, cudaMemcpyDeviceToHost);
            const int da = s->da;
            fprintf(stderr, "[ns] lock %d n_act %d run %d mode %d scale %.3g it %d evals %lld lnZ %.3f lmax %.3f cube %.0f ellipsoids %.0f lnV0 %.2f valid %d/%d diagL0:",
                    lock, n_act, r0, md, sc, it0, (long long)ne, z0, lm, B[1], B[0], B[NS_BOUND_HDR + da + da * da], valid, K);
            for (int j = 0; j < da; ++j) fprintf(stderr, " %.3g", B[NS_BOUND_HDR + da + j * da + j]);
            fprintf(stderr, "\n");
        }
    }
    if (rc == NF_OK) {
        ns_finalize_kernel<<<(unsigned)((R * 32 + 127) / 128), 128, 0, st>>>(
            s->nlive, s->live_th, s->live_l, s->dead_th, s->dead_l, s->dead_lw, s->lnZ, s->H, s->n_dead, s->it,
            s->lnZ_err, s->bestfit, s->mapfit, R, d, NL, s->dead_off, s->dead_cap);
        cudaError_t e = cudaStreamSynchronize(st);
        if (e == cudaSuccess) e = cudaGetLastError();
        if (e != cudaSuccess) rc = (int)e;
        s->launches += 1;
    }
    if (prof) {
        fprintf(stderr, "[ns-prof] ncomp %d runs %lld lock-steps %d: bounds %.1f ms, propose %.1f, transform+likelihood %.1f, "
                        "update %.1f, compact %.1f; sum of steps %.1f ms\n", s->ncomp, (long long)R, lock, pms[0], pms[1],
                pms[2], pms[3], pms[4], pwall);
        fprintf(stderr, "[ns-prof]   of which %d tail steps (n_act K < 8192): bounds %.1f ms, propose %.1f, transform+likelihood %.1f, "
                        "update %.1f, compact %.1f\n", ntail, ptail[0], ptail[1], ptail[2], ptail[3], ptail[4]);
        for (int i = 0; i < 6; ++i) cudaEventDestroy(pev[i]);
    }
    s->lock_iters = lock;
    if (prev >= 0) cudaSetDevice(prev);
    return rc;
}

int nf_ns_results(const nf_sampler *s, double *lnZ, double *lnZ_err, double *max_lnL, int32_t *n_samples,
                  int32_t *n_iter, int64_t *n_evals, double *bestfit, double *mapfit)
{
    if (!s) return NF_EINVAL;
    int prev = -1;
    cudaGetDevice(&prev);
    if (cudaSetDevice(s->device) != cudaSuccess) return NF_ENODEV;
    const size_t R = (size_t)s->n_run, D = (size_t)s->ndim;
    cudaError_t e = cudaSuccess;
    auto C = [&](void *dst, const void *src, size_t n) { if (dst && e == cudaSuccess) e = cudaMemcpy(dst, src, n, cudaMemcpyDeviceToHost); };
    C(lnZ, s->lnZ, R * 8); C(lnZ_err, s->lnZ_err, R * 8); C(max_lnL, s->lmax, R * 8);
    C(n_samples, s->n_dead, R * 4); C(n_iter, s->it, R * 4); C(n_evals, s->n_eval, R * 8);
    C(bestfit, s->bestfit, R * D * 8); C(mapfit, s->mapfit, R * D * 8);
    if (prev >= 0) cudaSetDevice(prev);
    return (int)e;
}

int nf_ns_posterior(const nf_sampler *s, int64_t run, int32_t capacity, float *theta, double *lnL, double *lnw)
{
    if (!s || run < 0 || run >= s->n_run || capacity < 0) return NF_EINVAL;
    int prev = -1;
    cudaGetDevice(&prev);
    if (cudaSetDevice(s->device) != cudaSuccess) return NF_ENODEV;
    int32_t n = 0;
    cudaError_t e = cudaMemcpy(&n, s->n_dead + run, 4, cudaMemcpyDeviceToHost);
    if (n > capacity) n = capacity;
    const size_t off = (size_t)(*s->h_dead_off)[(size_t)run], D = (size_t)s->ndim;
    if (e == cudaSuccess && theta) e = cudaMemcpy(theta, s->dead_th + off * D, (size_t)n * D * 4, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess && lnL) e = cudaMemcpy(lnL, s->dead_l + off, (size_t)n * 8, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess && lnw) e = cudaMemcpy(lnw, s->dead_lw + off, (size_t)n * 8, cudaMemcpyDeviceToHost);
    if (prev >= 0) cudaSetDevice(prev);
    return (int)e;
}


int nf_ns_products_rows(nf_sampler *s, int64_t *row_offsets)
{
    if (!s || !row_offsets) return NF_EINVAL;
    int prev = -1;
    cudaGetDevice(&prev);
    if (cudaSetDevice(s->device) != cudaSuccess) return NF_ENODEV;
    const int64_t R = s->n_run;
    ns_keep_count_kernel<<<(unsigned)((R * 32 + 127) / 128), 128, 0, s->stream>>>(s->dead_l, s->dead_off, s->n_dead,
                                                                                s->keep_n, R);
    std::vector<int32_t> keep((size_t)R);
    cudaError_t e = cudaMemcpyAsync(keep.data(), s->keep_n, (size_t)R * 4, cudaMemcpyDeviceToHost, s->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s->stream);
    if (e == cudaSuccess) {
        std::vector<int64_t> &off = *s->h_post_off;
        off[0] = 0;
        for (int64_t r = 0; r < R; ++r) off[(size_t)r + 1] = off[(size_t)r] + keep[(size_t)r];
        std::memcpy(row_offsets, off.data(), ((size_t)R + 1) * sizeof(int64_t));
        e = cudaMemcpyAsync(s->post_off, off.data(), ((size_t)R + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, s->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(s->stream);
    }
    s->post_ready = e == cudaSuccess;
    s->launches += 1;
    if (prev >= 0) cudaSetDevice(prev);
    return (int)e;
}

int nf_ns_products(nf_sampler *s, const double *quantiles, int n_q, float *post, double *marginals)
{
    if (!s || n_q < 0 || n_q > 64 || (n_q > 0 && (!quantiles || !marginals))) return NF_EINVAL;
    int prev = -1;
    cudaGetDevice(&prev);
    if (cudaSetDevice(s->device) != cudaSuccess) return NF_ENODEV;
    const int64_t R = s->n_run;
    const int d = s->ndim, w = d + 2;
    const std::vector<int64_t> &off = *s->h_post_off;
    const int64_t rows = off[(size_t)R];
    cudaStream_t st = s->stream;
    float *d_post = nullptr, *d_scratch = nullptr;
    double *d_q = nullptr, *d_marg = nullptr;
    int32_t *d_list = nullptr;
    cudaError_t e = cudaSuccess;
    auto A = [&](cudaError_t x) { if (e == cudaSuccess) e = x; };
    A(ns_scratch_alloc((void **)&d_post, (size_t)(rows > 0 ? rows : 1) * w * sizeof(float), st));
    if (e == cudaSuccess) {
        ns_pack_post_kernel<<<(unsigned)((R * 32 + 127) / 128), 128, 0, st>>>(s->dead_th, s->dead_l, s->dead_lw, s->dead_off,
                                                                            s->n_dead, s->lnZ, s->post_off, d_post, R, d);
        s->launches += 1;
    }
    if (e == cudaSuccess && n_q > 0) {
        // runs whose column fits in shared memory (<= 32768 rows) and the others (sorted in global scratch)
        const int SMEM_ROWS = 32768;
        std::vector<int32_t> small, big;
        int big_np2 = 0, small_np2 = 1;
        for (int64_t r = 0; r < R; ++r) {
            const int64_t n = off[(size_t)r + 1] - off[(size_t)r];
            int np2 = 1;
            while (np2 < n) np2 <<= 1;
            if (n <= SMEM_ROWS) { small.push_back((int32_t)r); small_np2 = np2 > small_np2 ? np2 : small_np2; }
            else { big.push_back((int32_t)r); big_np2 = np2 > big_np2 ? np2 : big_np2; }
        }
        A(ns_scratch_alloc((void **)&d_q, (size_t)n_q * sizeof(double), st));
        A(ns_scratch_alloc((void **)&d_marg, (size_t)R * n_q * d * sizeof(double), st));
        A(ns_scratch_alloc((void **)&d_list, (size_t)R * sizeof(int32_t), st));
        A(cudaMemcpyAsync(d_q, quantiles, (size_t)n_q * sizeof(double), cudaMemcpyHostToDevice, st));
        if (e == cudaSuccess && !small.empty()) {
            const size_t smem = (size_t)small_np2 * sizeof(float);
            A(nf_ensure_dyn_smem((const void *)ns_marginals_kernel, smem));
            A(cudaMemcpyAsync(d_list, small.data(), small.size() * sizeof(int32_t), cudaMemcpyHostToDevice, st));
            if (e == cudaSuccess)
                ns_marginals_kernel<<<(unsigned)(small.size() * d), 512, smem, st>>>(d_post, s->post_off, d_list, (int)small.size(), d,
                                                                                     d_q, n_q, d_marg, nullptr, 0);
            A(cudaStreamSynchronize(st));          // `small` must outlive the copy
            s->launches += 1;
        }
        // bounded scratch: the long runs go through in batches
        for (size_t b0 = 0; e == cudaSuccess && b0 < big.size();) {
            const size_t per = (size_t)big_np2 * d * sizeof(float);
            size_t nb = (size_t)(1ull << 31) / per;
            if (nb < 1) nb = 1;
            if (nb > big.size() - b0) nb = big.size() - b0;
            A(ns_scratch_alloc((void **)&d_scratch, nb * per, st));
            A(cudaMemcpyAsync(d_list, big.data() + b0, nb * sizeof(int32_t), cudaMemcpyHostToDevice, st));
            if (e == cudaSuccess)
                ns_marginals_kernel<<<(unsigned)(nb * d), 512, 0, st>>>(d_post, s->post_off, d_list, (int)nb, d, d_q, n_q,
                                                                       d_marg, d_scratch, big_np2);
            A(cudaStreamSynchronize(st));
            ns_scratch_free(d_scratch, st);
            d_scratch = nullptr;
            s->launches += 1;
            b0 += nb;
        }
        A(cudaMemcpyAsync(marginals, d_marg, (size_t)R * n_q * d * sizeof(double), cudaMemcpyDeviceToHost, st));
    }
    if (e == cudaSuccess && post && rows > 0)
        A(cudaMemcpyAsync(post, d_post, (size_t)rows * w * sizeof(float), cudaMemcpyDeviceToHost, st));
    A(cudaStreamSynchronize(st));
    if (e == cudaSuccess) e = cudaGetLastError();
    ns_scratch_free(d_post, st);
    ns_scratch_free(d_q, st);
    ns_scratch_free(d_marg, st);
    ns_scratch_free(d_list, st);
    cudaStreamSynchronize(st);
    if (prev >= 0) cudaSetDevice(prev);
    return (int)e;
}

int nf_ns_intensity(nf_sampler *s, const double *quantiles, int n_q, double *peak_q, double *integ_q)
{
    if (!s || !s->post_ready || n_q < 1 || n_q > 64 || !quantiles) return NF_EINVAL;
    const nf_pixels *px = s->px;
    if (px->model != NF_MODEL_NH3 && px->model != NF_MODEL_N2HP) return NF_EINVAL;
    int prev = -1;
    cudaGetDevice(&prev);
    if (cudaSetDevice(s->device) != cudaSuccess) return NF_ENODEV;
    const int64_t R = s->n_run;
    const int d = s->ndim, ncomp = s->ncomp, nm = d / ncomp, n_spec = px->n_spec;
    const std::vector<int64_t> &off = *s->h_post_off;
    cudaStream_t st = s->stream;
    // runs go through in groups of contiguous rows whose vectors fit the scratch (a run larger than that alone):
    // 2^23 vectors, about 0.4 GB of scratch at ncomp x 6 parameters and two spectra
    int64_t max_rows = 0;
    for (int64_t r = 0; r < R; ++r) max_rows = std::max(max_rows, off[(size_t)r + 1] - off[(size_t)r]);
    const int64_t cap_vec = std::max((int64_t)1 << 23, max_rows * ncomp);
    const int64_t cap_rows = cap_vec / ncomp;
    const size_t out_n = (size_t)R * n_q * n_spec * ncomp;
    float *d_vec = nullptr, *d_peak = nullptr, *d_wt = nullptr;
    double *d_sum = nullptr, *d_q = nullptr, *d_pq = nullptr, *d_iq = nullptr, *d_scratch = nullptr;
    int32_t *d_vpix = nullptr, *d_list = nullptr;
    cudaError_t e = cudaSuccess;
    auto A = [&](cudaError_t x) { if (e == cudaSuccess) e = x; };
    A(ns_scratch_alloc((void **)&d_vec, (size_t)cap_vec * nm * sizeof(float), st));
    A(ns_scratch_alloc((void **)&d_vpix, (size_t)cap_vec * sizeof(int32_t), st));
    A(ns_scratch_alloc((void **)&d_peak, (size_t)cap_vec * n_spec * sizeof(float), st));
    A(ns_scratch_alloc((void **)&d_sum, (size_t)cap_vec * n_spec * sizeof(double), st));
    A(ns_scratch_alloc((void **)&d_wt, (size_t)cap_rows * sizeof(float), st));
    A(ns_scratch_alloc((void **)&d_q, (size_t)n_q * sizeof(double), st));
    A(ns_scratch_alloc((void **)&d_pq, out_n * sizeof(double), st));
    A(ns_scratch_alloc((void **)&d_iq, out_n * sizeof(double), st));
    A(ns_scratch_alloc((void **)&d_list, (size_t)R * sizeof(int32_t), st));
    A(cudaMemcpyAsync(d_q, quantiles, (size_t)n_q * sizeof(double), cudaMemcpyHostToDevice, st));
    // moments of single-component vectors: the model kernel's moments mode, the block's axes and flags
    NfLikeArgs a;
    std::memset(&a, 0, sizeof(a));
    a.inv2s2 = px->inv2s2; a.params = d_vec; a.pix_of_vec = d_vpix; a.vecs_per_pix = 1;
    a.pix_stride = (int64_t)n_spec * px->n_pad; a.param_f64 = 0; a.ncomp = 1;
    a.n_spec = n_spec; a.n_chan = px->n_chan; a.n_pad = px->n_pad;
    a.cold = (s->flags & NF_FLAG_COLD) != 0; a.lte = (s->flags & NF_FLAG_LTE) != 0;
    for (int k = 0; k < n_spec; ++k) a.spec[k] = px->spec[k];
    a.pixmeta = px->pixmeta; a.mom_peak = d_peak; a.mom_sum = d_sum;
    const int SMEM_ROWS = 8192;                    // 16-byte entries (value, {weight, row}): at most 128 KB of shared memory
    static_assert(8192 <= (1 << 14), "size classes 0..14 cover the shared-memory runs");
    const int per_run = n_spec * ncomp * 2;
    // the run lists of every group, in one host array that outlives all the copies from it: group [r0, r1) uses
    // entries [r0, r1) here and in d_list, so no group waits for the one before
    std::vector<int32_t> h_list((size_t)R), big;
    for (int64_t r0 = 0; e == cudaSuccess && r0 < R;) {
        int64_t r1 = r0 + 1;
        while (r1 < R && off[(size_t)r1 + 1] - off[(size_t)r0] <= cap_rows) ++r1;
        const int64_t rows = off[(size_t)r1] - off[(size_t)r0], n_r = r1 - r0;
        if (rows > 0) {
            ns_int_gather_kernel<<<(unsigned)((n_r * 32 + 127) / 128), 128, 0, st>>>(
                s->dead_th, s->dead_l, s->dead_lw, s->dead_off, s->n_dead, s->lnZ, s->post_off, s->pix_ids, r0, n_r, d,
                ncomp, d_vec, d_vpix, d_wt);
            A(cudaGetLastError());
            a.B = rows * ncomp;
            if (e == cudaSuccess) A(px->model == NF_MODEL_NH3 ? nf_launch_nh3(a, st) : nf_launch_n2hp(a, st));
            s->launches += 2;
        }
        // runs that fit shared memory go through one launch per power-of-two size class, each with the shared
        // memory of its class (a long run does not lower the occupancy of the short ones); the others are sorted in
        // global scratch
        big.clear();
        std::vector<int32_t> cls_n(15, 0);              // runs per class, class k: np2 = 2^k <= SMEM_ROWS
        std::vector<int> run_cls((size_t)(r1 - r0), -1);
        int big_np2 = 1;
        for (int64_t r = r0; r < r1; ++r) {
            const int64_t n = off[(size_t)r + 1] - off[(size_t)r];
            int k = 0;
            while ((int64_t)1 << k < n) ++k;
            if (n <= SMEM_ROWS) { run_cls[(size_t)(r - r0)] = k; ++cls_n[(size_t)k]; }
            else { big.push_back((int32_t)r); big_np2 = std::max(big_np2, 1 << k); }
        }
        std::vector<int32_t> cls_off(16, 0);
        for (int k = 0; k < 15; ++k) cls_off[(size_t)k + 1] = cls_off[(size_t)k] + cls_n[(size_t)k];
        int32_t *small = h_list.data() + r0, *d_small = d_list + r0;
        const int32_t n_small = cls_off[15];
        {
            std::vector<int32_t> at(cls_off.begin(), cls_off.end() - 1);
            for (int64_t r = r0; r < r1; ++r) {
                const int k = run_cls[(size_t)(r - r0)];
                if (k >= 0) small[at[(size_t)k]++] = (int32_t)r;
            }
        }
        if (e == cudaSuccess && n_small > 0) {
            A(cudaMemcpyAsync(d_small, small, (size_t)n_small * sizeof(int32_t), cudaMemcpyHostToDevice, st));
            for (int k = 0; k < 15 && e == cudaSuccess; ++k) {
                const int nk = cls_n[(size_t)k];
                if (nk == 0) continue;
                const size_t smem = ((size_t)1 << k) * 2 * sizeof(double);
                A(nf_ensure_dyn_smem((const void *)ns_wquant_kernel, smem));
                if (e == cudaSuccess)
                    ns_wquant_kernel<<<(unsigned)((int64_t)nk * per_run), 512, smem, st>>>(
                        d_peak, d_sum, d_wt, s->post_off, off[(size_t)r0], d_small + cls_off[(size_t)k], nk, n_spec,
                        ncomp, d_q, n_q, d_pq, d_iq, nullptr, 0);
                A(cudaGetLastError());
                s->launches += 1;
            }
        }
        // bounded scratch: the long runs go through in batches
        for (size_t b0 = 0; e == cudaSuccess && b0 < big.size();) {
            const size_t per = (size_t)big_np2 * 2 * sizeof(double) * per_run;
            size_t nb = (size_t)(1ull << 31) / per;
            if (nb < 1) nb = 1;
            if (nb > big.size() - b0) nb = big.size() - b0;
            A(ns_scratch_alloc((void **)&d_scratch, nb * per, st));
            std::copy(big.begin() + b0, big.begin() + b0 + nb, h_list.begin() + r0 + n_small + b0);
            A(cudaMemcpyAsync(d_small + n_small + b0, small + n_small + b0, nb * sizeof(int32_t),
                              cudaMemcpyHostToDevice, st));
            if (e == cudaSuccess)
                ns_wquant_kernel<<<(unsigned)(nb * per_run), 512, 0, st>>>(
                    d_peak, d_sum, d_wt, s->post_off, off[(size_t)r0], d_small + n_small + b0, (int)nb, n_spec, ncomp,
                    d_q, n_q, d_pq, d_iq, d_scratch, big_np2);
            A(cudaGetLastError());
            A(cudaStreamSynchronize(st));
            ns_scratch_free(d_scratch, st);
            d_scratch = nullptr;
            s->launches += 1;
            b0 += nb;
        }
        r0 = r1;
    }
    if (peak_q) A(cudaMemcpyAsync(peak_q, d_pq, out_n * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (integ_q) A(cudaMemcpyAsync(integ_q, d_iq, out_n * sizeof(double), cudaMemcpyDeviceToHost, st));
    A(cudaStreamSynchronize(st));
    for (void *p : {(void *)d_vec, (void *)d_vpix, (void *)d_peak, (void *)d_sum, (void *)d_wt, (void *)d_q,
                    (void *)d_pq, (void *)d_iq, (void *)d_list})
        ns_scratch_free(p, st);
    cudaStreamSynchronize(st);
    if (prev >= 0) cudaSetDevice(prev);
    return (int)e;
}

int nf_ns_stats(const nf_sampler *s, int32_t *lock_iters, int64_t *launches)
{
    if (!s) return NF_EINVAL;
    if (lock_iters) *lock_iters = s->lock_iters;
    if (launches) *launches = s->launches;
    return NF_OK;
}

}  // extern "C"
