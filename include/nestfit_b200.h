/*
 * nestfit_b200.h -- C ABI of the B200-native NestFit likelihood hot path.
 *
 * Plain C, pointers and sizes only; no torch / CUDA types in any signature
 * (streams are passed as `void*` holding a cudaStream_t, 0 = default stream).
 * Every entry point returns an int status: 0 = NF_OK, negative = NF_E*, positive
 * = a cudaError_t.  No exceptions cross the boundary.  NaN parameters give NaN
 * (or null-model) log-likelihoods exactly like the reference's `void` callbacks.
 *
 * Reference interfaces replaced (paths relative to the reference tree):
 *   - `Runner.c_loglikelihood(double *utheta, double *lnL)`  nestfit/core/core.pxd:72,
 *     `AmmoniaRunner.c_loglikelihood`                        nestfit/models/ammonia.pyx:423-432
 *       -> nf_prior_transform + nf_nh3_loglike (batched: B vectors per call)
 *   - `amm_predict` / `AmmoniaRunner.predict`                nestfit/models/ammonia.pyx:364-366,437-447
 *       -> nf_nh3_predict
 *   - `gauss_predict` / `GaussianRunner.c_loglikelihood`     nestfit/models/gaussian.pyx:53-54,98-102
 *       -> nf_gauss_predict / nf_gauss_loglike
 *   - `nnhp_predict` / `DiazenyliumRunner.c_loglikelihood`   nestfit/models/diazenylium.pyx:140-158,206-215
 *       -> nf_n2hp_predict / nf_n2hp_loglike
 *   - `AmmoniaSpectrum.__init__`, `Spectrum.__init__`        nestfit/models/ammonia.pyx:245-277, nestfit/core/core.pyx:488-520
 *       -> nf_pixels_create (+ nf_pixels_null_lnz); spectra on their own axes and lengths
 *          (one Runner each, run_multinest per Runner) -> nf_pixels_create_axes
 *   - `PriorTransformer.c_transform`                         nestfit/core/core.pyx:459-476
 *       -> nf_priors_create + nf_prior_transform
 *   - MultiNest `run(...)` + `LogLike`/`dumper` callbacks    nestfit/core/cmultinest.pxd:5-33,
 *     `run_multinest`, `mn_dump`                             nestfit/core/core.pyx:627-823
 *       -> nf_ns_* (batched lock-step nested sampling over a block of pixels)
 *
 * Layouts: parameter vectors are parameter-major / component-minor,
 * `[p0c0,p0c1,..,p1c0,..]` (ammonia.pyx:337-343); NH3 order voff,trot,tex,ntot,
 * sigm,orth; Gaussian order voff,sigm,peak (gaussian.pyx:27-30); N2H+ order
 * voff,tex,ltau,sigm (diazenylium.pyx:148-153).
 */
#ifndef NESTFIT_B200_H
#define NESTFIT_B200_H

#include <stdint.h>
#include "nf_priors.h"

#ifdef __cplusplus
extern "C" {
#endif

#define NF_ABI_VERSION 2

enum {
    NF_OK = 0,
    NF_EINVAL = -1,   /* bad argument (size, NULL, unsupported configuration) */
    NF_ENOMEM = -2,   /* host allocation failed                               */
    NF_ENODEV = -3    /* no usable CUDA device                                */
};

enum { NF_MODEL_NH3 = 1, NF_MODEL_GAUSS = 2, NF_MODEL_N2HP = 3 };
enum { NF_F32 = 0, NF_F64 = 1 };
/* flags of the NH3 model (ammonia.pyx:344-347) */
enum { NF_FLAG_COLD = 1, NF_FLAG_LTE = 2 };

#define NF_MAX_SPEC 6       /* spectra (transitions) scored together per pixel */
#define NF_MAX_NCOMP_NH3 4  /* velocity components of the fused NH3 kernel      */
#define NF_MAX_NCOMP_GAUSS 32
/* Widest spectrum the hyperfine models (NH3, N2H+) accept, as (nu_last - nu_first) / nu_first (about 240 km/s).
 * Their kernel makes the brightness amplitude T0 (G(T0/tex) - tbg) linear in the channel; the error of that grows
 * with the square of the band, and up to this width it stays inside 1e-5 of a spectrum's peak for tex down to
 * 2.8 K.  The pixel-block constructors return NF_EINVAL for a wider hyperfine spectrum. */
#define NF_MAX_BAND_FRAC 8e-4

typedef struct nf_pixels nf_pixels; /* opaque: a block of pixels resident in HBM */
typedef struct nf_priors nf_priors; /* opaque: a prior plan resident in HBM      */
typedef struct nf_sampler nf_sampler; /* opaque: batched nested-sampling state   */

int nf_abi_version(void);
const char *nf_error_string(int code);
int nf_device_count(int *count);

/* ---- pixel blocks ------------------------------------------------------- */
/*
 * Upload a block of `n_pix` pixels, each with `n_spec` spectra of `n_chan`
 * channels on uniform ascending frequency axes x_j = nu_min[s] + j*nu_chan[s]
 * (Spectrum.__init__, core.pyx:503-514).  `data` is host memory
 * [n_pix][n_spec][n_chan] of `dtype` (NF_F32 / NF_F64), `noise` host
 * [n_pix][n_spec] (one scalar rms per spectrum, core.pyx:507).
 * model == NF_MODEL_NH3: `trans_id[s]` in 1..9 selects the (J,K) inversion
 * transition (ammonia.pyx:245-271), `rest_freq` ignored.
 * model == NF_MODEL_GAUSS: n_spec must be 1 and `rest_freq[0]` is the line rest
 * frequency in Hz (gaussian.pyx:31-32).
 * model == NF_MODEL_N2HP: `trans_id[s]` in 1..3 selects J = 1-0, 2-1, 3-2
 * (diazenylium.pyx:105-138), `rest_freq` ignored.
 * Data are stored as FP32 in HBM, channel-contiguous, rows padded to 32.
 */
int nf_pixels_create(int device, int model, int64_t n_pix, int n_spec, int n_chan,
                     const double *nu_min, const double *nu_chan,
                     const int *trans_id, const double *rest_freq,
                     const void *data, int dtype, const double *noise,
                     nf_pixels **out);
/* Same, but `data_dev` (FP32 [n_pix][n_spec][n_chan]) and `noise_dev`
 * (FP64 [n_pix][n_spec]) already live on `device`; they are copied. */
int nf_pixels_create_from_device(int device, int model, int64_t n_pix, int n_spec,
                                 int n_chan, const double *nu_min,
                                 const double *nu_chan, const int *trans_id,
                                 const double *rest_freq, const float *data_dev,
                                 const double *noise_dev, nf_pixels **out);
/* Same, but every (pixel, spectrum) has its own uniform ascending axis
 * x_j = nu_min[p][s] + j*nu_chan[p][s] and its own channel count
 * 2 <= n_chan[p][s] <= n_chan_max <= 65535: a catalogue of pointed
 * observations, or spectra cut from cubes with different set-ups.  `data` is
 * [n_pix][n_spec][n_chan_max]; channels past a spectrum's own n_chan are
 * stored as zero whatever the caller passed there.  The transitions
 * `trans_id[n_spec]` are shared by all pixels; the Gaussian model (n_spec = 1)
 * takes one `rest_freq[n_pix]` per pixel.  The *_loglike[_host] entry points
 * work unchanged on such a block; predictions need a pixel per vector and go
 * through nf_predict_pix[_host] (the *_predict[_host] calls return NF_EINVAL). */
int nf_pixels_create_axes(int device, int model, int64_t n_pix, int n_spec, int n_chan_max,
                          const double *nu_min, const double *nu_chan, const int *n_chan,
                          const int *trans_id, const double *rest_freq,
                          const void *data, int dtype, const double *noise, nf_pixels **out);
int nf_pixels_free(nf_pixels *px);
/* null-model evidence per pixel, -sum_s sum_j d^2/(2 sigma_s^2)
 * (core.pyx:518-520, ammonia.pyx:411-415) -> host double[n_pix]. */
int nf_pixels_null_lnz(const nf_pixels *px, double *out_host);

/* ---- likelihood / prediction: device-pointer entry points --------------- */
/*
 * Score B parameter vectors.  `params_dev` is [B][n_model*ncomp] of
 * `param_dtype` in physical units.  Vector b belongs to pixel
 * pix_of_vec_dev[b] (int32, device) or, when that is NULL, to pixel
 * b / vecs_per_pix.  Vectors of one pixel should be contiguous (the pixel's
 * spectra are then staged once per CTA in shared memory); any order is correct.
 * `lnL_dev` receives B doubles:  -sum (d-m)^2 / (2 sigma^2)  (core.pyx:522-530).
 * Asynchronous on `stream`.
 */
int nf_nh3_loglike(const nf_pixels *px, const void *params_dev, int param_dtype,
                   const int32_t *pix_of_vec_dev, int64_t vecs_per_pix, int64_t B,
                   int ncomp, int flags, double *lnL_dev, void *stream);
/* Model spectra only: pred_dev [B][n_spec][n_chan] FP32 (ammonia.pyx:437-447).
 * `px` supplies the axes/transitions; its data are not read. */
int nf_nh3_predict(const nf_pixels *px, const void *params_dev, int param_dtype,
                   int64_t B, int ncomp, int flags, float *pred_dev, void *stream);
int nf_gauss_loglike(const nf_pixels *px, const void *params_dev, int param_dtype,
                     const int32_t *pix_of_vec_dev, int64_t vecs_per_pix, int64_t B,
                     int ncomp, double *lnL_dev, void *stream);
/* N2H+: params [B][4*ncomp] = voff, tex, log10(tau_main), sigm (diazenylium.pyx:140-154) */
int nf_n2hp_loglike(const nf_pixels *px, const void *params_dev, int param_dtype,
                    const int32_t *pix_of_vec_dev, int64_t vecs_per_pix, int64_t B,
                    int ncomp, double *lnL_dev, void *stream);
int nf_n2hp_predict(const nf_pixels *px, const void *params_dev, int param_dtype,
                    int64_t B, int ncomp, float *pred_dev, void *stream);
int nf_gauss_predict(const nf_pixels *px, const void *params_dev, int param_dtype,
                     int64_t B, int ncomp, float *pred_dev, void *stream);
/* Model spectra of any block's model, vector b on the axes of pixel
 * pix_of_vec_dev[b] (required): pred_dev [B][n_spec][n_chan] FP32, n_chan
 * being the block's longest spectrum; channels past a spectrum's own length
 * are 0.  `flags` as for NH3 (ignored by the other models). */
int nf_predict_pix(const nf_pixels *px, const void *params_dev, int param_dtype,
                   const int32_t *pix_of_vec_dev, int64_t B, int ncomp, int flags,
                   float *pred_dev, void *stream);
/* Moments of single-component model spectra (hyperfine models only; NF_EINVAL
 * for the Gaussian model): `params_dev` [B][n_model] of `param_dtype`; vector b
 * is synthesised exactly as the *_predict calls do, on the axes of pixel
 * pix_of_vec_dev[b] (required on a block with per-pixel axes, may be NULL on a
 * shared-axis block), and reduced over the spectrum's own channels to
 * peak_dev [B][n_spec] FP32 = its maximum (K) and sum_dev [B][n_spec] FP64 =
 * its sum (K channel, accumulated in FP64).  No model row is written.  `flags`
 * as for NH3 (ignored by N2H+). */
int nf_predict_moments(const nf_pixels *px, const void *params_dev, int param_dtype,
                       const int32_t *pix_of_vec_dev, int64_t B, int flags,
                       float *peak_dev, double *sum_dev, void *stream);

/* ---- host-buffer entry points (the call a reference-side binding makes) -- */
/* params_host [B][ndim] of param_dtype, pix_of_vec_host may be NULL (then
 * vecs_per_pix is used), lnL_host double[B].  Copies are pipelined with the
 * kernel over internal streams; the call returns when lnL_host is complete.
 * Page-locked (cudaHostAlloc / cudaHostRegister) buffers are copied from and
 * into directly; pageable ones (plain numpy arrays) are bounced through a
 * page-locked ring owned by the block, so they are safe to pass and cost one
 * extra host copy that overlaps the kernel. */
int nf_nh3_loglike_host(const nf_pixels *px, const void *params_host, int param_dtype,
                        const int32_t *pix_of_vec_host, int64_t vecs_per_pix,
                        int64_t B, int ncomp, int flags, double *lnL_host);
int nf_gauss_loglike_host(const nf_pixels *px, const void *params_host, int param_dtype,
                          const int32_t *pix_of_vec_host, int64_t vecs_per_pix,
                          int64_t B, int ncomp, double *lnL_host);
int nf_nh3_predict_host(const nf_pixels *px, const void *params_host, int param_dtype,
                        int64_t B, int ncomp, int flags, float *pred_host);
int nf_gauss_predict_host(const nf_pixels *px, const void *params_host, int param_dtype,
                          int64_t B, int ncomp, float *pred_host);
int nf_n2hp_loglike_host(const nf_pixels *px, const void *params_host, int param_dtype,
                         const int32_t *pix_of_vec_host, int64_t vecs_per_pix,
                         int64_t B, int ncomp, double *lnL_host);
int nf_n2hp_predict_host(const nf_pixels *px, const void *params_host, int param_dtype,
                         int64_t B, int ncomp, float *pred_host);
int nf_predict_pix_host(const nf_pixels *px, const void *params_host, int param_dtype,
                        const int32_t *pix_of_vec_host, int64_t B, int ncomp, int flags,
                        float *pred_host);
int nf_predict_moments_host(const nf_pixels *px, const void *params_host, int param_dtype,
                            const int32_t *pix_of_vec_host, int64_t B, int flags,
                            float *peak_host, double *sum_host);

/* ---- prior transform ---------------------------------------------------- */
int nf_priors_create(int device, const nf_prior_desc *priors, int n_prior,
                     const nf_dist_desc *dists, int n_dist, const double *tables,
                     int64_t n_tables, int n_model, nf_priors **out);
int nf_priors_free(nf_priors *pr);
/* In place, unit cube -> physical: u_dev [B][n_model*ncomp] doubles. */
int nf_prior_transform(const nf_priors *pr, double *u_dev, int64_t B, int ncomp,
                       void *stream);
int nf_prior_transform_host(const nf_priors *pr, double *u_host, int64_t B, int ncomp);

/* ---- batched nested sampling (replaces the per-pixel MultiNest loop) ------ */
/*
 * MultiNest's `run(IS, mmodal, ceff, nlive, tol, efr, ndims, nPar, ..., LogLike,
 * dumper, context)` (cmultinest.pxd:5-33) fits ONE pixel per call through a C
 * callback.  nf_ns_* fits a block of "runs" (pixel, ncomp) in lock-step: every
 * iteration draws `n_prop` proposals per in-flight run from the constrained
 * prior, maps them through the device prior transform and scores all of them
 * with one launch of the fused likelihood kernel.  The knobs keep MultiNest's
 * names and meaning where they exist (run_multinest, core.pyx:727-732).
 */
typedef struct nf_ns_config {
    int32_t nlive_max;   /* capacity of the live set; per-run nlive <= nlive_max       */
    int32_t n_prop;      /* proposals per run per lock-step iteration (K)              */
    int32_t max_iter;    /* `maxiter`: cap on nested-sampling iterations per run       */
    int32_t max_samples; /* capacity of the posterior sample (dead + final live pts)   */
    int32_t bound_update_interval; /* `walks`: random-walk steps per new point (<=1: 20 + active dims) */
    int32_t flags;       /* bits 0-1: 0 auto: ellipsoidal rejection, random walk once it stalls;
                            1 random walk from the start; 2 ellipsoidal rejection only.
                            bit 2 (4): keep the dimensions the priors overwrite (ConstantPrior rows,
                            DuplicatePrior's second row) inside the bounding ellipsoid / walk metric
                            instead of drawing them uniformly on their own;
                            bit 3 (8): ONE bounding ellipsoid instead of the MultiNest-style
                            decomposition into up to 8 (`mmodal`, core.pyx:727-732)          */
    double tol;          /* `tol`: stop when ln(Z + Lmax X) - ln Z < tol               */
    double efr;          /* `efr`: target sampling efficiency (ellipsoid enlargement)  */
    uint64_t seed;       /* counter-based RNG seed: results are reproducible           */
    int32_t n_prop_max;  /* most proposals a run may get per lock-step once few runs remain
                            (rounded down to a multiple of n_prop; <= n_prop: fixed K)       */
    int32_t target_batch; /* vectors per likelihood launch aimed at in that regime (0: 65536) */
} nf_ns_config;

/* pix_ids[n_run], nlive[n_run] are host arrays (nlive per run: main.py:445-447).
 * `model_flags` = NF_FLAG_COLD | NF_FLAG_LTE for the NH3 model. */
int nf_ns_create(const nf_pixels *px, const nf_priors *pr, int ncomp, int model_flags,
                 const nf_ns_config *cfg, int64_t n_run, const int32_t *pix_ids,
                 const int32_t *nlive, nf_sampler **out);
int nf_ns_run(nf_sampler *s);
int nf_ns_free(nf_sampler *s);
/* What the reference's dumper receives per run (core.pyx:627-687): ln Z
 * (`global_lnZ`), its error sqrt(H/nlive), max log-likelihood, number of posterior
 * samples, plus iteration / likelihood-evaluation counts; bestfit = maximum-
 * likelihood sample, mapfit = sample of largest posterior weight.  All host arrays
 * of n_run (x ndim) entries; any may be NULL. */
int nf_ns_results(const nf_sampler *s, double *lnZ, double *lnZ_err, double *max_lnL,
                  int32_t *n_samples, int32_t *n_iter, int64_t *n_evals,
                  double *bestfit, double *mapfit);
/* Posterior sample of one run: theta [n][ndim] FP32 (the reference stores the
 * posterior as float32, core.pyx:680), lnL [n], ln prior-mass weight lnw [n];
 * posterior weight p_i = exp(lnL_i + lnw_i - lnZ).  n = min(n_samples, capacity). */
int nf_ns_posterior(const nf_sampler *s, int64_t run, int32_t capacity, float *theta,
                    double *lnL, double *lnw);
/* Posterior products of ALL runs in two calls (what the reference's dumper writes per run,
 * core.pyx:645-687), replacing one nf_ns_posterior round trip per run:
 *   nf_ns_products_rows: row_offsets[n_run + 1] (host) -- run r owns rows [off[r], off[r+1]) of the pool:
 *     its dead points and final live points in death order, logZero points (lnL = -inf) dropped;
 *   nf_ns_products: `post` (host, may be pageable) receives the float32 pool [rows][ndim + 2] laid out like
 *     the reference's `posteriors` dataset (theta, lnL, posterior weight; core.pyx:680) with one device-to-host
 *     copy; `marginals` [n_run][n_q][ndim] = numpy.quantile(theta columns, quantiles) -- unweighted, linear
 *     interpolation, like Dumper.calc_marginals (core.pyx:596-598) -- sorted on the device.  Either may be NULL. */
int nf_ns_products_rows(nf_sampler *s, int64_t *row_offsets);
int nf_ns_products(nf_sampler *s, const double *quantiles, int n_q, float *post, double *marginals);
/* Credible intervals of each component's peak and integrated intensity (hyperfine models; NF_EINVAL for the
 * Gaussian model and before nf_ns_products_rows).  Every posterior row of every run (the rows
 * nf_ns_products_rows counts) is split into its `ncomp` single-component vectors, which are synthesised on the
 * run's pixel as nf_predict_moments does; then, per (run, spectrum, component), the posterior-weighted quantiles
 * of the peak (K) and of the channel sum (K channel), with the float32 weights of the `posteriors` rows and the
 * rule of numpy.interp(q, cumsum(w_sorted) / sum(w), x_sorted).  peak_q, integ_q: host
 * [n_run][n_q][n_spec][ncomp] FP64; either may be NULL. */
int nf_ns_intensity(nf_sampler *s, const double *quantiles, int n_q, double *peak_q, double *integ_q);
int nf_ns_stats(const nf_sampler *s, int32_t *lock_iters, int64_t *launches);

/* ---- kernel timing helper (bench / roofline) ---------------------------- */
/* Milliseconds the last *_host call spent in kernels only (CUDA events on the
 * launching streams), and how many kernels it launched. */
int nf_last_call_stats(double *kernel_ms, int64_t *n_launches);

/* Measured roofline denominators on `device`: MUFU.EX2 results per second
 * (Gop/s) and FP32 FMA rate (GFLOP/s, 2 flop per FMA), register-resident loops. */
int nf_measure_peaks(int device, double *mufu_gops, double *ffma_gflops);

#ifdef __cplusplus
}
#endif
#endif /* NESTFIT_B200_H */
