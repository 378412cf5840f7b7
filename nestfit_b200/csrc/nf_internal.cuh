// Internal declarations shared by the translation units of libnestfit_b200.so.
#pragma once

#include <cstdint>
#include <mutex>
#include <cuda_runtime.h>

#include "../../include/nestfit_b200.h"

// Physical constants as compiled into the reference
// (includes/model_includes.pxi:27-36, nestfit/models/ammonia.pyx:15-18).
#define NF_CKMS 299792.458
#define NF_CCMS 29979245800.0
#define NF_H 6.62607015e-27
#define NF_KB 1.380649e-16
#define NF_TCMB 2.72548
#define NF_BROT 298192.92e6
#define NF_CROT 186695.86e6
#define NF_FWHM 2.3548200450309493

#define NF_WARPS_PER_CTA 8
#define NF_THREADS (NF_WARPS_PER_CTA * 32)
#define NF_TILE_VECS 64          // parameter vectors per CTA tile
#define NF_IEM_SIZE 1000         // 1/(e^x-1) table, nestfit/models/hyperfine.pyx:12

// Per-spectrum constants prepared on the host in FP64.
struct NfSpecMeta {
    double nu_min;      // x_0 [Hz]                       core.pyx:513
    double nu_chan;     // x_1 - x_0 [Hz]                 core.pyx:503
    double inv_chan;    // 1 / nu_chan
    double nu0;         // rest frequency [Hz]
    double fracterm;    // c^2 A / (8 pi nu0^2)           ammonia.pyx:358
    double width_c;     // c_kms / (nu0 sqrt(2 pi))       ammonia.pyx:359 (divided by sigma on device)
    double hnu_k;       // h nu0 / k_B                    ammonia.pyx:355
    double T0_first;    // h x_0 / k_B                    hyperfine.pyx:106
    double T0_last;     // h x_{N-1} / k_B
    double tbg0, tbg1;  // 1/expm1(T0_j/Tcmb) ~= tbg0 + tbg1*j   ammonia.pyx:273-277
    float t0a, t0b;     // T0_j = t0a + t0b*j
    int line_off;       // first line in the global line tables
    int nlines;         // hyperfine lines of this transition
    int J;              // rotational level J (=K), 1..9
    int para;           // para (K % 3 != 0) or ortho
};

// One (pixel, spectrum) of a block whose pixels have their own axes: the spectrum's constants and its own channel
// count (rows are zero past it up to the block's n_chan).
struct NfPixSpecMeta {
    NfSpecMeta m;
    int n_chan;
    int pad_;
};

#define NF_HOST_SLOTS 3         // chunks in flight in a host-buffer call (ring of streams and staging buffers)

struct nf_pixels {
    int device;
    int model;
    int64_t n_pix;
    int n_spec, n_chan, n_pad;      // n_pad: channels per row in HBM (multiple of 64)
    float *data;                    // [n_pix][n_spec][n_pad]
    double *inv2s2;                 // [n_pix][n_spec]  1/(2 sigma^2)
    double *null_lnz;               // [n_pix]
    float *d2chunk;                 // [n_pix][n_spec][n_pad/32]  sum of d^2 over each 32-channel chunk
    NfSpecMeta spec[NF_MAX_SPEC];   // per-pixel axes: pixel 0's (the transitions are shared by all pixels)
    NfPixSpecMeta *pixmeta;         // [n_pix][n_spec] on the device when every pixel has its own axes, else NULL
    // pipelined host-call resources (one host-buffer call at a time per block: guarded by host_mu)
    std::mutex *host_mu;
    cudaStream_t streams[NF_HOST_SLOTS];
    void *stage_dev[NF_HOST_SLOTS];
    void *stage_host[NF_HOST_SLOTS];            // page-locked twins of stage_dev, allocated on the first call with pageable buffers
    size_t stage_bytes, stage_host_bytes;
};

struct nf_priors {
    int device;
    int n_prior, n_dist, n_model;
    int max_stride;
    int64_t n_tables;
    nf_prior_desc *priors;   // device
    nf_dist_desc *dists;     // device
    double *tables;          // device
    nf_prior_desc *h_priors; // host copies (validation)
    nf_dist_desc *h_dists;
};

struct NfLikeArgs {
    const float *data;          // may be NULL (predict only)
    const double *inv2s2;
    const float *d2chunk;       // per pixel, spectrum and 32-channel chunk: sum of d^2 (Gaussian-model kernel)
    const void *params;
    const int32_t *pix_of_vec;  // may be NULL
    int64_t vecs_per_pix;
    int64_t B;
    const int32_t *B_dev;       // optional: device-resident vector count (<= B, which then only sizes the grid)
    int64_t pix_stride;         // floats per pixel = n_spec * n_pad
    double *lnL;                // may be NULL
    float *pred;                // may be NULL: [B][n_spec][n_chan]
    int param_f64;
    int ncomp, n_spec, n_chan, n_pad;
    int cold, lte;
    int tile_vecs;              // parameter vectors per CTA tile (0 -> NF_TILE_VECS)
    int npair;                  // hyperfine kernel: line records per component (set by the launcher)
    int stage;                  // the tile's pixel is staged in shared memory (set by the launcher)
    int nkey;                   // hyperfine kernel: line keys per component (set by the launcher)
    NfSpecMeta spec[NF_MAX_SPEC];
    const NfPixSpecMeta *pixmeta;   // per-pixel axes [n_pix][n_spec] (NULL: every pixel uses spec[]); n_chan is then the
                                    // longest spectrum and pred rows are that long
    float *mom_peak;            // may be NULL: hyperfine kernel, ncomp 1, [B][n_spec] maximum of the model over the
    double *mom_sum;            // spectrum's own channels, and its sum (replaces pred)
};

// launchers (nf_model.cu)
cudaError_t nf_launch_nh3(const NfLikeArgs &a, cudaStream_t st);          // nf_nh3.cu
cudaError_t nf_launch_n2hp(const NfLikeArgs &a, cudaStream_t st);         // nf_nh3.cu (N2H+ front end)
cudaError_t nf_launch_gauss(const NfLikeArgs &a, cudaStream_t st);
cudaError_t nf_launch_null_lnz(const float *data, const double *inv2s2, double *out,
                               int64_t n_pix, int n_spec, int n_chan, int n_pad,
                               cudaStream_t st);
cudaError_t nf_launch_d2chunk(const float *data, float *out, int64_t n_rows, int n_pad, cudaStream_t st);
cudaError_t nf_launch_pack_rows(const void *src, int src_f64, float *dst, int64_t rows,
                                int n_chan, int n_pad, cudaStream_t st);
// nf_priors.cu
cudaError_t nf_launch_prior_transform(const nf_priors *pr, double *u, int64_t B, int ncomp,
                                      cudaStream_t st, const int32_t *B_dev = nullptr);

// The dynamic shared-memory limit of a kernel is state of the (device, function) pair, shared by all host threads:
// raise it monotonically under a lock (a thread that lowered it would fail the launches of another).  nf_capi.cu
cudaError_t nf_ensure_dyn_smem(const void *func, size_t bytes);

extern thread_local double g_nf_last_kernel_ms;
extern thread_local int64_t g_nf_last_launches;
