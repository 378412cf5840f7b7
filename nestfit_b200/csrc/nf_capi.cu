// extern "C" boundary of libnestfit_b200.so (see include/nestfit_b200.h).
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <new>
#include <map>
#include <thread>
#include <utility>
#include <vector>

#include "nf_internal.cuh"
#include "../../include/nf_nh3_tables.h"
#include "../../include/nf_n2hp_tables.h"

cudaError_t nf_ensure_dyn_smem(const void *func, size_t bytes)
{
    static std::mutex mu;
    static std::map<std::pair<int, const void *>, size_t> limit;
    int device = 0;
    cudaError_t e = cudaGetDevice(&device);
    if (e != cudaSuccess) return e;
    std::lock_guard<std::mutex> lock(mu);
    size_t &cur = limit[std::make_pair(device, func)];
    if (bytes <= cur) return cudaSuccess;
    e = cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e == cudaSuccess) cur = bytes;
    return e;
}

thread_local double g_nf_last_kernel_ms = 0.0;
thread_local int64_t g_nf_last_launches = 0;

namespace {

const double kNu[NF_NH3_NTRANS] = NF_NH3_REST_FREQ_INIT;
const double kEa[NF_NH3_NTRANS] = NF_NH3_EINSTEIN_A_INIT;
const int kOff[NF_NH3_NTRANS + 1] = NF_NH3_LINE_OFFSET_INIT;
const double kNuN2hp[NF_N2HP_NTRANS] = NF_N2HP_REST_FREQ_INIT;
const int kOffN2hp[NF_N2HP_NTRANS + 1] = NF_N2HP_LINE_OFFSET_INIT;

inline bool is_hyperfine(int model) { return model == NF_MODEL_NH3 || model == NF_MODEL_N2HP; }
inline int model_nparams(int model) { return model == NF_MODEL_NH3 ? 6 : (model == NF_MODEL_N2HP ? 4 : 3); }
inline cudaError_t launch_model(int model, const NfLikeArgs &a, cudaStream_t st)
{
    switch (model) {
    case NF_MODEL_NH3: return nf_launch_nh3(a, st);
    case NF_MODEL_N2HP: return nf_launch_n2hp(a, st);
    default: return nf_launch_gauss(a, st);
    }
}

struct DeviceGuard {
    int prev = -1;
    bool ok = false;
    explicit DeviceGuard(int dev)
    {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        ok = cudaSetDevice(dev) == cudaSuccess;
    }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

#define NF_CUDA(expr) do { cudaError_t e__ = (expr); if (e__ != cudaSuccess) return (int)e__; } while (0)

// Constants of one spectrum of n channels on the axis x_j = nu_min + j nu_chan; `t` is its transition id (hyperfine
// models) and `rest_freq` its rest frequency (Gaussian model, may be NULL otherwise).
int fill_spec_meta(int model, int n, double nu_min, double nu_chan, int t, const double *rest_freq, NfSpecMeta &m)
{
    std::memset(&m, 0, sizeof(m));
    if (!(nu_chan > 0.0) || !std::isfinite(nu_min)) return NF_EINVAL;       // core.pyx:504
    m.nu_min = nu_min;
    m.nu_chan = nu_chan;
    m.inv_chan = 1.0 / nu_chan;
    const double x_last = nu_min + (double)(n - 1) * nu_chan;
    if (model != NF_MODEL_GAUSS && !((x_last - nu_min) / nu_min <= NF_MAX_BAND_FRAC)) return NF_EINVAL;
    m.T0_first = NF_H * nu_min / NF_KB;
    m.T0_last = NF_H * x_last / NF_KB;
    const double nm1 = n > 1 ? (double)(n - 1) : 1.0;
    m.t0a = (float)m.T0_first;
    m.t0b = (float)((m.T0_last - m.T0_first) / nm1);
    m.tbg0 = 1.0 / std::expm1(m.T0_first / NF_TCMB);
    m.tbg1 = (1.0 / std::expm1(m.T0_last / NF_TCMB) - m.tbg0) / nm1;
    if (model == NF_MODEL_NH3) {
        if (t < 1 || t > NF_NH3_NTRANS) return NF_EINVAL;                   // ammonia.pyx:268
        m.J = t;
        m.para = (t % 3) != 0;
        m.nu0 = kNu[t - 1];
        m.line_off = kOff[t - 1];
        m.nlines = kOff[t] - kOff[t - 1];
        m.fracterm = NF_CCMS * NF_CCMS * kEa[t - 1] / (8.0 * M_PI * m.nu0 * m.nu0);
        m.width_c = NF_CKMS / (m.nu0 * std::sqrt(2.0 * M_PI));
        m.hnu_k = NF_H * m.nu0 / NF_KB;
    } else if (model == NF_MODEL_N2HP) {
        if (t < 1 || t > NF_N2HP_NTRANS) return NF_EINVAL;                  // diazenylium.pyx:128
        m.J = t;
        m.nu0 = kNuN2hp[t - 1];
        m.line_off = NF_NH3_NLINES_TOTAL + kOffN2hp[t - 1];                 // flat line list of nf_nh3.cu
        m.nlines = kOffN2hp[t] - kOffN2hp[t - 1];
        m.hnu_k = NF_H * m.nu0 / NF_KB;
    } else {
        if (!rest_freq || !(*rest_freq > 0.0)) return NF_EINVAL;
        m.nu0 = *rest_freq;
        m.nlines = 1;
    }
    return NF_OK;
}

int fill_meta(nf_pixels *px, const double *nu_min, const double *nu_chan, const int *trans_id,
              const double *rest_freq)
{
    for (int s = 0; s < px->n_spec; ++s) {
        const int rc = fill_spec_meta(px->model, px->n_chan, nu_min[s], nu_chan[s], trans_id ? trans_id[s] : 0,
                                      rest_freq ? rest_freq + s : nullptr, px->spec[s]);
        if (rc != NF_OK) return rc;
    }
    return NF_OK;
}

int pixels_alloc(int device, int model, int64_t n_pix, int n_spec, int n_chan, const double *nu_min,
                 const double *nu_chan, const int *trans_id, const double *rest_freq, nf_pixels **out)
{
    if (!out) return NF_EINVAL;
    *out = nullptr;
    if (n_pix <= 0 || n_spec <= 0 || n_spec > NF_MAX_SPEC || n_chan < 2 || n_chan > 65535) return NF_EINVAL;
    if (model != NF_MODEL_NH3 && model != NF_MODEL_GAUSS && model != NF_MODEL_N2HP) return NF_EINVAL;
    if (model == NF_MODEL_GAUSS && n_spec != 1) return NF_EINVAL;
    if (!nu_min || !nu_chan) return NF_EINVAL;
    nf_pixels *px = new (std::nothrow) nf_pixels();
    if (!px) return NF_ENOMEM;
    std::memset(px, 0, sizeof(*px));
    px->host_mu = new (std::nothrow) std::mutex();
    if (!px->host_mu) { delete px; return NF_ENOMEM; }
    px->device = device;
    px->model = model;
    px->n_pix = n_pix;
    px->n_spec = n_spec;
    px->n_chan = n_chan;
    // the hyperfine kernel walks 64-channel chunks, the Gaussian kernel 128-channel chunks
    px->n_pad = model == NF_MODEL_GAUSS ? ((n_chan + 127) / 128) * 128 : ((n_chan + 63) / 64) * 64;
    int rc = fill_meta(px, nu_min, nu_chan, trans_id, rest_freq);
    if (rc != NF_OK) { delete px->host_mu; delete px; return rc; }
    cudaError_t e;
    const size_t nrow = (size_t)n_pix * n_spec;
    if ((e = cudaMalloc(&px->data, nrow * px->n_pad * sizeof(float))) != cudaSuccess ||
        (e = cudaMalloc(&px->inv2s2, nrow * sizeof(double))) != cudaSuccess ||
        (e = cudaMalloc(&px->null_lnz, (size_t)n_pix * sizeof(double))) != cudaSuccess ||
        (e = cudaMalloc(&px->d2chunk, nrow * (px->n_pad / 32) * sizeof(float))) != cudaSuccess) {
        nf_pixels_free(px);
        return (int)e;
    }
    for (int i = 0; i < NF_HOST_SLOTS; ++i)
        if ((e = cudaStreamCreateWithFlags(&px->streams[i], cudaStreamNonBlocking)) != cudaSuccess) {
            nf_pixels_free(px);
            return (int)e;
        }
    *out = px;
    return NF_OK;
}

int upload_noise(nf_pixels *px, const double *noise_host)
{
    const size_t nrow = (size_t)px->n_pix * px->n_spec;
    std::vector<double> inv(nrow);
    for (size_t i = 0; i < nrow; ++i) {
        const double s = noise_host[i];
        inv[i] = 1.0 / (2.0 * s * s);       // core.pyx:530
    }
    NF_CUDA(cudaMemcpy(px->inv2s2, inv.data(), nrow * sizeof(double), cudaMemcpyHostToDevice));
    return NF_OK;
}

// raw host rows [n_pix * n_spec][n_chan] of dtype -> device scratch -> padded FP32 rows, in bounded pieces
int upload_host_rows(nf_pixels *px, const void *data, int dtype)
{
    const int n_chan = px->n_chan;
    const size_t esz = dtype == NF_F64 ? 8 : 4;
    const int64_t rows = px->n_pix * px->n_spec;
    int64_t piece = (int64_t)((size_t)64 << 20) / ((size_t)n_chan * esz);
    if (piece < 1) piece = 1;
    if (piece > rows) piece = rows;
    void *scratch = nullptr;
    cudaError_t e = cudaMalloc(&scratch, (size_t)piece * n_chan * esz);
    for (int64_t r0 = 0; e == cudaSuccess && r0 < rows; r0 += piece) {
        const int64_t nr = rows - r0 < piece ? rows - r0 : piece;
        e = cudaMemcpy(scratch, (const unsigned char *)data + (size_t)r0 * n_chan * esz,
                       (size_t)nr * n_chan * esz, cudaMemcpyHostToDevice);
        if (e == cudaSuccess)
            e = nf_launch_pack_rows(scratch, dtype == NF_F64, px->data + (size_t)r0 * px->n_pad, nr, n_chan,
                                    px->n_pad, 0);
        if (e == cudaSuccess) e = cudaDeviceSynchronize();
    }
    if (scratch) cudaFree(scratch);
    return (int)e;
}

int finish_pixels(nf_pixels *px)
{
    NF_CUDA(nf_launch_null_lnz(px->data, px->inv2s2, px->null_lnz, px->n_pix, px->n_spec, px->n_chan,
                               px->n_pad, 0));
    NF_CUDA(nf_launch_d2chunk(px->data, px->d2chunk, px->n_pix * px->n_spec, px->n_pad, 0));
    NF_CUDA(cudaDeviceSynchronize());
    return NF_OK;
}

int ensure_stage(const nf_pixels *cpx, size_t bytes)
{
    nf_pixels *px = const_cast<nf_pixels *>(cpx);
    if (px->stage_bytes >= bytes) return NF_OK;
    for (int i = 0; i < NF_HOST_SLOTS; ++i) {
        if (px->stage_dev[i]) cudaFree(px->stage_dev[i]);
        px->stage_dev[i] = nullptr;
    }
    px->stage_bytes = 0;
    for (int i = 0; i < NF_HOST_SLOTS; ++i) NF_CUDA(cudaMalloc(&px->stage_dev[i], bytes));
    px->stage_bytes = bytes;
    return NF_OK;
}

// Page-locked twin of the device staging buffers, for callers that hand over pageable memory (plain numpy arrays).
int ensure_stage_host(const nf_pixels *cpx, size_t bytes)
{
    nf_pixels *px = const_cast<nf_pixels *>(cpx);
    if (px->stage_host_bytes >= bytes) return NF_OK;
    for (int i = 0; i < NF_HOST_SLOTS; ++i) {
        if (px->stage_host[i]) cudaFreeHost(px->stage_host[i]);
        px->stage_host[i] = nullptr;
    }
    px->stage_host_bytes = 0;
    for (int i = 0; i < NF_HOST_SLOTS; ++i) NF_CUDA(cudaHostAlloc(&px->stage_host[i], bytes, cudaHostAllocDefault));
    px->stage_host_bytes = bytes;
    return NF_OK;
}

// true when the driver can DMA straight from / into the buffer (page-locked, registered or managed memory)
bool host_ptr_is_pinned(const void *p)
{
    if (!p) return true;
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return at.type == cudaMemoryTypeHost || at.type == cudaMemoryTypeManaged;
}

// host copy between a pageable buffer and the page-locked ring: a few threads, one thread cannot feed the kernel
void host_copy(void *dst, const void *src, size_t bytes)
{
    const size_t part_min = (size_t)1 << 20;
    unsigned hw = std::thread::hardware_concurrency();
    size_t nt = hw >= 8 ? 4 : (hw >= 4 ? 2 : 1);
    if (bytes / part_min < nt) nt = bytes / part_min;
    if (nt <= 1) {
        std::memcpy(dst, src, bytes);
        return;
    }
    const size_t part = ((bytes / nt) + 4095) & ~(size_t)4095;
    std::vector<std::thread> th;
    th.reserve(nt - 1);
    for (size_t i = 1; i < nt; ++i) {
        const size_t o = i * part;
        if (o >= bytes) break;
        const size_t n = bytes - o < part ? bytes - o : part;
        th.emplace_back([=] { std::memcpy((unsigned char *)dst + o, (const unsigned char *)src + o, n); });
    }
    std::memcpy(dst, src, part < bytes ? part : bytes);
    for (auto &t : th) t.join();
}

int make_args(const nf_pixels *px, const void *params, int param_dtype, const int32_t *pix_of_vec,
              int64_t vecs_per_pix, int64_t B, int ncomp, int flags, double *lnL, float *pred,
              bool use_data, NfLikeArgs *a)
{
    if (!px || !params || B < 0 || ncomp < 1) return NF_EINVAL;
    if (param_dtype != NF_F32 && param_dtype != NF_F64) return NF_EINVAL;
    if (is_hyperfine(px->model) && ncomp > NF_MAX_NCOMP_NH3) return NF_EINVAL;
    if (px->model == NF_MODEL_GAUSS && ncomp > NF_MAX_NCOMP_GAUSS) return NF_EINVAL;
    if (is_hyperfine(px->model) && ncomp * px->n_spec > 32) return NF_EINVAL;
    if (use_data && !pix_of_vec && vecs_per_pix < 1) return NF_EINVAL;
    std::memset(a, 0, sizeof(*a));
    a->data = use_data ? px->data : nullptr;
    a->inv2s2 = px->inv2s2;
    a->d2chunk = use_data ? px->d2chunk : nullptr;
    a->params = params;
    a->pix_of_vec = (use_data || px->pixmeta) ? pix_of_vec : nullptr;   // predictions on per-pixel axes need the map
    a->vecs_per_pix = vecs_per_pix > 0 ? vecs_per_pix : 1;
    a->B = B;
    a->pix_stride = (int64_t)px->n_spec * px->n_pad;
    a->lnL = lnL;
    a->pred = pred;
    a->param_f64 = param_dtype == NF_F64;
    a->ncomp = ncomp;
    a->n_spec = px->n_spec;
    a->n_chan = px->n_chan;
    a->n_pad = px->n_pad;
    a->cold = (flags & NF_FLAG_COLD) != 0;
    a->lte = (flags & NF_FLAG_LTE) != 0;
    for (int s = 0; s < px->n_spec; ++s) a->spec[s] = px->spec[s];
    a->pixmeta = px->pixmeta;
    return NF_OK;
}

int run_device(const nf_pixels *px, const NfLikeArgs &a, void *stream)
{
    DeviceGuard g(px->device);
    if (!g.ok) return NF_ENODEV;
    cudaStream_t st = (cudaStream_t)stream;
    return (int)launch_model(px->model, a, st);
}

// Host-buffer call: chunks of vectors rotate over a ring of streams and staging buffers so the H2D
// copy of chunk k+1 overlaps the kernel of chunk k and the D2H of chunk k-1.
// Page-locked caller buffers are copied from / into directly.  Pageable ones (plain numpy arrays: what a
// reference-side caller hands over) would serialise the pipeline -- a device-to-host copy into pageable memory
// returns only when the kernel before it has finished -- so the log-likelihood call bounces them through a
// page-locked ring: the host copies chunk k+1 into the ring while the kernel of chunk k runs.
// Moments (peak_host / sum_host, [B][n_spec]) take the place of lnL_host and bounce like it.
int run_host(const nf_pixels *px, int model, const void *params_host, int param_dtype,
             const int32_t *pix_host, int64_t vecs_per_pix, int64_t B, int ncomp, int flags,
             double *lnL_host, float *pred_host, float *peak_host = nullptr, double *sum_host = nullptr)
{
    if (!px || px->model != model) return NF_EINVAL;
    if (B == 0) return NF_OK;
    const bool want_mom = peak_host != nullptr;
    if (want_mom && (!sum_host || lnL_host || pred_host)) return NF_EINVAL;
    if (!params_host || (!lnL_host && !pred_host && !want_mom)) return NF_EINVAL;
    DeviceGuard g(px->device);
    if (!g.ok) return NF_ENODEV;
    const int n_model = model_nparams(model);
    const int ndim = n_model * ncomp;
    const size_t psz = param_dtype == NF_F64 ? 8 : 4;
    const bool want_pred = pred_host != nullptr;
    const size_t pred_per_vec = want_pred ? (size_t)px->n_spec * px->n_chan * sizeof(float) : 0;
    // chunk size: a multiple of the CTA tile and, when pixels are implicit, of vecs_per_pix
    int64_t chunk = want_pred ? 8192 : 131072;
    if (!pix_host && vecs_per_pix > 0 && !want_pred) {
        int64_t unit = vecs_per_pix;
        while (unit % NF_TILE_VECS) unit *= 2;
        chunk = ((chunk + unit - 1) / unit) * unit;
    }
    if (chunk > B) chunk = B;
    const size_t off_pix = (((size_t)chunk * ndim * psz) + 255) / 256 * 256;
    const size_t off_lnl = off_pix + (((size_t)chunk * 4) + 255) / 256 * 256;
    const size_t mom_peak_per_vec = want_mom ? (size_t)px->n_spec * 4 : 0;
    const size_t off_mpk = off_lnl + (((size_t)chunk * 8) + 255) / 256 * 256;
    const size_t off_msum = off_mpk + (((size_t)chunk * mom_peak_per_vec) + 255) / 256 * 256;
    const size_t off_pred = off_msum + (((size_t)chunk * 2 * mom_peak_per_vec) + 255) / 256 * 256;
    const size_t total = off_pred + (size_t)chunk * pred_per_vec;
    // the block's two streams and staging buffers serve one host-buffer call at a time
    std::lock_guard<std::mutex> host_lock(*px->host_mu);
    int rc = ensure_stage(px, total);
    if (rc != NF_OK) return rc;
    const bool bounce = !want_pred && (!host_ptr_is_pinned(params_host) || !host_ptr_is_pinned(pix_host) ||
                                       !host_ptr_is_pinned(lnL_host) || !host_ptr_is_pinned(peak_host) ||
                                       !host_ptr_is_pinned(sum_host));
    if (bounce && (rc = ensure_stage_host(px, off_pred)) != NF_OK) return rc;

    constexpr int S = NF_HOST_SLOTS;
    cudaEvent_t ev0[S] = {}, ev1[S] = {};
    double kernel_ms = 0.0;
    int64_t launches = 0;
    bool pending[S] = {};
    int64_t pend_b0[S] = {}, pend_nb[S] = {};
    int status = NF_OK;
    // the slot's previous chunk has drained its buffers: account its kernel time, hand its results over
    auto drain = [&](int slot) {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, ev0[slot], ev1[slot]);
        kernel_ms += ms;
        if (bounce && lnL_host)
            std::memcpy(lnL_host + pend_b0[slot], (const unsigned char *)px->stage_host[slot] + off_lnl,
                        (size_t)pend_nb[slot] * 8);
        if (bounce && want_mom) {
            std::memcpy((unsigned char *)peak_host + (size_t)pend_b0[slot] * mom_peak_per_vec,
                        (const unsigned char *)px->stage_host[slot] + off_mpk, (size_t)pend_nb[slot] * mom_peak_per_vec);
            std::memcpy((unsigned char *)sum_host + (size_t)pend_b0[slot] * 2 * mom_peak_per_vec,
                        (const unsigned char *)px->stage_host[slot] + off_msum,
                        (size_t)pend_nb[slot] * 2 * mom_peak_per_vec);
        }
        pending[slot] = false;
    };
    // errors inside the pipeline leave through `status` so that the events are always destroyed
#define NF_STEP(expr) { cudaError_t e__ = (expr); if (e__ != cudaSuccess) { status = (int)e__; break; } }
    for (int i = 0; i < NF_HOST_SLOTS && status == NF_OK; ++i) {
        NF_STEP(cudaEventCreate(&ev0[i]));
        NF_STEP(cudaEventCreate(&ev1[i]));
    }
    int64_t k = 0;
    for (int64_t b0 = 0; b0 < B && status == NF_OK; b0 += chunk, ++k) {
        const int slot = (int)(k % S);
        cudaStream_t st = px->streams[slot];
        const int64_t nb = (B - b0 < chunk) ? B - b0 : chunk;
        if (pending[slot]) {
            NF_STEP(cudaStreamSynchronize(st));
            drain(slot);
        }
        unsigned char *dev = (unsigned char *)px->stage_dev[slot];
        unsigned char *ring = bounce ? (unsigned char *)px->stage_host[slot] : nullptr;
        const unsigned char *p_src = (const unsigned char *)params_host + (size_t)b0 * ndim * psz;
        if (bounce) {
            host_copy(ring, p_src, (size_t)nb * ndim * psz);
            p_src = ring;
        }
        NF_STEP(cudaMemcpyAsync(dev, p_src, (size_t)nb * ndim * psz, cudaMemcpyHostToDevice, st));
        const int32_t *pix_dev = nullptr;
        if (pix_host) {
            const void *x_src = pix_host + b0;
            if (bounce) {
                std::memcpy(ring + off_pix, x_src, (size_t)nb * 4);
                x_src = ring + off_pix;
            }
            NF_STEP(cudaMemcpyAsync(dev + off_pix, x_src, (size_t)nb * 4, cudaMemcpyHostToDevice, st));
            pix_dev = (const int32_t *)(dev + off_pix);
        }
        NfLikeArgs a;
        rc = make_args(px, dev, param_dtype, pix_dev, vecs_per_pix, nb, ncomp, flags,
                       lnL_host ? (double *)(dev + off_lnl) : nullptr,
                       want_pred ? (float *)(dev + off_pred) : nullptr, lnL_host != nullptr, &a);
        if (rc != NF_OK) { status = rc; break; }
        if (want_mom) {
            a.mom_peak = (float *)(dev + off_mpk);
            a.mom_sum = (double *)(dev + off_msum);
        }
        if (!pix_host && lnL_host) {
            // implicit pixel map continues across chunks: shift by whole pixels
            a.data = px->data + (b0 / a.vecs_per_pix) * a.pix_stride;
            a.inv2s2 = px->inv2s2 + (b0 / a.vecs_per_pix) * px->n_spec;
            a.d2chunk = px->d2chunk + (b0 / a.vecs_per_pix) * px->n_spec * (px->n_pad / 32);
            if (px->pixmeta) a.pixmeta = px->pixmeta + (b0 / a.vecs_per_pix) * px->n_spec;
        }
        NF_STEP(cudaEventRecord(ev0[slot], st));
        NF_STEP(launch_model(model, a, st));
        NF_STEP(cudaEventRecord(ev1[slot], st));
        ++launches;
        pending[slot] = true;
        pend_b0[slot] = b0;
        pend_nb[slot] = nb;
        if (lnL_host)
            NF_STEP(cudaMemcpyAsync(bounce ? (void *)(ring + off_lnl) : (void *)(lnL_host + b0), dev + off_lnl,
                                    (size_t)nb * 8, cudaMemcpyDeviceToHost, st));
        if (want_pred)
            NF_STEP(cudaMemcpyAsync((unsigned char *)pred_host + (size_t)b0 * pred_per_vec, dev + off_pred,
                                    (size_t)nb * pred_per_vec, cudaMemcpyDeviceToHost, st));
        if (want_mom) {
            NF_STEP(cudaMemcpyAsync(bounce ? (void *)(ring + off_mpk)
                                           : (void *)((unsigned char *)peak_host + (size_t)b0 * mom_peak_per_vec),
                                    dev + off_mpk, (size_t)nb * mom_peak_per_vec, cudaMemcpyDeviceToHost, st));
            NF_STEP(cudaMemcpyAsync(bounce ? (void *)(ring + off_msum)
                                           : (void *)((unsigned char *)sum_host + (size_t)b0 * 2 * mom_peak_per_vec),
                                    dev + off_msum, (size_t)nb * 2 * mom_peak_per_vec, cudaMemcpyDeviceToHost, st));
        }
    }
#undef NF_STEP
    // the chunks still in flight, oldest first
    for (int i = 0; i < S; ++i) {
        const int slot = (int)((k + i) % S);
        cudaError_t e = cudaStreamSynchronize(px->streams[slot]);
        if (e != cudaSuccess && status == NF_OK) status = (int)e;
        if (pending[slot] && e == cudaSuccess) drain(slot);
    }
    for (int i = 0; i < NF_HOST_SLOTS; ++i) {
        if (ev0[i]) cudaEventDestroy(ev0[i]);
        if (ev1[i]) cudaEventDestroy(ev1[i]);
    }
    g_nf_last_kernel_ms = kernel_ms;
    g_nf_last_launches = launches;
    return status;
}

}  // namespace

extern "C" {

int nf_abi_version(void) { return NF_ABI_VERSION; }

const char *nf_error_string(int code)
{
    switch (code) {
    case NF_OK: return "ok";
    case NF_EINVAL: return "invalid argument";
    case NF_ENOMEM: return "host allocation failed";
    case NF_ENODEV: return "no usable CUDA device";
    default: break;
    }
    if (code > 0) return cudaGetErrorString((cudaError_t)code);
    return "unknown error";
}

int nf_device_count(int *count)
{
    if (!count) return NF_EINVAL;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) { *count = 0; return (int)e; }
    *count = n;
    return NF_OK;
}

int nf_pixels_create(int device, int model, int64_t n_pix, int n_spec, int n_chan, const double *nu_min,
                     const double *nu_chan, const int *trans_id, const double *rest_freq,
                     const void *data, int dtype, const double *noise, nf_pixels **out)
{
    if (!data || !noise || (dtype != NF_F32 && dtype != NF_F64)) return NF_EINVAL;
    DeviceGuard g(device);
    if (!g.ok) return NF_ENODEV;
    nf_pixels *px = nullptr;
    int rc = pixels_alloc(device, model, n_pix, n_spec, n_chan, nu_min, nu_chan, trans_id, rest_freq, &px);
    if (rc != NF_OK) return rc;
    // noise must be positive (core.pyx:502)
    for (int64_t i = 0; i < n_pix * n_spec; ++i)
        if (!(noise[i] > 0.0)) { nf_pixels_free(px); return NF_EINVAL; }
    rc = upload_noise(px, noise);
    if (rc == NF_OK) rc = upload_host_rows(px, data, dtype);
    if (rc == NF_OK) rc = finish_pixels(px);
    if (rc != NF_OK) { nf_pixels_free(px); return rc; }
    *out = px;
    return NF_OK;
}

int nf_pixels_create_axes(int device, int model, int64_t n_pix, int n_spec, int n_chan_max, const double *nu_min,
                          const double *nu_chan, const int *n_chan, const int *trans_id, const double *rest_freq,
                          const void *data, int dtype, const double *noise, nf_pixels **out)
{
    if (!out) return NF_EINVAL;
    *out = nullptr;
    if (!data || !noise || !n_chan || !nu_min || !nu_chan || (dtype != NF_F32 && dtype != NF_F64)) return NF_EINVAL;
    if (n_pix <= 0 || n_spec <= 0 || n_spec > NF_MAX_SPEC || n_chan_max < 2 || n_chan_max > 65535) return NF_EINVAL;
    if (model == NF_MODEL_GAUSS && (n_spec != 1 || !rest_freq)) return NF_EINVAL;
    const int64_t rows = n_pix * n_spec;
    std::vector<NfPixSpecMeta> meta((size_t)rows);
    for (int64_t p = 0; p < n_pix; ++p)
        for (int sp = 0; sp < n_spec; ++sp) {
            const int64_t r = p * n_spec + sp;
            const int n = n_chan[r];
            if (n < 2 || n > n_chan_max || !(noise[r] > 0.0)) return NF_EINVAL;       // core.pyx:502
            std::memset(&meta[(size_t)r], 0, sizeof(NfPixSpecMeta));
            meta[(size_t)r].n_chan = n;
            const int rc = fill_spec_meta(model, n, nu_min[r], nu_chan[r], trans_id ? trans_id[sp] : 0,
                                          model == NF_MODEL_GAUSS ? rest_freq + p : nullptr, meta[(size_t)r].m);
            if (rc != NF_OK) return rc;
        }
    // channels past a spectrum's own end are zero in HBM, whatever the caller left there: the null evidence, the
    // per-chunk sums of d^2 and the residual pass then need no channel counts
    const size_t esz = dtype == NF_F64 ? 8 : 4, row_bytes = (size_t)n_chan_max * esz;
    std::vector<unsigned char> rows_zf((size_t)rows * row_bytes);
    std::memcpy(rows_zf.data(), data, rows_zf.size());
    for (int64_t r = 0; r < rows; ++r)
        std::memset(rows_zf.data() + (size_t)r * row_bytes + (size_t)n_chan[r] * esz, 0,
                    (size_t)(n_chan_max - n_chan[r]) * esz);
    DeviceGuard g(device);
    if (!g.ok) return NF_ENODEV;
    nf_pixels *px = nullptr;
    int rc = pixels_alloc(device, model, n_pix, n_spec, n_chan_max, nu_min, nu_chan, trans_id, rest_freq, &px);
    if (rc != NF_OK) return rc;
    for (int sp = 0; sp < n_spec; ++sp) px->spec[sp] = meta[(size_t)sp].m;    // pixel 0: the shared transitions
    cudaError_t e = cudaMalloc(&px->pixmeta, (size_t)rows * sizeof(NfPixSpecMeta));
    if (e == cudaSuccess)
        e = cudaMemcpy(px->pixmeta, meta.data(), (size_t)rows * sizeof(NfPixSpecMeta), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) rc = (int)e;
    if (rc == NF_OK) rc = upload_noise(px, noise);
    if (rc == NF_OK) rc = upload_host_rows(px, rows_zf.data(), dtype);
    if (rc == NF_OK) rc = finish_pixels(px);
    if (rc != NF_OK) { nf_pixels_free(px); return rc; }
    *out = px;
    return NF_OK;
}

int nf_pixels_create_from_device(int device, int model, int64_t n_pix, int n_spec, int n_chan,
                                 const double *nu_min, const double *nu_chan, const int *trans_id,
                                 const double *rest_freq, const float *data_dev, const double *noise_dev,
                                 nf_pixels **out)
{
    if (!data_dev || !noise_dev) return NF_EINVAL;
    DeviceGuard g(device);
    if (!g.ok) return NF_ENODEV;
    nf_pixels *px = nullptr;
    int rc = pixels_alloc(device, model, n_pix, n_spec, n_chan, nu_min, nu_chan, trans_id, rest_freq, &px);
    if (rc != NF_OK) return rc;
    const size_t nrow = (size_t)n_pix * n_spec;
    std::vector<double> noise(nrow);
    cudaError_t e = cudaMemcpy(noise.data(), noise_dev, nrow * sizeof(double), cudaMemcpyDeviceToHost);
    if (e == cudaSuccess) {
        for (size_t i = 0; i < nrow; ++i)
            if (!(noise[i] > 0.0)) { nf_pixels_free(px); return NF_EINVAL; }
        rc = upload_noise(px, noise.data());
    }
    if (e == cudaSuccess && rc == NF_OK)
        e = nf_launch_pack_rows(data_dev, 0, px->data, (int64_t)nrow, n_chan, px->n_pad, 0);
    if (rc == NF_OK && e != cudaSuccess) rc = (int)e;
    if (rc == NF_OK) rc = finish_pixels(px);
    if (rc != NF_OK) { nf_pixels_free(px); return rc; }
    *out = px;
    return NF_OK;
}

int nf_pixels_free(nf_pixels *px)
{
    if (!px) return NF_OK;
    DeviceGuard g(px->device);
    if (px->data) cudaFree(px->data);
    if (px->inv2s2) cudaFree(px->inv2s2);
    if (px->null_lnz) cudaFree(px->null_lnz);
    if (px->d2chunk) cudaFree(px->d2chunk);
    if (px->pixmeta) cudaFree(px->pixmeta);
    for (int i = 0; i < NF_HOST_SLOTS; ++i) {
        if (px->stage_dev[i]) cudaFree(px->stage_dev[i]);
        if (px->stage_host[i]) cudaFreeHost(px->stage_host[i]);
        if (px->streams[i]) cudaStreamDestroy(px->streams[i]);
    }
    delete px->host_mu;
    delete px;
    return NF_OK;
}

int nf_pixels_null_lnz(const nf_pixels *px, double *out_host)
{
    if (!px || !out_host) return NF_EINVAL;
    DeviceGuard g(px->device);
    if (!g.ok) return NF_ENODEV;
    NF_CUDA(cudaMemcpy(out_host, px->null_lnz, (size_t)px->n_pix * sizeof(double), cudaMemcpyDeviceToHost));
    return NF_OK;
}

int nf_nh3_loglike(const nf_pixels *px, const void *params_dev, int param_dtype,
                   const int32_t *pix_of_vec_dev, int64_t vecs_per_pix, int64_t B, int ncomp, int flags,
                   double *lnL_dev, void *stream)
{
    if (!px || px->model != NF_MODEL_NH3 || !lnL_dev) return NF_EINVAL;
    NfLikeArgs a;
    int rc = make_args(px, params_dev, param_dtype, pix_of_vec_dev, vecs_per_pix, B, ncomp, flags, lnL_dev,
                       nullptr, true, &a);
    if (rc != NF_OK) return rc;
    return run_device(px, a, stream);
}

int nf_nh3_predict(const nf_pixels *px, const void *params_dev, int param_dtype, int64_t B, int ncomp,
                   int flags, float *pred_dev, void *stream)
{
    if (!px || px->model != NF_MODEL_NH3 || !pred_dev || px->pixmeta) return NF_EINVAL;
    NfLikeArgs a;
    int rc = make_args(px, params_dev, param_dtype, nullptr, 1, B, ncomp, flags, nullptr, pred_dev, false, &a);
    if (rc != NF_OK) return rc;
    return run_device(px, a, stream);
}

int nf_n2hp_loglike(const nf_pixels *px, const void *params_dev, int param_dtype,
                    const int32_t *pix_of_vec_dev, int64_t vecs_per_pix, int64_t B, int ncomp, double *lnL_dev,
                    void *stream)
{
    if (!px || px->model != NF_MODEL_N2HP || !lnL_dev) return NF_EINVAL;
    NfLikeArgs a;
    int rc = make_args(px, params_dev, param_dtype, pix_of_vec_dev, vecs_per_pix, B, ncomp, 0, lnL_dev,
                       nullptr, true, &a);
    if (rc != NF_OK) return rc;
    return run_device(px, a, stream);
}

int nf_n2hp_predict(const nf_pixels *px, const void *params_dev, int param_dtype, int64_t B, int ncomp,
                    float *pred_dev, void *stream)
{
    if (!px || px->model != NF_MODEL_N2HP || !pred_dev || px->pixmeta) return NF_EINVAL;
    NfLikeArgs a;
    int rc = make_args(px, params_dev, param_dtype, nullptr, 1, B, ncomp, 0, nullptr, pred_dev, false, &a);
    if (rc != NF_OK) return rc;
    return run_device(px, a, stream);
}

int nf_n2hp_loglike_host(const nf_pixels *px, const void *params_host, int param_dtype,
                         const int32_t *pix_of_vec_host, int64_t vecs_per_pix, int64_t B, int ncomp,
                         double *lnL_host)
{
    if (!lnL_host) return NF_EINVAL;
    return run_host(px, NF_MODEL_N2HP, params_host, param_dtype, pix_of_vec_host, vecs_per_pix, B, ncomp, 0,
                    lnL_host, nullptr);
}

int nf_n2hp_predict_host(const nf_pixels *px, const void *params_host, int param_dtype, int64_t B, int ncomp,
                         float *pred_host)
{
    if (!pred_host || (px && px->pixmeta)) return NF_EINVAL;
    return run_host(px, NF_MODEL_N2HP, params_host, param_dtype, nullptr, 1, B, ncomp, 0, nullptr, pred_host);
}

int nf_gauss_loglike(const nf_pixels *px, const void *params_dev, int param_dtype,
                     const int32_t *pix_of_vec_dev, int64_t vecs_per_pix, int64_t B, int ncomp,
                     double *lnL_dev, void *stream)
{
    if (!px || px->model != NF_MODEL_GAUSS || !lnL_dev) return NF_EINVAL;
    NfLikeArgs a;
    int rc = make_args(px, params_dev, param_dtype, pix_of_vec_dev, vecs_per_pix, B, ncomp, 0, lnL_dev,
                       nullptr, true, &a);
    if (rc != NF_OK) return rc;
    return run_device(px, a, stream);
}

int nf_gauss_predict(const nf_pixels *px, const void *params_dev, int param_dtype, int64_t B, int ncomp,
                     float *pred_dev, void *stream)
{
    if (!px || px->model != NF_MODEL_GAUSS || !pred_dev || px->pixmeta) return NF_EINVAL;
    NfLikeArgs a;
    int rc = make_args(px, params_dev, param_dtype, nullptr, 1, B, ncomp, 0, nullptr, pred_dev, false, &a);
    if (rc != NF_OK) return rc;
    return run_device(px, a, stream);
}

int nf_nh3_loglike_host(const nf_pixels *px, const void *params_host, int param_dtype,
                        const int32_t *pix_of_vec_host, int64_t vecs_per_pix, int64_t B, int ncomp,
                        int flags, double *lnL_host)
{
    if (!lnL_host) return NF_EINVAL;
    return run_host(px, NF_MODEL_NH3, params_host, param_dtype, pix_of_vec_host, vecs_per_pix, B, ncomp, flags,
                    lnL_host, nullptr);
}

int nf_gauss_loglike_host(const nf_pixels *px, const void *params_host, int param_dtype,
                          const int32_t *pix_of_vec_host, int64_t vecs_per_pix, int64_t B, int ncomp,
                          double *lnL_host)
{
    if (!lnL_host) return NF_EINVAL;
    return run_host(px, NF_MODEL_GAUSS, params_host, param_dtype, pix_of_vec_host, vecs_per_pix, B, ncomp, 0,
                    lnL_host, nullptr);
}

int nf_nh3_predict_host(const nf_pixels *px, const void *params_host, int param_dtype, int64_t B, int ncomp,
                        int flags, float *pred_host)
{
    if (!pred_host || (px && px->pixmeta)) return NF_EINVAL;
    return run_host(px, NF_MODEL_NH3, params_host, param_dtype, nullptr, 1, B, ncomp, flags, nullptr, pred_host);
}

int nf_gauss_predict_host(const nf_pixels *px, const void *params_host, int param_dtype, int64_t B, int ncomp,
                          float *pred_host)
{
    if (!pred_host || (px && px->pixmeta)) return NF_EINVAL;
    return run_host(px, NF_MODEL_GAUSS, params_host, param_dtype, nullptr, 1, B, ncomp, 0, nullptr, pred_host);
}

int nf_predict_pix(const nf_pixels *px, const void *params_dev, int param_dtype, const int32_t *pix_of_vec_dev,
                   int64_t B, int ncomp, int flags, float *pred_dev, void *stream)
{
    if (!px || !pred_dev || !pix_of_vec_dev) return NF_EINVAL;
    NfLikeArgs a;
    int rc = make_args(px, params_dev, param_dtype, pix_of_vec_dev, 1, B, ncomp, flags, nullptr, pred_dev, false, &a);
    if (rc != NF_OK) return rc;
    return run_device(px, a, stream);
}

int nf_predict_pix_host(const nf_pixels *px, const void *params_host, int param_dtype, const int32_t *pix_of_vec_host,
                        int64_t B, int ncomp, int flags, float *pred_host)
{
    if (!px || !pred_host || !pix_of_vec_host) return NF_EINVAL;
    return run_host(px, px->model, params_host, param_dtype, pix_of_vec_host, 1, B, ncomp, flags, nullptr, pred_host);
}

int nf_predict_moments(const nf_pixels *px, const void *params_dev, int param_dtype, const int32_t *pix_of_vec_dev,
                       int64_t B, int flags, float *peak_dev, double *sum_dev, void *stream)
{
    if (!px || !is_hyperfine(px->model) || !peak_dev || !sum_dev || (px->pixmeta && !pix_of_vec_dev)) return NF_EINVAL;
    NfLikeArgs a;
    int rc = make_args(px, params_dev, param_dtype, pix_of_vec_dev, 1, B, 1, px->model == NF_MODEL_NH3 ? flags : 0,
                       nullptr, nullptr, false, &a);
    if (rc != NF_OK) return rc;
    a.mom_peak = peak_dev;
    a.mom_sum = sum_dev;
    return run_device(px, a, stream);
}

int nf_predict_moments_host(const nf_pixels *px, const void *params_host, int param_dtype,
                            const int32_t *pix_of_vec_host, int64_t B, int flags, float *peak_host, double *sum_host)
{
    if (!px || !is_hyperfine(px->model) || !peak_host || !sum_host || (px->pixmeta && !pix_of_vec_host))
        return NF_EINVAL;
    return run_host(px, px->model, params_host, param_dtype, pix_of_vec_host, 1, B, 1,
                    px->model == NF_MODEL_NH3 ? flags : 0, nullptr, nullptr, peak_host, sum_host);
}

int nf_last_call_stats(double *kernel_ms, int64_t *n_launches)
{
    if (kernel_ms) *kernel_ms = g_nf_last_kernel_ms;
    if (n_launches) *n_launches = g_nf_last_launches;
    return NF_OK;
}

}  // extern "C"
