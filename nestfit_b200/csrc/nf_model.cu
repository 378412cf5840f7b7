// Fused multi-component Gaussian model + chi-square kernel (sm_100a) and the small
// pixel-block helpers (null evidence, per-chunk sum of squares, row packing).
//
// One warp scores one parameter vector against one pixel:
//   lanes <-> components during the FP64 set-up (window with the reference's floor rule),
//   lanes <-> channels during the FP32 main loop: 128-channel chunks, lane l owns channels 128 g + l
//   + {0, 32, 64, 96} (packed FP32x2 across channel pairs): most chunks are touched by one component, so
//   four channels per lane spread the per-chunk work (record fetch, residual) over more terms.
// A CTA (8 warps) works on a tile of consecutive vectors; the pixel of the tile's first vector
// is staged once in shared memory with a TMA bulk copy (cp.async.bulk + mbarrier), unless the row is too long to
// fit (more than 51840 channels): every pixel is then read from HBM / L2.  Components
// are unordered and have unequal widths: per super-block of 32 chunks the (chunk, component) pairs that
// overlap are compacted into a flat, channel-ordered work list (lanes <-> chunks: every lane collects the
// components covering its chunk from the other lanes' chunk masks, a warp scan places its entries), and the
// main loop walks that list -- one entry = one component on the lane's four channels of one chunk.  Chunks no
// component touches are never visited: they contribute their sum of d^2 from the per-pixel table built at
// upload (`d2chunk`).
//
// Reference arithmetic restated here (paths relative to the reference tree):
//   c_gauss_predict      nestfit/models/gaussian.pyx:17-50 (__APPROX window rule 35-46)
//   Spectrum.c_loglikelihood nestfit/core/core.pyx:522-530
//   FastExp semantics    nestfit/core/fastexp.c:234-283 (exp(-x); 0 for x >= 32) -> MUFU.EX2 with
//                        log2(e) folded in.
// The NH3 / N2H+ hyperfine kernel lives in nf_nh3.cu.

#include <cmath>
#include <cstdio>
#include <vector>

#include "nf_internal.cuh"
#include "nf_device.cuh"

#define NF_GAUSS_MIN_CTAS 4

// One component: 32 bytes, read with one LDS.128 + one LDS.32.  The window [lo, hi) is stored
// symmetric about its own midpoint R' (a multiple of 1/2): channel j is inside <=> |j - R'| <= h.
struct __align__(32) GaussRec {
    float4 a;   // {-R', -k2, 2 k2 phi', peak * 2^(-k2 phi'^2)},  phi' = centre - R'
    float h;
    float pad[3];
};

#define NF_GAUSS_LIST_CAP 256        // work-list entries resident per pass (the list is built in passes if longer)

struct __align__(32) GaussScratch {
    GaussRec rec[NF_MAX_NCOMP_GAUSS];
    uint2 list[NF_GAUSS_LIST_CAP];  // {record smem address | last-of-chunk << 31, float(first channel of the chunk)}
};

__device__ __forceinline__ float gauss_lds_f32(uint32_t addr)
{
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr) : "memory");
    return v;
}
__device__ __forceinline__ uint2 gauss_lds64u(uint32_t addr)
{
    uint2 v;
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(addr) : "memory");
    return v;
}
__device__ __forceinline__ float4 gauss_lds128(uint32_t addr)
{
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr) : "memory");
    return v;
}

// Index of the lowest set bit without FLO/BREV (they execute on the XU pipe, which the exponentials need):
// de Bruijn multiplication, table in constant memory, scaled by sizeof(GaussRec).
__constant__ uint32_t g_lsb_rec_off[32] = {
    0 * 32, 1 * 32, 28 * 32, 2 * 32, 29 * 32, 14 * 32, 24 * 32, 3 * 32, 30 * 32, 22 * 32, 20 * 32, 15 * 32, 25 * 32,
    17 * 32, 4 * 32, 8 * 32, 31 * 32, 27 * 32, 13 * 32, 23 * 32, 21 * 32, 19 * 32, 16 * 32, 7 * 32, 26 * 32, 12 * 32,
    18 * 32, 6 * 32, 11 * 32, 5 * 32, 10 * 32, 9 * 32};
static_assert(sizeof(GaussRec) == 32, "g_lsb_rec_off is scaled by the record size");

// Four channels of a pixel row that is not the CTA's staged pixel (tiles straddling two pixels, rows too long to
// stage).  Kept out of line so that the compiler does not predicate these loads into the common path.
__device__ __noinline__ float4 gauss_row4_global(const float *p)
{
    return make_float4(__ldg(p), __ldg(p + 32), __ldg(p + 64), __ldg(p + 96));
}

// channels of the spectrum of pixel pix
template <bool PIXAX>
__device__ __forceinline__ int gauss_nchan_of(const NfLikeArgs &a, int64_t pix)
{
    if constexpr (PIXAX) return a.pixmeta[pix].n_chan;
    else return a.n_chan;
}

// WRITE_PRED = false: log-likelihood against the pixel's data (a.data, a.lnL);
// WRITE_PRED = true : model spectra only (a.pred), no data are read.
// PIXAX: every pixel has its own axis and channel count (a.pixmeta); a.n_chan is the longest spectrum.
template <bool WRITE_PRED, typename PT, bool PIXAX>
__global__ void __launch_bounds__(NF_THREADS, NF_GAUSS_MIN_CTAS)
nf_gauss_kernel(const __grid_constant__ NfLikeArgs a)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    uint64_t *bar = reinterpret_cast<uint64_t *>(smem_raw);
    float *sdata = reinterpret_cast<float *>(smem_raw + 128);
    const int data_floats = a.stage ? a.n_pad : 0;       // one spectrum per pixel (gaussian.pyx:94-96)
    GaussScratch *scr_all = reinterpret_cast<GaussScratch *>(smem_raw + 128 + (((size_t)data_floats * 4 + 127) / 128) * 128);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    GaussScratch &sc = scr_all[warp];
    const uint32_t rec_addr = smem_u32(sc.rec);

    const int tile = a.tile_vecs > 0 ? a.tile_vecs : NF_TILE_VECS;
    const int64_t b0 = (int64_t)blockIdx.x * tile;
    // the vector count may live on the device (lock-step sampler): a.B then only sized the grid
    const int64_t B = a.B_dev ? min(a.B, (int64_t)__ldg(a.B_dev)) : a.B;
    if (b0 >= B) return;
    constexpr bool have_data = !WRITE_PRED;
    int64_t pix0 = -1;
    if (have_data && a.stage) {
        pix0 = a.pix_of_vec ? (int64_t)__ldg(a.pix_of_vec + b0) : b0 / a.vecs_per_pix;
        if (tid == 0) mbar_init(bar, 1);
        __syncthreads();
        if (tid == 0)
            tma_load_1d(sdata, a.data + pix0 * a.pix_stride, (uint32_t)(data_floats * 4), bar);
    }
    bool data_ready = !(have_data && a.stage);

    const int ncomp = a.ncomp;
    const int ndim = 3 * ncomp;
    const int nchunks = (a.n_chan + 127) >> 7;       // 128-channel chunks (rows are padded to a multiple of 128)
    const NfSpecMeta &sm = a.spec[0];                  // PIXAX: the vector's pixel's entry of a.pixmeta instead
    const double nu_min_b = sm.nu_min, inv_chan_b = sm.inv_chan, f0_b = sm.nu0;
    const float lane_f = (float)lane;

    for (int64_t b = b0 + warp; b < b0 + tile && b < B; b += NF_WARPS_PER_CTA) {
        const int64_t pbase = b * ndim;
        int64_t pix = 0;
        if (have_data || PIXAX) pix = a.pix_of_vec ? (int64_t)__ldg(a.pix_of_vec + b) : b / a.vecs_per_pix;
        const NfPixSpecMeta *pm = PIXAX ? a.pixmeta + pix : nullptr;
        const double nu_min = PIXAX ? pm->m.nu_min : nu_min_b, inv_chan = PIXAX ? pm->m.inv_chan : inv_chan_b;
        const double f0 = PIXAX ? pm->m.nu0 : f0_b;

        // ---- set-up, lanes <-> components (gaussian.pyx:25-46) ----
        int lo = 0, hi = 0;
        bool on = false;
        {
            const bool act = lane < ncomp;
            const int cl = act ? lane : 0;
            const double voff = ld_param<PT>(a.params, pbase + cl);
            const double sigm = ld_param<PT>(a.params, pbase + ncomp + cl);
            const float peak = act ? (float)ld_param<PT>(a.params, pbase + 2 * ncomp + cl) : 0.0f;
            const double w = sigm / NF_CKMS * f0;               // gaussian.pyx:31
            const double nucen = f0 * (1.0 - voff / NF_CKMS);   // gaussian.pyx:32
            const double cut = 5.0 * fabs(w);                   // sqrt(12.5 / (0.5 / w^2)), gaussian.pyx:35
            const double rel = nucen - nu_min;
            // floor((nu_cen - nu_min -/+ cut) / nu_chan), gaussian.pyx:36-40.  cvt.rmi saturates and maps
            // NaN to 0, so non-finite parameters end up with an empty window.
            lo = __double2int_rd((rel - cut) * inv_chan);
            hi = __double2int_rd((rel + cut) * inv_chan);
            on = act && !(hi < 0 || lo > gauss_nchan_of<PIXAX>(a, pix) - 1);   // gaussian.pyx:41
            lo = max(lo, 0);
            hi = min(hi, gauss_nchan_of<PIXAX>(a, pix) - 1);
            on = on && hi > lo;                                 // loop j in [lo, hi)
            GaussRec r;
            r.a = make_float4(0.f, 0.f, 0.f, 0.f);
            r.h = -1.0f;
            if (on) {
                const int r2 = lo + hi - 1;                     // twice the window midpoint
                const float phi = (float)(rel * inv_chan - 0.5 * (double)r2);
                const float sch = (float)(w * inv_chan);
                const float k2 = __fdividef(0.5f * (float)NF_LOG2E, sch * sch);
                r.a = make_float4(-0.5f * (float)r2, -k2, 2.0f * k2 * phi, peak * ex2_approx(-k2 * phi * phi));
                r.h = 0.5f * (float)(hi - 1 - lo);
            }
            sc.rec[lane].a = r.a;
            sc.rec[lane].h = r.h;
        }
        __syncwarp();
        if (!data_ready) { mbar_wait(bar, 0); data_ready = true; }

        const bool staged = have_data && pix == pix0;
        const uint32_t srow = smem_u32(sdata) + (uint32_t)lane * 4u;
        const float *grow = have_data ? a.data + pix * a.pix_stride + lane : nullptr;
        float *prow = WRITE_PRED ? a.pred + b * (int64_t)a.n_chan : nullptr;
        if (WRITE_PRED)       // chunks without components stay zero; the others are overwritten by the same lane
            for (int j = lane; j < a.n_chan; j += 32) prow[j] = 0.0f;
        float acc = 0.0f;
        const uint32_t list_addr = smem_u32(sc.list);
        const uint64_t l2a = pack2(lane_f, lane_f + 32.0f), l2b = pack2(lane_f + 64.0f, lane_f + 96.0f);
        for (int sb = 0; sb < nchunks; sb += 32) {
            // chunks [sb, sb+32) touched by this lane's component
            uint32_t cm = 0u;
            {
                int c_lo = (lo >> 7) - sb, c_hi = ((hi - 1) >> 7) - sb;
                if (on && c_hi >= 0 && c_lo < 32) {
                    c_lo = max(c_lo, 0);
                    c_hi = min(c_hi, 31);
                    cm = (0xffffffffu >> (31 - c_hi)) & (0xffffffffu << c_lo);
                }
            }
            // lanes <-> chunks: the components covering chunk sb + lane (bit c = component c)
            uint32_t mine = 0u;
            for (int c = 0; c < ncomp; ++c) mine |= ((__shfl_sync(NF_FULL, cm, c) >> lane) & 1u) << c;
            const int n_mine = __popc(mine);
            if (have_data) {          // a chunk no component touches contributes its sum of d^2
                const int g = sb + lane;
                if (g < nchunks && n_mine == 0) {
                    const float4 q = __ldg(reinterpret_cast<const float4 *>(a.d2chunk + pix * (int64_t)(a.n_pad >> 5)) + g);
                    acc += (q.x + q.y) + (q.z + q.w);
                }
            }
            int incl = n_mine;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int u = __shfl_up_sync(NF_FULL, incl, o);
                if (lane >= o) incl += u;
            }
            const int n_tot = __shfl_sync(NF_FULL, incl, 31);
            const int first = incl - n_mine;                  // position of this chunk's first entry
            const uint32_t xbits = __float_as_uint((float)((sb + lane) << 7));
            float m0 = 0.0f, m1 = 0.0f, m2 = 0.0f, m3 = 0.0f;
            // the list is consumed in passes of NF_GAUSS_LIST_CAP entries (one pass unless > 8 components overlap
            // everywhere); a chunk's entries may straddle two passes: the model sums m0..m3 carry over
            for (int p0 = 0; p0 < n_tot; p0 += NF_GAUSS_LIST_CAP) {
                __syncwarp();
                {
                    uint32_t rest = mine;
                    int at = first - p0;
                    while (rest) {
                        const uint32_t lsb = rest & (0u - rest);
                        rest ^= lsb;
                        if (at >= 0 && at < NF_GAUSS_LIST_CAP)
                            sc.list[at] = make_uint2((rec_addr + g_lsb_rec_off[(lsb * 0x077CB531u) >> 27]) |
                                                     (rest == 0u ? 0x80000000u : 0u), xbits);
                        ++at;
                    }
                }
                __syncwarp();
                const int n_here = min(n_tot - p0, NF_GAUSS_LIST_CAP);
                uint32_t sa = list_addr;
                const uint32_t send = sa + (uint32_t)n_here * 8u;
#pragma unroll 1
                for (; sa != send; sa += 8u) {
                    const uint2 ent = gauss_lds64u(sa);
                    const uint32_t ra = ent.x & 0x7fffffffu;
                    const float4 A = gauss_lds128(ra);
                    const float h = gauss_lds_f32(ra + 16);
                    const float s0 = __uint_as_float(ent.y) + A.x;                     // chunk base - R' (exact)
                    const uint64_t S2 = pack2(s0, s0), K2 = pack2(A.y, A.y), B2 = pack2(A.z, A.z);
                    const uint64_t da2 = add2(l2a, S2), db2 = add2(l2b, S2);          // exact: multiples of 1/2
                    const uint64_t ta2 = fma2(K2, da2, B2), tb2 = fma2(K2, db2, B2);
                    float d0, d1, d2, d3, e0, e1, e2, e3;
                    unpack2(da2, d0, d1);
                    unpack2(db2, d2, d3);
                    unpack2(mul2(ta2, da2), e0, e1);    // -k2 (d^2 - 2 phi' d) log2(e); 2^(-k2 phi'^2) is in A.w
                    unpack2(mul2(tb2, db2), e2, e3);
                    e0 = ex2_approx(e0);
                    e1 = ex2_approx(e1);
                    e2 = ex2_approx(e2);
                    e3 = ex2_approx(e3);
                    if (fabsf(d0) <= h) m0 = fmaf(A.w, e0, m0);
                    if (fabsf(d1) <= h) m1 = fmaf(A.w, e1, m1);
                    if (fabsf(d2) <= h) m2 = fmaf(A.w, e2, m2);
                    if (fabsf(d3) <= h) m3 = fmaf(A.w, e3, m3);
                    if ((int)ent.x < 0) {            // last component of this chunk: residual
                        const int j0 = (int)__uint_as_float(ent.y);
                        if (WRITE_PRED) {
                            const int j = j0 + lane;
                            if (j < gauss_nchan_of<PIXAX>(a, pix)) prow[j] = m0;
                            if (j + 32 < gauss_nchan_of<PIXAX>(a, pix)) prow[j + 32] = m1;
                            if (j + 64 < gauss_nchan_of<PIXAX>(a, pix)) prow[j + 64] = m2;
                            if (j + 96 < gauss_nchan_of<PIXAX>(a, pix)) prow[j + 96] = m3;
                        } else {
                            float q0, q1, q2, q3;
                            if (staged) {
                                const uint32_t da = srow + (uint32_t)j0 * 4u;
                                q0 = gauss_lds_f32(da);
                                q1 = gauss_lds_f32(da + 128u);
                                q2 = gauss_lds_f32(da + 256u);
                                q3 = gauss_lds_f32(da + 384u);
                            } else {
                                const float4 q = gauss_row4_global(grow + j0);
                                q0 = q.x; q1 = q.y; q2 = q.z; q3 = q.w;
                            }
                            q0 -= m0; q1 -= m1; q2 -= m2; q3 -= m3;
                            acc = fmaf(q0, q0, acc);
                            acc = fmaf(q1, q1, acc);
                            acc = fmaf(q2, q2, acc);
                            acc = fmaf(q3, q3, acc);
                        }
                        m0 = 0.0f; m1 = 0.0f; m2 = 0.0f; m3 = 0.0f;
                    }
                }
            }
        }
        if (have_data) {
            const double tot = warp_sum((double)acc);
            if (lane == 0) a.lnL[b] = -tot * __ldg(a.inv2s2 + pix);
        }
        __syncwarp();
    }
    // a CTA whose warps all ran out of vectors must still drain the bulk copy
    if (!data_ready) mbar_wait(bar, 0);
}

template <bool WP, typename PT, bool PIXAX>
static cudaError_t gauss_launch_one(const NfLikeArgs &a0, cudaStream_t st)
{
    auto kern = nf_gauss_kernel<WP, PT, PIXAX>;
    NfLikeArgs a = a0;
    // the tile's pixel is staged in shared memory by one bulk copy; rows too long for that are read from HBM / L2
    a.stage = WP ? 0 : 1;
    auto smem_bytes = [&] {
        return 128 + (a.stage ? (((size_t)a.n_pad * 4 + 127) / 128) * 128 : 0) + sizeof(GaussScratch) * NF_WARPS_PER_CTA;
    };
    size_t smem = smem_bytes();
    if (smem > 227 * 1024 && a.stage) {
        a.stage = 0;
        smem = smem_bytes();
    }
    if (smem > 227 * 1024) return cudaErrorInvalidConfiguration;
    cudaError_t e = nf_ensure_dyn_smem((const void *)kern, smem);
    if (e) return e;
    const int tile = a.tile_vecs > 0 ? a.tile_vecs : NF_TILE_VECS;
    const int64_t grid = (a.B + tile - 1) / tile;
    if (grid <= 0) return cudaSuccess;
    kern<<<(unsigned)grid, NF_THREADS, smem, st>>>(a);
    return cudaGetLastError();
}

template <bool PIXAX>
static cudaError_t gauss_launch_ax(const NfLikeArgs &a, cudaStream_t st)
{
    const bool wp = a.pred != nullptr;
    if (a.param_f64)
        return wp ? gauss_launch_one<true, double, PIXAX>(a, st) : gauss_launch_one<false, double, PIXAX>(a, st);
    return wp ? gauss_launch_one<true, float, PIXAX>(a, st) : gauss_launch_one<false, float, PIXAX>(a, st);
}

cudaError_t nf_launch_gauss(const NfLikeArgs &a, cudaStream_t st)
{
    if (a.ncomp < 1 || a.ncomp > NF_MAX_NCOMP_GAUSS || a.n_spec != 1) return cudaErrorInvalidValue;
    return a.pixmeta ? gauss_launch_ax<true>(a, st) : gauss_launch_ax<false>(a, st);
}

// ---- pixel-block helpers ----------------------------------------------------
// null_lnZ = -sum_s sum_j d^2 / (2 sigma_s^2)   (core.pyx:518-520, ammonia.pyx:411-415)
__global__ void nf_null_lnz_kernel(const float *data, const double *inv2s2, double *out,
                                   int64_t n_pix, int n_spec, int n_chan, int n_pad)
{
    const int lane = threadIdx.x & 31;
    const int64_t p = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (p >= n_pix) return;
    double tot = 0.0;
    for (int s = 0; s < n_spec; ++s) {
        const float *row = data + (p * n_spec + s) * (int64_t)n_pad;
        double acc = 0.0;
        for (int j = lane; j < n_chan; j += 32) { double d = (double)row[j]; acc += d * d; }
        acc = warp_sum(acc);
        tot -= acc * inv2s2[p * n_spec + s];
    }
    if (lane == 0) out[p] = tot;
}

cudaError_t nf_launch_null_lnz(const float *data, const double *inv2s2, double *out, int64_t n_pix,
                               int n_spec, int n_chan, int n_pad, cudaStream_t st)
{
    const int wpb = 8;
    int64_t grid = (n_pix + wpb - 1) / wpb;
    if (grid <= 0) return cudaSuccess;
    nf_null_lnz_kernel<<<(unsigned)grid, wpb * 32, 0, st>>>(data, inv2s2, out, n_pix, n_spec, n_chan, n_pad);
    return cudaGetLastError();
}

// sum of d^2 over every 32-channel chunk of every (pixel, spectrum) row: one warp per chunk
__global__ void nf_d2chunk_kernel(const float *data, float *out, int64_t n_chunks_total)
{
    const int lane = threadIdx.x & 31;
    const int64_t g = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (g >= n_chunks_total) return;
    const float d = data[g * 32 + lane];
    const float v = warp_sum_f32(d * d);
    if (lane == 0) out[g] = v;
}

cudaError_t nf_launch_d2chunk(const float *data, float *out, int64_t n_rows, int n_pad, cudaStream_t st)
{
    const int64_t total = n_rows * (n_pad / 32);
    if (total <= 0) return cudaSuccess;
    const int wpb = 8;
    nf_d2chunk_kernel<<<(unsigned)((total + wpb - 1) / wpb), wpb * 32, 0, st>>>(data, out, total);
    return cudaGetLastError();
}

// rows of n_chan (f32 or f64) -> zero-padded FP32 rows of n_pad
template <typename T>
__global__ void nf_pack_rows_kernel(const T *src, float *dst, int64_t rows, int n_chan, int n_pad)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t total = rows * n_pad;
    for (; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        int64_t r = i / n_pad;
        int j = (int)(i - r * n_pad);
        dst[i] = j < n_chan ? (float)src[r * n_chan + j] : 0.0f;
    }
}

cudaError_t nf_launch_pack_rows(const void *src, int src_f64, float *dst, int64_t rows, int n_chan,
                                int n_pad, cudaStream_t st)
{
    int64_t total = rows * n_pad;
    if (total <= 0) return cudaSuccess;
    int64_t grid = (total + 255) / 256;
    if (grid > 148 * 32) grid = 148 * 32;
    if (src_f64)
        nf_pack_rows_kernel<double><<<(unsigned)grid, 256, 0, st>>>((const double *)src, dst, rows, n_chan, n_pad);
    else
        nf_pack_rows_kernel<float><<<(unsigned)grid, 256, 0, st>>>((const float *)src, dst, rows, n_chan, n_pad);
    return cudaGetLastError();
}
