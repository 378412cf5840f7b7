// Fused hyperfine synthesis + radiative transfer + chi-square kernel (sm_100a) for the NH3
// (J,K) inversion lines and N2H+ J = 1-0, 2-1, 3-2.
//
// One warp scores one parameter vector against one pixel, in four phases:
//   S  set-up, batched over the warp's next few vectors: lanes <-> (vector, component,
//      spectrum); partition function, main-line optical depth and the brightness
//      amplitude in FP64                                   (ammonia.pyx:289-361,
//                                                           diazenylium.pyx:140-154)
//   L  per (vector, spectrum): lanes <-> (component, hyperfine line), flattened; window
//      [lo, hi) with the reference's floor rule in FP64, one 24-byte record per line
//                                                          (hyperfine.pyx:68-96)
//   T  item list of a super-block (1024 channels of one spectrum): lanes <-> four consecutive
//      8-channel blocks; the lines reaching a block are a contiguous run of the frequency-
//      sorted records (counting + warp scan); the non-empty (component, block) items are
//      counting-sorted by the length of their run
//   M  rounds of 32 items: a lane owns ONE 8-channel block of ONE component, walks its run
//      of lines (one record fetch per line, eight windowed Gaussians in packed FP32x2
//      FADD2/FFMA2 + MUFU.EX2, one compare per term) with the optical depth of its eight
//      channels in registers, applies the radiative transfer to them and adds the result
//      to the model of the super-block in shared memory; then the residual of the whole
//      super-block, four channels per lane             (hyperfine.pyx:98-113, core.pyx:522-530)
//
// Arithmetic identities used (all exact up to FP32 rounding):
//   tau_j = sum_i tau_main w_i exp(-k_i (j - c_i)^2) is accumulated as
//   tp_j = -log2(e) tau_j = sum_i mA_i 2^((B_i - k2_i d) d + L_i),  d = j - R'_i (exact),
//   with R' the midpoint of the line's window (so the window test is |d| <= h), B = 2 k2 phi',
//   L = -k2 phi'^2 and mA_i = -log2(e) tau_main w_i kept OUTSIDE the exponent: the exponent
//   vanishes at the line centre, where its rounding matters most.  exp(-tau_j) = 2^tp_j.
//   FastExp semantics (nestfit/core/fastexp.c:234-283): exp(-x) of the float-rounded
//   argument -> MUFU.EX2; Taylor-3 branch below 2^-5 kept for 1 - exp(-tau).

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <mutex>
#include <vector>

#include "nf_internal.cuh"
#include "nf_device.cuh"
#include "../../include/nf_nh3_tables.h"
#include "../../include/nf_n2hp_tables.h"

#define NH3_WARPS NF_WARPS_PER_CTA
#define NH3_KEY_NEVER 30000     // chunk key of a line above the band

// ---- device tables ---------------------------------------------------------
// NH3 lines first, then the N2H+ lines (NfSpecMeta::line_off indexes this flat list)
#define NH3_NLINES_ALL (NF_NH3_NLINES_TOTAL + NF_N2HP_NLINES_TOTAL)
__device__ double n_line_freq[NH3_NLINES_ALL];  // (1 - voff_i/c) * nu0   hyperfine.pyx:70
__device__ float n_line_w[NH3_NLINES_ALL];      // the tau weights  ammonia.pyx:168-228, diazenylium.pyx:66-92
__device__ double n_iem_y[NF_IEM_SIZE];              // 1/(exp(x_k)-1)         hyperfine.pyx:19
__constant__ double n_iem_xmin, n_iem_xmax, n_iem_step, n_iem_inv_dx;

static const double hn_nu[NF_NH3_NTRANS] = NF_NH3_REST_FREQ_INIT;
static const int hn_off[NF_NH3_NTRANS + 1] = NF_NH3_LINE_OFFSET_INIT;
static const double hn_voff[NF_NH3_NLINES_TOTAL] = NF_NH3_LINE_VOFF_INIT;
static const double hn_wt[NF_NH3_NLINES_TOTAL] = NF_NH3_LINE_WEIGHT_INIT;
static const double hd_nu[NF_N2HP_NTRANS] = NF_N2HP_REST_FREQ_INIT;
static const int hd_off[NF_N2HP_NTRANS + 1] = NF_N2HP_LINE_OFFSET_INIT;
static const double hd_voff[NF_N2HP_NLINES_TOTAL] = NF_N2HP_LINE_VOFF_INIT;
static const double hd_wt[NF_N2HP_NLINES_TOTAL] = NF_N2HP_LINE_WEIGHT_INIT;

static cudaError_t nh3_upload_device_tables();

// The tables are uploaded once per device, whichever host thread gets there first (samplers of several
// streams call in concurrently).
static cudaError_t nh3_init_device_tables()
{
    int device = 0;
    cudaError_t e = cudaGetDevice(&device);
    if (e) return e;
    if (device < 0 || device >= 64) return nh3_upload_device_tables();
    static std::once_flag once[64];
    static cudaError_t result[64];
    std::call_once(once[device], [device] { result[device] = nh3_upload_device_tables(); });
    return result[device];
}

static cudaError_t nh3_upload_device_tables()
{
    cudaError_t e = cudaSuccess;
    double freq[NH3_NLINES_ALL];
    float wt[NH3_NLINES_ALL];
    for (int t = 0; t < NF_NH3_NTRANS; ++t)
        for (int i = hn_off[t]; i < hn_off[t + 1]; ++i) {
            freq[i] = (1.0 - hn_voff[i] / NF_CKMS) * hn_nu[t];
            wt[i] = (float)hn_wt[i];
        }
    for (int t = 0; t < NF_N2HP_NTRANS; ++t)
        for (int i = hd_off[t]; i < hd_off[t + 1]; ++i) {
            freq[NF_NH3_NLINES_TOTAL + i] = (1.0 - hd_voff[i] / NF_CKMS) * hd_nu[t];
            wt[NF_NH3_NLINES_TOTAL + i] = (float)hd_wt[i];
        }
    if ((e = cudaMemcpyToSymbol(n_line_freq, freq, sizeof(freq)))) return e;
    if ((e = cudaMemcpyToSymbol(n_line_w, wt, sizeof(wt)))) return e;
    // hyperfine.pyx:12-20: x = linspace(XMIN, XMAX, 1000), y = 1/(exp(x)-1)
    std::vector<double> y(NF_IEM_SIZE);
    const double lo = NF_H * 23.0e9 / NF_KB, hi = NF_H * 28.0e9 / NF_KB;
    const double xmin = lo / 8.0, xmax = hi / 2.7;
    const double step = (xmax - xmin) / (double)(NF_IEM_SIZE - 1);
    const double x1 = xmin + step, inv_dx = 1.0 / (x1 - xmin);
    for (int k = 0; k < NF_IEM_SIZE; ++k) {
        const double x = (k == NF_IEM_SIZE - 1) ? xmax : xmin + (double)k * step;
        y[k] = 1.0 / (std::exp(x) - 1.0);
    }
    if ((e = cudaMemcpyToSymbol(n_iem_y, y.data(), sizeof(double) * NF_IEM_SIZE))) return e;
    if ((e = cudaMemcpyToSymbol(n_iem_xmin, &xmin, sizeof(double)))) return e;
    if ((e = cudaMemcpyToSymbol(n_iem_xmax, &xmax, sizeof(double)))) return e;
    if ((e = cudaMemcpyToSymbol(n_iem_step, &step, sizeof(double)))) return e;
    if ((e = cudaMemcpyToSymbol(n_iem_inv_dx, &inv_dx, sizeof(double)))) return e;
    // legacy-stream copies: make them visible before any kernel on a non-blocking stream can run
    return cudaDeviceSynchronize();
}

// 1/(exp(x)-1) exactly as the reference evaluates it (table lerp inside the table
// domain, expm1 outside), hyperfine.pyx:23-45.  FP64.
__device__ double nh3_iemtex(double x)
{
    if (n_iem_xmin < x && x < n_iem_xmax) {
        int k = (int)((x - n_iem_xmin) * n_iem_inv_dx);
        k = min(k, NF_IEM_SIZE - 2);
        const double xk = n_iem_xmin + (double)k * n_iem_step;
        const double yk = n_iem_y[k], yk1 = n_iem_y[k + 1];
        return (yk1 - yk) * n_iem_inv_dx * (x - xk) + yk;
    }
    return 1.0 / expm1(x);
}

// (2J+1) * h (B J(J+1) + (C-B) J^2) / k_B in kelvin, FP32 (levels other than J = 1, 2)
#define NH3_BK_F ((float)(NF_HK * NF_BROT))
#define NH3_CK_F ((float)(NF_HK * (NF_CROT - NF_BROT)))

// ---- per-pixel axes (PIXAX) ------------------------------------------------------
// Spectrum s of pixel pix: the block's shared constants, or that pixel's own entry in HBM.
template <bool PIXAX>
__device__ __forceinline__ const NfSpecMeta &nh3_spec_of(const NfLikeArgs &a, int64_t pix, int s)
{
    if constexpr (PIXAX) return a.pixmeta[pix * a.n_spec + s].m;
    else return a.spec[s];
}
template <bool PIXAX>
__device__ __forceinline__ int nh3_nchan_of(const NfLikeArgs &a, int64_t pix, int s)
{
    if constexpr (PIXAX) return a.pixmeta[pix * a.n_spec + s].n_chan;
    else return a.n_chan;
}
__device__ __forceinline__ int64_t nh3_pix_of(const NfLikeArgs &a, int64_t b)
{
    return a.pix_of_vec ? (int64_t)__ldg(a.pix_of_vec + b) : b / a.vecs_per_pix;
}

// ---- S: batched set-up, lanes <-> (vector, component, spectrum) -----------------
// MODEL 0: NH3 (voff, trot, tex, ntot, sigm, orth; ammonia.pyx:326-361);
// MODEL 1: N2H+ (voff, tex, ltau, sigm; diazenylium.pyx:140-154).
// PIXAX: every lane reads the axis of its own vector's pixel.
template <int MODEL, int NC, bool PIXAX, typename PT, typename SC>
__device__ __noinline__ void nh3_setup_batch(const NfLikeArgs &a, SC &sc, int64_t bb, int nb, int lane)
{
    const int n_spec = a.n_spec;
    const int ipv = NC * n_spec;
    const int kk = lane / ipv;
    const int r = lane - kk * ipv;
    const int c = r / n_spec, s = r - c * n_spec;
    const bool valid = kk < nb;
    const int64_t pbase = (bb + (valid ? kk : 0)) * ((MODEL == 0 ? 6 : 4) * NC);
    const int64_t pix = PIXAX ? nh3_pix_of(a, bb + (valid ? kk : 0)) : 0;
    const NfSpecMeta &sm = nh3_spec_of<PIXAX>(a, pix, s);
    const double voff = ld_param<PT>(a.params, pbase + 0 * NC + c);
    double tex, sigm, tau_main;
    if constexpr (MODEL == 1) {
        tex = ld_param<PT>(a.params, pbase + 1 * NC + c);
        const double ltau = ld_param<PT>(a.params, pbase + 2 * NC + c);
        sigm = ld_param<PT>(a.params, pbase + 3 * NC + c);
        tau_main = exp10(ltau);                                          // hyperfine.pyx:63
    } else {
    double trot = ld_param<PT>(a.params, pbase + 1 * NC + c);
    tex = ld_param<PT>(a.params, pbase + 2 * NC + c);
    const double ntot = ld_param<PT>(a.params, pbase + 3 * NC + c);
    sigm = ld_param<PT>(a.params, pbase + 4 * NC + c);
    const double orth = ld_param<PT>(a.params, pbase + 5 * NC + c);
    if (a.cold)  // swift_convert, ammonia.pyx:280-286
        trot = trot / (1.0 + (trot / 41.18) * log(1.0 + 0.6 * exp(-15.7 / trot)));
    if (a.lte) tex = trot;                                              // ammonia.pyx:346-347
    // partition function (ammonia.pyx:289-315): levels J = 1, 2 carry all but ~1e-3 of
    // Q_para and are added in FP64; the others go through MUFU.EX2 in FP32, summed while
    // any lane's level is inside FastExp's range (x < 32)
    const int my_J = sm.J, my_para = sm.para;
    const float itr = 1.0f / (float)trot;
    float q32 = 0.0f;
    for (int J = 0; J <= 50; ++J) {
        if (J == 1 || J == 2) continue;
        const float Jf = (float)J;
        const float x = (NH3_BK_F * Jf * (Jf + 1.0f) + NH3_CK_F * Jf * Jf) * itr;
        const bool live = x < 32.0f;
        if (!__any_sync(NF_FULL, live && valid)) break;
        const float lev = live ? (2.0f * Jf + 1.0f) * ex2_approx(-(float)NF_LOG2E * x) : 0.0f;
        const bool ortho_J = (J % 3) == 0;
        if (my_para ? !ortho_J : ortho_J) q32 += my_para ? lev : 2.0f * lev;
    }
    const double a1 = NF_HK * (2.0 * NF_BROT + (NF_CROT - NF_BROT));
    const double a2 = NF_HK * (6.0 * NF_BROT + 4.0 * (NF_CROT - NF_BROT));
    const double lev1 = 3.0 * fastexp_f64(a1 / trot);
    const double lev2 = 5.0 * fastexp_f64(a2 / trot);
    double zlev = my_J == 1 ? lev1 : lev2;
    if (my_J > 2) {
        const double J = (double)my_J;
        zlev = (2.0 * J + 1.0) * fastexp_f64(NF_HK * (NF_BROT * J * (J + 1.0) + (NF_CROT - NF_BROT) * J * J) / trot);
    }
    const double qtot = my_para ? lev1 + lev2 + (double)q32 : (double)q32;
    const double frac = my_para ? 1.0 - orth : orth;
    const double pop = exp10(ntot) * frac * zlev / qtot;          // ammonia.pyx:353
    const double e = exp(-sm.hnu_k / tex);                        // ammonia.pyx:354-357
    tau_main = pop * sm.fracterm * ((1.0 - e) / (1.0 + e)) * (sm.width_c / sigm);
    }
    // T_B amplitude T0_j * (G(T0_j/tex) - tbg_j), hyperfine.pyx:106-113, as the max of two
    // lines in j: the reference's G is a convex piecewise-linear table, and the lines of the
    // table segments at the two band edges reproduce it exactly while the band crosses at most
    // one knot (about 1e-3 of nu); beyond, G is underestimated between the outer knots.  With
    // tbg and T0 made linear in j the amplitude is within 6.2e-6 of its peak up to
    // NF_MAX_BAND_FRAC over tex >= 2.8 K, error growing as the band squared (the pixel-block
    // constructors refuse wider hyperfine spectra; tests/test_amplitude_model.py).
    const double nm1 = (double)(nh3_nchan_of<PIXAX>(a, pix, s) - 1);
    const double xL = sm.T0_first / tex, xR = sm.T0_last / tex;
    const double dxdj = (xR - xL) / nm1;
    double aL, bL, aR, bR;
    const bool inL = n_iem_xmin < xL && xL < n_iem_xmax;
    const bool inR = n_iem_xmin < xR && xR < n_iem_xmax;
    if (inL && inR) {
        const int kL = min((int)((xL - n_iem_xmin) * n_iem_inv_dx), NF_IEM_SIZE - 2);
        const int kR = min((int)((xR - n_iem_xmin) * n_iem_inv_dx), NF_IEM_SIZE - 2);
        double xk = n_iem_xmin + (double)kL * n_iem_step;
        double sl = (n_iem_y[kL + 1] - n_iem_y[kL]) * n_iem_inv_dx;
        aL = n_iem_y[kL] + sl * (xL - xk);
        bL = sl * dxdj;
        xk = n_iem_xmin + (double)kR * n_iem_step;
        sl = (n_iem_y[kR + 1] - n_iem_y[kR]) * n_iem_inv_dx;
        aR = n_iem_y[kR] + sl * (xL - xk);
        bR = sl * dxdj;
    } else {
        const double gL = nh3_iemtex(xL), gR = nh3_iemtex(xR);
        aL = aR = gL;
        bL = bR = (gR - gL) / nm1;
    }
    // fold T0_j = T0_first + (T0_last - T0_first) j / (N-1) into both lines through their
    // end-channel values (the j^2 term of the product is dropped: it grows as the band squared)
    const double pL0 = sm.T0_first * (aL - sm.tbg0);
    const double pL1 = sm.T0_last * (aL + bL * nm1 - sm.tbg0 - sm.tbg1 * nm1);
    const double pR0 = sm.T0_first * (aR - sm.tbg0);
    const double pR1 = sm.T0_last * (aR + bR * nm1 - sm.tbg0 - sm.tbg1 * nm1);
    if (valid) {
        sc.amp[lane] = make_float4((float)pL0, (float)pR0, (float)((pL1 - pL0) / nm1), (float)((pR1 - pR0) / nm1));
        sc.set_tau(lane, tau_main);
        sc.soc[lane] = sigm / NF_CKMS;
        sc.voc[lane] = voff / NF_CKMS;
    }
}

__device__ __forceinline__ float4 lds128(uint32_t addr)
{
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr) : "memory");
    return v;
}
__device__ __forceinline__ float2 lds64(uint32_t addr)
{
    float2 v;
    asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(addr) : "memory");
    return v;
}

// ---- the fused kernel ---------------------------------------------------------
// Why the items are sorted: the 32 items of a round run for as many trips as the longest of their runs, and runs
// range from 1 line (the edge of an outer satellite) to a dozen (overlapping main groups).  Within a class the items
// keep the order (component, lane, block), so the lanes of a round mostly read the same line records (broadcast)
// and usually own blocks of one component; items of different components can own the same channels, in which
// case the components of the round add to the model in turn.
#ifndef BLK_MINCTA
#define BLK_MINCTA 3
#endif
#ifndef BLK_GRP
#define BLK_GRP 4               // neighbouring blocks of a lane that enter the item list together (4, 2 or 1)
#endif
#define BLK_SB 128              // blocks per super-block
#define BLK_STRIDE 132          // counting-array stride per component (slot 128 = beyond the super-block)
#define BLK_PLANE 528           // bytes per plane of the model array: 32 float4 entries + 16 bytes of skew
#define BLK_M_BYTES (8 * BLK_PLANE)

template <int NC>
struct __align__(16) BlkScratch {
    // model spectrum of the current super-block (all zero between uses), as eight planes of float4: the half
    // (channels 8 blk + 4 half ... + 3) of block blk lives in plane (blk & 3) * 2 + half at entry blk >> 2.  Lanes that
    // own blocks 4 l + q (accumulation) and lanes that read channels 128 i + 4 l ... (residual) both hit 8 different
    // 16-byte bank groups per quarter warp.
    float m[BLK_M_BYTES / 4];
    uint32_t items[NC * BLK_STRIDE];      // sorted items: block | component << 7 | first line << 9 | lines << 15;
                                          // doubles as the counting array cnt[NC][BLK_STRIDE] while the list is built
    // (the 2 x 16 counters of the counting sort by run length -- class 15 - min(lines, 15) -- live in the skew words
    // of the model planes: hist[k] in plane k / 4, base[k] in plane 4 + k / 4)
    float4 amp[32];                       // per set-up item: T_B amplitude as the max of two lines in j
    double soc[32], voc[32];              // sigma / c_kms, voff / c_kms
    float tauA[32];                       // log2(e) * tau_main
    __device__ __forceinline__ void set_tau(int i, double tau_main) { tauA[i] = (float)(tau_main * NF_LOG2E); }
};

// tp += e * mA for a channel inside the line's window, |d| <= h
__device__ __forceinline__ void masked_fma(float &tp, float e, float mA, float d, float h)
{
    asm("{\n"
        ".reg .pred p;\n"
        ".reg .f32 ad;\n"
        "abs.f32 ad, %3;\n"
        "setp.le.f32 p, ad, %4;\n"
        "@p fma.rn.f32 %0, %1, %2, %0;\n"
        "}\n"
        : "+f"(tp)
        : "f"(e), "f"(mA), "f"(d), "f"(h));
}

__device__ __forceinline__ void sts128(uint32_t addr, float4 v)
{
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

// the counters of the counting sort: four per plane, in the 16 skew bytes behind its 32 entries
__device__ __forceinline__ uint32_t *blk_counter(float *m, int which, int k)
{
    return reinterpret_cast<uint32_t *>(m) + ((which * 4 + (k >> 2)) * BLK_PLANE + 512) / 4 + (k & 3);
}

// byte offset of the first half of block blk in the model array (second half: + BLK_PLANE)
__device__ __forceinline__ uint32_t blk_m_off(int blk)
{
    return (uint32_t)((blk & 3) * (2 * BLK_PLANE) + (blk >> 2) * 16);
}

// m[block] += val, both halves
__device__ __forceinline__ void blk_m_add(uint32_t ma, const float (&val)[8])
{
    float4 u = lds128(ma), v = lds128(ma + BLK_PLANE);
    unpack2(add2(pack2(u.x, u.y), pack2(val[0], val[1])), u.x, u.y);
    unpack2(add2(pack2(u.z, u.w), pack2(val[2], val[3])), u.z, u.w);
    unpack2(add2(pack2(v.x, v.y), pack2(val[4], val[5])), v.x, v.y);
    unpack2(add2(pack2(v.z, v.w), pack2(val[6], val[7])), v.z, v.w);
    sts128(ma, u);
    sts128(ma + BLK_PLANE, v);
}

// PIXAX: every pixel has its own axes and channel counts (a.pixmeta); a.n_chan is the longest spectrum, and the
// super-blocks and the residual run to it (data and model are zero past a spectrum's own end).
// MOM (with WRITE_PRED): instead of the model row, its maximum and its sum over the spectrum's own channels per
// (vector, spectrum) -> a.mom_peak (FP32) and a.mom_sum (FP64, summed in FP64 per lane and across the warp).
template <int MODEL, int NC, bool WRITE_PRED, typename PT, bool PIXAX, bool MOM = false>
__global__ void __launch_bounds__(NF_THREADS, (NC <= 3 ? BLK_MINCTA : 2))
nf_nh3_kernel(const __grid_constant__ NfLikeArgs a)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    uint64_t *bar = reinterpret_cast<uint64_t *>(smem_raw);
    float *sdata = reinterpret_cast<float *>(smem_raw + 128);
    const int data_floats = a.stage ? a.n_spec * a.n_pad : 0;      // the tile's pixel is staged unless it does not fit
    typedef BlkScratch<NC> Scratch;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nrec = a.npair;                              // records per component (lines of the widest transition; even)
    const int nkey = a.nkey;                               // line keys per component (multiple of 4; 0: one super-block)
    const size_t rec4_bytes = (size_t)NC * nrec * 16, rec2_bytes = (size_t)NC * nrec * 8;
    const size_t key_bytes = (size_t)NC * nkey * sizeof(short2);
    const size_t warp_bytes = rec4_bytes + rec2_bytes + key_bytes + sizeof(Scratch);
    unsigned char *wbase = smem_raw + 128 + (((size_t)data_floats * 4 + 127) / 128) * 128 + warp * warp_bytes;
    float4 *rec4 = reinterpret_cast<float4 *>(wbase);                      // {-R', -k2, B, L} per (component, line)
    float2 *rec2 = reinterpret_cast<float2 *>(wbase + rec4_bytes);        // {h, -log2(e) tau_main w}
    short2 *keys = reinterpret_cast<short2 *>(wbase + rec4_bytes + rec2_bytes);   // first block, first block after the window
    Scratch &sc = *reinterpret_cast<Scratch *>(wbase + rec4_bytes + rec2_bytes + key_bytes);
    uint32_t *cw = sc.items;                               // cnt[c][slot] = cw[c * BLK_STRIDE + slot]
    const uint32_t rec4_addr = smem_u32(rec4), rec2_addr = smem_u32(rec2), m_addr = smem_u32(sc.m);

    const int tile = a.tile_vecs > 0 ? a.tile_vecs : NF_TILE_VECS;
    const int64_t b0 = (int64_t)blockIdx.x * tile;
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
    for (int idx = lane; idx < BLK_M_BYTES / 4; idx += 32) sc.m[idx] = 0.0f;

    const int n_spec = a.n_spec;
    const int ipv = NC * n_spec;
    const int nwarps = blockDim.x >> 5;
    const int vpw = (tile + nwarps - 1) / nwarps;
    const int vb = min(32 / ipv, 8);
    int64_t bw_end = b0 + (int64_t)(warp + 1) * vpw;
    if (bw_end > b0 + tile) bw_end = b0 + tile;
    if (bw_end > B) bw_end = B;
    const int n_sb = (a.n_chan + BLK_SB * 8 - 1) / (BLK_SB * 8);
    // the lane's float4 of the model array in the residual pass: channels 128 i + 4 lane ... of the super-block
    const uint32_t m_lane = m_addr + (uint32_t)((lane & 7) * BLK_PLANE + (lane >> 3) * 16);

    // FastExp's Taylor branch for 1 - exp(-tau), tau < 2^-5 (fastexp.c:265-270), in tp = -log2(e) tau
    const float kC1 = -(float)NF_LN2, kC2 = -(float)(0.5 * NF_LN2 * NF_LN2),
                kC3 = -(float)(NF_LN2 * NF_LN2 * NF_LN2 / 6.0);
    const float kThr = -(float)(0.03125 * NF_LOG2E);

    for (int64_t bb = b0 + (int64_t)warp * vpw; bb < bw_end; bb += vb) {
        const int nb = (int)min((int64_t)vb, bw_end - bb);
        nh3_setup_batch<MODEL, NC, PIXAX, PT, Scratch>(a, sc, bb, nb, lane);
        __syncwarp();

        for (int k = 0; k < nb; ++k) {
            const int64_t b = bb + k;
            int64_t pix = 0;
            if (have_data || PIXAX) pix = a.pix_of_vec ? (int64_t)__ldg(a.pix_of_vec + b) : b / a.vecs_per_pix;
            const bool staged = have_data && pix == pix0;
            double lnl = 0.0;
            for (int s = 0; s < n_spec; ++s) {
                const NfSpecMeta &sm = nh3_spec_of<PIXAX>(a, pix, s);
                const int n_own = nh3_nchan_of<PIXAX>(a, pix, s);     // channels of this spectrum
                const int NL = sm.nlines, nitems_l = NC * NL;
                // ---- L: line records, lanes <-> (component, line) flattened; counts of super-block 0 ----
                for (int idx = lane; idx < NC * BLK_STRIDE; idx += 32) cw[idx] = 0u;
                __syncwarp();
                {
                    const double nu_min = sm.nu_min, inv_chan = sm.inv_chan;
                    for (int t0 = 0; t0 < nitems_l; t0 += 32) {
                        const int t = t0 + lane;
                        const bool act = t < nitems_l;
                        int c = 0;
                        if (NC > 1) c += t >= NL;
                        if (NC > 2) c += t >= 2 * NL;
                        if (NC > 3) c += t >= 3 * NL;
                        int i = t - c * NL;
                        if (!act) { c = 0; i = 0; }
                        const int it = k * ipv + c * n_spec + s;
                        const double f = n_line_freq[sm.line_off + i];
                        const double w = sc.soc[it] * f;                 // hyperfine.pyx:71
                        const double nucen = f - sc.voc[it] * f;         // hyperfine.pyx:72-73
                        const double cut = 5.0 * fabs(w);                // sqrt(12.5 / (0.5 / w^2)), hyperfine.pyx:82
                        const double rel = nucen - nu_min;
                        // floor((nu_cen - nu_min -/+ cut) / nu_chan), hyperfine.pyx:83-87.  cvt.rmi saturates
                        // and maps NaN to 0, so non-finite parameters end up with an empty window.
                        int lo = __double2int_rd((rel - cut) * inv_chan);
                        int hi = __double2int_rd((rel + cut) * inv_chan);
                        const bool inband = !(hi < 0 || lo > n_own - 1);      // hyperfine.pyx:88
                        const bool below = hi < 0;
                        lo = max(lo, 0);
                        hi = min(hi, n_own - 1);
                        const bool on = inband && hi > lo;                    // loop j in [lo, hi)
                        // block keys, ascending in the (frequency-sorted) line index.  An in-band line with an
                        // empty window keeps a nominal one-channel extent so that both keys stay sorted.
                        const int hi_n = max(hi, lo + 1);
                        const int kE = below ? -1 : (inband ? (lo >> 3) : NH3_KEY_NEVER);
                        const int kF = below ? -1 : (inband ? ((hi_n - 1) >> 3) + 1 : NH3_KEY_NEVER);
                        float4 r4 = make_float4(0.f, 0.f, 0.f, 0.f);
                        float2 r2v = make_float2(-1.0f, 0.f);
                        if (on) {
                            const int r2 = lo + hi - 1;                       // twice the window midpoint
                            const double jc = rel * inv_chan;
                            const float phi = (float)(jc - 0.5 * (double)r2);
                            const float sch = (float)(w * inv_chan);
                            const float k2 = __fdividef(0.5f * (float)NF_LOG2E, sch * sch);
                            r4 = make_float4(-0.5f * (float)r2, -k2, 2.0f * k2 * phi, -k2 * phi * phi);
                            r2v = make_float2(0.5f * (float)(hi - 1 - lo), -(sc.tauA[it] * n_line_w[sm.line_off + i]));
                        }
                        if (act) {
                            if (nkey) keys[c * nkey + i] = make_short2((short)kE, (short)kF);
                            atomicAdd(&cw[c * BLK_STRIDE + min(max(kE, 0), BLK_SB)], 1u);
                            atomicAdd(&cw[c * BLK_STRIDE + min(max(kF, 0), BLK_SB)], 0x100u);
                            rec4[c * nrec + i] = r4;
                            rec2[c * nrec + i] = r2v;
                        }
                    }
                }
                __syncwarp();

                const char *grow = nullptr;
                if (have_data) grow = reinterpret_cast<const char *>(a.data + pix * a.pix_stride + (int64_t)s * a.n_pad);
                uint64_t acc_a = 0ull, acc_b = 0ull;        // packed FP32x2 sums of squared residuals
                [[maybe_unused]] float mom_pk = -INFINITY;  // MOM: the lane's maximum and FP64 sum of the model
                [[maybe_unused]] double mom_sum = 0.0;
                for (int sbk = 0; sbk < n_sb; ++sbk) {
                    const int blk0 = sbk * BLK_SB;
                    // ---- T: items of the super-block, lanes <-> four consecutive blocks ----
                    if (sbk > 0) {   // later super-blocks (n_chan > 1024): recount from the stored keys
                        for (int idx = lane; idx < NC * BLK_STRIDE; idx += 32) cw[idx] = 0u;
                        __syncwarp();
                        for (int t0 = 0; t0 < nitems_l; t0 += 32) {
                            const int t = t0 + lane;
                            if (t < nitems_l) {
                                int c = 0;
                                if (NC > 1) c += t >= NL;
                                if (NC > 2) c += t >= 2 * NL;
                                if (NC > 3) c += t >= 3 * NL;
                                const int i = t - c * NL;
                                const short2 ky = keys[c * nkey + i];
                                atomicAdd(&cw[c * BLK_STRIDE + min(max((int)ky.x - blk0, 0), BLK_SB)], 1u);
                                atomicAdd(&cw[c * BLK_STRIDE + min(max((int)ky.y - blk0, 0), BLK_SB)], 0x100u);
                            }
                        }
                        __syncwarp();
                    }
                    if (lane < 16) *blk_counter(sc.m, 0, lane) = 0u;
                    // inclusive prefix of {lines started, lines ended} at the lane's blocks 4 lane .. 4 lane + 3:
                    // the lines reaching block g are the run [#ended(g), #started(g)) of the sorted records
                    uint32_t pre[NC][4];
#pragma unroll
                    for (int c = 0; c < NC; ++c) {
                        const uint4 q = *reinterpret_cast<const uint4 *>(&cw[c * BLK_STRIDE + 4 * lane]);
                        const uint32_t s0 = q.x, s1 = s0 + q.y, s2 = s1 + q.z, s3 = s2 + q.w;
                        uint32_t incl = s3;
#pragma unroll
                        for (int o = 1; o < 32; o <<= 1) {
                            const uint32_t u = __shfl_up_sync(NF_FULL, incl, o);
                            if (lane >= o) incl += u;
                        }
                        const uint32_t excl = incl - s3;
                        pre[c][0] = excl + s0; pre[c][1] = excl + s1; pre[c][2] = excl + s2; pre[c][3] = excl + s3;
                    }
                    __syncwarp();     // every lane has read its counts: the item list may overwrite them
                    // The four blocks of a lane (one component) enter the list together, in the class of the longest
                    // of their runs: neighbouring blocks have nearly the same lines, and one shared-memory atomic per
                    // (component, lane) instead of four keeps the dependent chain of the placement short.
                    constexpr int NG = 4 / BLK_GRP;      // groups of BLK_GRP neighbouring blocks per lane and component
                    int qn[NC][NG], qk[NC][NG];          // items of the group, its class
#pragma unroll
                    for (int c = 0; c < NC; ++c)
#pragma unroll
                        for (int g = 0; g < NG; ++g) {
                            int nmax = 0, cnt = 0;
#pragma unroll
                            for (int q = g * BLK_GRP; q < (g + 1) * BLK_GRP; ++q) {
                                const int n = (int)(pre[c][q] & 0xffu) - (int)((pre[c][q] >> 8) & 0xffu);
                                nmax = max(nmax, n);
                                cnt += n > 0;
                            }
                            qn[c][g] = cnt;
                            qk[c][g] = 15 - min(nmax, 15);
                            if (cnt > 0) atomicAdd(blk_counter(sc.m, 0, qk[c][g]), (uint32_t)cnt);
                        }
                    __syncwarp();
                    int nit;
                    {
                        const uint32_t hv = lane < 16 ? *blk_counter(sc.m, 0, lane) : 0u;
                        uint32_t incl = hv;
#pragma unroll
                        for (int o = 1; o < 16; o <<= 1) {
                            const uint32_t u = __shfl_up_sync(NF_FULL, incl, o);
                            if (lane >= o) incl += u;
                        }
                        if (lane < 16) *blk_counter(sc.m, 1, lane) = incl - hv;
                        nit = (int)__shfl_sync(NF_FULL, incl, 15);
                    }
                    __syncwarp();
                    // placement: classes in descending run length; the blocks of a group stay together
                    uint32_t qpos[NC][NG];
#pragma unroll
                    for (int c = 0; c < NC; ++c)
#pragma unroll
                        for (int g = 0; g < NG; ++g) {
                            qpos[c][g] = 0u;
                            if (qn[c][g] > 0) qpos[c][g] = atomicAdd(blk_counter(sc.m, 1, qk[c][g]), (uint32_t)qn[c][g]);
                        }
#pragma unroll
                    for (int c = 0; c < NC; ++c)
#pragma unroll
                        for (int g = 0; g < NG; ++g) {
                            uint32_t pos = qpos[c][g];
#pragma unroll
                            for (int q = g * BLK_GRP; q < (g + 1) * BLK_GRP; ++q) {
                                const uint32_t first = (pre[c][q] >> 8) & 0xffu;
                                const int n = (int)(pre[c][q] & 0xffu) - (int)first;
                                if (n > 0) {
                                    sc.items[pos] = (uint32_t)(4 * lane + q) | ((uint32_t)c << 7) | (first << 9) | ((uint32_t)n << 15);
                                    ++pos;
                                }
                            }
                        }
                    __syncwarp();

                    // ---- M: rounds of 32 items ----
                    for (int r0 = 0; r0 < nit; r0 += 32) {
                        const uint32_t item = r0 + lane < nit ? sc.items[r0 + lane] : 0u;   // idle lanes: no lines
                        const int n = (int)((item >> 15) & 63u), c = (int)((item >> 7) & 3u);
                        const int blk = (int)(item & 127u), first = (int)((item >> 9) & 63u);
                        const int T = __reduce_max_sync(NF_FULL, n);
                        const float j0 = (float)((blk0 + blk) << 3);       // first channel of the block
                        uint64_t x[4];
#pragma unroll
                        for (int q = 0; q < 4; ++q) x[q] = pack2(j0 + (float)(2 * q), j0 + (float)(2 * q + 1));
                        const int ri = c * nrec + first;
                        uint32_t ra4 = rec4_addr + (uint32_t)(ri * 16), ra2 = rec2_addr + (uint32_t)(ri * 8);
                        float tp[8];
#pragma unroll
                        for (int q = 0; q < 8; ++q) tp[q] = 0.0f;
#pragma unroll 1
                        for (int t = 0; t < T; ++t, ra4 += 16u, ra2 += 8u) {
                            const float4 A = lds128(ra4);
                            const float2 H = lds64(ra2);
                            const float h = t < n ? H.x : -1.0f;       // lanes whose run is shorter sit the trip out
                            const uint64_t R2 = pack2(A.x, A.x), K2 = pack2(A.y, A.y), B2 = pack2(A.z, A.z), L2 = pack2(A.w, A.w);
#pragma unroll
                            for (int q = 0; q < 4; ++q) {
                                const uint64_t d2 = add2(x[q], R2);                 // exact: multiples of 1/2
                                const uint64_t a2 = fma2(fma2(K2, d2, B2), d2, L2);
                                float d0, d1, a0, a1;
                                unpack2(d2, d0, d1);
                                unpack2(a2, a0, a1);
                                const float e0 = ex2_approx(a0), e1 = ex2_approx(a1);
                                masked_fma(tp[2 * q], e0, H.y, d0, h);
                                masked_fma(tp[2 * q + 1], e1, H.y, d1, h);
                            }
                        }
                        // radiative transfer on the lane's eight channels: 1 - exp(-tau) with FastExp's Taylor branch
                        // below 2^-5 (fastexp.c:265-270), times the T_B amplitude (max of two lines in j)
                        const float4 am = sc.amp[k * ipv + c * n_spec + s];        // {i_L, i_R, s_L, s_R}
                        float val[8];
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            const uint64_t tp2 = pack2(tp[2 * q], tp[2 * q + 1]);
                            float es0, es1, aL0, aL1, aR0, aR1;
                            unpack2(mul2(tp2, fma2(tp2, fma2(tp2, pack2(kC3, kC3), pack2(kC2, kC2)), pack2(kC1, kC1))), es0, es1);
                            const float el0 = 1.0f - ex2_approx(tp[2 * q]), el1 = 1.0f - ex2_approx(tp[2 * q + 1]);
                            const float e0 = tp[2 * q] > kThr ? es0 : el0, e1 = tp[2 * q + 1] > kThr ? es1 : el1;
                            unpack2(fma2(pack2(am.z, am.z), x[q], pack2(am.x, am.x)), aL0, aL1);
                            unpack2(fma2(pack2(am.w, am.w), x[q], pack2(am.y, am.y)), aR0, aR1);
                            val[2 * q] = fmaxf(aL0, aR0) * e0;
                            val[2 * q + 1] = fmaxf(aL1, aR1) * e1;
                        }
                        // accumulate into the model.  Items of ONE component own different blocks (the usual round);
                        // a round that holds several components adds them in turn
                        const uint32_t ma = m_addr + blk_m_off(blk);
                        if (NC == 1) {
                            if (n > 0) blk_m_add(ma, val);
                            __syncwarp();
                        } else {
                            const int c_first = __shfl_sync(NF_FULL, c, 0);
                            if (__all_sync(NF_FULL, n == 0 || c == c_first)) {
                                if (n > 0) blk_m_add(ma, val);
                                __syncwarp();
                            } else {
#pragma unroll
                                for (int cc = 0; cc < NC; ++cc) {
                                    if (!__any_sync(NF_FULL, c == cc && n > 0)) continue;
                                    if (c == cc && n > 0) blk_m_add(ma, val);
                                    __syncwarp();
                                }
                            }
                        }
                    }

                    // ---- residual over the whole super-block, four channels per lane; the model goes back to zero ----
                    const int ch0 = blk0 << 3;
                    const int nch = min(BLK_SB * 8, a.n_pad - ch0);      // padded channels (data and model are zero there)
                    if (WRITE_PRED) {
                        if constexpr (MOM) {
                            // the channels WRITE_PRED writes, without those past the spectrum's end (0 there)
                            const int nreal = min(BLK_SB * 8, (PIXAX ? n_own : a.n_chan) - ch0);
                            for (int j = lane; j < nreal; j += 32) {
                                const int bq = j >> 3;
                                const float mv = sc.m[(blk_m_off(bq) + ((j >> 2) & 1) * BLK_PLANE) / 4 + (j & 3)];
                                mom_pk = fmaxf(mom_pk, mv);
                                mom_sum += (double)mv;
                            }
                        } else {
                        float *row = a.pred + (b * n_spec + s) * (int64_t)a.n_chan;
                        const int nreal = min(BLK_SB * 8, a.n_chan - ch0);
                        for (int j = lane; j < nreal; j += 32) {
                            const int bq = j >> 3;
                            const float mv = sc.m[(blk_m_off(bq) + ((j >> 2) & 1) * BLK_PLANE) / 4 + (j & 3)];
                            row[ch0 + j] = (PIXAX && ch0 + j >= n_own) ? 0.0f : mv;   // past the spectrum's end
                        }
                        }
                        __syncwarp();
                        for (int idx = lane; idx < BLK_M_BYTES / 4; idx += 32) sc.m[idx] = 0.0f;
                    } else {
                        if (!data_ready) { mbar_wait(bar, 0); data_ready = true; }
                        const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
                        const uint64_t neg1 = pack2(-1.0f, -1.0f);
                        if (staged) {
                            const uint32_t dl = smem_u32(sdata + s * a.n_pad + ch0) + (uint32_t)lane * 16u;
#pragma unroll 4
                            for (int j4 = lane * 4, i = 0; j4 < nch; j4 += 128, ++i) {
                                const float4 mv = lds128(m_lane + (uint32_t)i * 64u);
                                const float4 dv = lds128(dl + (uint32_t)i * 512u);
                                sts128(m_lane + (uint32_t)i * 64u, zero4);
                                const uint64_t ra_ = fma2(pack2(mv.x, mv.y), neg1, pack2(dv.x, dv.y));
                                const uint64_t rb_ = fma2(pack2(mv.z, mv.w), neg1, pack2(dv.z, dv.w));
                                acc_a = fma2(ra_, ra_, acc_a);
                                acc_b = fma2(rb_, rb_, acc_b);
                            }
                        } else {
                            const float4 *dg = reinterpret_cast<const float4 *>(grow) + (ch0 >> 2) + lane;
#pragma unroll 4
                            for (int j4 = lane * 4, i = 0; j4 < nch; j4 += 128, ++i) {
                                const float4 mv = lds128(m_lane + (uint32_t)i * 64u);
                                const float4 dv = __ldg(dg + i * 32);
                                sts128(m_lane + (uint32_t)i * 64u, zero4);
                                const uint64_t ra_ = fma2(pack2(mv.x, mv.y), neg1, pack2(dv.x, dv.y));
                                const uint64_t rb_ = fma2(pack2(mv.z, mv.w), neg1, pack2(dv.z, dv.w));
                                acc_a = fma2(ra_, ra_, acc_a);
                                acc_b = fma2(rb_, rb_, acc_b);
                            }
                        }
                    }
                    __syncwarp();
                }
                if (have_data) {
                    float a0, a1, a2, a3;
                    unpack2(acc_a, a0, a1);
                    unpack2(acc_b, a2, a3);
                    const double tot = warp_sum((double)((a0 + a1) + (a2 + a3)));
                    lnl -= tot * __ldg(a.inv2s2 + pix * n_spec + s);
                }
                if constexpr (MOM) {
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) mom_pk = fmaxf(mom_pk, __shfl_xor_sync(NF_FULL, mom_pk, o));
                    const double tot = warp_sum(mom_sum);
                    if (lane == 0) {
                        a.mom_peak[b * n_spec + s] = mom_pk;
                        a.mom_sum[b * n_spec + s] = tot;
                    }
                }
                __syncwarp();
            }
            if (a.lnL && lane == 0) a.lnL[b] = lnl;
        }
        __syncwarp();
    }
    // a CTA whose warps all ran out of vectors must still drain the bulk copy
    if (!data_ready) mbar_wait(bar, 0);
}

template <int NC>
static size_t nh3_smem_bytes(const NfLikeArgs &a, int nwarps)
{
    const size_t data = a.stage ? (((size_t)a.n_spec * a.n_pad * 4 + 127) / 128) * 128 : 0;
    return 128 + data + ((size_t)NC * a.npair * 24 + (size_t)NC * a.nkey * sizeof(short2) + sizeof(BlkScratch<NC>)) * nwarps;
}

template <int MODEL, int NC, bool WP, typename PT, bool PIXAX, bool MOM = false>
static cudaError_t nh3_launch_one(const NfLikeArgs &a0, cudaStream_t st)
{
    NfLikeArgs a = a0;
    int max_lines = 1;
    for (int s = 0; s < a.n_spec; ++s) max_lines = a.spec[s].nlines > max_lines ? a.spec[s].nlines : max_lines;
    a.npair = (max_lines + 1) & ~1;                            // records per component (even: 16-byte aligned arrays)
    a.nkey = a.n_chan > BLK_SB * 8 ? ((max_lines + 3) & ~3) : 0;   // line keys are only re-read by later super-blocks
    auto kern = nf_nh3_kernel<MODEL, NC, WP, PT, PIXAX, MOM>;
    // the tile's pixel is staged in shared memory by one bulk copy; rows too long for that are read from HBM / L2
    a.stage = WP ? 0 : 1;
    size_t smem = nh3_smem_bytes<NC>(a, NH3_WARPS);
    if (smem > 227 * 1024 && a.stage) {
        a.stage = 0;
        smem = nh3_smem_bytes<NC>(a, NH3_WARPS);
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

template <int MODEL, int NC, bool PIXAX>
static cudaError_t nh3_launch_ax(const NfLikeArgs &a, cudaStream_t st)
{
    if (a.mom_peak) {       // moments of single-component models only
        if constexpr (NC == 1)
            return a.param_f64 ? nh3_launch_one<MODEL, 1, true, double, PIXAX, true>(a, st)
                               : nh3_launch_one<MODEL, 1, true, float, PIXAX, true>(a, st);
        return cudaErrorInvalidValue;
    }
    const bool wp = a.pred != nullptr;
    if (a.param_f64)
        return wp ? nh3_launch_one<MODEL, NC, true, double, PIXAX>(a, st)
                  : nh3_launch_one<MODEL, NC, false, double, PIXAX>(a, st);
    return wp ? nh3_launch_one<MODEL, NC, true, float, PIXAX>(a, st) : nh3_launch_one<MODEL, NC, false, float, PIXAX>(a, st);
}

template <int MODEL, int NC>
static cudaError_t nh3_launch_nc(const NfLikeArgs &a, cudaStream_t st)
{
    return a.pixmeta ? nh3_launch_ax<MODEL, NC, true>(a, st) : nh3_launch_ax<MODEL, NC, false>(a, st);
}

cudaError_t nf_launch_nh3(const NfLikeArgs &a, cudaStream_t st)
{
    cudaError_t e = nh3_init_device_tables();
    if (e) return e;
    switch (a.ncomp) {
    case 1: return nh3_launch_nc<0, 1>(a, st);
    case 2: return nh3_launch_nc<0, 2>(a, st);
    case 3: return nh3_launch_nc<0, 3>(a, st);
    case 4: return nh3_launch_nc<0, 4>(a, st);
    default: return cudaErrorInvalidValue;
    }
}

// N2H+ (diazenylium.pyx): same hyperfine kernel, 4-parameter front end
cudaError_t nf_launch_n2hp(const NfLikeArgs &a, cudaStream_t st)
{
    cudaError_t e = nh3_init_device_tables();
    if (e) return e;
    switch (a.ncomp) {
    case 1: return nh3_launch_nc<1, 1>(a, st);
    case 2: return nh3_launch_nc<1, 2>(a, st);
    case 3: return nh3_launch_nc<1, 3>(a, st);
    case 4: return nh3_launch_nc<1, 4>(a, st);
    default: return cudaErrorInvalidValue;
    }
}
