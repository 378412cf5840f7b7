"""numpy model of the FP32 arithmetic of the fused likelihood kernel (nestfit_b200/csrc/nf_nh3.cu, phases L and M):
the same line records (symmetric window about its midpoint R', single compare |d| <= h, weight folded into the
exponent), the same FP32 operation order in the pair term and the radiative-transfer step (Taylor branch below
2^-5), with MUFU.EX2's relative error modelled as a random 2^-22 perturbation.  The FP64 set-up (partition function,
main-line optical depth, brightness amplitude) is taken from the C oracle, so a comparison with the oracle's
spectra isolates the error budget of the FP32 part -- a CPU test bed for changes to the record algebra before they
cost GPU time.  `amplitude` restates the set-up's brightness amplitude (nf_capi.cu fill_spec_meta, nf_nh3.cu
nh3_setup_batch and the radiative-transfer step of phase M) on its own, so that its error can be compared with the
oracle's per-channel T0_j (G(T0_j / tex) - tbg_j).  Development tool and test infrastructure: nothing under
nestfit_b200/ imports it.

  python tools/kernel_model.py [n_vectors]     error statistics against the oracle for prior-drawn vectors
"""
import re
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

F32 = np.float32
# physical constants as in nestfit_b200/csrc/nf_internal.cuh (the reference's, model_includes.pxi:20-38)
H, KB, CKMS, CCMS, TCMB = 6.62607015e-27, 1.380649e-16, 299792.458, 29979245800.0, 2.72548
LOG2E, LN2 = 1.4426950408889634, 0.6931471805599453


def _macro(text, name):
    body = re.search(r'#define ' + name + r' \{(.*?)\}', text, re.S).group(1)
    body = re.sub(r'/\*.*?\*/', '', body).replace('\\', ' ')
    return np.array([float(v) for v in body.replace('\n', ' ').split(',') if v.strip()])


def load_tables():
    """Rest frequencies, Einstein A, line offsets / weights from include/nf_nh3_tables.h (lines sorted by frequency)."""
    text = (ROOT / 'include' / 'nf_nh3_tables.h').read_text()
    return dict(nu=_macro(text, 'NF_NH3_REST_FREQ_INIT'), ea=_macro(text, 'NF_NH3_EINSTEIN_A_INIT'),
                off=_macro(text, 'NF_NH3_LINE_OFFSET_INIT').astype(int), voff=_macro(text, 'NF_NH3_LINE_VOFF_INIT'),
                wts=_macro(text, 'NF_NH3_LINE_WEIGHT_INIT'))


# the 1/(e^x - 1) table of hyperfine.pyx:12-20 as nf_nh3.cu uploads it
IEM_SIZE = 1000
IEM_XMIN = H * 23.0e9 / KB / 8.0
IEM_XMAX = H * 28.0e9 / KB / 2.7
IEM_STEP = (IEM_XMAX - IEM_XMIN) / (IEM_SIZE - 1)
IEM_INV_DX = 1.0 / ((IEM_XMIN + IEM_STEP) - IEM_XMIN)
IEM_Y = 1.0 / (np.exp(np.append(IEM_XMIN + np.arange(IEM_SIZE - 1) * IEM_STEP, IEM_XMAX)) - 1.0)


def _iemtex(x):
    """nh3_iemtex: table lerp inside the table's domain, 1/expm1 outside."""
    if IEM_XMIN < x < IEM_XMAX:
        k = min(int((x - IEM_XMIN) * IEM_INV_DX), IEM_SIZE - 2)
        return (IEM_Y[k + 1] - IEM_Y[k]) * IEM_INV_DX * (x - (IEM_XMIN + k * IEM_STEP)) + IEM_Y[k]
    return 1.0 / np.expm1(x)


def amplitude(nu_min, nu_chan, n, tex):
    """The brightness amplitude T0_j (G(T0_j / tex) - tbg_j) of channels j = 0 .. n-1 of the axis
    nu_min + j nu_chan the way the kernel evaluates it (float32 [n]): the set-up (FP64) makes tbg and T0 linear in j
    and G the larger of two lines taken from the table segments at the two band edges; phase M evaluates both lines
    with one FP32 FMA each and takes their maximum."""
    # fill_spec_meta (nf_capi.cu)
    T0_first = H * nu_min / KB
    T0_last = H * (nu_min + (n - 1) * nu_chan) / KB
    nm1 = float(n - 1)
    tbg0 = 1.0 / np.expm1(T0_first / TCMB)
    tbg1 = (1.0 / np.expm1(T0_last / TCMB) - tbg0) / nm1
    # nh3_setup_batch (nf_nh3.cu)
    xL, xR = T0_first / tex, T0_last / tex
    dxdj = (xR - xL) / nm1
    if IEM_XMIN < xL < IEM_XMAX and IEM_XMIN < xR < IEM_XMAX:
        lines = []
        for xe in (xL, xR):
            k = min(int((xe - IEM_XMIN) * IEM_INV_DX), IEM_SIZE - 2)
            sl = (IEM_Y[k + 1] - IEM_Y[k]) * IEM_INV_DX
            lines.append((IEM_Y[k] + sl * (xL - (IEM_XMIN + k * IEM_STEP)), sl * dxdj))
        (aL, bL), (aR, bR) = lines
    else:
        gL, gR = _iemtex(xL), _iemtex(xR)
        aL = aR = gL
        bL = bR = (gR - gL) / nm1
    pL0 = T0_first * (aL - tbg0)
    pL1 = T0_last * (aL + bL * nm1 - tbg0 - tbg1 * nm1)
    pR0 = T0_first * (aR - tbg0)
    pR1 = T0_last * (aR + bR * nm1 - tbg0 - tbg1 * nm1)
    am = np.array([pL0, pR0, (pL1 - pL0) / nm1, (pR1 - pR0) / nm1]).astype(F32)
    # phase M: fma2(slope, j, intercept) per line, then the larger of the two
    j = np.arange(n, dtype=F32)
    fL = (am[2].astype(np.float64) * j + am[0]).astype(F32)       # one rounding: an FMA
    fR = (am[3].astype(np.float64) * j + am[1]).astype(F32)
    return np.maximum(fL, fR)


def _ex2(a, rng):
    """FP32 2^a with MUFU.EX2's ~2^-22 relative error (flush to zero below 2^-126)."""
    e = np.exp2(a.astype(np.float64))
    if rng is not None:
        e = e * (1.0 + rng.uniform(-1, 1, size=e.shape) * 2.0**-22)
    e = e.astype(F32)
    e[a < -126] = 0
    return e


def predict(xarrs, trans_ids, params, ncomp, tables=None, rng=None, orc=None, amp_outside=True):
    """Model spectra [n_spec, n_chan] (float32) of one parameter vector [6 ncomp] the way the kernel computes them."""
    if orc is None:
        from oracle import oracle as orc
    lib = orc.load()
    tb = tables or load_tables()
    params = np.asarray(params, dtype=np.float64).reshape(6, ncomp)
    out = []
    for x, tid in zip(xarrs, trans_ids):
        x = np.asarray(x, dtype=np.float64)
        n = x.shape[0]
        nu_min, inv_chan = x[0], 1.0 / (x[1] - x[0])
        nu0, ea = tb['nu'][tid - 1], tb['ea'][tid - 1]
        lo_i, hi_i = tb['off'][tid - 1], tb['off'][tid]
        para = (tid % 3) != 0
        T0 = H * x / KB
        tbg = 1.0 / np.expm1(T0 / TCMB)
        j = np.arange(n, dtype=F32)
        pred = np.zeros(n, dtype=F32)
        for c in range(ncomp):
            voff, trot, tex, ntot, sigm, orth = params[:, c]
            # ---- S (FP64, ammonia.pyx:326-361) ----
            zlev = lib.nfo_partition_level(int(tid), trot)
            qtot = lib.nfo_partition_func(int(para), trot)
            pop = 10.0**ntot * ((1.0 - orth) if para else orth) * zlev / qtot
            e = np.exp(-(H * nu0 / KB) / tex)
            tau_main = pop * (CCMS**2 * ea / (8 * np.pi * nu0**2)) * ((1 - e) / (1 + e)) * (CKMS / (nu0 * np.sqrt(2 * np.pi)) / sigm)
            tauL = np.log2(F32(tau_main * LOG2E))                                   # float
            amp = np.array([T0[k] * (lib.nfo_iemtex_interp(T0[k] / tex) - tbg[k]) for k in range(n)]).astype(F32)
            # ---- L: line records ----
            tp = np.zeros(n, dtype=F32)                                             # -log2(e) tau per channel
            for i in range(lo_i, hi_i):
                f = nu0 * (1.0 - tb['voff'][i] / CKMS)                              # hyperfine.pyx:70
                w = sigm / CKMS * f
                nucen = f - voff / CKMS * f
                cut = 5.0 * abs(w)
                rel = nucen - nu_min
                lo = int(np.floor((rel - cut) * inv_chan))
                hi = int(np.floor((rel + cut) * inv_chan))
                if hi < 0 or lo > n - 1:
                    continue
                lo, hi = max(lo, 0), min(hi, n - 1)
                if hi <= lo:
                    continue
                r2 = lo + hi - 1
                phi = F32(rel * inv_chan - 0.5 * r2)
                sch = F32(w * inv_chan)
                k2 = F32(0.5 * LOG2E) / (sch * sch)
                mR, mk2 = F32(-0.5 * r2), -k2
                Bq = F32(2.0) * k2 * phi
                Lq = (tauL + np.log2(F32(tb['wts'][i]))) - k2 * phi * phi
                if amp_outside:     # block-owner kernel: the line amplitude multiplies the exponential
                    Lq = -k2 * phi * phi
                    mA = -(F32(tau_main * LOG2E) * F32(tb['wts'][i]))
                hh = F32(0.5 * (hi - 1 - lo))
                # ---- M: pair term ----
                d = j + mR
                t = (mk2 * d + Bq).astype(F32)
                a = (t * d + Lq).astype(F32)
                ev = _ex2(a, rng)
                inside = np.abs(d) <= hh
                if amp_outside:
                    tp = np.where(inside, (ev * mA + tp).astype(F32), tp)
                else:
                    tp = np.where(inside, (tp - ev).astype(F32), tp)
            # ---- radiative transfer: 1 - exp(-tau), FastExp's Taylor branch below 2^-5 ----
            c1, c2, c3 = F32(-LN2), F32(-0.5 * LN2 * LN2), F32(-LN2**3 / 6.0)
            small = tp * (c1 + tp * (c2 + tp * c3))
            large = F32(1.0) - _ex2(tp, rng)
            e1 = np.where(tp > F32(-0.03125 * LOG2E), small, large).astype(F32)
            pred = (pred + amp * e1).astype(F32)
        out.append(pred)
    return np.stack(out)


def error_stats(n_vec=64, ncomp=3, n_chan=1000, dv=0.07, seed=0, amp_outside=True):
    """Worst spectrum error of the model against the oracle, in units of the spectrum peak."""
    import nestfit_b200 as nb
    from oracle import oracle as orc
    rng = np.random.default_rng(seed)
    ut = nb.get_irdc_priors()
    xs = [orc.bench_axis(1, n_chan, dv), orc.bench_axis(2, n_chan, dv)]
    P = orc.prior_transform(ut.pack(), rng.uniform(size=(2 * n_vec, 6 * ncomp)), ncomp)
    P = P[np.isfinite(P).all(axis=1)][:n_vec]
    want = orc.nh3_batch(xs, [1, 2], P, ncomp, want_pred=True)["pred"]
    tb = load_tables()
    worst = 0.0
    for b in range(P.shape[0]):
        got = predict(xs, [1, 2], P[b], ncomp, tables=tb, rng=rng, orc=orc, amp_outside=amp_outside)
        peak = np.abs(want[b]).max()
        if peak > 0:
            worst = max(worst, float(np.abs(got - want[b]).max() / peak))
    return worst


if __name__ == '__main__':
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 64
    for ao in (False, True):
        print(f"amplitude {'outside' if ao else 'inside '} the exponent: worst |model - oracle| / peak over {n} prior-drawn "
              f"3-component vectors: {error_stats(n, amp_outside=ao):.3e} (bound 1e-5)")
