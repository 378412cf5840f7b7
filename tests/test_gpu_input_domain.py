"""GPU tests of the likelihood kernels against the float64 C oracle (oracle/nf_oracle.c) across the inputs a pixel
block accepts, away from the benchmark shape: hyperfine rows too long to stage in shared memory, six spectra and
every NH3 / N2H+ transition, 9 to 32 Gaussian components (including a work list built in two passes), Gaussian rows
too long to stage, and wide bands up to the hyperfine models' fractional-bandwidth limit.

Bounds as in tests/test_gpu_parity.py: spectra within 1e-5 of each spectrum's peak, lnL within 1e-3 + 2e-6 |lnL|.
Every case runs with float64 and float32 parameters and a ragged, unsorted pixel map, on a shared-axis block
(PixelBlock) and, where it applies, on a per-pixel-axes block (PixelBlock.from_spectra).  Each check prints its
worst error as a fraction of its bound (pytest -s)."""
import ctypes as C
from types import SimpleNamespace

import numpy as np
import pytest

from oracle import oracle as orc

pytestmark = pytest.mark.gpu

SPEC_TOL = 1e-5
LNL_ABS, LNL_REL = 1e-3, 2e-6
SMEM_MAX = 227 * 1024            # dynamic shared memory a CTA may have on sm_100a
WARPS = 8                        # NF_WARPS_PER_CTA
NH3_NLINES = [18, 21, 26, 7, 7, 7, 7, 7, 1]      # include/nf_nh3_tables.h, (1,1) .. (9,9)
N2HP_NLINES = [15, 40, 45]                       # include/nf_n2hp_tables.h, J 1-0, 2-1, 3-2
# priors of get_irdc_priors
TEX = (2.8, 12.06)
# The reference evaluates 1 - exp(-tau) as 1 - FastExp(tau) in FP64, which keeps only 1e-16 / tau of relative
# precision: a spectrum whose peak is below ~1e-8 K (tau below ~1e-8) has no reference value accurate to 1e-5 of its
# peak, and is left out of the spectrum comparison (its lnL is still compared).
THIN_PEAK = 1e-8
DTYPES = (np.float64, np.float32)


def assert_spectra(err, what, tol=SPEC_TOL):
    """err: the worst |got - want| / (peak of want) over the spectra compared."""
    print(f"\n  {what}: spectra max error {err:.2e} of peak = {err / tol:.3f} of bound", end="")
    assert err < tol, f"{what}: max spectrum error {err:.3e} of peak"


def assert_lnl(got, want, what):
    err = np.abs(got - want)
    lim = LNL_ABS + LNL_REL * np.abs(want)
    r = (err / lim).max()
    print(f"\n  {what}: lnL max |error| {err.max():.2e} = {r:.3f} of bound", end="")
    assert (err <= lim).all(), f"{what}: max lnL error {err.max():.3e} (worst ratio {r:.2f})"


def axis(nu0, n, dv, v0=0.0):
    """Ascending frequency axis of n channels of dv km/s centred on velocity v0."""
    v = v0 + (np.arange(n) - 0.5 * (n - 1)) * dv
    return np.sort(nu0 * (1.0 - v / orc.CKMS))


def rest_freqs(model, tids):
    return [orc.NU[t - 1] if model == "ammonia" else orc.N2HP_NU[t - 1] for t in tids]


def ragged_pix(rng, n_pix, B):
    """Every pixel, unequal runs, mostly sorted with every 7th entry moved elsewhere."""
    pix = np.sort(np.concatenate([np.arange(n_pix), rng.integers(0, n_pix, B - n_pix)]))
    pix[::7] = rng.integers(0, n_pix, pix[::7].shape)
    return pix.astype(np.int32)


def nh3_smem_bytes(nc, n_spec, n_chan, max_lines, stage=True):
    """nh3_smem_bytes of nf_nh3.cu: bulk-copy buffer of the staged pixel + per warp the line records, line keys
    and BlkScratch<nc>."""
    n_pad = -(-n_chan // 64) * 64
    npair = (max_lines + 1) & ~1
    nkey = (max_lines + 3) & ~3 if n_chan > 1024 else 0
    scratch = 8 * 528 + nc * 132 * 4 + 32 * 16 + 2 * 32 * 8 + 32 * 4
    data = -(-(n_spec * n_pad * 4) // 128) * 128 if stage else 0
    return 128 + data + (nc * npair * 24 + nc * nkey * 4 + scratch) * WARPS


def gauss_smem_bytes(n_chan):
    """Shared memory of the Gaussian kernel with the pixel staged: bulk-copy buffer + one GaussScratch per warp."""
    n_pad = -(-n_chan // 128) * 128
    return 128 + n_pad * 4 + WARPS * (32 * 32 + 256 * 8)


# ---- parameters ------------------------------------------------------------------------------------------------
def nh3_params(rng, n, ncomp, vspan=4.0, trot=(7.0, 30.0), tex=TEX, ntot=(12.5, 16.5), ortho=True):
    P = np.concatenate([rng.uniform(-vspan, vspan, (n, ncomp)), rng.uniform(*trot, (n, ncomp)),
                        rng.uniform(*tex, (n, ncomp)), rng.uniform(*ntot, (n, ncomp)),
                        rng.uniform(0.067, 2.067, (n, ncomp)),
                        rng.uniform(0.0, 0.9, (n, ncomp)) if ortho else np.zeros((n, ncomp))], axis=1)
    return P


def n2hp_params(rng, n, ncomp, vspan=3.0, tex=(3.0, 10.0)):
    return np.concatenate([rng.uniform(-vspan, vspan, (n, ncomp)), rng.uniform(*tex, (n, ncomp)),
                           rng.uniform(-1, 1, (n, ncomp)), rng.uniform(0.1, 1.0, (n, ncomp))], axis=1)


def gauss_params(rng, n, ncomp, vspan, sigma):
    return np.concatenate([rng.uniform(-vspan, vspan, (n, ncomp)), rng.uniform(*sigma, (n, ncomp)),
                           rng.uniform(0.1, 5.0, (n, ncomp))], axis=1)


# ---- the oracle on one pixel's own axes --------------------------------------------------------------------------
def oracle_pixel(model, xs, tids, P, ncomp, data=None, noise=None, cold=False, lte=False, rest=None):
    """lnL [B] of P against one pixel (data[s] on axis xs[s]) or, without data, its model spectra [B][s][n_s]."""
    lnl = np.zeros(P.shape[0])
    preds = []
    for s, x in enumerate(xs):
        kw = dict(want_pred=data is None)
        if data is not None:
            kw.update(data=np.asarray(data[s], dtype=np.float64)[None, None], noise=noise[s])
        if model == "ammonia":
            o = orc.nh3_batch([x], [tids[s]], P, ncomp, cold=cold, lte=lte, **kw)
        elif model == "diazenylium":
            o = orc.n2hp_batch([x], [tids[s]], P, ncomp, **kw)
        else:
            if data is not None:
                kw["data"] = kw["data"][0]
            o = orc.gauss_batch(x, rest, P, ncomp, **kw)
            o["pred"] = None if o["pred"] is None else o["pred"][:, None]
        if data is not None:
            lnl += o["lnL"]
        else:
            preds.append(o["pred"][:, 0])
    return lnl if data is not None else preds


class Problem:
    """Pixels with their own axes xs[p][s] (all equal for a shared-axis block), float32 data drawn around the
    oracle's model of a truth vector per pixel, and the blocks under test."""

    def __init__(self, nb, model, xs, tids, ncomp, truth, rng, rest=None, shared=True, perpix=True):
        self.model, self.xs, self.tids, self.ncomp, self.rest = model, xs, tids, ncomp, rest
        self.n_pix, self.n_spec = len(xs), len(xs[0])
        self.noise = rng.uniform(0.05, 0.3, (self.n_pix, self.n_spec))
        self.data = []
        for p in range(self.n_pix):
            clean = oracle_pixel(model, xs[p], tids, truth[p:p + 1], ncomp, rest=self._rest(p))
            self.data.append([(c[0] + rng.normal(0, self.noise[p, s], c.shape[1])).astype(np.float32)
                              for s, c in enumerate(clean)])
        self.blocks = {}
        if shared:
            d = np.array(self.data)
            kw = dict(rest_freq=rest[0]) if model == "gaussian" else dict(trans_ids=tids)
            self.blocks["shared"] = nb.PixelBlock(model, xs[0], d, self.noise, **kw)
        if perpix:
            spectra = [[SimpleNamespace(xarr=xs[p][s], data=self.data[p][s].astype(np.float64),
                                        noise=self.noise[p, s], trans_id=None if tids is None else tids[s],
                                        rest_freq=self._rest(p))
                        for s in range(self.n_spec)] for p in range(self.n_pix)]
            self.blocks["per-pixel"] = nb.PixelBlock.from_spectra(model, spectra)

    def _rest(self, p):
        return None if self.rest is None else self.rest[p]

    def close(self):
        for b in self.blocks.values():
            b.close()

    def want_lnl(self, P, pv, cold=False, lte=False):
        out = np.empty(P.shape[0])
        for p in range(self.n_pix):
            rows = np.flatnonzero(pv == p)
            out[rows] = oracle_pixel(self.model, self.xs[p], self.tids, P[rows], self.ncomp, data=self.data[p],
                                     noise=self.noise[p], cold=cold, lte=lte, rest=self._rest(p))
        return out

    def want_null(self):
        return np.array([-sum((d.astype(np.float64) ** 2).sum() / (2 * self.noise[p, s] ** 2)
                              for s, d in enumerate(self.data[p])) for p in range(self.n_pix)])

    def check(self, P, pv, what, n_pred=32, flags=((False, False),), dtypes=DTYPES):
        """loglike, predict and null_lnZ of every block against the oracle."""
        for name, blk in self.blocks.items():
            np.testing.assert_allclose(blk.null_lnZ(), self.want_null(), rtol=1e-6)
        for dtype in dtypes:
            Pd = P.astype(dtype)
            Pr = Pd.astype(np.float64)
            pvp = pv[:n_pred]
            for cold, lte in flags:
                tag = f"{what} {np.dtype(dtype).name}" + (f" cold={cold:d} lte={lte:d}" if self.model == "ammonia" else "")
                want = self.want_lnl(Pr, pv, cold, lte)
                wp = [oracle_pixel(self.model, self.xs[p], self.tids, Pr[b:b + 1], self.ncomp, cold=cold, lte=lte,
                                   rest=self._rest(p)) for b, p in enumerate(pvp)]
                for name, blk in self.blocks.items():
                    assert_lnl(blk.loglike(Pd, self.ncomp, pix_of_vec=pv, cold=cold, lte=lte), want, f"{tag} {name}")
                    if name == "shared":
                        got = blk.predict(Pd[:n_pred], self.ncomp, cold=cold, lte=lte)
                    else:
                        got = blk.predict(Pd[:n_pred], self.ncomp, cold=cold, lte=lte, pix_of_vec=pvp)
                    err, n_cmp = 0.0, 0
                    for b in range(n_pred):
                        for s in range(self.n_spec):
                            w = wp[b][s][0]
                            n = w.shape[0]
                            assert (got[b, s, n:] == 0).all()
                            peak = np.abs(w).max()
                            if peak >= THIN_PEAK:
                                err = max(err, np.abs(got[b, s, :n] - w).max() / peak)
                                n_cmp += 1
                    assert n_cmp >= 0.5 * n_pred * self.n_spec, f"{tag} {name}: {n_cmp} spectra above {THIN_PEAK} K"
                    assert_spectra(err, f"{tag} {name}")


# ---- A. hyperfine rows too long to stage --------------------------------------------------------------------------
@pytest.mark.parametrize("ncomp", [1, 2, 3, 4])
def test_nh3_unstaged_rows(nb, ncomp):
    """NH3 (1,1)+(2,2), 2 x 29000 channels of 0.0069 km/s (200 km/s).  nh3_smem_bytes at NC = 1 (the smallest):
    per warp 22 records x 24 B + 24 keys x 4 B + BlkScratch<1> 5904 B = 6528 B, x 8 warps = 52224 B; the staged
    pixel adds 2 x 29056 x 4 = 232448 B: 284800 B = 1.23 x the 232448 B a CTA may have, so the launcher clears
    `stage` and the residual reads the data from HBM."""
    n, dv = 29000, 0.0069
    assert nh3_smem_bytes(ncomp, 2, n, 21) >= 1.2 * SMEM_MAX
    rng = np.random.default_rng(300 + ncomp)
    xs = [[axis(orc.NU[0], n, dv), axis(orc.NU[1], n, dv)]] * 3
    truth = nh3_params(rng, 3, ncomp, vspan=60)
    pb = Problem(nb, "ammonia", xs, [1, 2], ncomp, truth, rng)
    P = nh3_params(rng, 160, ncomp, vspan=80)
    pv = ragged_pix(rng, 3, 160)
    P[:3] = truth
    pb.check(P, pv, f"NH3 2x{n} NC={ncomp}", n_pred=12)
    pb.close()


def test_n2hp_unstaged_rows(nb):
    """N2H+ (1-0)+(3-2), NC = 4, 2 x 22400 channels of 0.0089 km/s (199 km/s).  nh3_smem_bytes: per warp
    4 x 46 records x 24 B + 4 x 48 keys x 4 B + BlkScratch<4> 7488 B = 12672 B, x 8 = 101376 B; the staged pixel
    adds 2 x 22400 x 4 = 179200 B: 280704 B = 1.21 x 232448 B, so the pixel is not staged."""
    n, dv, ncomp = 22400, 0.0089, 4
    assert nh3_smem_bytes(ncomp, 2, n, 45) >= 1.2 * SMEM_MAX
    rng = np.random.default_rng(31)
    xs = [[axis(orc.N2HP_NU[0], n, dv), axis(orc.N2HP_NU[2], n, dv)]] * 3
    truth = n2hp_params(rng, 3, ncomp, vspan=60)
    pb = Problem(nb, "diazenylium", xs, [1, 3], ncomp, truth, rng)
    P = n2hp_params(rng, 160, ncomp, vspan=80)
    P[:3] = truth
    pb.check(P, ragged_pix(rng, 3, 160), f"N2H+ 2x{n} NC={ncomp}", n_pred=12)
    pb.close()


def test_nh3_longest_row(nb):
    """One NH3 (1,1) spectrum of 65535 channels (the most a block takes) of 0.003 km/s (197 km/s): the staged
    pixel alone would take 65536 x 4 = 262144 B; with the NC = 2 warp scratch nh3_smem_bytes is 321920 B =
    1.38 x 232448 B."""
    n, dv, ncomp = 65535, 0.003, 2
    assert nh3_smem_bytes(ncomp, 1, n, 18) >= 1.2 * SMEM_MAX
    rng = np.random.default_rng(65535)
    xs = [[axis(orc.NU[0], n, dv)]] * 2
    truth = nh3_params(rng, 2, ncomp, vspan=60)
    pb = Problem(nb, "ammonia", xs, [1], ncomp, truth, rng)
    P = nh3_params(rng, 96, ncomp, vspan=90)
    P[:2] = truth
    pb.check(P, ragged_pix(rng, 2, 96), f"NH3 1x{n} NC={ncomp}", n_pred=8)
    pb.close()


@pytest.mark.parametrize("ncomp", [1, 3])
def test_long_pixel_unstages_short_pixels(nb, ncomp):
    """A per-pixel-axes block whose pixel 0 has 2 x 30000 channels (0.0066 km/s, 198 km/s) and whose other pixels
    have 300-1200: rows are as long as the longest spectrum, so at NC = 1 nh3_smem_bytes is 128 + 2 x 30016 x 4 +
    52224 = 292480 B = 1.26 x 232448 B and no pixel is staged, the short ones included."""
    assert nh3_smem_bytes(ncomp, 2, 30000, 21) >= 1.2 * SMEM_MAX
    rng = np.random.default_rng(70 + ncomp)
    xs = [[axis(orc.NU[0], 30000, 0.0066), axis(orc.NU[1], 30000, 0.0066)]]
    for p in range(3):
        xs.append([axis(orc.NU[t], int(rng.integers(300, 1201)), rng.uniform(0.05, 0.2), rng.uniform(-2, 2))
                   for t in (0, 1)])
    truth = nh3_params(rng, 4, ncomp)
    pb = Problem(nb, "ammonia", xs, [1, 2], ncomp, truth, rng, shared=False)
    assert pb.blocks["per-pixel"].n_chan_max == 30000
    P = nh3_params(rng, 200, ncomp)
    P[:4] = truth
    pb.check(P, ragged_pix(rng, 4, 200), f"NH3 per-pixel 30000 + short NC={ncomp}", n_pred=16)
    pb.close()


# ---- B. six spectra, every transition ---------------------------------------------------------------------------
ALL_FLAGS = ((False, False), (True, False), (False, True), (True, True))


def unequal_axes(rng, n_pix, nus, lo=300, hi=700):
    return [[axis(f, int(rng.integers(lo, hi + 1)), rng.uniform(0.06, 0.15), rng.uniform(-1, 1)) for f in nus]
            for _ in range(n_pix)]


@pytest.mark.parametrize("tids", [[1, 2, 3, 4, 5, 6], [4, 5, 6, 7, 8, 9]])
@pytest.mark.parametrize("ncomp", [1, 2, 3, 4])
def test_nh3_six_spectra(nb, tids, ncomp):
    """Six spectra per pixel (NF_MAX_SPEC): at NC = 4 the set-up batch has 24 lanes per vector and one vector per
    batch.  (4,4) .. (9,9) have their own J, para / ortho state and partition-function levels; warm gas (50-90 K)
    keeps their optical depths above THIN_PEAK.  All four cold / lte combinations, a free ortho fraction; the same
    pixels on a shared-axis and a per-pixel-axes block, then a per-pixel-axes block of unequal lengths."""
    rng = np.random.default_rng(600 + 10 * tids[0] + ncomp)
    trot = (7.0, 30.0) if tids[0] == 1 else (50.0, 90.0)
    nus = rest_freqs("ammonia", tids)
    gen = lambda n: nh3_params(rng, n, ncomp, trot=trot, ntot=(13.5, 16.5))     # noqa: E731
    truth = gen(3)
    for xs, shared, tag in (([[axis(f, 500, 0.1) for f in nus]] * 3, True, "equal"),
                            (unequal_axes(rng, 3, nus), False, "unequal")):
        pb = Problem(nb, "ammonia", xs, tids, ncomp, truth, rng, shared=shared)
        P = gen(128)
        P[:3] = truth
        pb.check(P, ragged_pix(rng, 3, 128), f"NH3 {tids} NC={ncomp} {tag}", n_pred=16, flags=ALL_FLAGS)
        pb.close()


@pytest.mark.parametrize("ncomp", [1, 2, 3, 4])
def test_n2hp_all_transitions(nb, ncomp):
    """N2H+ J 1-0, 2-1 and 3-2 together (15, 40 and 45 lines)."""
    rng = np.random.default_rng(700 + ncomp)
    nus = rest_freqs("diazenylium", [1, 2, 3])
    truth = n2hp_params(rng, 3, ncomp)
    for xs, shared, tag in (([[axis(f, 600, 0.08) for f in nus]] * 3, True, "equal"),
                            (unequal_axes(rng, 3, nus), False, "unequal")):
        pb = Problem(nb, "diazenylium", xs, [1, 2, 3], ncomp, truth, rng, shared=shared)
        P = n2hp_params(rng, 128, ncomp)
        P[:3] = truth
        pb.check(P, ragged_pix(rng, 3, 128), f"N2H+ [1,2,3] NC={ncomp} {tag}", n_pred=16)
        pb.close()


# ---- C. Gaussian components 9 .. 32 -----------------------------------------------------------------------------
GAUSS_N, GAUSS_DV = 4096, 0.05          # the benchmark's axis: 32 chunks of 128 channels, one super-block


def gauss_check(nb, rng, ncomp, P, truth, what, n=GAUSS_N, dv=GAUSS_DV, n_pred=32):
    """A per-pixel-axes block with a rest frequency per pixel, then both kinds of block with one rest frequency."""
    n_pix = truth.shape[0]
    xs = [[axis(orc.NU[0], n, dv)]] * n_pix
    rest = orc.NU[0] * (1.0 + rng.uniform(-1e-6, 1e-6, n_pix))
    pb = Problem(nb, "gaussian", xs, None, ncomp, truth, rng, rest=rest, shared=False)
    pb.check(P, ragged_pix(rng, n_pix, P.shape[0]), f"{what} per-pixel rest", n_pred=n_pred)
    pb.close()
    pb = Problem(nb, "gaussian", xs, None, ncomp, truth, rng, rest=[orc.NU[0]] * n_pix)
    pb.check(P, ragged_pix(rng, n_pix, P.shape[0]), what, n_pred=n_pred)
    pb.close()


@pytest.mark.parametrize("ncomp", [9, 16, 32])
@pytest.mark.parametrize("width", ["narrow", "wide"])
def test_gauss_many_components(nb, ncomp, width):
    """Components 9 .. 32 of nf_gauss_kernel: list entries whose record offsets come from g_lsb_rec_off past bit 7,
    narrow components scattered over the band and wide ones overlapping many chunks."""
    rng = np.random.default_rng(900 + ncomp + (width == "wide"))
    sigma = (0.1, 0.6) if width == "narrow" else (3.0, 15.0)
    P = gauss_params(rng, 192, ncomp, 95.0, sigma)
    gauss_check(nb, rng, ncomp, P, P[:3].copy(), f"Gauss NC={ncomp} {width}")


def gauss_list_passes(P, ncomp, x, rest):
    """For each vector, (entries of the work list of super-block 0, the chunk whose entries straddle entry 256 or
    -1): the window rule and the (chunk, component) overlap count of nf_gauss_kernel."""
    nu_min, inv_chan, n = x[0], 1.0 / (x[1] - x[0]), x.shape[0]
    out = []
    for row in P:
        voff, sig = row[:ncomp], row[ncomp:2 * ncomp]
        w = sig / orc.CKMS * rest
        rel = rest * (1.0 - voff / orc.CKMS) - nu_min
        lo = np.floor((rel - 5 * np.abs(w)) * inv_chan).astype(int)
        hi = np.floor((rel + 5 * np.abs(w)) * inv_chan).astype(int)
        on = ~((hi < 0) | (lo > n - 1))
        lo, hi = np.maximum(lo, 0), np.minimum(hi, n - 1)
        on &= hi > lo
        per_chunk = np.zeros(32, dtype=int)
        for c in np.flatnonzero(on):
            per_chunk[lo[c] >> 7:((hi[c] - 1) >> 7) + 1] += 1
        first = np.cumsum(per_chunk) - per_chunk
        split = np.flatnonzero((first < 256) & (first + per_chunk > 256))
        out.append((int(per_chunk.sum()), int(split[0]) if split.size else -1))
    return out


def test_gauss_work_list_second_pass(nb):
    """32 components, each about 10 of the 32 chunks of the super-block wide (window +-5 sigma = 1280 channels at
    sigma = 6.4 km/s on 0.05 km/s channels), centres spread over the band: about 320 (chunk, component) entries,
    more than the NF_GAUSS_LIST_CAP = 256 a pass holds.  The test counts the entries with the kernel's window rule
    and keeps the vectors for which there are more than 256 and one chunk's entries straddle entry 256, so that
    chunk's model sums carry from the first pass into the second (about 7 in 8 of the draws)."""
    rng = np.random.default_rng(256)
    ncomp, B = 32, 192
    x = axis(orc.NU[0], GAUSS_N, GAUSS_DV)
    centres = np.linspace(-85.0, 85.0, ncomp)
    P = np.concatenate([centres + rng.uniform(-3, 3, (B, ncomp)), rng.uniform(6.0, 6.8, (B, ncomp)),
                        rng.uniform(0.1, 5.0, (B, ncomp))], axis=1)
    P[:, :ncomp] = P[:, rng.permutation(ncomp)]          # components in no particular order
    passes = gauss_list_passes(P, ncomp, x, orc.NU[0])
    keep = np.array([n > 256 and split >= 0 for n, split in passes])
    P, passes = P[keep], [q for q, k in zip(passes, keep) if k]
    assert P.shape[0] >= 128
    print(f"\n  work list: {min(n for n, _ in passes)} .. {max(n for n, _ in passes)} entries, chunks "
          f"{sorted({s for _, s in passes})} straddle entry 256", end="")
    gauss_check(nb, rng, ncomp, P, P[:3].copy(), "Gauss NC=32 two-pass list")


def test_gauss_ncomp_33_refused(nb):
    from nestfit_b200 import _lib
    x = axis(orc.NU[0], 512, 0.1)
    blk = nb.PixelBlock("gaussian", [x], np.zeros((1, 1, 512)), 0.1, rest_freq=orc.NU[0])
    with pytest.raises(_lib.NfError):
        blk.loglike(np.zeros((4, 99)), 33, vecs_per_pix=4)
    with pytest.raises(_lib.NfError):
        blk.predict(np.zeros((4, 99)), 33)
    blk.close()


# ---- D. Gaussian rows too long to stage --------------------------------------------------------------------------
@pytest.mark.parametrize("n_chan", [51840, 65535])
def test_gauss_long_rows(nb, n_chan):
    """51840 channels is the longest row whose staged pixel fits: 128 + 51840 x 4 + 8 x 3072 = 232064 B <= 232448 B.
    65535 channels (the most a block takes) needs 286848 B staged, so the kernel reads every pixel from HBM."""
    assert (gauss_smem_bytes(n_chan) <= SMEM_MAX) == (n_chan == 51840)
    assert gauss_smem_bytes(51841) > SMEM_MAX
    rng = np.random.default_rng(n_chan)
    ncomp, dv = 8, 0.05
    half = 0.5 * n_chan * dv
    P = gauss_params(rng, 96, ncomp, 0.95 * half, (0.3, 20.0))
    gauss_check(nb, rng, ncomp, P, P[:2].copy(), f"Gauss {n_chan} ch", n=n_chan, dv=dv, n_pred=8)


# ---- E. wide bands ------------------------------------------------------------------------------------------------
def band_limit_kms():
    from nestfit_b200 import _lib
    return _lib.NF_MAX_BAND_FRAC * orc.CKMS


def wide_band_case(nb, model, tids, band_kms, seed):
    """4000 channels over `band_kms`, four optically thick components spread over the band (so the spectrum's peak
    sits where the brightness amplitude is evaluated), tex over the whole prior with a quarter of the vectors in
    [2.8, 3.5] K, where the amplitude's approximation is worst."""
    rng = np.random.default_rng(seed)
    n, ncomp, B = 4000, 4, 192
    dv = band_kms / (n - 1)
    xs = [[axis(f, n, dv) for f in rest_freqs(model, tids)]] * 3
    vspan = 0.4 * band_kms

    def gen(k):
        tex = np.where(np.arange(k)[:, None] % 4 == 0, rng.uniform(2.8, 3.5, (k, ncomp)), rng.uniform(*TEX, (k, ncomp)))
        if model == "ammonia":
            P = nh3_params(rng, k, ncomp, vspan=vspan, ntot=(14.5, 16.5), ortho=False)
            P[:, 2 * ncomp:3 * ncomp] = tex
        else:
            P = n2hp_params(rng, k, ncomp, vspan=vspan)
            P[:, ncomp:2 * ncomp] = tex
            P[:, 2 * ncomp:3 * ncomp] = rng.uniform(0.5, 1.5, (k, ncomp))
        return P
    truth = gen(3)
    pb = Problem(nb, model, xs, tids, ncomp, truth, rng)
    P = gen(B)
    P[:3] = truth
    pb.check(P, ragged_pix(rng, 3, B), f"{model} {tids} band {band_kms:.0f} km/s", n_pred=64)
    pb.close()


def accepted_bands():
    return [70.0, 150.0, 220.0, 0.995 * band_limit_kms()]


@pytest.mark.parametrize("model, tids", [("ammonia", [1, 2]), ("diazenylium", [1])])
@pytest.mark.parametrize("k_band", range(4))
def test_wide_band(nb, model, tids, k_band):
    """Bands from 70 km/s to just inside NF_MAX_BAND_FRAC: the kernel's brightness amplitude (T0 and tbg linear in
    the channel, G the larger of two lines from the table segments at the band edges) against the oracle's
    per-channel T0_j (G(T0_j / tex) - tbg_j)."""
    wide_band_case(nb, model, tids, accepted_bands()[k_band], seed=1000 + k_band)


@pytest.mark.parametrize("model, tid", [("ammonia", 1), ("ammonia", 9), ("diazenylium", 1), ("diazenylium", 3)])
def test_band_past_limit_refused(nb, model, tid):
    """An axis whose (nu_last - nu_first) / nu_first is 0.2 % past NF_MAX_BAND_FRAC is refused by PixelBlock,
    PixelBlock.from_spectra and the three C entry points that upload a block; one 0.2 % inside it is accepted."""
    import torch
    from nestfit_b200 import _lib
    lib = _lib.load()
    lim = _lib.NF_MAX_BAND_FRAC
    code = nb.pixels._MODELS[model]
    nu0 = rest_freqs(model, [tid])[0]
    n = 2000
    tids = np.array([tid], dtype=np.int32)
    noise = np.array([0.1])
    for scale, ok in ((0.998, True), (1.002, False)):
        nu_chan = nu0 * lim * scale / (n - 1)
        x = nu0 + np.arange(n) * nu_chan
        data = np.zeros((1, 1, n))
        spectra = [[SimpleNamespace(xarr=x, data=data[0, 0], noise=0.1, trans_id=tid, rest_freq=None)]]
        if ok:
            nb.PixelBlock(model, [x], data, 0.1, trans_ids=[tid]).close()
            nb.PixelBlock.from_spectra(model, spectra).close()
            continue
        with pytest.raises(ValueError, match="NF_MAX_BAND_FRAC"):
            nb.PixelBlock(model, [x], data, 0.1, trans_ids=[tid])
        with pytest.raises(ValueError, match="NF_MAX_BAND_FRAC"):
            nb.PixelBlock.from_spectra(model, spectra)
        nu_min, nu_ch = np.array([x[0]]), np.array([nu_chan])
        out = C.c_void_p()
        assert lib.nf_pixels_create(0, code, 1, 1, n, _lib.ptr(nu_min), _lib.ptr(nu_ch), _lib.ptr(tids), None,
                                    _lib.ptr(data), _lib.NF_F64, _lib.ptr(noise), C.byref(out)) == -1
        n_chan = np.array([n], dtype=np.int32)
        assert lib.nf_pixels_create_axes(0, code, 1, 1, n, _lib.ptr(nu_min), _lib.ptr(nu_ch), _lib.ptr(n_chan),
                                         _lib.ptr(tids), None, _lib.ptr(data), _lib.NF_F64, _lib.ptr(noise),
                                         C.byref(out)) == -1
        d_dev = torch.zeros(n, dtype=torch.float32, device="cuda:0")
        s_dev = torch.full((1,), 0.1, dtype=torch.float64, device="cuda:0")
        assert lib.nf_pixels_create_from_device(0, code, 1, 1, n, _lib.ptr(nu_min), _lib.ptr(nu_ch), _lib.ptr(tids),
                                                None, C.c_void_p(d_dev.data_ptr()), C.c_void_p(s_dev.data_ptr()),
                                                C.byref(out)) == -1
        assert not out.value
