"""GPU tests of the intensity credible intervals: the moments mode of the hyperfine kernel against the predicted
spectra and the oracle, and nf_ns_intensity (through CubeFitter, NestedSamplingBatch and run_multinest_batch)
against a host recomputation from the stored posteriors."""
import numpy as np
import pytest

from oracle import oracle as orc
from nestfit_b200.pixels import channel_kms
from nestfit_b200.sampler import weighted_quantiles
from nestfit_b200.store import INTENSITY_DATASETS, MARG_QUANTILES

pytestmark = pytest.mark.gpu
M = MARG_QUANTILES.size


def axis(nu0, n, dv, v0=0.0):
    """Ascending frequency axis of n channels of dv km/s centred on velocity v0."""
    v = v0 + (np.arange(n) - 0.5 * (n - 1)) * dv
    return np.sort(nu0 * (1.0 - v / orc.CKMS))


def prior_vectors(nb, model, rng, n):
    """Single-component vectors drawn from the priors; a quarter of them moved far outside the band."""
    if model == "ammonia":
        ut = nb.get_irdc_priors()
        P = orc.prior_transform(ut.pack(), rng.uniform(0.02, 0.98, size=(3 * n, 6)), 1)
        P = P[np.isfinite(P).all(axis=1)][:n]
    else:
        P = np.stack([rng.uniform(-4, 4, n), rng.uniform(3, 12, n), rng.uniform(-1, 1.3, n),
                      rng.uniform(0.08, 1.2, n)], axis=1)
    P[::4, 0] += rng.choice([-1, 1], P[::4].shape[0]) * rng.uniform(60, 150, P[::4].shape[0])
    return P


def spectra_of(nb, model, xs, data, noise, tids):
    cls = nb.AmmoniaSpectrum if model == "ammonia" else nb.DiazenyliumSpectrum
    return [[cls(xs[p][s], data[p][s], noise, tids[s]) for s in range(len(tids))] for p in range(len(xs))]


@pytest.mark.parametrize("model", ["ammonia", "diazenylium"])
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("per_pixel_axes", [False, True])
def test_moments_kernel(nb, model, dtype, per_pixel_axes):
    rng = np.random.default_rng(7 + per_pixel_axes + 2 * (dtype == np.float32) + 4 * (model == "ammonia"))
    tids = [1, 2]
    nu = orc.NU[:2] if model == "ammonia" else orc.N2HP_NU[:2]
    n_pix, n = 5, 600
    if per_pixel_axes:         # unequal lengths, one spectrum past the 1024-channel super-block
        lens = rng.integers(150, 1100, size=(n_pix, 2))
        lens[0] = [1100, 1030]
        xs = [[axis(nu[s], int(lens[p, s]), rng.uniform(0.05, 0.2), rng.uniform(-2, 2)) for s in range(2)]
              for p in range(n_pix)]
        data = [[np.zeros(len(x)) for x in xp] for xp in xs]
        blk = nb.PixelBlock.from_spectra(model, spectra_of(nb, model, xs, data, 0.1, tids))
    else:
        xs = [[axis(f, 1100, 0.1 + 0.02 * s) for s, f in enumerate(nu)]] * n_pix
        blk = nb.PixelBlock(model, xs[0], np.zeros((n_pix, 2, 1100), np.float32), 0.1, trans_ids=tids)
    P = prior_vectors(nb, model, rng, n).astype(dtype)
    pv = rng.integers(0, n_pix, n).astype(np.int32)
    peak, total = blk.moments(P, pix_of_vec=pv)
    pred = blk.predict(P, 1, pix_of_vec=pv)
    assert peak.dtype == np.float32 and total.dtype == np.float64 and peak.shape == (n, 2)
    if not per_pixel_axes:            # without a map: the same numbers
        p2, t2 = blk.moments(P)
        np.testing.assert_array_equal(p2, peak)
        np.testing.assert_array_equal(t2, total)
    oracle = orc.nh3_batch if model == "ammonia" else orc.n2hp_batch
    P64 = P.astype(np.float64)
    n_out = 0
    for s in range(2):
        for p in range(n_pix):
            sel = np.flatnonzero(pv == p)
            nch = len(xs[p][s])
            row = pred[sel, s, :nch]
            np.testing.assert_array_equal(peak[sel, s], row.max(axis=1))
            want_sum = row.sum(axis=1, dtype=np.float64)
            assert (np.abs(total[sel, s] - want_sum) <= 1e-12 * np.abs(row).sum(axis=1, dtype=np.float64)).all()
            wp = oracle([xs[p][s]], [tids[s]], P64[sel], 1, want_pred=True)["pred"][:, 0]
            wpk = wp.max(axis=1)
            scale = np.maximum(np.abs(wp).max(axis=1), 1e-30)
            assert (np.abs(peak[sel, s] - wpk) <= 1e-5 * scale).all()
            assert (np.abs(total[sel, s] - wp.sum(axis=1)) <= 1e-5 * scale * nch).all()
            n_out += int((np.abs(wp).max(axis=1) < 1e-12).sum())
    assert n_out > 0                                                 # components outside the band were scored
    blk.close()


def stable_weighted_quantiles(x, w, q):
    """sampler.weighted_quantiles with equal values kept in row order (argsort kind='stable').  Duplicate posterior
    rows (a final live point equal to a dead point) give equal values with different weights, and the interpolation
    then depends on their order, which numpy's default argsort leaves unspecified; the device keeps row order."""
    out = np.empty((len(q), x.shape[1]))
    for j in range(x.shape[1]):
        o = np.argsort(x[:, j], kind="stable")
        cw = np.cumsum(w[o])
        cw /= cw[-1]
        out[:, j] = np.interp(q, cw, x[o, j])
    return out


def test_stable_variant_is_weighted_quantiles_without_ties():
    rng = np.random.default_rng(0)
    x, w = rng.normal(size=(500, 3)), rng.exponential(size=500)
    np.testing.assert_array_equal(stable_weighted_quantiles(x, w, MARG_QUANTILES),
                                  weighted_quantiles(x, w, MARG_QUANTILES))


def host_intensity(blk, post, ncomp, pix, n_own, kms, cold=False, lte=False):
    """The run's intensity quantiles from its posterior rows (theta, lnL, weight), on the host: PixelBlock.predict
    of each row's components, max / FP64 sum over the spectrum's own channels, (stable) weighted_quantiles."""
    n_model = blk.n_model
    th = np.ascontiguousarray(post[:, :n_model * ncomp], dtype=np.float32)
    w = post[:, -1].astype(np.float64)
    out = {k: np.empty((M, blk.n_spec, ncomp)) for k in INTENSITY_DATASETS}
    rng_of = {k: np.empty((blk.n_spec, ncomp)) for k in INTENSITY_DATASETS}
    for c in range(ncomp):
        P = np.ascontiguousarray(th[:, c::ncomp])
        pv = np.full(P.shape[0], pix, dtype=np.int32) if blk.per_pixel_axes else None
        pred = blk.predict(P, 1, cold=cold, lte=lte, pix_of_vec=pv)
        for s in range(blk.n_spec):
            row = pred[:, s, :n_own[s]]
            for name, x in (("peak_intensity_marginals", row.max(axis=1).astype(np.float64)),
                            ("integrated_intensity_marginals", row.sum(axis=1, dtype=np.float64) * kms[s])):
                out[name][:, s, c] = stable_weighted_quantiles(x[:, None], w, MARG_QUANTILES)[:, 0]
                rng_of[name][s, c] = x.max() - x.min() + 1e-13 * np.abs(x).max()
    return out, rng_of


def assert_close(got, want, rng_of):
    for name in INTENSITY_DATASETS:
        assert got[name].shape == want[name].shape
        err = np.abs(np.asarray(got[name]) - want[name])
        assert (err <= 1e-9 * rng_of[name][None] + 1e-300).all(), (name, (err / rng_of[name][None]).max())


def _fit(nb, stack, ut, path, intensity):
    from nestfit_b200.models import ammonia
    fitter = nb.CubeFitter(stack, ut, ammonia.AmmoniaRunner, ncomp_max=2, mn_kwargs={'nlive': 80}, n_prop=32,
                           lnZ_thresh=11, seed=5, intensity_marginals=intensity)
    return fitter.fit_cube(str(path), nproc=1)[0]


def test_cube_fit_intensity(nb, tmp_path):
    from nestfit_b200.synth import make_synth_stack
    ut = nb.get_irdc_priors()
    rng = np.random.default_rng(11)
    ncomp_map = rng.integers(0, 3, size=(8, 8))
    stack = make_synth_stack((8, 8), ut, ncomp_map=ncomp_map, n_chan=400, dv=0.158, noise=0.1, seed=12)
    on = _fit(nb, stack, ut, tmp_path / 'on', True)
    off = _fit(nb, stack, ut, tmp_path / 'off', False)
    assert on['intensity_seconds'] > 0 and off['intensity_seconds'] == 0
    np.testing.assert_array_equal(on['nbest'], off['nbest'])
    np.testing.assert_array_equal(on['lnZ'], off['lnZ'])
    s_on, s_off = nb.HdfStore(str(tmp_path / 'on')), nb.HdfStore(str(tmp_path / 'off'))
    blk = nb.PixelBlock("ammonia", [c.xarr for c in stack.cubes], np.zeros((1, 2, 400), np.float32), 1.0,
                        trans_ids=[c.trans_id for c in stack.cubes])
    kms = np.array([c.dv for c in stack.cubes])
    n_runs = 0
    for g in s_on.iter_pix_groups():
        g_off = s_off.hdf[f"/pix/{g.attrs['i_lon']}/{g.attrs['i_lat']}"]
        for key in g:
            run, run_off = g[key], g_off[key]
            for name in ('posteriors', 'marginals', 'bestfit_params', 'map_params'):       # nothing else moves
                np.testing.assert_array_equal(np.asarray(run[name]), np.asarray(run_off[name]))
            assert run.attrs['global_lnZ'] == run_off.attrs['global_lnZ']
            assert not any(name in run_off for name in INTENSITY_DATASETS)
            ncomp = int(key)
            want, rng_of = host_intensity(blk, np.asarray(run['posteriors']), ncomp, 0, [400, 400], kms)
            assert_close({n: np.asarray(run[n]) for n in INTENSITY_DATASETS}, want, rng_of)
            n_runs += 1
    assert n_runs >= 64
    nb.aggregate_run_attributes(s_on)
    nb.aggregate_intensity_marginals(s_on)
    pk = np.asarray(s_on.hdf[f'{s_on.dpath}/nbest_peak_intensity_marginals'])
    assert pk.shape == (2, 2, M, 8, 8)
    nbest = on['nbest'].reshape(8, 8)
    lon, lat = np.argwhere(nbest == nbest.max())[0]
    run = s_on.hdf[f'/pix/{lon}/{lat}/{nbest.max()}']
    np.testing.assert_array_equal(pk[:, :nbest.max(), :, lat, lon],
                                  np.asarray(run['peak_intensity_marginals']).transpose(1, 2, 0))
    s_on.close()
    s_off.close()
    blk.close()


def test_large_run_uses_global_scratch(nb):
    from nestfit_b200 import _lib
    from nestfit_b200.sampler import NestedSamplingBatch
    rng = np.random.default_rng(21)
    xs = [axis(orc.NU[0], 500, 0.158), axis(orc.NU[1], 500, 0.158)]
    truth = np.array([0.3, 14.0, 7.0, 15.0, 0.45, 0.0])
    clean = orc.nh3_batch(xs, [1, 2], truth[None], 1, want_pred=True)["pred"][0]
    data = (clean[None] + rng.normal(0, 0.05, (2,) + clean.shape)).astype(np.float32)
    blk = nb.PixelBlock("ammonia", xs, data, 0.05, trans_ids=[1, 2])
    ns = NestedSamplingBatch(blk, nb.get_irdc_priors(), 1, nlive=[1000, 100], tol=0.5, n_prop=32, seed=3)
    ns.run()
    q = np.ascontiguousarray(MARG_QUANTILES)
    out = np.empty((2, M, 2, 1))
    # before nf_ns_products_rows there are no row offsets to work from
    assert _lib.load().nf_ns_intensity(ns.handle, _lib.ptr(q), M, _lib.ptr(out), _lib.ptr(out)) == -1
    prod = ns.products_all(marginals=False, posteriors=True)
    off = prod["row_offsets"]
    assert off[1] - off[0] > 8192 >= off[2] - off[1]                 # one run beyond the shared-memory sort
    got = ns.intensity_marginals()
    kms = np.array([channel_kms(x) for x in xs])
    for r in range(2):
        want, rng_of = host_intensity(blk, prod["posteriors"][off[r]:off[r + 1]], 1, r, [500, 500], kms)
        assert_close({n: got[n][r] for n in INTENSITY_DATASETS}, want, rng_of)
    ns.close()
    blk.close()


def test_run_multinest_batch_intensity(nb):
    from nestfit_b200.sampler import Dumper
    from nestfit_b200.store import MemGroup
    rng = np.random.default_rng(31)
    ut = nb.get_irdc_priors()
    runners, xss = [], []
    for k in range(4):
        vs = rng.uniform(-1, 1)
        truth = np.array([vs, 13.0, 6.0, 14.7, 0.4, 0.0])
        xs = [axis(orc.NU[t], int(rng.integers(300, 900)), rng.uniform(0.08, 0.2), vs) for t in (0, 1)]
        spec = [[x, orc.nh3_batch([x], [s + 1], truth[None], 1, want_pred=True)["pred"][0, 0]
                 + rng.normal(0, 0.15, len(x)), 0.15, s + 1] for s, x in enumerate(xs)]
        runners.append(nb.AmmoniaRunner.from_data(spec, ut, ncomp=1))
        xss.append(xs)
    groups = [MemGroup(f"/pix/{i}/0/1") for i in range(4)]
    nb.run_multinest_batch(runners, [Dumper(g) for g in groups], nlive=100, seed=4, tol=1.0,
                           intensity_marginals=True)
    for r, g, xs in zip(runners, groups, xss):
        kms = np.array([channel_kms(x) for x in xs])
        blk = r._block
        want, rng_of = host_intensity(blk, np.asarray(g['posteriors']), 1, 0, [len(x) for x in xs], kms)
        assert_close({n: g[n] for n in INTENSITY_DATASETS}, want, rng_of)
        assert g['integrated_intensity_marginals'].shape == (M, 2, 1)


def test_run_multinest_batch_intensity_n2hp(nb):
    """The N2H+ branch of nf_ns_intensity: J = 1-0 and 3-2 spectra of unequal lengths, two components."""
    from nestfit_b200.models import diazenylium as dz
    from nestfit_b200.sampler import Dumper
    from nestfit_b200.store import MemGroup
    rng = np.random.default_rng(41)
    size = 200
    u = np.linspace(0, 1, size)
    flat = np.ones(size) / size
    ut = nb.PriorTransformer(np.array([
        nb.OrderedPrior(nb.Distribution(12 * u - 6, flat), 0), nb.Prior(nb.Distribution(22 * u + 3, flat), 1),
        nb.Prior(nb.Distribution(3 * u - 1.5, flat), 2), nb.Prior(nb.Distribution(1.5 * u + 0.07, flat), 3)],
        dtype=object))
    truth = np.array([-1.2, 1.4, 8.0, 6.0, 0.3, -0.2, 0.35, 0.5])
    runners, xss = [], []
    for k in range(3):
        xs = [axis(orc.N2HP_NU[t - 1], int(rng.integers(300, 800)), rng.uniform(0.08, 0.16), rng.uniform(-1, 1))
              for t in (1, 3)]
        spec = [[x, orc.n2hp_batch([x], [t], truth[None], 2, want_pred=True)["pred"][0, 0]
                 + rng.normal(0, 0.1, len(x)), 0.1, t] for x, t in zip(xs, (1, 3))]
        runners.append(dz.DiazenyliumRunner.from_data(spec, ut, ncomp=2))
        xss.append(xs)
    groups = [MemGroup(f"/pix/{i}/0/2") for i in range(3)]
    nb.run_multinest_batch(runners, [Dumper(g) for g in groups], nlive=100, seed=6, tol=1.0,
                           intensity_marginals=True)
    for r, g, xs in zip(runners, groups, xss):
        kms = np.array([channel_kms(x) for x in xs])
        want, rng_of = host_intensity(r._block, np.asarray(g['posteriors']), 2, 0, [len(x) for x in xs], kms)
        assert_close({n: g[n] for n in INTENSITY_DATASETS}, want, rng_of)
        assert g['peak_intensity_marginals'].shape == (M, 2, 2)
        # the brighter component's median peak is well above the noise
        assert np.asarray(g['peak_intensity_marginals'])[4].max() > 0.5
