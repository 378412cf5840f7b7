"""GPU tests of pixel blocks whose spectra each have their own axis and length (PixelBlock.from_spectra,
nf_pixels_create_axes) and of run_multinest_batch, the batched form of run_multinest over a list of runners:
bit-identity with the shared-axis block when every pixel has the same axis, parity with the C oracle on
per-pixel axes, runners with spectra of unequal lengths, and the batched fit of a catalogue."""
import numpy as np
import pytest

from oracle import oracle as orc

pytestmark = pytest.mark.gpu


def axis(nu0, n, dv, v0=0.0):
    """Ascending frequency axis of n channels of dv km/s centred on velocity v0."""
    v = v0 + (np.arange(n) - 0.5 * (n - 1)) * dv
    return np.sort(nu0 * (1.0 - v / orc.CKMS))


def spectra_of(nb, model, xs, data, noise, tids=None, rest_freq=None):
    """Pixel p's spectra as the package's Spectrum objects: xs[p][s], data[p][s], noise[p][s]."""
    out = []
    for p in range(len(xs)):
        if model == "gaussian":
            out.append([nb.Spectrum(xs[p][0], data[p][0], noise[p][0], rest_freq=rest_freq[p])])
        else:
            cls = nb.AmmoniaSpectrum if model == "ammonia" else nb.DiazenyliumSpectrum
            out.append([cls(xs[p][s], data[p][s], noise[p][s], tids[s]) for s in range(len(tids))])
    return out


def nh3_params(nb, rng, n, ncomp):
    ut = nb.get_irdc_priors()
    P = orc.prior_transform(ut.pack(), rng.uniform(0.05, 0.95, size=(3 * n, 6 * ncomp)), ncomp)
    return P[np.isfinite(P).all(axis=1)][:n]


def n2hp_params(rng, n, ncomp):
    return np.concatenate([rng.uniform(-3, 3, (n, ncomp)), rng.uniform(3, 10, (n, ncomp)),
                           rng.uniform(-1, 1, (n, ncomp)), rng.uniform(0.1, 1.0, (n, ncomp))], axis=1)


def gauss_params(rng, n, ncomp):
    return np.concatenate([rng.uniform(-5, 5, (n, ncomp)), rng.uniform(0.3, 2.0, (n, ncomp)),
                           rng.uniform(0.0, 3.0, (n, ncomp))], axis=1)


CASES = [("ammonia", 1), ("ammonia", 2), ("ammonia", 3), ("ammonia", 4), ("diazenylium", 2), ("gaussian", 3)]


def shared_problem(nb, model, ncomp, rng, n_pix=5, vpp=64):
    """A shared-axis block and the same pixels as a per-pixel-axes block."""
    if model == "ammonia":
        tids, nu = [1, 2], [orc.NU[0], orc.NU[1]]
        P = nh3_params(nb, rng, n_pix * vpp, ncomp)
    elif model == "diazenylium":
        tids, nu = [1, 2], orc.N2HP_NU[:2]
        P = n2hp_params(rng, n_pix * vpp, ncomp)
    else:
        tids, nu = None, [orc.NU[0]]
        P = gauss_params(rng, n_pix * vpp, ncomp)
    xs = [axis(f, 700, 0.1) for f in nu]
    data = rng.normal(0.0, 0.3, (n_pix, len(xs), 700)).astype(np.float32)
    noise = rng.uniform(0.1, 0.3, (n_pix, len(xs)))
    if model == "gaussian":
        shared = nb.PixelBlock(model, xs, data, noise, rest_freq=orc.NU[0])
    else:
        shared = nb.PixelBlock(model, xs, data, noise, trans_ids=tids)
    spectra = spectra_of(nb, model, [xs] * n_pix, data.astype(np.float64), noise, tids, [orc.NU[0]] * n_pix)
    return shared, nb.PixelBlock.from_spectra(model, spectra), P


@pytest.mark.parametrize("model, ncomp", CASES)
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_shared_axes_bit_identical(nb, model, ncomp, dtype):
    rng = np.random.default_rng(ncomp + 10 * len(model))
    n_pix, vpp = 5, 64
    shared, perpix, P = shared_problem(nb, model, ncomp, rng, n_pix, vpp)
    P = P.astype(dtype)
    assert perpix.per_pixel_axes and perpix.n_chan.shape == (n_pix, shared.n_spec)
    np.testing.assert_array_equal(perpix.null_lnZ(), shared.null_lnZ())
    for pv in (np.repeat(np.arange(n_pix), vpp), np.tile(np.arange(n_pix), vpp)):     # contiguous, interleaved
        pv = pv.astype(np.int32)
        a = shared.loglike(P, ncomp, pix_of_vec=pv)
        b = perpix.loglike(P, ncomp, pix_of_vec=pv)
        assert np.isfinite(a).all()
        np.testing.assert_array_equal(a, b)
    np.testing.assert_array_equal(shared.loglike(P, ncomp, vecs_per_pix=vpp), perpix.loglike(P, ncomp, vecs_per_pix=vpp))
    pv = np.tile(np.arange(n_pix), vpp)[:96].astype(np.int32)
    want = shared.predict(P[:96], ncomp)
    np.testing.assert_array_equal(perpix.predict(P[:96], ncomp, pix_of_vec=pv), want)
    np.testing.assert_array_equal(shared.predict(P[:96], ncomp, pix_of_vec=pv), want)
    with pytest.raises(ValueError):
        perpix.predict(P[:4], ncomp)
    shared.close()
    perpix.close()


def test_existing_predict_refuses_per_pixel_axes(nb):
    from nestfit_b200 import _lib
    shared, perpix, P = shared_problem(nb, "ammonia", 1, np.random.default_rng(1), n_pix=2, vpp=4)
    P = np.ascontiguousarray(P)
    out = np.empty((P.shape[0], 2, 700), dtype=np.float32)
    rc = _lib.load().nf_nh3_predict_host(perpix.handle, _lib.ptr(P), _lib.NF_F64, P.shape[0], 1, 0, _lib.ptr(out))
    assert rc == -1                                               # NF_EINVAL: no pixel map
    shared.close()
    perpix.close()


def test_sampler_identical_on_both_blocks(nb):
    from nestfit_b200.sampler import NestedSamplingBatch
    rng = np.random.default_rng(5)
    xs = [orc.bench_axis(1, 400, 0.158), orc.bench_axis(2, 400, 0.158)]
    truth = np.array([0.5, 14.0, 6.0, 14.6, 0.45, 0.0])
    clean = orc.nh3_batch(xs, [1, 2], truth[None], 1, want_pred=True)["pred"][0]
    data = (clean[None] + rng.normal(0, 0.1, (3,) + clean.shape)).astype(np.float32)
    shared = nb.PixelBlock("ammonia", xs, data, 0.1, trans_ids=[1, 2])
    perpix = nb.PixelBlock.from_spectra("ammonia", spectra_of(nb, "ammonia", [xs] * 3, data.astype(np.float64),
                                                                np.full((3, 2), 0.1), [1, 2]))
    ut = nb.get_irdc_priors()
    res = [NestedSamplingBatch(b, ut, 1, nlive=100, tol=1.0, n_prop=32, seed=11).run() for b in (shared, perpix)]
    for key in ("lnZ", "n_evals", "bestfit", "n_samples"):
        np.testing.assert_array_equal(res[0][key], res[1][key])


def catalogue_axes(rng, n_pix, nu, lo=200, hi=1100, vspan=20.0):
    """Per pixel and spectrum: velocity offset, channel width and length of its own."""
    v0 = rng.uniform(-vspan, vspan, n_pix)
    xs = []
    for p in range(n_pix):
        n = rng.integers(lo, hi + 1, size=len(nu))
        if p == 0:
            n[:] = [1100, 1030][:len(nu)]          # one spectrum past the 1024-channel super-block
        if p == 1 and len(nu) > 1:
            n[:] = [379, 381]
        dv = rng.uniform(0.05, 0.2, size=len(nu))
        xs.append([axis(f, int(n[s]), dv[s], v0[p] + rng.uniform(-1, 1)) for s, f in enumerate(nu)])
    return xs, v0


def oracle_model(model, x, tid, P, ncomp, data=None, noise=None, rest_freq=None):
    kw = dict(data=None if data is None else data[None, None], noise=noise, want_pred=data is None)
    if model == "ammonia":
        o = orc.nh3_batch([x], [tid], P, ncomp, **kw)
    elif model == "diazenylium":
        o = orc.n2hp_batch([x], [tid], P, ncomp, **kw)
    else:
        kw["data"] = None if data is None else data[None]
        o = orc.gauss_batch(x, rest_freq, P, ncomp, **kw)
        return o["lnL"] if data is not None else o["pred"]
    return o["lnL"] if data is not None else o["pred"][:, 0]


@pytest.mark.parametrize("model, ncomp", [("ammonia", 1), ("ammonia", 3), ("diazenylium", 2), ("gaussian", 2)])
def test_per_pixel_axes_against_oracle(nb, model, ncomp):
    rng = np.random.default_rng(100 + ncomp)
    n_pix, vpp = 8, 96
    tids = {"ammonia": [1, 2], "diazenylium": [1, 2], "gaussian": [None]}[model]
    nu = {"ammonia": orc.NU[:2], "diazenylium": orc.N2HP_NU[:2], "gaussian": [orc.NU[0]]}[model]
    xs, v0 = catalogue_axes(rng, n_pix, nu)
    gen = {"ammonia": lambda n: nh3_params(nb, rng, n, ncomp), "diazenylium": lambda n: n2hp_params(rng, n, ncomp),
           "gaussian": lambda n: gauss_params(rng, n, ncomp)}[model]
    truth = gen(n_pix)
    truth[:, :ncomp] += v0[:, None]
    # per pixel: the truth, the truth perturbed on scales 1e-4 .. 0.3, and plain draws around the pixel's velocity
    P = np.repeat(truth, vpp, axis=0)
    scale = 10.0 ** rng.uniform(-4, -0.5, size=(n_pix * vpp, 1))
    P = P * (1 + scale * rng.normal(size=P.shape))
    far = np.tile(np.arange(vpp) >= vpp // 2, n_pix)
    P[far] = gen(int(far.sum()))
    P[far, :ncomp] += np.repeat(v0, vpp // 2)[:, None]
    P[::vpp] = truth
    rest = (1.0 + rng.uniform(-1e-5, 1e-5, n_pix)) * orc.NU[0]        # Gaussian model: a rest frequency per pixel
    noise = rng.uniform(0.05, 0.2, (n_pix, len(nu)))
    data = []
    for p in range(n_pix):
        row = []
        for s in range(len(nu)):
            clean = oracle_model(model, xs[p][s], tids[s], truth[p:p + 1], ncomp, rest_freq=rest[p])[0]
            row.append((clean + rng.normal(0, noise[p, s], clean.shape)).astype(np.float32).astype(np.float64))
        data.append(row)
    blk = nb.PixelBlock.from_spectra(model, spectra_of(nb, model, xs, data, noise, tids, rest))
    assert blk.n_chan_max == 1100 and (blk.n_chan == np.array([[len(x) for x in xp] for xp in xs])).all()
    pv = np.tile(np.arange(n_pix), vpp).astype(np.int32)          # interleaved pixels
    perm = np.argsort(pv, kind="stable")                           # rows of P in interleaved order
    Pi = np.empty_like(P)
    Pi[perm] = P
    got = blk.loglike(Pi, ncomp, pix_of_vec=pv)[perm]
    pred = blk.predict(Pi, ncomp, pix_of_vec=pv)[perm]
    want = np.zeros(P.shape[0])
    for p in range(n_pix):
        sl = slice(p * vpp, (p + 1) * vpp)
        for s in range(len(nu)):
            n = len(xs[p][s])
            want[sl] += oracle_model(model, xs[p][s], tids[s], P[sl], ncomp, data=data[p][s], noise=noise[p, s],
                                     rest_freq=rest[p])
            wp = oracle_model(model, xs[p][s], tids[s], P[sl], ncomp, rest_freq=rest[p])
            peak = np.maximum(np.abs(wp).max(axis=1, keepdims=True), 1e-30)
            assert (np.abs(pred[sl, s, :n] - wp) / peak).max() < 1e-5
            assert (pred[sl, s, n:] == 0).all()
    err = np.abs(got - want)
    near = np.repeat(want.reshape(n_pix, vpp).max(axis=1), vpp) - want <= 1e3
    assert near.sum() >= n_pix
    assert err[near].max() <= 1e-3, f"bulk max |dlnL| {err[near].max():.3e}"
    assert (err[~near] <= 1e-6 * np.abs(want[~near])).all()
    blk.close()


def test_runner_with_unequal_lengths(nb):
    rng = np.random.default_rng(3)
    ut = nb.get_irdc_priors()
    xs = [axis(orc.NU[0], 379, 0.158), axis(orc.NU[1], 381, 0.15, 1.0)]
    truth = np.array([0.5, 14.0, 6.0, 14.6, 0.45, 0.0])
    data = [oracle_model("ammonia", x, t, truth[None], 1)[0] + rng.normal(0, 0.2, len(x)) for x, t in zip(xs, (1, 2))]
    runner = nb.AmmoniaRunner.from_data([[xs[0], data[0], 0.2, 1], [xs[1], data[1], 0.2, 2]], ut, ncomp=1)
    assert runner.n_chan_tot == 760 and runner._block.per_pixel_axes
    d32 = [d.astype(np.float32).astype(np.float64) for d in data]
    got, want = [], []
    for k in range(64):
        u = rng.uniform(0.05, 0.95, 6) if k else np.full(6, 0.5)
        lnl = runner.loglikelihood(u)                             # u is transformed in place
        if not np.isfinite(u).all():
            continue
        got.append(lnl)
        want.append(sum(oracle_model("ammonia", xs[s], s + 1, u[None], 1, data=d32[s], noise=0.2)[0] for s in range(2)))
    got, want = np.array(got), np.array(want)
    err = np.abs(got - want)
    near = want.max() - want <= 1e3
    assert (err[near] <= 1e-3).all() and (err[~near] <= 1e-6 * np.abs(want[~near])).all()
    runner.predict(truth)
    for s, spec in enumerate(runner.spectra):
        wp = oracle_model("ammonia", xs[s], s + 1, truth[None], 1)[0]
        assert spec.pred.shape == (len(xs[s]),)
        assert np.abs(spec.pred - wp).max() < 1e-5 * np.abs(wp).max()


def nh3_source(rng, ncomp_true, noise):
    """A (1,1)+(2,2) source on axes of its own (velocity centre, channel width, length 300-1100), with a
    known 1- or 2-component truth."""
    vsrc = rng.uniform(-1.5, 1.5)
    if ncomp_true == 1:
        truth = np.array([vsrc, rng.uniform(11, 16), rng.uniform(5, 7), rng.uniform(14.4, 14.8), rng.uniform(0.3, 0.6),
                          0.0])
    else:
        truth = np.array([vsrc - 1.3, vsrc + 1.3, 10, 15, 5, 6, 14.6, 14.9, 0.3, 0.5, 0, 0], dtype=float)
    xs = [axis(orc.NU[t - 1], int(rng.integers(300, 1101)), rng.uniform(0.08, 0.2), vsrc + rng.uniform(-3, 3))
          for t in (1, 2)]
    spec = []
    for s, x in enumerate(xs):
        clean = oracle_model("ammonia", x, s + 1, truth[None], ncomp_true)[0]
        spec.append([x, clean + rng.normal(0, noise, len(x)), noise, s + 1])
    return spec, truth


def test_run_multinest_batch_dumper_contract(nb):
    from nestfit_b200.sampler import Dumper, MARG_COLS
    from nestfit_b200.store import MemGroup
    rng = np.random.default_rng(8)
    ut = nb.get_irdc_priors()
    srcs = [nh3_source(rng, 1, 0.15)[0] for _ in range(4)]
    runners = [nb.AmmoniaRunner.from_data(s, ut, ncomp=1) for s in srcs]
    groups = [MemGroup(f"/pix/{i}/0/1") for i in range(4)]
    dumpers = [Dumper(g) for g in groups]
    res = nb.run_multinest_batch(runners, dumpers, nlive=[100, 120, 100, 120], seed=5, tol=1.0, max_runs_per_batch=3)
    assert res["lnZ"].shape == (4,) and not res["truncated"].any()
    for r, g, d, nl in zip(runners, groups, dumpers, (100, 120, 100, 120)):
        assert np.isfinite(r.run_lnZ) and r.run_lnZ == g.attrs['global_lnZ']
        for key in ('ncomp', 'null_lnZ', 'n_chan_tot', 'n_samples', 'n_live', 'n_params', 'global_lnZ',
                    'global_lnZ_err', 'max_loglike', 'marg_cols', 'marg_quantiles', 'BIC', 'AIC', 'AICc',
                    'null_BIC', 'null_AIC', 'null_AICc'):
            assert key in g.attrs
        assert g.attrs['n_chan_tot'] == r.n_chan_tot == sum(sp.size for sp in r.spectra) and g.attrs['null_lnZ'] == pytest.approx(r.null_lnZ)
        assert g.attrs['n_params'] == 6 and g.attrs['n_live'] == nl
        assert list(g.attrs['marg_cols']) == MARG_COLS
        n = g.attrs['n_samples']
        assert d.n_calls == 1 and d.n_samples == n
        assert g['posteriors'].shape == (n, 8) and g['posteriors'].dtype == np.float32
        assert g['marginals'].shape == (15, 6)
        assert g['bestfit_params'].shape == (6,) and g['map_params'].shape == (6,)
        k, nn, maxL = 6.0, float(r.n_chan_tot), g.attrs['max_loglike']
        assert g.attrs['BIC'] == pytest.approx(np.log(nn) * k - 2 * maxL)
    assert len({r.n_chan_tot for r in runners}) > 1


def test_run_multinest_batch_agrees_with_serial(nb):
    rng = np.random.default_rng(9)
    ut = nb.get_irdc_priors()
    srcs = [nh3_source(rng, 1, 0.15)[0] for _ in range(8)]
    batch = [nb.AmmoniaRunner.from_data(s, ut, ncomp=1) for s in srcs]
    res = nb.run_multinest_batch(batch, nlive=200, seed=1, tol=0.5)
    for i, s in enumerate(srcs):
        r = nb.AmmoniaRunner.from_data(s, ut, ncomp=1)
        one = nb.run_multinest(r, None, nlive=200, seed=100 + i, tol=0.5)
        tol = 4 * np.hypot(res["lnZ_err"][i], one["lnZ_err"][0])
        assert abs(batch[i].run_lnZ - r.run_lnZ) < tol, (i, batch[i].run_lnZ, r.run_lnZ, tol)


def test_catalogue_escalation(nb):
    """64 sources on axes of their own, 1 or 2 true components: the caller's escalation loop over
    run_multinest_batch at lnZ_thresh = 11 picks the true ncomp, and recovers velocity and width."""
    from nestfit_b200.sampler import Dumper
    from nestfit_b200.store import MemGroup
    rng = np.random.default_rng(64)
    ut = nb.get_irdc_priors()
    n_src, thresh = 64, 11.0
    true_nc = np.where(np.arange(n_src) % 3 == 0, 2, 1)
    cat = [nh3_source(rng, int(k), 0.12) for k in true_nc]
    best = np.zeros(n_src, dtype=int)
    lnZ_best = np.empty(n_src)
    active = np.arange(n_src)
    groups = {}
    for ncomp in (1, 2, 3):
        batch = [nb.AmmoniaRunner.from_data(cat[i][0], ut, ncomp=ncomp) for i in active]
        dumpers = None
        if ncomp == 1:
            groups = {i: MemGroup(f"/pix/{i}/0/1") for i in active}
            dumpers = [Dumper(groups[i]) for i in active]
        nb.run_multinest_batch(batch, dumpers, nlive=150, seed=ncomp, tol=0.5)
        lnZ = np.array([r.run_lnZ for r in batch])
        ref = np.array([r.null_lnZ for r in batch]) if ncomp == 1 else lnZ_best[active]
        better = lnZ - ref > thresh
        best[active[better]] = ncomp
        lnZ_best[active[better]] = lnZ[better]
        active = active[better]
        if active.size == 0:
            break
    hit = best == true_nc
    print(f"\nescalation: {hit.sum()}/{n_src} sources get their true ncomp")
    assert hit.mean() >= 0.9
    for i in np.flatnonzero(true_nc == 1):
        post = groups[i]['posteriors'].astype(np.float64)
        w = post[:, -1] / post[:, -1].sum()
        mean = (post[:, :6] * w[:, None]).sum(0)
        std = np.sqrt((w[:, None] * (post[:, :6] - mean) ** 2).sum(0))
        truth = cat[i][1]
        for k in (0, 4):
            assert abs(mean[k] - truth[k]) < 5 * std[k] + 0.01, (i, k, mean[k], truth[k], std[k])
