"""CPU tests: the C oracle (oracle/nf_oracle.c) against the committed golden
fixtures generated from the compiled reference, against the reference's own
known-answer values, and -- when oracle/_ref is present -- against the compiled
reference directly."""
import numpy as np
import pytest

from oracle import oracle as orc
from oracle import ref as oref

GOLDEN = __import__('pathlib').Path(__file__).resolve().parent / 'golden'


def test_kat_swift_convert():
    # reference test_swift_convert, nestfit/models/ammonia.pyx:517-521
    np.testing.assert_almost_equal(orc.load().nfo_swift_convert(15.0), 14.023487575888257, decimal=8)


def test_kat_partition(nh3_golden):
    lib = orc.load()
    got = np.array([lib.nfo_partition_level(1, 10.0), lib.nfo_partition_func(1, 10.0),
                    lib.nfo_partition_func(0, 10.0)])
    np.testing.assert_allclose(got, nh3_golden["kat_partition"], rtol=1e-13)
    # SURVEY.md Appendix B values of the compiled reference
    np.testing.assert_allclose(got, [0.2927352107367582, 0.3006679571980005, 2.000060176241782], rtol=1e-12)


def test_kat_iemtex(nh3_golden):
    lib = orc.load()
    got = np.array([lib.nfo_iemtex_interp(x) for x in nh3_golden["kat_iemtex_x"]])
    np.testing.assert_allclose(got, nh3_golden["kat_iemtex_y"], rtol=1e-13)
    # reference test_iemtex_interp, hyperfine.pyx:147-152: table error < 1.5e-5
    x = np.linspace(0.1381, 0.4975, 5000)
    tab = np.array([lib.nfo_iemtex_interp(v) for v in x])
    assert np.max(np.abs(tab * np.expm1(x) - 1.0)) < 1.5e-5


def test_fast_expn_semantics():
    lib = orc.load()
    f = lib.nfo_fast_expn
    assert f(0.0) == 1.0
    assert f(32.0) == 0.0 and f(1e3) == 0.0
    assert f(-1.0) == pytest.approx(np.e, rel=1e-15)
    x = np.linspace(0.04, 31.9, 2001)
    got = np.array([f(v) for v in x])
    assert np.max(np.abs(got / np.exp(-x) - 1.0)) < 1e-6     # float-cast argument (SURVEY App. C)
    xs = np.linspace(1e-6, 0.031, 500)
    got = np.array([f(v) for v in xs])
    assert np.max(np.abs(got / np.exp(-xs) - 1.0)) < 5e-8    # Taylor-3 region


@pytest.mark.parametrize("ncomp", [1, 2, 3, 4])
def test_nh3_against_golden(nh3_golden, ncomp):
    g = nh3_golden
    xs = [g["x11"], g["x22"]]
    out = orc.nh3_batch(xs, [1, 2], g[f"params{ncomp}"], ncomp, data=g[f"data{ncomp}"][None], noise=0.1,
                        want_pred=True)
    peak = np.abs(g[f"pred{ncomp}"]).max(axis=2, keepdims=True)
    assert np.max(np.abs(out["pred"] - g[f"pred{ncomp}"]) / peak) < 1e-11
    np.testing.assert_allclose(out["lnL"], g[f"lnL{ncomp}"], rtol=1e-11)


@pytest.mark.parametrize("name", ["hand1", "hand2", "hand3", "edge1", "narrow1", "ortho1"])
def test_nh3_hand_vectors(nh3_golden, name):
    g = nh3_golden
    p = g[f"{name}_p"]
    ncomp = p.size // 6
    for cold, lte in ((0, 0), (1, 0), (0, 1)):
        out = orc.nh3_batch([g["x11"], g["x22"]], [1, 2], p[None], ncomp, cold=cold, lte=lte, want_pred=True)
        want = g[f"{name}_c{cold}l{lte}"]
        scale = max(np.abs(want).max(), 1e-300)
        assert np.max(np.abs(out["pred"][0] - want)) / scale < 1e-11


def test_nh3_survey_appendix_b(nh3_golden):
    # numbers quoted in SURVEY.md Appendix B for the compiled reference
    g = nh3_golden
    out = orc.nh3_batch([g["x11"], g["x22"]], [1, 2], g["hand2_p"][None], 2, data=np.zeros((1, 2, 1000)),
                        noise=0.1, want_pred=True)
    assert out["pred"][0, 0].sum() == pytest.approx(3.687872850e+02, rel=1e-9)
    assert out["pred"][0, 1].sum() == pytest.approx(6.513799533e+01, rel=1e-9)
    assert int(np.count_nonzero(out["pred"][0, 0])) == 534
    assert int(out["pred"][0, 0].argmax()) == 478
    assert out["lnL"][0] == pytest.approx(-2.9987458219e+04 - 3.2488042253e+03, rel=1e-9)


def test_nh3_ortho_transition(nh3_golden):
    g = nh3_golden
    out = orc.nh3_batch([g["x33"]], [3], g["ortho1_p"][None], 1, want_pred=True)
    assert np.max(np.abs(out["pred"][0, 0] - g["ortho1_33"])) / g["ortho1_33"].max() < 1e-11


def test_gauss_against_golden(gauss_golden):
    g = gauss_golden
    out = orc.gauss_batch(g["x"], float(g["rest_freq"]), g["params"], 8, data=g["data"][None], noise=0.1,
                          want_pred=True)
    assert np.max(np.abs(out["pred"] - g["pred"])) / g["pred"].max() < 1e-11
    np.testing.assert_allclose(out["lnL"], g["lnL"], rtol=1e-11)
    # SURVEY.md Appendix B: sum, max and support of the fixed 8-component vector
    assert out["pred"][0].sum() == pytest.approx(1.534055611e+03, rel=1e-9)
    assert int(np.count_nonzero(out["pred"][0])) == 2110


@pytest.mark.parametrize("name,ncomps", [("irdc", (1, 2, 3, 4)), ("synth", (1, 2))])
def test_prior_transform_against_golden(prior_golden, name, ncomps):
    import nestfit_b200.prior_constructors as pc
    ut = pc.get_irdc_priors() if name == "irdc" else pc.get_synth_priors()
    packed = ut.pack()
    for ncomp in ncomps:
        U, want = prior_golden[f"{name}_u{ncomp}"], prior_golden[f"{name}_p{ncomp}"]
        got = orc.prior_transform(packed, U, ncomp)
        ok = np.isfinite(want)
        assert (np.isfinite(got) == ok).all()
        np.testing.assert_allclose(got[ok], want[ok], rtol=0, atol=1e-11)


@pytest.mark.parametrize("name", ["ordered", "spaced", "censep"])
def test_prior_kinds_against_golden(name):
    """OrderedPrior, SpacedPrior, CenSepPrior (core.pyx:241-318) against fixtures of the compiled reference
    (tests/golden/make_golden.py --only-prior-kinds): the packed plan of nestfit_b200.core through the C oracle."""
    import sys
    import nestfit_b200.core as nbcore
    sys.path.insert(0, str(GOLDEN))
    from prior_kind_sets import kind_prior_sets
    g = np.load(GOLDEN / "prior_kinds_golden.npz")
    packed = kind_prior_sets(nbcore)[name].pack()
    for ncomp in (1, 2, 3, 4):
        U, want = g[f"{name}_u{ncomp}"], g[f"{name}_p{ncomp}"]
        got = orc.prior_transform(packed, U, ncomp)
        ok = np.isfinite(want)
        assert (np.isfinite(got) == ok).all()
        np.testing.assert_allclose(got[ok], want[ok], rtol=0, atol=1e-11)
    if name == "censep":      # ncomp > 2 is not parametrised: the unit-cube values stay in place (core.pyx:313-318)
        assert np.array_equal(g["censep_p3"][:, :3], g["censep_u3"][:, :3])


def test_prior_distribution_kat():
    # reference test_distribution, core.pyx:830-840
    import nestfit_b200 as nb
    x = np.linspace(-4, 4, 201)
    d = nb.Distribution(x, np.exp(-0.5 * x**2))
    assert abs(d.ppf[100]) < 1e-15
    ut = nb.PriorTransformer(np.array([nb.Prior(d, 0)], dtype=object))
    got = orc.prior_transform(ut.pack(), np.array([[0.5]]), 1)
    assert abs(got[0, 0]) < 1e-15


def test_oracle_equals_compiled_reference(nh3_golden, prior_golden):
    """The oracle's get_irdc_priors transform and NH3 spectra against the compiled reference: live when oracle/_ref
    is built, otherwise against the reference's own transforms and amm_predict spectra stored by
    tests/golden/make_golden.py (ncomp 1..3, same tolerances)."""
    import nestfit_b200.prior_constructors as pc
    packed = pc.get_irdc_priors().pack()
    if not oref.available():
        xs = [nh3_golden["x11"], nh3_golden["x22"]]
        for ncomp in (1, 2, 3):
            P = orc.prior_transform(packed, prior_golden[f"irdc_u{ncomp}"], ncomp)
            np.testing.assert_allclose(P, prior_golden[f"irdc_p{ncomp}"], atol=1e-11, rtol=0)
            out = orc.nh3_batch(xs, [1, 2], nh3_golden[f"params{ncomp}"], ncomp, want_pred=True)
            for b, want_b in enumerate(nh3_golden[f"pred{ncomp}"]):
                for t in (0, 1):
                    want = want_b[t]
                    assert np.max(np.abs(out["pred"][b, t] - want)) <= 1e-11 * max(want.max(), 1e-30)
        return
    m = oref.load()
    rng = np.random.default_rng(3)
    ut_ref = oref.make_irdc_priors(m.core)
    xs = [oref.bench_axis(oref.NU11, 380, 0.158), oref.bench_axis(oref.NU22, 380, 0.158)]
    for ncomp in (1, 2, 3):
        U = rng.uniform(size=(40, 6 * ncomp))
        P = orc.prior_transform(packed, U, ncomp)
        Pr = U.copy()
        for row in Pr:
            ut_ref.transform(row, ncomp)
        np.testing.assert_allclose(P, Pr, atol=1e-11, rtol=0)
        out = orc.nh3_batch(xs, [1, 2], P, ncomp, want_pred=True)
        for t in (0, 1):
            s = m.ammonia.AmmoniaSpectrum(xs[t], np.zeros(380), 0.2, trans_id=t + 1)
            for b in range(P.shape[0]):
                m.ammonia.amm_predict(s, P[b].copy())
                want = s.get_spec()
                assert np.max(np.abs(out["pred"][b, t] - want)) <= 1e-11 * max(want.max(), 1e-30)


@pytest.mark.parametrize("trans", [1, 2, 3])
def test_n2hp_against_golden(n2hp_golden, trans):
    """N2H+ (diazenylium.pyx:140-154) restatement against the compiled reference's fixtures."""
    g = n2hp_golden
    for ncomp in (1, 2, 3):
        P = g[f"params{trans}_{ncomp}"]
        o = orc.n2hp_batch([g[f"x{trans}"]], [trans], P, ncomp, data=g[f"data{trans}_{ncomp}"][None, None],
                           noise=0.1, want_pred=True)
        want = g[f"pred{trans}_{ncomp}"]
        peak = np.abs(want).max(axis=1, keepdims=True)
        assert (np.abs(o["pred"][:, 0] - want) <= 1e-12 * peak).all()
        np.testing.assert_allclose(o["lnL"], g[f"lnL{trans}_{ncomp}"], rtol=1e-10, atol=1e-8)
