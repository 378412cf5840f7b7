"""CPU tests of the intensity credible intervals: argument checks that refuse before any device work, the store
round trip of waves with and without the intensity datasets, and aggregate_intensity_marginals on a fabricated
store."""
import numpy as np
import pytest

from nestfit_b200.store import INTENSITY_DATASETS, MARG_QUANTILES, RUN_ATTR_COLUMNS, RUN_DATASETS, Wave

M = MARG_QUANTILES.size


@pytest.fixture
def no_device(monkeypatch):
    from nestfit_b200 import _lib, pixels

    def refuse(*args, **kwargs):
        raise AssertionError("the device was touched before the arguments were checked")
    monkeypatch.setattr(_lib, "load", refuse)
    monkeypatch.setattr(pixels.PixelBlock, "from_spectra", classmethod(refuse))


def _block(model, per_pixel_axes=False):
    """A PixelBlock with the attributes the checks read, uploaded nowhere."""
    from nestfit_b200 import PixelBlock
    from nestfit_b200.pixels import _MODELS, _N_MODEL
    b = PixelBlock.__new__(PixelBlock)
    b.model = _MODELS[model]
    b.n_model, b.n_spec, b.n_pix = _N_MODEL[b.model], 2 if model != "gaussian" else 1, 4
    b.per_pixel_axes = per_pixel_axes
    return b


def test_moments_argument_checks(no_device):
    with pytest.raises(ValueError, match="Gaussian"):
        _block("gaussian").moments(np.zeros((3, 3)))
    for model, n_model in (("ammonia", 6), ("diazenylium", 4)):
        with pytest.raises(ValueError, match="single-component"):
            _block(model).moments(np.zeros((3, 2 * n_model)))        # two components
        with pytest.raises(ValueError, match="single-component"):
            _block(model).moments(np.zeros(n_model))
        with pytest.raises(ValueError, match="pix_of_vec"):
            _block(model, per_pixel_axes=True).moments(np.zeros((3, n_model)))
        with pytest.raises(ValueError, match="out of range"):
            _block(model).moments(np.zeros((2, n_model)), pix_of_vec=[0, 4])


def test_sampler_and_fitters_refuse_gaussian(no_device):
    from nestfit_b200 import CubeFitter, GaussianRunner, NestedSamplingBatch, run_multinest, run_multinest_batch
    ns = NestedSamplingBatch.__new__(NestedSamplingBatch)
    ns.block = _block("gaussian")
    with pytest.raises(ValueError, match="Gaussian"):
        ns.intensity_marginals()
    r = GaussianRunner.__new__(GaussianRunner)
    r.utrans, r.ncomp, r.n_spec, r.ndim, r.n_params = object(), 1, 1, 3, 3
    r._block = _block("gaussian")
    with pytest.raises(ValueError, match="Gaussian"):
        run_multinest_batch([r], intensity_marginals=True)
    with pytest.raises(ValueError, match="Gaussian"):
        run_multinest(r, None, intensity_marginals=True)
    fitter = CubeFitter(None, None, GaussianRunner, intensity_marginals=True)
    with pytest.raises(ValueError, match="Gaussian"):
        fitter.fit_block((np.array([0]), np.array([0])))


def test_quantile_count_checked_before_device(no_device):
    from nestfit_b200 import NestedSamplingBatch
    ns = NestedSamplingBatch.__new__(NestedSamplingBatch)
    ns.block = _block("ammonia")
    for q in (np.zeros(0), np.linspace(0, 1, 65), np.zeros((2, 2))):
        with pytest.raises(ValueError, match="quantiles"):
            ns.intensity_marginals(q)


def test_c_entry_points_refuse_bad_handles(nb):
    from nestfit_b200 import _lib
    lib = _lib.load()
    q = np.ascontiguousarray(MARG_QUANTILES)
    out = np.empty(M)
    assert lib.nf_ns_intensity(None, _lib.ptr(q), M, _lib.ptr(out), _lib.ptr(out)) == -1
    p, pk, sm = np.zeros((1, 6)), np.empty((1, 2), np.float32), np.empty((1, 2))
    assert lib.nf_predict_moments(None, _lib.ptr(p), _lib.NF_F64, None, 1, 0, _lib.ptr(pk), _lib.ptr(sm), None) == -1
    assert lib.nf_predict_moments_host(None, _lib.ptr(p), _lib.NF_F64, None, 1, 0, _lib.ptr(pk), _lib.ptr(sm)) == -1


class _FakeSamplerLib:
    """Stands in for the library behind NestedSamplingBatch: nf_ns_intensity refuses (NF_EINVAL) until
    nf_ns_products_rows has been called, as the C entry point does."""

    def __init__(self):
        self.calls = []

    def nf_ns_products_rows(self, handle, off):
        self.calls.append("nf_ns_products_rows")
        return 0

    def nf_ns_intensity(self, handle, q, n_q, peak, integ):
        self.calls.append("nf_ns_intensity")
        return 0 if "nf_ns_products_rows" in self.calls else -1

    def nf_error_string(self, code):
        return b"invalid argument"


def _batch(model="ammonia"):
    from nestfit_b200 import NestedSamplingBatch
    ns = NestedSamplingBatch.__new__(NestedSamplingBatch)
    ns.block = _block(model)
    ns.block.chan_kms = np.array([0.07, 0.07])
    ns.n_run, ns.ncomp, ns.pix_ids, ns.handle = 3, 2, np.arange(3, dtype=np.int32), None
    ns._results, ns._batch = {}, None
    return ns


def test_intensity_needs_the_row_offsets_first(monkeypatch):
    """nf_ns_intensity works from the row offsets of nf_ns_products_rows: the wrapper asks for them first, and a
    refusal of the library surfaces as NfError."""
    from nestfit_b200 import _lib
    fake = _FakeSamplerLib()
    monkeypatch.setattr(_lib, "load", lambda: fake)
    out = _batch().intensity_marginals()
    assert fake.calls == ["nf_ns_products_rows", "nf_ns_intensity"]
    assert out["peak_intensity_marginals"].shape == (3, M, 2, 2)
    fake.calls = []
    ns = _batch()
    ns._batch = {}              # offsets believed present: the library's own guard refuses
    with pytest.raises(_lib.NfError, match="nf_ns_intensity"):
        ns.intensity_marginals()
    assert fake.calls == ["nf_ns_intensity"]


def _wave(ncomp, lon, lat, rng, intensity=True, n_spec=2, posteriors=True):
    n = len(lon)
    ndim = 6 * ncomp
    n_rows = rng.integers(3, 7, n)
    off = np.concatenate([[0], np.cumsum(n_rows)])
    cols = {k: rng.normal(size=n) for k in RUN_ATTR_COLUMNS}
    post = rng.normal(size=(off[-1], ndim + 2)).astype(np.float32) if posteriors else None
    inten = None
    if intensity:
        inten = {k: rng.normal(size=(n, M, n_spec, ncomp)) for k in INTENSITY_DATASETS}
    return Wave(ncomp, ndim, 800, lon, lat, cols, off, post, rng.normal(size=(n, M, ndim)),
                rng.normal(size=(n, ndim)), rng.normal(size=(n, ndim)), inten)


def test_slab_round_trip(tmp_path):
    from nestfit_b200.store import SlabSink, slab_pix_tree
    rng = np.random.default_rng(0)
    with_i = _wave(2, [0, 1], [0, 0], rng)
    without = _wave(1, [0, 1], [1, 1], rng, intensity=False, posteriors=False)
    sink = SlabSink(tmp_path / "chunk0")
    sink.add_wave(with_i)
    sink.add_wave(without)
    sink.add_pixels([0, 1, 0, 1], [0, 0, 1, 1], [2, 2, 1, 1])
    sink.close()
    pix = slab_pix_tree([tmp_path / "chunk0"])
    for r, lon in enumerate((0, 1)):
        g = pix[str(lon)]["0"]["2"]
        assert list(g) == list(RUN_DATASETS) + list(INTENSITY_DATASETS)
        for name in INTENSITY_DATASETS:
            np.testing.assert_array_equal(g[name], with_i.intensity[name][r])
            assert g[name].shape == (M, 2, 2)
        np.testing.assert_array_equal(g["posteriors"], with_i.run_dataset(r, "posteriors"))
        # a wave written without the datasets reads as before: no new names
        g1 = pix[str(lon)]["1"]["1"]
        assert list(g1) == [n for n in RUN_DATASETS if n != "posteriors"]
        np.testing.assert_array_equal(g1["marginals"], without.marginals[r])


def test_group_sink_writes_run_datasets():
    from nestfit_b200.store import GroupSink, MemGroup
    rng = np.random.default_rng(1)
    root = MemGroup("/")
    w = _wave(2, [3], [4], rng)
    GroupSink(root).add_wave(w)
    GroupSink(root).add_wave(_wave(1, [3], [4], rng, intensity=False))
    g = root["/pix/3/4/2"]
    for name in INTENSITY_DATASETS:
        assert g[name].shape == (M, 2, 2)
        np.testing.assert_array_equal(g[name], w.intensity[name][0])
    assert not any(name in root["/pix/3/4/1"] for name in INTENSITY_DATASETS)
    assert RUN_DATASETS == ('posteriors', 'marginals', 'bestfit_params', 'map_params')


def _store(tmp_path, rng, intensity=True):
    """A 3 x 2 store: runs of ncomp 1 and 2 at (0, 0), (1, 0), (2, 1); (0, 1) and (1, 1) have none."""
    from nestfit_b200.store import HdfStore
    store = HdfStore(str(tmp_path / "s"), nchunks=1)
    store.hdf.attrs.update(naxis1=3, naxis2=2, n_max_components=2)
    sink = store.chunk_sink(0)
    lon, lat = [0, 1, 2], [0, 0, 1]
    waves = [_wave(1, lon, lat, rng, intensity), _wave(2, lon, lat, rng, intensity)]
    for w in waves:
        sink.add_wave(w)
    sink.add_pixels(lon + [0, 1], lat + [1, 1], [2, 1, 0, 0, 0])
    sink.close()
    store.link_files()
    nbest = np.full((2, 3), -1, dtype=np.int32)                  # (b, l)
    nbest[0, 0], nbest[0, 1], nbest[1, 2] = 2, 1, 0
    store.create_dataset("nbest", nbest, group=store.dpath)
    return store, waves


def test_aggregate_picks_the_preferred_run(tmp_path):
    from nestfit_b200 import aggregate_intensity_marginals
    store, waves = _store(tmp_path, np.random.default_rng(2))
    aggregate_intensity_marginals(store)
    for name in INTENSITY_DATASETS:
        got = np.asarray(store.hdf[f"{store.dpath}/nbest_{name}"])
        assert got.shape == (2, 2, M, 2, 3)                        # (t, m, M, b, l)
        np.testing.assert_array_equal(got[:, :, :, 0, 0], waves[1].intensity[name][0].transpose(1, 2, 0))
        np.testing.assert_array_equal(got[:, :1, :, 0, 1], waves[0].intensity[name][1].transpose(1, 2, 0))
        assert np.isnan(got[:, 1, :, 0, 1]).all()                  # component 2 of a 1-component pixel
        assert np.isnan(got[:, :, :, 1, 2]).all()                  # nbest 0
        assert np.isnan(got[:, :, :, 1, :2]).all()                 # no runs
    # with a convolved model selection, that one decides
    conv = np.full((2, 3), -1, dtype=np.int32)
    conv[0, 0] = 1
    store.create_dataset("conv_nbest", conv, group=store.dpath)
    with pytest.warns(RuntimeWarning):
        aggregate_intensity_marginals(store)
    for name in INTENSITY_DATASETS:
        got = np.asarray(store.hdf[f"{store.dpath}/nbest_{name}"])
        np.testing.assert_array_equal(got[:, :1, :, 0, 0], waves[0].intensity[name][0].transpose(1, 2, 0))
        assert np.isnan(got[:, 1, :, 0, 0]).all() and np.isnan(got[:, :, :, 0, 1]).all()
    store.close()


def test_aggregate_refuses_store_without_intensity(tmp_path):
    from nestfit_b200 import aggregate_intensity_marginals
    store, _ = _store(tmp_path, np.random.default_rng(3), intensity=False)
    with pytest.raises(ValueError, match="intensity"):
        aggregate_intensity_marginals(store)
    store.close()
