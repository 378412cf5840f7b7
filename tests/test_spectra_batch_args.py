"""CPU tests of run_multinest_batch's argument checks: every mismatch among the runners is refused with
ValueError before any device call (the library loader and the block upload are made to fail if reached)."""
import numpy as np
import pytest


class _Spec:
    def __init__(self, n, trans_id):
        self.size = n
        self.trans_id = trans_id


def _runner(cls, utrans, ncomp=1, tids=(1, 2), sizes=(379, 381), cold=False, lte=False):
    """A runner object with the attributes the checks read, built without uploading anything."""
    r = cls.__new__(cls)
    r.spectra = np.array([_Spec(n, t) for n, t in zip(sizes, tids)], dtype=object)
    r.utrans, r.ncomp, r.n_spec = utrans, ncomp, len(tids)
    r.n_model = 6
    r.n_params = r.ndim = 6 * ncomp
    r.cold, r.lte = cold, lte
    return r


@pytest.fixture
def no_device(monkeypatch):
    from nestfit_b200 import _lib, pixels

    def refuse(*args, **kwargs):
        raise AssertionError("the device was touched before the arguments were checked")
    monkeypatch.setattr(_lib, "load", refuse)
    monkeypatch.setattr(pixels.PixelBlock, "from_spectra", classmethod(refuse))


def test_empty_list(no_device):
    from nestfit_b200 import run_multinest_batch
    with pytest.raises(ValueError, match="at least one runner"):
        run_multinest_batch([])


@pytest.mark.parametrize("change, what", [
    (dict(ncomp=2), "ncomp"),
    (dict(tids=(1, 2, 3), sizes=(379, 381, 400)), "number of spectra"),
    (dict(tids=(1, 3)), "transition ids"),
    (dict(cold=True), "cold"),
    (dict(lte=True), "lte"),
])
def test_runners_must_agree(no_device, change, what):
    from nestfit_b200 import AmmoniaRunner, run_multinest_batch
    ut = object()
    runners = [_runner(AmmoniaRunner, ut), _runner(AmmoniaRunner, ut, sizes=(500, 300)),
               _runner(AmmoniaRunner, ut, **change)]
    with pytest.raises(ValueError, match=f"runner 2 differs from runner 0 in its {what}"):
        run_multinest_batch(runners)


def test_runner_class_and_prior_transformer(no_device):
    from nestfit_b200 import AmmoniaRunner, DiazenyliumRunner, run_multinest_batch
    ut = object()
    with pytest.raises(ValueError, match="class"):
        run_multinest_batch([_runner(AmmoniaRunner, ut), _runner(DiazenyliumRunner, ut)])
    with pytest.raises(ValueError, match="prior transformer"):
        run_multinest_batch([_runner(AmmoniaRunner, ut), _runner(AmmoniaRunner, object())])


def test_sampler_arguments(no_device):
    from nestfit_b200 import AmmoniaRunner, Dumper, run_multinest_batch
    ut = object()
    runners = [_runner(AmmoniaRunner, ut) for _ in range(3)]
    for kwargs in (dict(nlive=[100, 200]), dict(nlive=[[100] * 3]), dict(nlive=0), dict(nlive=[100, 0, 100]),
                   dict(tol=0.0), dict(efr=1.5), dict(maxiter=-1), dict(max_runs_per_batch=0),
                   dict(dumpers=[Dumper(None)]), dict(nClsPar=7)):
        with pytest.raises(ValueError):
            run_multinest_batch(runners, **kwargs)
