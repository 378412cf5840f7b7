"""The hyperfine kernel's brightness amplitude, restated in numpy (tools/kernel_model.amplitude), against the C
oracle's per-channel T0_j (G(T0_j / tex) - tbg_j) on the CPU.  The kernel makes T0 and tbg linear in the channel and
takes G as the larger of two lines from the table segments at the band edges; the error of that grows with the
square of the band.  Up to NF_MAX_BAND_FRAC it takes at most 0.7 of the suite's 1e-5-of-peak spectrum bound over
the whole tex prior of get_irdc_priors, leaving the rest to the FP32 line synthesis; past it the error is allowed
to exceed the bound, which is why wider hyperfine spectra are refused."""
import re
import sys
from pathlib import Path
from types import SimpleNamespace

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT / "tools"))

TEX = np.concatenate([np.linspace(2.8, 3.5, 36), np.linspace(3.5, 12.06, 40)])     # get_irdc_priors' tex range
NH3_NU = [23.6944955e9, 23.722633335e9, 27.477943e9]        # (1,1), (2,2), (9,9)
N2HP_NU = [93173.7637e6, 279511.8325e6]                     # J 1-0, 3-2


def amplitude_error(nu0, frac, n=2001):
    """Worst |kernel - oracle| amplitude over the channels, as a fraction of the largest |oracle| amplitude,
    over TEX, for an axis of n channels starting at nu0 and spanning frac nu0."""
    import kernel_model as km
    from oracle import oracle as orc
    lib = orc.load()
    nu_chan = nu0 * frac / (n - 1)
    x = nu0 + np.arange(n) * nu_chan
    T0 = km.H * x / km.KB
    tbg = 1.0 / np.expm1(T0 / km.TCMB)
    worst = 0.0
    for tex in TEX:
        want = np.array([T0[j] * (lib.nfo_iemtex_interp(T0[j] / tex) - tbg[j]) for j in range(n)])
        got = km.amplitude(nu0, nu_chan, n, tex)
        worst = max(worst, float(np.abs(got - want).max() / np.abs(want).max()))
    return worst


def band_limit():
    from nestfit_b200 import _lib
    return _lib.NF_MAX_BAND_FRAC


def test_limit_mirrors_header():
    from nestfit_b200 import _lib
    text = (ROOT / "include" / "nestfit_b200.h").read_text()
    assert float(re.search(r"#define NF_MAX_BAND_FRAC (\S+)", text).group(1)) == _lib.NF_MAX_BAND_FRAC


@pytest.mark.parametrize("nu0", NH3_NU + N2HP_NU)
def test_amplitude_inside_limit(nu0):
    for frac in (70.0 / 299792.458, 0.5 * band_limit(), band_limit()):
        err = amplitude_error(nu0, frac)
        print(f"\n  nu0 {nu0 / 1e9:.3f} GHz, band {frac:.2e}: amplitude error {err:.2e} of peak", end="")
        assert err < 0.7e-5


def test_amplitude_error_past_limit():
    """Three times the limit, the (1,1) amplitude alone is off by more than the spectrum bound."""
    assert amplitude_error(NH3_NU[0], 3 * band_limit()) > 1e-5


@pytest.fixture
def no_device(monkeypatch):
    from nestfit_b200 import _lib

    def refuse(*args, **kwargs):
        raise AssertionError("the library was reached before the axis was checked")
    monkeypatch.setattr(_lib, "load", refuse)


@pytest.mark.parametrize("model, nu0, tid", [("ammonia", NH3_NU[0], 1), ("diazenylium", N2HP_NU[0], 1)])
def test_wide_hyperfine_axis_refused_before_upload(no_device, model, nu0, tid):
    from nestfit_b200 import PixelBlock
    n = 1000
    x = nu0 * (1.0 + 1.002 * band_limit() * np.arange(n) / (n - 1))
    with pytest.raises(ValueError, match="NF_MAX_BAND_FRAC"):
        PixelBlock(model, [x], np.zeros((1, 1, n)), 0.1, trans_ids=[tid])
    spec = SimpleNamespace(xarr=x, data=np.zeros(n), noise=0.1, trans_id=tid, rest_freq=None)
    with pytest.raises(ValueError, match="NF_MAX_BAND_FRAC"):
        PixelBlock.from_spectra(model, [[spec]])
    # the Gaussian model has no such limit: the same axis gets as far as the library
    with pytest.raises(AssertionError, match="library was reached"):
        PixelBlock("gaussian", [x], np.zeros((1, 1, n)), 0.1, rest_freq=nu0)
