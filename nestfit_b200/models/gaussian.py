"""Multi-component Gaussian emission model: host mirror of
``nestfit.models.gaussian`` (reference nestfit/models/gaussian.pyx:17-148)."""
import numpy as np

from ..core import Runner, Spectrum
from ..pixels import PixelBlock

N_PARAMS = 3


def _block_from_spectrum(s, device=0):
    return PixelBlock("gaussian", [s.xarr], s.data[None, None, :], np.array([[s.noise]]),
                      rest_freq=s.rest_freq, device=device)


def gauss_predict(s, params):
    """Fill ``s.pred`` for physical params [voff.., sigm.., peak..] (gaussian.pyx:17-54)."""
    params = np.ascontiguousarray(params, dtype=np.float64)
    ncomp = params.shape[0] // N_PARAMS
    blk = getattr(s, "_block", None)
    if blk is None:
        blk = _block_from_spectrum(s)
        s._block = blk
    s.pred[:] = blk.predict(params.reshape(1, -1), ncomp)[0, 0]


class GaussianRunner(Runner):
    """Likelihood operator for one spectrum (gaussian.pyx:57-112)."""
    model_name = 'gaussian'

    def __init__(self, spectrum, utrans, ncomp=1):
        assert ncomp > 0
        self.n_model = N_PARAMS
        self.spectrum = spectrum
        self.utrans = utrans
        self.ncomp = ncomp
        self.n_spec = 1
        self.n_params = self.n_model * ncomp
        self.ndim = self.n_params
        self.null_lnZ = spectrum.null_lnZ
        self.n_chan_tot = spectrum.size
        self.run_lnZ = np.nan
        self._block = _block_from_spectrum(spectrum)

    @classmethod
    def from_data(cls, spec_data, utrans, **kwargs):
        # flat (xarr, data, noise, rest_freq) like the reference (gaussian.pyx:94-96)
        return cls(Spectrum(*spec_data), utrans, **kwargs)

    def loglikelihood(self, utheta):
        utheta = np.asarray(utheta)
        self.utrans.transform_batch(utheta.reshape(1, -1), self.ncomp)
        return float(self._block.loglike(utheta.reshape(1, -1), self.ncomp, vecs_per_pix=1)[0])

    def loglikelihood_batch(self, uthetas):
        self.utrans.transform_batch(uthetas, self.ncomp)
        return self._block.loglike(uthetas, self.ncomp, vecs_per_pix=uthetas.shape[0])

    def get_spectrum(self):
        return np.array(self.spectrum)

    def predict(self, params):
        params = np.ascontiguousarray(params, dtype=np.float64)
        if params.shape[0] != self.ndim:
            ncomp = self.ncomp
            shape = params.shape[0]
            raise ValueError(f'Invalid shape for ncomp={ncomp}: {shape}')
        self.spectrum.pred[:] = self._block.predict(params.reshape(1, -1), self.ncomp)[0, 0]


N = N_PARAMS
IX_VCEN = 0
IX_SIGM = 1
NAME = 'gaussian'
model_predict = gauss_predict
ModelSpectrum = Spectrum
ModelRunner = GaussianRunner

PAR_NAMES = ['voff', 'sigm', 'peak']
PAR_NAMES_SHORT = ['v', 's', 'pk']

TEX_LABELS = [
    r'$v_\mathrm{lsr}$',
    r'$\sigma_\mathrm{v}$',
    r'$T_\mathrm{pk}$',
]

TEX_LABELS_WITH_UNITS = [
    r'$v_\mathrm{lsr} \ [\mathrm{km\, s^{-1}}]$',
    r'$\sigma_\mathrm{v} \ [\mathrm{km\, s^{-1}}]$',
    r'$T_\mathrm{pk} \ [\mathrm{K}]$',
]


def get_par_names(ncomp=None):
    if ncomp is None:
        return PAR_NAMES_SHORT
    return [f'{label}{n}' for label in PAR_NAMES_SHORT for n in range(1, ncomp + 1)]
