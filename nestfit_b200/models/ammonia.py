"""NH3 (J,K) inversion-line model: host mirror of ``nestfit.models.ammonia``
(reference nestfit/models/ammonia.pyx:244-489).  Synthesis, radiative transfer
and chi-square run in the fused CUDA kernel; these classes keep the reference's
names, arguments, attributes and error behaviour.
"""
import numpy as np

from .. import _lib
from ..core import HyperfineSpectrum, Runner
from ..pixels import PixelBlock

N_LEVELS = 9
N_PARAMS = 6


class AmmoniaSpectrum(HyperfineSpectrum):
    """Spectrum of one NH3 transition; ``trans_id`` 1..9 = (1,1)..(9,9)
    (ammonia.pyx:244-277)."""

    def __init__(self, xarr, data, noise, trans_id=1):
        assert trans_id in range(1, N_LEVELS + 1)
        super().__init__(xarr, data, noise, rest_freq=0, trans_id=trans_id)


def _block_from_spectra(spectra, device=0):
    if len({s.size for s in spectra}) > 1:      # spectra of different lengths: each on its own axis
        return PixelBlock.from_spectra("ammonia", [spectra], device=device)
    xarrs = [s.xarr for s in spectra]
    data = np.stack([s.data for s in spectra])[None, :, :]
    noise = np.array([[s.noise for s in spectra]])
    tids = [s.trans_id for s in spectra]
    return PixelBlock("ammonia", xarrs, data, noise, trans_ids=tids, device=device)


def amm_predict(s, params, cold=False, lte=False):
    """Fill ``s.pred`` with the model spectrum for physical ``params``
    (parameter-major, component-minor; ammonia.pyx:326-366)."""
    params = np.ascontiguousarray(params, dtype=np.float64)
    ncomp = params.shape[0] // N_PARAMS
    blk = getattr(s, "_block", None)
    if blk is None:
        blk = _block_from_spectra([s])
        s._block = blk
    s.pred[:] = blk.predict(params.reshape(1, -1), ncomp, cold=cold, lte=lte)[0, 0]


class AmmoniaRunner(Runner):
    """Likelihood operator over one pixel's NH3 spectra (ammonia.pyx:369-447)."""
    model_name = 'ammonia'

    def __init__(self, spectra, utrans, ncomp=1, cold=False, lte=False):
        assert ncomp > 0
        self.n_model = N_PARAMS
        self.spectra = np.asarray(spectra, dtype=object)
        self.utrans = utrans
        self.ncomp = ncomp
        self.cold = bool(cold)
        self.lte = bool(lte)
        self.n_spec = len(spectra)
        self.n_params = self.n_model * ncomp
        self.ndim = self.n_params  # no nuisance parameters
        self.null_lnZ = float(sum(s.null_lnZ for s in self.spectra))
        self.n_chan_tot = int(sum(s.size for s in self.spectra))
        self.run_lnZ = np.nan
        self._block = _block_from_spectra(list(self.spectra))

    @classmethod
    def from_data(cls, spec_data, utrans, **kwargs):
        spectra = np.array([AmmoniaSpectrum(*args) for args in spec_data], dtype=object)
        return cls(spectra, utrans, **kwargs)

    def loglikelihood(self, utheta):
        """Unit-cube vector in (overwritten with physical parameters), lnL out
        (ammonia.pyx:423-432, core.pyx:558-561)."""
        utheta = np.asarray(utheta)
        self.utrans.transform_batch(utheta.reshape(1, -1), self.ncomp)
        return float(self._block.loglike(utheta.reshape(1, -1), self.ncomp, vecs_per_pix=1,
                                         cold=self.cold, lte=self.lte)[0])

    def loglikelihood_batch(self, uthetas):
        """Batched extension: uthetas [B, ndim] transformed in place -> lnL [B]."""
        self.utrans.transform_batch(uthetas, self.ncomp)
        return self._block.loglike(uthetas, self.ncomp, vecs_per_pix=uthetas.shape[0],
                                   cold=self.cold, lte=self.lte)

    def get_spectra(self):
        return np.array(self.spectra)

    def predict(self, params):
        params = np.ascontiguousarray(params, dtype=np.float64)
        if params.shape[0] != self.ndim:
            ncomp = self.ncomp
            shape = params.shape[0]
            raise ValueError(f'Invalid shape for ncomp={ncomp}: {shape}')
        pix = [0] if self._block.per_pixel_axes else None
        pred = self._block.predict(params.reshape(1, -1), self.ncomp, cold=self.cold, lte=self.lte, pix_of_vec=pix)[0]
        for i, spec in enumerate(self.spectra):
            spec.pred[:] = pred[i, :spec.size]


# Aliases and metadata consumed by the store (ammonia.pyx:451-489, main.py:369-377)
N = N_PARAMS
IX_VCEN = 0
IX_SIGM = 4
NAME = 'ammonia'
model_predict = amm_predict
ModelSpectrum = AmmoniaSpectrum
ModelRunner = AmmoniaRunner

PAR_NAMES = ['voff', 'trot', 'tex', 'ntot', 'sigm', 'orth']
PAR_NAMES_SHORT = ['v', 'Tk', 'Tx', 'N', 's', 'o']

TEX_LABELS = [
    r'$v_\mathrm{lsr}$',
    r'$T_\mathrm{rot}$',
    r'$T_\mathrm{ex}$',
    r'$\log(N_\mathrm{p})$',
    r'$\sigma_\mathrm{v}$',
    r'$f_\mathrm{o}$',
]

TEX_LABELS_WITH_UNITS = [
    r'$v_\mathrm{lsr} \ [\mathrm{km\, s^{-1}}]$',
    r'$T_\mathrm{rot} \ [\mathrm{K}]$',
    r'$T_\mathrm{ex} \ [\mathrm{K}]$',
    r'$\log(N) \ [\log(\mathrm{cm^{-2}})]$',
    r'$\sigma_\mathrm{v} \ [\mathrm{km\, s^{-1}}]$',
    r'$f_\mathrm{o}$',
]


def get_par_names(ncomp=None):
    if ncomp is None:
        return PAR_NAMES_SHORT
    return [f'{label}{n}' for label in PAR_NAMES_SHORT for n in range(1, ncomp + 1)]
