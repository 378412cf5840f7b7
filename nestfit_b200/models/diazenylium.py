"""N2H+ J = 1-0, 2-1, 3-2 model: host mirror of ``nestfit.models.diazenylium``
(reference nestfit/models/diazenylium.pyx:105-272).  The hyperfine synthesis,
radiative transfer and chi-square run in the same fused CUDA kernel as NH3 with
the N2H+ line tables and the four-parameter front end (voff, tex, ltau, sigm).
"""
import numpy as np

from ..core import HyperfineSpectrum, Runner
from ..pixels import PixelBlock

N_LEVELS = 3
N_PARAMS = 4


class DiazenyliumSpectrum(HyperfineSpectrum):
    """Spectrum of one N2H+ transition; ``trans_id`` 1..3 = (1-0), (2-1), (3-2)
    (diazenylium.pyx:105-138)."""

    def __init__(self, xarr, data, noise, trans_id=1):
        assert trans_id in range(1, N_LEVELS + 1)
        super().__init__(xarr, data, noise, rest_freq=0, trans_id=trans_id)


def _block_from_spectra(spectra, device=0):
    if len({s.size for s in spectra}) > 1:      # spectra of different lengths: each on its own axis
        return PixelBlock.from_spectra("diazenylium", [spectra], device=device)
    xarrs = [s.xarr for s in spectra]
    data = np.stack([s.data for s in spectra])[None, :, :]
    noise = np.array([[s.noise for s in spectra]])
    return PixelBlock("diazenylium", xarrs, data, noise, trans_ids=[s.trans_id for s in spectra], device=device)


def nnhp_predict(s, params):
    """Fill ``s.pred`` with the model spectrum for physical ``params``
    (parameter-major, component-minor; diazenylium.pyx:140-158)."""
    params = np.ascontiguousarray(params, dtype=np.float64)
    ncomp = params.shape[0] // N_PARAMS
    blk = getattr(s, "_block", None)
    if blk is None:
        blk = _block_from_spectra([s])
        s._block = blk
    s.pred[:] = blk.predict(params.reshape(1, -1), ncomp)[0, 0]


class DiazenyliumRunner(Runner):
    """Likelihood operator over one pixel's N2H+ spectra (diazenylium.pyx:161-232)."""
    model_name = 'diazenylium'

    def __init__(self, spectra, utrans, ncomp=1):
        assert ncomp > 0
        self.n_model = N_PARAMS
        self.spectra = np.asarray(spectra, dtype=object)
        self.utrans = utrans
        self.ncomp = ncomp
        self.n_spec = len(spectra)
        self.n_params = self.n_model * ncomp
        self.ndim = self.n_params  # no nuisance parameters
        self.null_lnZ = float(sum(s.null_lnZ for s in self.spectra))
        self.n_chan_tot = int(sum(s.size for s in self.spectra))
        self.run_lnZ = np.nan
        self._block = _block_from_spectra(list(self.spectra))

    @classmethod
    def from_data(cls, spec_data, utrans, **kwargs):
        spectra = np.array([DiazenyliumSpectrum(*args) for args in spec_data], dtype=object)
        return cls(spectra, utrans, **kwargs)

    def loglikelihood(self, utheta):
        """Unit-cube vector in (overwritten with physical parameters), lnL out
        (diazenylium.pyx:206-215, core.pyx:558-561)."""
        utheta = np.asarray(utheta)
        self.utrans.transform_batch(utheta.reshape(1, -1), self.ncomp)
        return float(self._block.loglike(utheta.reshape(1, -1), self.ncomp, vecs_per_pix=1)[0])

    def loglikelihood_batch(self, uthetas):
        """Batched extension: uthetas [B, ndim] transformed in place -> lnL [B]."""
        self.utrans.transform_batch(uthetas, self.ncomp)
        return self._block.loglike(uthetas, self.ncomp, vecs_per_pix=uthetas.shape[0])

    def get_spectra(self):
        return np.array(self.spectra)

    def predict(self, params):
        params = np.ascontiguousarray(params, dtype=np.float64)
        if params.shape[0] != self.ndim:
            ncomp = self.ncomp
            shape = params.shape[0]
            raise ValueError(f'Invalid shape for ncomp={ncomp}: {shape}')
        pix = [0] if self._block.per_pixel_axes else None
        pred = self._block.predict(params.reshape(1, -1), self.ncomp, pix_of_vec=pix)[0]
        for i, spec in enumerate(self.spectra):
            spec.pred[:] = pred[i, :spec.size]


# Aliases and metadata consumed by the store (diazenylium.pyx:235-272, main.py:369-377)
N = N_PARAMS
IX_VCEN = 0
IX_SIGM = 3
NAME = 'diazenylium'
model_predict = nnhp_predict
ModelSpectrum = DiazenyliumSpectrum
ModelRunner = DiazenyliumRunner

PAR_NAMES = ['voff', 'tex', 'ltau', 'sigm']
PAR_NAMES_SHORT = ['v', 'Tx', 'lt', 's']

TEX_LABELS = [
    r'$v_\mathrm{lsr}$',
    r'$T_\mathrm{ex}$',
    r'$\log(\tau_0)$',
    r'$\sigma_\mathrm{v}$',
]

TEX_LABELS_WITH_UNITS = [
    r'$v_\mathrm{lsr} \ [\mathrm{km\, s^{-1}}]$',
    r'$T_\mathrm{ex} \ [\mathrm{K}]$',
    r'$\log(\tau_0)$',
    r'$\sigma_\mathrm{v} \ [\mathrm{km\, s^{-1}}]$',
]


def get_par_names(ncomp=None):
    if ncomp is None:
        return PAR_NAMES_SHORT
    return [f'{label}{n}' for label in PAR_NAMES_SHORT for n in range(1, ncomp + 1)]
