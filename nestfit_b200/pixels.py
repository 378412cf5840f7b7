"""`PixelBlock`: a block of pixels (spectra + noise) resident in HBM.

Thin Python owner of an opaque ``nf_pixels*`` handle (include/nestfit_b200.h).
It is the batched counterpart of the reference's per-pixel ``Spectrum`` /
``AmmoniaSpectrum`` objects (nestfit/core/core.pyx:486-520,
nestfit/models/ammonia.pyx:244-277): the cube's ``data[lon, lat, chan]`` slab
(nestfit/main.py:152) is uploaded once and every likelihood call references
pixels by index.  ``PixelBlock.from_spectra`` uploads spectra that do not form a
cube -- a catalogue of pointed observations, where every (pixel, spectrum) has
its own axis and length.
"""
import ctypes as C

import numpy as np

from . import _lib

C_KMS = 299792.458


def channel_kms(x):
    """Channel width of the ascending uniform axis x [Hz] in km/s, |dnu| / mean(nu) * c (DataCube.dv)."""
    return abs(x[1] - x[0]) / x.mean() * C_KMS


_MODELS = {"ammonia": _lib.NF_MODEL_NH3, "gaussian": _lib.NF_MODEL_GAUSS, "diazenylium": _lib.NF_MODEL_N2HP}
_N_MODEL = {_lib.NF_MODEL_NH3: 6, _lib.NF_MODEL_N2HP: 4, _lib.NF_MODEL_GAUSS: 3}


def _check_band(model, x):
    """The hyperfine models' brightness amplitude is linear in the channel, which holds to the suite's accuracy up
    to a fractional bandwidth of NF_MAX_BAND_FRAC (include/nestfit_b200.h)."""
    if model != _lib.NF_MODEL_GAUSS:
        frac = (x[-1] - x[0]) / x[0]
        if not frac <= _lib.NF_MAX_BAND_FRAC:
            raise ValueError(f"spectrum spans {frac:.4g} of its lowest frequency; the hyperfine models accept at most "
                             f"NF_MAX_BAND_FRAC = {_lib.NF_MAX_BAND_FRAC:g} (about "
                             f"{_lib.NF_MAX_BAND_FRAC * 299792.458:.0f} km/s)")


class PixelBlock:
    per_pixel_axes = False

    def __init__(self, model, xarrs, data, noise, trans_ids=None, rest_freq=None, device=0):
        """
        model     : 'ammonia' | 'gaussian' | 'diazenylium'
        xarrs     : sequence of n_spec ascending uniform frequency axes [Hz], equal length
        data      : array [n_pix, n_spec, n_chan] (float32 or float64)
        noise     : array [n_pix, n_spec] rms per spectrum
        trans_ids : NH3 transition ids (1..9) / N2H+ transition ids (1..3) per spectrum
        rest_freq : Gaussian-model rest frequency [Hz]
        """
        from .core import check_uniform_axis
        self.model_name = model
        self.model = _MODELS[model]
        xarrs = [np.ascontiguousarray(x, dtype=np.float64) for x in xarrs]
        self.n_spec = len(xarrs)
        self.n_chan = int(xarrs[0].shape[0])
        for x in xarrs:
            if x.shape[0] != self.n_chan:
                raise ValueError("all spectra of a block must have the same number of channels")
            check_uniform_axis(x)
            _check_band(self.model, x)
        lib = _lib.load()
        self.xarrs = xarrs
        data = np.asarray(data)
        if data.dtype not in (np.float32, np.float64):
            data = data.astype(np.float64)
        data = np.ascontiguousarray(data)
        if data.ndim != 3 or data.shape[1] != self.n_spec or data.shape[2] != self.n_chan:
            raise ValueError(f"data must be [n_pix, {self.n_spec}, {self.n_chan}], got {data.shape}")
        self.n_pix = int(data.shape[0])
        noise = np.ascontiguousarray(np.broadcast_to(np.asarray(noise, dtype=np.float64),
                                                     (self.n_pix, self.n_spec)))
        nu_min = np.array([x[0] for x in xarrs], dtype=np.float64)
        nu_chan = np.array([x[1] - x[0] for x in xarrs], dtype=np.float64)
        tid = None
        rf = None
        if self.model in (_lib.NF_MODEL_NH3, _lib.NF_MODEL_N2HP):
            tid = np.ascontiguousarray(trans_ids, dtype=np.int32)
            if tid.shape != (self.n_spec,):
                raise ValueError("trans_ids must have one entry per spectrum")
        else:
            rf = np.ascontiguousarray(np.broadcast_to(np.asarray(rest_freq, dtype=np.float64), (self.n_spec,)))
        self.trans_ids, self.rest_freq = tid, rf
        self.chan_kms = np.array([channel_kms(x) for x in xarrs])           # [n_spec]
        self.device = device
        out = C.c_void_p()
        dtype = _lib.NF_F64 if data.dtype == np.float64 else _lib.NF_F32
        _lib.check(lib.nf_pixels_create(device, self.model, self.n_pix, self.n_spec, self.n_chan,
                                        _lib.ptr(nu_min), _lib.ptr(nu_chan), _lib.ptr(tid), _lib.ptr(rf),
                                        _lib.ptr(data), dtype, _lib.ptr(noise), C.byref(out)),
                   "nf_pixels_create")
        self.handle = out
        self.n_model = _N_MODEL[self.model]

    @classmethod
    def from_spectra(cls, model, spectra, device=0):
        """Block in which every (pixel, spectrum) has its own uniform ascending axis and length.

        spectra[p] is pixel p's list of Spectrum-like objects (``xarr``, ``data``, ``noise``, ``trans_id``; the
        Gaussian model takes one spectrum per pixel and its ``rest_freq``).  All pixels have the same number of
        spectra and the same transitions.  ``n_chan`` is then [n_pix, n_spec] and ``n_chan_max`` its maximum;
        ``predict`` needs ``pix_of_vec`` and returns rows of ``n_chan_max`` channels, zero past each spectrum's end.
        """
        from .core import check_uniform_axis
        self = cls.__new__(cls)
        self.model_name = model
        self.model = _MODELS[model]
        self.per_pixel_axes = True
        spectra = [list(sp) for sp in spectra]
        n_pix = len(spectra)
        if n_pix == 0:
            raise ValueError("from_spectra needs at least one pixel")
        n_spec = len(spectra[0])
        if n_spec < 1 or any(len(sp) != n_spec for sp in spectra):
            raise ValueError("every pixel must have the same number of spectra")
        if n_spec > _lib.NF_MAX_SPEC:
            raise ValueError(f"at most {_lib.NF_MAX_SPEC} spectra per pixel")
        if self.model == _lib.NF_MODEL_GAUSS and n_spec != 1:
            raise ValueError("the Gaussian model takes one spectrum per pixel")
        n_chan = np.array([[int(np.asarray(s.xarr).shape[0]) for s in sp] for sp in spectra], dtype=np.int32)
        n_chan_max = int(n_chan.max())
        nu_min = np.empty((n_pix, n_spec))
        nu_chan = np.empty((n_pix, n_spec))
        noise = np.empty((n_pix, n_spec))
        chan_kms = np.empty((n_pix, n_spec))
        data = np.zeros((n_pix, n_spec, n_chan_max))
        for p, sp in enumerate(spectra):
            for k, s in enumerate(sp):
                x = np.ascontiguousarray(s.xarr, dtype=np.float64)
                check_uniform_axis(x)
                _check_band(self.model, x)
                d = np.asarray(s.data, dtype=np.float64)
                if d.shape != x.shape:
                    raise ValueError(f"pixel {p} spectrum {k}: data and axis lengths differ")
                nu_min[p, k], nu_chan[p, k] = x[0], x[1] - x[0]
                chan_kms[p, k] = channel_kms(x)
                noise[p, k] = s.noise
                data[p, k, :x.shape[0]] = d
        tid = rf = None
        if self.model in (_lib.NF_MODEL_NH3, _lib.NF_MODEL_N2HP):
            tid = np.array([s.trans_id for s in spectra[0]], dtype=np.int32)
            if any([s.trans_id for s in sp] != list(tid) for sp in spectra):
                raise ValueError("all pixels of a block must have the same transitions")
        else:
            rf = np.array([sp[0].rest_freq for sp in spectra], dtype=np.float64)
        self.n_pix, self.n_spec = n_pix, n_spec
        self.n_chan, self.n_chan_max = n_chan, n_chan_max
        self.xarrs = None
        self.chan_kms = chan_kms                                            # [n_pix, n_spec]
        self.trans_ids, self.rest_freq = tid, rf
        self.device = device
        self.n_model = _N_MODEL[self.model]
        lib = _lib.load()
        out = C.c_void_p()
        _lib.check(lib.nf_pixels_create_axes(device, self.model, n_pix, n_spec, n_chan_max, _lib.ptr(nu_min),
                                             _lib.ptr(nu_chan), _lib.ptr(n_chan), _lib.ptr(tid), _lib.ptr(rf),
                                             _lib.ptr(data), _lib.NF_F64, _lib.ptr(noise), C.byref(out)),
                   "nf_pixels_create_axes")
        self.handle = out
        return self

    def close(self):
        if getattr(self, "handle", None):
            _lib.load().nf_pixels_free(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def null_lnZ(self):
        out = np.empty(self.n_pix, dtype=np.float64)
        _lib.check(_lib.load().nf_pixels_null_lnz(self.handle, _lib.ptr(out)), "nf_pixels_null_lnz")
        return out

    @staticmethod
    def _params(params):
        params = np.asarray(params)
        if params.dtype not in (np.float32, np.float64):
            params = params.astype(np.float64)
        params = np.ascontiguousarray(params)
        return params, (_lib.NF_F64 if params.dtype == np.float64 else _lib.NF_F32)

    def loglike(self, params, ncomp, pix_of_vec=None, vecs_per_pix=0, cold=False, lte=False, out=None):
        """Host-buffer likelihood call: params [B, n_model*ncomp] physical units -> lnL [B]."""
        lib = _lib.load()
        params, dt = self._params(params)
        if params.ndim != 2 or params.shape[1] != self.n_model * ncomp:
            raise ValueError(f'Invalid shape for ncomp={ncomp}: {params.shape}')
        B = params.shape[0]
        if out is None:
            out = np.empty(B, dtype=np.float64)
        pv = None
        if pix_of_vec is not None:
            pv = np.ascontiguousarray(pix_of_vec, dtype=np.int32)
            if pv.shape != (B,):
                raise ValueError("pix_of_vec must have one entry per vector")
            if B and (pv.min() < 0 or pv.max() >= self.n_pix):
                raise ValueError("pix_of_vec out of range")
        else:
            if vecs_per_pix < 1:
                vecs_per_pix = max(1, -(-B // self.n_pix))
            if (B + vecs_per_pix - 1) // vecs_per_pix > self.n_pix:
                raise ValueError("more vectors than pixels * vecs_per_pix")
        if self.model == _lib.NF_MODEL_NH3:
            flags = (_lib.NF_FLAG_COLD if cold else 0) | (_lib.NF_FLAG_LTE if lte else 0)
            rc = lib.nf_nh3_loglike_host(self.handle, _lib.ptr(params), dt, _lib.ptr(pv), vecs_per_pix, B,
                                         ncomp, flags, _lib.ptr(out))
        elif self.model == _lib.NF_MODEL_N2HP:
            rc = lib.nf_n2hp_loglike_host(self.handle, _lib.ptr(params), dt, _lib.ptr(pv), vecs_per_pix, B,
                                          ncomp, _lib.ptr(out))
        else:
            rc = lib.nf_gauss_loglike_host(self.handle, _lib.ptr(params), dt, _lib.ptr(pv), vecs_per_pix, B,
                                           ncomp, _lib.ptr(out))
        _lib.check(rc, "loglike")
        return out

    def predict(self, params, ncomp, cold=False, lte=False, pix_of_vec=None):
        """Model spectra for params [B, n_model*ncomp] -> float32 [B, n_spec, n_chan].

        With ``pix_of_vec`` (required on a block from ``from_spectra``) vector b is synthesised on the axes of pixel
        pix_of_vec[b]; rows then have ``n_chan_max`` channels and are zero past each spectrum's own length."""
        lib = _lib.load()
        params, dt = self._params(params)
        if params.ndim != 2 or params.shape[1] != self.n_model * ncomp:
            raise ValueError(f'Invalid shape for ncomp={ncomp}: {params.shape}')
        B = params.shape[0]
        if self.per_pixel_axes and pix_of_vec is None:
            raise ValueError("a block with per-pixel axes needs pix_of_vec to predict")
        flags = (_lib.NF_FLAG_COLD if cold else 0) | (_lib.NF_FLAG_LTE if lte else 0)
        if pix_of_vec is not None:
            pv = np.ascontiguousarray(pix_of_vec, dtype=np.int32)
            if pv.shape != (B,):
                raise ValueError("pix_of_vec must have one entry per vector")
            if B and (pv.min() < 0 or pv.max() >= self.n_pix):
                raise ValueError("pix_of_vec out of range")
            n_row = self.n_chan_max if self.per_pixel_axes else self.n_chan
            out = np.empty((B, self.n_spec, n_row), dtype=np.float32)
            if self.model != _lib.NF_MODEL_NH3:
                flags = 0
            _lib.check(lib.nf_predict_pix_host(self.handle, _lib.ptr(params), dt, _lib.ptr(pv), B, ncomp, flags,
                                               _lib.ptr(out)), "predict")
            return out
        out = np.empty((B, self.n_spec, self.n_chan), dtype=np.float32)
        if self.model == _lib.NF_MODEL_NH3:
            rc = lib.nf_nh3_predict_host(self.handle, _lib.ptr(params), dt, B, ncomp, flags, _lib.ptr(out))
        elif self.model == _lib.NF_MODEL_N2HP:
            rc = lib.nf_n2hp_predict_host(self.handle, _lib.ptr(params), dt, B, ncomp, _lib.ptr(out))
        else:
            rc = lib.nf_gauss_predict_host(self.handle, _lib.ptr(params), dt, B, ncomp, _lib.ptr(out))
        _lib.check(rc, "predict")
        return out

    def moments(self, params, cold=False, lte=False, pix_of_vec=None):
        """Peak and channel sum of single-component model spectra (NH3 and N2H+ blocks): params [B, n_model] ->
        (peak float32 [B, n_spec] in K, sum float64 [B, n_spec] in K channel), each over the spectrum's own
        channels.  The spectra are those ``predict`` synthesises; only their maximum and FP64 sum leave the device.
        ``pix_of_vec`` as for ``predict`` (required on a block from ``from_spectra``)."""
        if self.model == _lib.NF_MODEL_GAUSS:
            raise ValueError("moments: the Gaussian model's peak and area are its own parameters")
        params, dt = self._params(params)
        if params.ndim != 2 or params.shape[1] != self.n_model:
            raise ValueError(f"moments takes single-component vectors [B, {self.n_model}], got {params.shape}")
        B = params.shape[0]
        pv = None
        if pix_of_vec is not None:
            pv = np.ascontiguousarray(pix_of_vec, dtype=np.int32)
            if pv.shape != (B,):
                raise ValueError("pix_of_vec must have one entry per vector")
            if B and (pv.min() < 0 or pv.max() >= self.n_pix):
                raise ValueError("pix_of_vec out of range")
        elif self.per_pixel_axes:
            raise ValueError("a block with per-pixel axes needs pix_of_vec for moments")
        flags = (_lib.NF_FLAG_COLD if cold else 0) | (_lib.NF_FLAG_LTE if lte else 0)
        peak = np.empty((B, self.n_spec), dtype=np.float32)
        total = np.empty((B, self.n_spec), dtype=np.float64)
        _lib.check(_lib.load().nf_predict_moments_host(self.handle, _lib.ptr(params), dt, _lib.ptr(pv), B, flags,
                                                        _lib.ptr(peak), _lib.ptr(total)), "moments")
        return peak, total

    def last_call_stats(self):
        ms = C.c_double()
        n = C.c_int64()
        _lib.load().nf_last_call_stats(C.byref(ms), C.byref(n))
        return ms.value, n.value
