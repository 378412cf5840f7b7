"""Cube orchestration behind the reference's ``nestfit.main`` fitting API (NoiseMap, DataCube, CubeStack,
CubeFitter, get_multiproc_indices; reference nestfit/main.py:39-223,380-526,565-571).

The reference walks pixels one at a time per forked process and calls MultiNest per (pixel, ncomp).  Here a
contiguous block of pixels is uploaded to one GPU and all its pixels advance in lock-step through the batched
sampler, one *wave* per number of components; the ncomp-escalation rule (main.py:450-469) selects which pixels
enter the next wave.  A finished wave leaves the device as one posterior pool plus attribute columns and is
written to the store by a background thread while the next wave runs.  Multi-GPU = disjoint contiguous pixel
blocks handed out to one process per GPU, one store chunk per process, no collective.
"""
import os
import queue as _queue
import threading
import time

import numpy as np

from .pixels import PixelBlock
from .sampler import NestedSamplingBatch
from .store import GroupSink, HdfStore, Wave, chunk_sink, run_attr_columns


def nans(shape, dtype=None):
    return np.full(shape, np.nan, dtype=dtype)


class NoiseMap:
    """Per-pixel rms in the cube's (lon, lat) order.  Like the reference's class (main.py:39-65) it is built from
    an image in (lat, lon) order; `get_noise` takes scalar or array indices (the GPU path asks for whole blocks)."""
    shape = None

    def __init__(self, data):
        self.data = np.swapaxes(np.asarray(data, dtype=np.float64), 0, 1)
        self.shape = self.data.shape

    @classmethod
    def from_pbimg(cls, rms, pb_img):
        """rms / primary-beam response; the plane is the last two axes of a 2-, 3- or 4-axis image, pixels where
        the response vanishes get infinite noise."""
        pb = np.asarray(pb_img, dtype=np.float64)
        if not 2 <= pb.ndim <= 4:
            raise ValueError(f'Cannot parse shape : {pb.shape}')
        plane = pb.reshape(pb.shape[-2:]) if pb.size == pb.shape[-2] * pb.shape[-1] else pb[(0,) * (pb.ndim - 2)]
        with np.errstate(divide='ignore', invalid='ignore'):
            img = rms / plane
        return cls(np.where(np.isfinite(img), img, np.inf))

    def get_noise(self, i_lon, i_lat):
        return self.data[i_lon, i_lat]


class NoiseMapUniform(NoiseMap):
    """One rms for every pixel (main.py:68-74); `shape` is None so that any cube accepts it."""

    def __init__(self, rms):
        self.rms = rms

    def get_noise(self, i_lon, i_lat):
        return self.rms


class DataCube:
    """Channel-contiguous cube ``data[lon, lat, chan]`` on an ascending Hz axis with
    scalar noise per pixel: the array contract of the reference's DataCube
    (main.py:77-172).  Built from arrays (`from_arrays`); FITS ingestion through
    spectral_cube stays with the reference (those packages are optional)."""

    def __init__(self, cube=None, noise_map=None, trans_id=None, *, data=None, xarr=None, header=None):
        if cube is not None:
            data, xarr, header = self._from_spectral_cube(cube)
        if isinstance(noise_map, (float, int)):
            self.noise_map = NoiseMapUniform(noise_map)
        else:
            self.noise_map = noise_map
        self.trans_id = trans_id
        self._header = dict(header or {})
        xarr = np.ascontiguousarray(xarr, dtype=np.float64)
        data = np.asarray(data)
        if xarr[1] < xarr[0]:                      # ascending frequency axis (main.py:146-149)
            xarr = xarr[::-1].copy()
            data = data[..., ::-1]
        self.data = np.ascontiguousarray(data)
        self.xarr = xarr
        self.shape = self.data.shape
        self.spatial_shape = (self.shape[0], self.shape[1])
        self.nchan = self.shape[2]
        self.dv = abs(xarr[1] - xarr[0]) / xarr.mean() * 299792.458
        if self.noise_map.shape is not None:
            assert self.spatial_shape == self.noise_map.shape

    @classmethod
    def from_arrays(cls, data, xarr, noise_map, trans_id=None, header=None):
        return cls(None, noise_map, trans_id, data=data, xarr=xarr, header=header)

    @staticmethod
    def _from_spectral_cube(cube):  # pragma: no cover - optional dependency
        from astropy import units
        if cube.unit == '':
            cube._unit = units.K
        elif cube.unit != 'K':
            cube = cube.to('K')
        if cube.spectral_axis.unit != 'Hz':
            cube = cube.with_spectral_unit('Hz')
        axis = cube.spectral_axis.value.copy()
        data = cube._data.transpose().copy()       # (s, b, l) -> (l, b, s)
        return data, axis, dict(cube.header)

    @property
    def full_header(self):
        return self._header

    @property
    def simple_header(self):
        keys = ('SIMPLE', 'BITPIX', 'NAXIS', 'NAXIS1', 'NAXIS2', 'WCSAXES', 'CRPIX1', 'CRPIX2', 'CDELT1', 'CDELT2',
                'CUNIT1', 'CUNIT2', 'CTYPE1', 'CTYPE2', 'CRVAL1', 'CRVAL2', 'RADESYS', 'EQUINOX')
        hdict = {k: self._header[k] for k in keys if k in self._header}
        hdict['NAXIS'] = 2
        hdict['WCSAXES'] = 2
        return hdict

    def get_spec_data(self, i_lon, i_lat):
        arr = self.data[i_lon, i_lat, :]
        noise = self.noise_map.get_noise(i_lon, i_lat)
        has_nans = np.isnan(arr).any() or np.isnan(noise)
        return self.xarr, arr, noise, self.trans_id, has_nans


class CubeStack:
    """The cubes fitted together (one per transition; main.py:175-223).  The batched view `block_arrays` is what
    the GPU path consumes; the reference's per-pixel accessors are thin views of it."""

    def __init__(self, cubes):
        self.cubes = list(cubes)
        if not self.cubes:
            raise ValueError('CubeStack needs at least one cube')
        self.n_cubes = len(self.cubes)
        first = self.cubes[0]
        # the stack reports the geometry and headers of its first cube
        self.shape, self.spatial_shape = first.shape, first.spatial_shape

    def __iter__(self):
        return iter(self.cubes)

    full_header = property(lambda self: self.cubes[0].full_header)
    simple_header = property(lambda self: self.cubes[0].simple_header)

    def block_arrays(self, lon, lat):
        """data [n, n_cubes, n_chan], noise [n, n_cubes], valid [n] for pixel lists."""
        lon, lat = np.asarray(lon), np.asarray(lat)
        data = np.stack([c.data[lon, lat, :] for c in self.cubes], axis=1)
        noise = np.stack([np.broadcast_to(np.asarray(c.noise_map.get_noise(lon, lat), dtype=np.float64), lon.shape)
                          for c in self.cubes], axis=1)
        valid = ~(np.isnan(data).any(axis=(1, 2)) | np.isnan(noise).any(axis=1))
        return data, noise, valid

    def block_max_snr(self, lon, lat):
        """Largest peak signal-to-noise over the cubes, per pixel (the quantity nlive scales with, main.py:445-447)."""
        data, noise, _ = self.block_arrays(lon, lat)
        return np.maximum((data.max(axis=2) / noise).max(axis=1), 0.0)

    def get_arrays(self, i_lon, i_lat):
        return list(self.block_arrays([i_lon], [i_lat])[0][0])

    def get_spec_data(self, i_lon, i_lat):
        data, noise, valid = self.block_arrays([i_lon], [i_lat])
        rows = [[c.xarr, data[0, k], noise[0, k].item(), c.trans_id] for k, c in enumerate(self.cubes)]
        return rows, not bool(valid[0])

    def get_max_snr(self, i_lon, i_lat):
        return float(self.block_max_snr([i_lon], [i_lat])[0])


def get_multiproc_indices(shape, nproc):
    """The reference's row striping `lon_ix[i::nproc]` (main.py:565-571)."""
    lon_ix, lat_ix = np.indices(shape)
    return [(lon_ix[i::nproc, ...].flatten(), lat_ix[i::nproc, ...].flatten()) for i in range(nproc)]


def get_block_indices(shape, nblocks):
    """Contiguous pixel blocks of the (lon, lat) grid in C order, one per GPU."""
    lon_ix, lat_ix = np.indices(shape)
    lon_ix, lat_ix = lon_ix.ravel(), lat_ix.ravel()
    bounds = np.linspace(0, lon_ix.size, nblocks + 1).astype(int)
    return [(lon_ix[a:b], lat_ix[a:b]) for a, b in zip(bounds[:-1], bounds[1:])]


class _WaveWriter:
    """Background thread that turns finished samplers into store waves: the device pass over the posterior
    products, the one device-to-host copy and the file write of wave N overlap the sampling of wave N + 1."""

    def __init__(self, sink, store_posteriors, intensity=False):
        self.sink, self.store_posteriors, self.intensity = sink, store_posteriors, intensity
        self.q = _queue.Queue(maxsize=1)          # at most one finished sampler waits with its device pool
        self.error = None
        self.seconds = 0.0
        self.intensity_seconds = 0.0
        self.rows = 0
        self.thread = threading.Thread(target=self._loop, daemon=True)
        self.thread.start()

    def _loop(self):
        while True:
            job = self.q.get()
            if job is None:
                return
            ns, sel, meta = job
            try:
                if self.error is None:
                    t0 = time.perf_counter()
                    wave = make_wave(ns, sel, self.store_posteriors, intensity=self.intensity, **meta)
                    self.intensity_seconds += wave.intensity_seconds
                    self.sink.add_wave(wave)
                    self.seconds += time.perf_counter() - t0
            except BaseException as exc:          # surfaces in the fitting thread at the next submit / close
                self.error = exc
            finally:
                ns.close()

    def submit(self, ns, sel, **meta):
        if self.error is not None:
            ns.close()
            raise self.error
        self.q.put((ns, sel, meta))

    def close(self):
        self.q.put(None)
        self.thread.join()
        if self.error is not None:
            raise self.error


def make_wave(ns, sel, store_posteriors, i_lon, i_lat, null_lnZ, n_chan_tot, intensity=False):
    """The runs `sel` (None = all) of a finished sampler as a store `Wave`; with `intensity` it carries the runs'
    intensity credible intervals (NestedSamplingBatch.intensity_marginals), computed before the sampler closes."""
    res = ns.results
    prod = ns.products_all(marginals=True, posteriors=store_posteriors)
    t_i = time.perf_counter()
    inten = ns.intensity_marginals() if intensity else None
    t_i = time.perf_counter() - t_i
    off = prod['row_offsets']
    n_samples = np.diff(off)
    cols = run_attr_columns(ns.ndim, n_chan_tot, ns.nlive, null_lnZ, res, n_samples)
    post, marg, best, mapf = prod['posteriors'], prod['marginals'], res['bestfit'], res['mapfit']
    if sel is not None:
        sel = np.asarray(sel, dtype=np.int64)
        cols = {k: v[sel] for k, v in cols.items()}
        if post is not None:
            post = np.concatenate([post[off[r]:off[r + 1]] for r in sel]) if sel.size else post[:0]
        off = np.concatenate([[0], np.cumsum(n_samples[sel])])
        marg, best, mapf = marg[sel], best[sel], mapf[sel]
        i_lon, i_lat = np.asarray(i_lon)[sel], np.asarray(i_lat)[sel]
        if inten is not None:
            inten = {k: v[sel] for k, v in inten.items()}
    wave = Wave(ns.ncomp, ns.ndim, n_chan_tot, i_lon, i_lat, cols, off, post, marg, best, mapf, inten)
    wave.intensity_seconds = t_i if intensity else 0.0
    return wave


class CubeFitter:
    mn_default_kwargs = {
        'nlive': 100,
        'tol': 1.0,
        'efr': 0.3,
        'updInt': 2000,
    }

    def __init__(self, stack, utrans, runner_cls, runner_kwargs=None, lnZ_thresh=11, ncomp_max=2, mn_kwargs=None,
                 nlive_snr_fact=5, n_prop=32, max_pixels_per_wave=16384, seed=1234, store_posteriors=True,
                 n_streams=1, pixels_per_stream=1024, retry_margin=None, retry_chi2_sigma=6.0,
                 intensity_marginals=False):
        """Same arguments as the reference (main.py:388-421) plus the batching knobs
        `n_prop` (proposals per pixel per lock-step iteration), `max_pixels_per_wave`
        (pixels in flight per device wave), `n_streams` (host threads / CUDA streams that
        escalate sub-blocks of `pixels_per_stream` pixels concurrently), `seed`, and the optional lost-mode
        guard `retry_margin` (default None = off, one run per (pixel, ncomp) like the reference; e.g. 10):
        an N-component run whose maximum likelihood falls more than this below the (N-1)-component run's
        has lost the dominant mode and is repeated once with twice the live points, as is a run (N >= 2)
        that fails the evidence threshold while its best chi-square is more than `retry_chi2_sigma` sigma
        above the channel count.  The repeats are a small extra wave per ncomp (~1-2 s of latency each).
        Sampler options ride in `mn_kwargs`: 'walks', 'method', 'max_samples_per_live' (rows of the posterior pool
        per live point, default 64; runs that fill their share are repeated with four times as many).
        `intensity_marginals` (NH3 / N2H+): every run written to the store also carries the posterior-weighted
        quantiles of each component's peak and integrated intensity ('peak_intensity_marginals',
        'integrated_intensity_marginals', (M, n_spec, ncomp)), computed on the device by the store writer before the
        run's posterior leaves it; `aggregate_intensity_marginals` gathers them into maps."""
        self.stack = stack
        self.utrans = utrans
        self.runner_cls = runner_cls
        self.runner_kwargs = {} if runner_kwargs is None else runner_kwargs
        self.lnZ_thresh = lnZ_thresh
        self.ncomp_max = ncomp_max
        self.mn_kwargs = self.mn_default_kwargs.copy()
        if mn_kwargs is not None:
            self.mn_kwargs.update(mn_kwargs)
        self.nlive_snr_fact = nlive_snr_fact
        self.n_prop = n_prop
        self.max_pixels_per_wave = max_pixels_per_wave
        self.n_streams = n_streams
        self.pixels_per_stream = pixels_per_stream
        self.retry_margin = retry_margin
        self.retry_chi2_sigma = retry_chi2_sigma
        self.seed = seed
        self.store_posteriors = store_posteriors
        self.intensity_marginals = intensity_marginals
        self.stats = {}

    def __getstate__(self):
        # what a spawned worker needs: no open store, no device binding, no results of earlier fits
        state = self.__dict__.copy()
        for k in ('_store', '_device'):
            state.pop(k, None)
        state['stats'] = {}
        return state

    def _model_name(self):
        import inspect
        return inspect.getmodule(self.runner_cls).NAME

    def _sampler(self, blk, ncomp, pix, nlive, seed, per_live=None):
        kw = {k: v for k, v in self.runner_kwargs.items() if k in ('cold', 'lte')}
        if self.mn_kwargs.get('walks'):
            kw['walks'] = int(self.mn_kwargs['walks'])       # random-walk steps per new point
        if self.mn_kwargs.get('method'):
            kw['method'] = self.mn_kwargs['method']
        if 'mmodal' in self.mn_kwargs:                       # MultiNest's switch (core.pyx:729): ellipsoid decomposition
            kw['mmodal'] = bool(self.mn_kwargs['mmodal'])
        per_live = int(per_live or self.mn_kwargs.get('max_samples_per_live', 64))
        return NestedSamplingBatch(blk, self.utrans, ncomp, pix_ids=pix, nlive=nlive, tol=self.mn_kwargs['tol'],
                                   efr=self.mn_kwargs['efr'], n_prop=self.n_prop, seed=seed,
                                   max_iter=self.mn_kwargs.get('maxiter', 1_000_000),
                                   max_samples=per_live * int(np.max(nlive)), **kw)

    def fit_block(self, indices, device=0, group_root=None, verbose=False):
        """Fit the pixels (all_lon, all_lat) on one GPU.  Returns a dict of per-pixel arrays (nbest,
        lnZ[ncomp_max+1], ...).  `group_root` receives the results: a store sink (``HdfStore.chunk_sink``) takes
        whole waves; an h5py-like group gets the reference's /pix/<lon>/<lat>/<ncomp> groups one by one."""
        all_lon, all_lat = (np.asarray(a) for a in indices)
        n_tot = all_lon.size
        model = self._model_name()
        if self.intensity_marginals and model not in ('ammonia', 'diazenylium'):
            raise ValueError("intensity_marginals: the Gaussian model's peak and area are its own parameters")
        sink = None
        if group_root is not None:
            sink = group_root if hasattr(group_root, 'add_wave') else GroupSink(group_root, self.store_posteriors)
            if hasattr(sink, 'store_posteriors'):
                sink.store_posteriors = self.store_posteriors
        writer = _WaveWriter(sink, self.store_posteriors, self.intensity_marginals) if sink is not None else None
        n_evals = 0
        out = dict(i_lon=all_lon, i_lat=all_lat, nbest=np.full(n_tot, -1, dtype=np.int32),
                   lnZ=nans((n_tot, self.ncomp_max + 1)), lnZ_err=nans((n_tot, self.ncomp_max + 1)),
                   max_loglike=nans((n_tot, self.ncomp_max + 1)), n_samples=np.zeros((n_tot, self.ncomp_max + 1), int),
                   n_retried=0, n_rescued=0, n_truncated=0, evals_by_ncomp=np.zeros(self.ncomp_max + 1, dtype=np.int64),
                   seconds_by_ncomp=np.zeros(self.ncomp_max + 1))
        n_lat = int(self.stack.spatial_shape[1])
        t0 = time.perf_counter()
        try:
            for w0 in range(0, n_tot, self.max_pixels_per_wave):
                sl = slice(w0, min(n_tot, w0 + self.max_pixels_per_wave))
                lon, lat = all_lon[sl], all_lat[sl]
                data, noise, valid = self.stack.block_arrays(lon, lat)
                if not valid.any():
                    continue
                vidx = np.flatnonzero(valid)
                dv = data[vidx]
                xarrs = [c.xarr for c in self.stack.cubes]
                if model in ('ammonia', 'diazenylium'):
                    blk = PixelBlock(model, xarrs, dv, noise[vidx], trans_ids=[c.trans_id for c in self.stack.cubes],
                                     device=device)
                else:
                    blk = PixelBlock('gaussian', xarrs, dv, noise[vidx],
                                     rest_freq=self.runner_kwargs.get('rest_freq', xarrs[0].mean()), device=device)
                null = blk.null_lnZ()
                # live points scale with the peak SNR (main.py:445-447)
                max_snr = np.maximum(np.max(dv.max(axis=2) / noise[vidx], axis=1), 0.0)
                nlive = self.mn_kwargs['nlive'] + (self.nlive_snr_fact * max_snr).astype(int)
                n_chan_tot = blk.n_spec * blk.n_chan
                old_lnZ = null.copy()
                nbest = np.zeros(vidx.size, dtype=np.int32)
                out['lnZ'][w0 + vidx, 0] = null
                lock = threading.Lock()
                # the random streams are keyed on (seed, run, ...): every block gets its own seed from the
                # cube-wide index of its first pixel, so equal run numbers of different blocks differ
                block_key = 1000003 * (int(lon[0]) * n_lat + int(lat[0]) + 1)

                def fit_sub(active, tag):
                    """ncomp escalation (main.py:450-469) of one sub-block of the wave's pixels."""
                    nonlocal n_evals
                    for ncomp in range(1, self.ncomp_max + 1):
                        if active.size == 0:
                            break
                        if verbose:
                            print(f'-- wave {w0}.{tag}: N = {ncomp}: {active.size} pixels')
                        t_n = time.perf_counter()
                        seed = self.seed + 7919 * ncomp + 104729 * tag + block_key
                        ns = self._sampler(blk, ncomp, active, nlive[active], seed)
                        res = ns.run()
                        evals = int(res['n_evals'].sum())
                        assert np.isfinite(res['lnZ']).all()           # main.py:463
                        gi = w0 + vidx[active]
                        extra = []          # (sampler, positions of its runs in `active`, its rows to keep or None = all)
                        # A run that filled its share of the posterior pool stopped before its evidence
                        # converged (very bright pixels: H > ~60 nats): repeat those with a four times larger share
                        trunc = np.flatnonzero(res['truncated'])
                        if trunc.size:
                            ns_t = self._sampler(blk, ncomp, active[trunc], nlive[active[trunc]], seed + 32452843,
                                                 per_live=4 * int(self.mn_kwargs.get('max_samples_per_live', 64)))
                            res_t = ns_t.run()
                            evals += int(res_t['n_evals'].sum())
                            for key in ('lnZ', 'lnZ_err', 'max_loglike', 'n_samples'):
                                res[key][trunc] = res_t[key]
                            extra.append((ns_t, trunc, None))
                            with lock:
                                out['n_truncated'] += int(trunc.size)
                        # Lost-mode guard (a few per cent of 3-component runs at nlive ~ 300 end in a secondary
                        # mode).  Two symptoms: (i) an N-component model can always reproduce the (N-1)-component
                        # fit, so a best likelihood clearly *below* the previous wave's is a lost mode; (ii) the
                        # run does not pass the evidence threshold although its best fit is far from the noise
                        # (chi-square many sigma above the channel count, the noise being known).  Such runs are
                        # repeated once with twice the live points and a new seed; the repeat replaces the run
                        # when its evidence is higher.
                        if ncomp >= 2 and self.retry_margin is not None:
                            suspect = res['max_loglike'] < out['max_loglike'][gi, ncomp - 1] - self.retry_margin
                            if self.retry_chi2_sigma is not None:
                                chi2_max = n_chan_tot + self.retry_chi2_sigma * np.sqrt(2.0 * n_chan_tot)
                                suspect |= ((-2.0 * res['max_loglike'] > chi2_max) &
                                            (res['lnZ'] - old_lnZ[active] < self.lnZ_thresh))
                            lost = np.flatnonzero(suspect)
                            if lost.size:
                                ns_r = self._sampler(blk, ncomp, active[lost], 2 * nlive[active[lost]], seed + 15485863)
                                res2 = ns_r.run()
                                evals += int(res2['n_evals'].sum())
                                better = np.flatnonzero(res2['lnZ'] > res['lnZ'][lost])
                                for key in ('lnZ', 'lnZ_err', 'max_loglike', 'n_samples'):
                                    res[key][lost[better]] = res2[key][better]
                                extra.append((ns_r, lost, better))
                                with lock:
                                    out['n_retried'] += int(lost.size)
                                    out['n_rescued'] += int(better.size)
                        out['lnZ'][gi, ncomp] = res['lnZ']
                        out['lnZ_err'][gi, ncomp] = res['lnZ_err']
                        out['max_loglike'][gi, ncomp] = res['max_loglike']
                        out['n_samples'][gi, ncomp] = res['n_samples']
                        # hand the finished samplers to the writer (a later wave of the same (pixel, ncomp)
                        # replaces the earlier one in the store); without a store they are simply released
                        for s_obj, pos, rows in [(ns, np.arange(active.size), None)] + extra:
                            if writer is None or (rows is not None and len(rows) == 0):
                                s_obj.close()
                                continue
                            px = active[pos]
                            writer.submit(s_obj, rows, i_lon=lon[vidx[px]], i_lat=lat[vidx[px]], null_lnZ=null[px],
                                          n_chan_tot=n_chan_tot)
                        improved = res['lnZ'] - old_lnZ[active] >= self.lnZ_thresh     # main.py:464-469
                        old_lnZ[active[improved]] = res['lnZ'][improved]
                        nbest[active[improved]] = ncomp
                        with lock:
                            n_evals += evals
                            out['evals_by_ncomp'][ncomp] += evals
                            out['seconds_by_ncomp'][ncomp] += time.perf_counter() - t_n
                        active = active[improved]

                # Sub-blocks of the wave escalate independently, each on its own stream, picked from a
                # queue by `n_streams` host threads (the sampler call releases the GIL).  The workers
                # drift apart, so the thin tail of one sub-block's run overlaps the bulk of another's
                # instead of idling the GPU.
                n_sub = max(1, vidx.size // max(1, self.pixels_per_stream)) if self.n_streams > 1 else 1
                subs = np.array_split(np.arange(vidx.size), n_sub)
                if n_sub == 1:
                    fit_sub(subs[0], 0)
                else:
                    errors = []
                    todo = list(enumerate(subs))[::-1]

                    def worker():
                        while True:
                            with lock:
                                if not todo or errors:
                                    return
                                tag, sub = todo.pop()
                            try:
                                fit_sub(sub, tag)
                            except BaseException as exc:   # re-raised in the caller's thread
                                errors.append(exc)

                    threads = [threading.Thread(target=worker) for _ in range(min(self.n_streams, n_sub))]
                    for th in threads:
                        th.start()
                    for th in threads:
                        th.join()
                    if errors:
                        raise errors[0]
                out['nbest'][w0 + vidx] = nbest
                if sink is not None:
                    sink.add_pixels(lon[vidx], lat[vidx], nbest)
                if writer is not None:          # the block's device rows must outlive its samplers
                    t_w = time.perf_counter()
                    writer.close()
                    # time the writer worked (mostly hidden behind the next wave) and time the fit waited for it
                    out['store_seconds'] = out.get('store_seconds', 0.0) + writer.seconds
                    out['store_wait_seconds'] = out.get('store_wait_seconds', 0.0) + time.perf_counter() - t_w
                    out['intensity_seconds'] = out.get('intensity_seconds', 0.0) + writer.intensity_seconds
                    writer = _WaveWriter(sink, self.store_posteriors, self.intensity_marginals)
                blk.close()
        except BaseException:
            if writer is not None:
                try:
                    writer.close()
                except BaseException:
                    pass
            raise
        if writer is not None:
            writer.close()
        out['seconds'] = time.perf_counter() - t0
        out['n_evals'] = n_evals
        return out

    def fit(self, *args):
        """Reference-compatible worker entry (main.py:423-474): ((all_lon, all_lat), chunk_path)."""
        (all_lon, all_lat), chunk_path = args
        store = getattr(self, "_store", None)
        device = getattr(self, "_device", 0)
        if store is not None:
            i = [str(p) for p in store.chunk_paths].index(str(chunk_path))
            root = store.open_chunk(i)
            try:
                res = self.fit_block((all_lon, all_lat), device=device, group_root=root)
            finally:
                store.close_chunk(i, root)
            return res
        return self.fit_block((all_lon, all_lat), device=device)

    def _check_partition(self, nproc, blocks_per_gpu, devices):
        n_lon = self.stack.spatial_shape[0]
        if nproc > n_lon:
            raise ValueError(f'The pixel width of the image in longitude ({n_lon}) ' +
                             f'must be greater than or equal to the number of processes ({nproc}).')
        if blocks_per_gpu < 1:
            raise ValueError(f'blocks_per_gpu must be positive: {blocks_per_gpu}')
        devices = list(range(nproc)) if devices is None else [int(d) for d in devices]
        if len(devices) != nproc:
            raise ValueError(f'devices must name one CUDA device per process: {devices}')
        return devices

    def _new_store(self, store_name, nproc):
        store = HdfStore(store_name, nchunks=nproc)
        store.insert_header(self.stack)
        store.insert_fitter_pars(self)
        store.insert_model_metadata(self.runner_cls)
        return store

    def fit_cube(self, store_name='run/test_cube', nproc=1, timeout=None, blocks_per_gpu=1, devices=None):
        """Fit every pixel and write the store.  `nproc` = number of GPUs: one process per GPU, one chunk
        per process (main.py:476-526).  With `blocks_per_gpu` = 1 every process fits one contiguous pixel
        block; with more, the cube is cut into `nproc * blocks_per_gpu` contiguous blocks that the processes
        take from a shared queue as they finish (pixels differ in cost: nlive grows with the SNR and the
        number of model runs with the number of components, SURVEY.md 8e).  `devices` lists the CUDA device
        of each process (default 0 .. nproc-1).  Returns one result dict per fitted block."""
        devices = self._check_partition(nproc, blocks_per_gpu, devices)
        store = self._new_store(store_name, nproc)
        n_blocks = store.nchunks * int(blocks_per_gpu)
        n_pix = int(np.prod(self.stack.spatial_shape))
        indices = get_block_indices(self.stack.spatial_shape, min(n_blocks, n_pix))
        results = []
        if store.nchunks == 1:
            self._store, self._device = store, devices[0]
            try:
                lon = np.concatenate([b[0] for b in indices])
                lat = np.concatenate([b[1] for b in indices])
                results.append(self.fit((lon, lat), store.chunk_paths[0]))
            finally:
                self._store = None
        else:
            import multiprocessing as mp
            ctx = mp.get_context('spawn')
            work = None
            if blocks_per_gpu > 1:
                work = ctx.Queue()
                for j in range(len(indices)):
                    work.put(j)
                for _ in range(store.nchunks):
                    work.put(None)                 # one stop mark per process
            done = ctx.Queue()
            procs = [ctx.Process(target=_fit_worker,
                                 args=(self, str(store.store_dir), store.nchunks, i, devices[i],
                                       indices if work is not None else indices[i], work, done))
                     for i in range(store.nchunks)]
            for proc in procs:
                proc.start()
            failed = None
            t_end = None if timeout is None else time.monotonic() + timeout
            live = list(procs)
            while live and failed is None:
                try:                               # drain the (small) per-block summaries while the workers run
                    results.append(done.get(timeout=0.2))
                except _queue.Empty:
                    pass
                for proc in list(live):
                    if not proc.is_alive():
                        live.remove(proc)
                        if proc.exitcode != 0:
                            failed = proc.exitcode
                if t_end is not None and time.monotonic() > t_end:
                    break
            if failed is not None:
                for proc in procs:          # do not leave the other workers running behind the error
                    if proc.is_alive():
                        proc.terminate()
                raise RuntimeError(f'GPU worker failed with exit code {failed}')
            while True:
                try:
                    results.append(done.get(timeout=0.2))
                except _queue.Empty:
                    break
        store.link_files()
        store.close()
        self.stats['results'] = results
        return results

    def fit_cube_rank(self, store_name, rank, world, blocks_per_gpu=8, device=0, barrier=None, concurrent_blocks=2,
                      pixels_in_flight=8192):
        """SPMD form of `fit_cube` for processes that already exist, one per GPU (torchrun): every rank calls this
        with its `rank`; blocks are claimed through the store directory (exclusive file creation), rank 0 creates
        the store and links the chunks at the end.  `barrier()` (e.g. torch.distributed.barrier) separates
        creation, fitting and linking.

        The blocks of an over-decomposed cube are small, and one small block alone leaves the GPU underfilled (fewer
        runs per lock-step than the device has warps, and a thin tail per wave).  So a rank (i) claims several
        blocks at a time and fits them as ONE wave sequence -- as many as bring about `pixels_in_flight` pixels onto
        the device, but never more than half of its fair share of the cube, so that the second half of the work
        is handed out dynamically -- and (ii) keeps `concurrent_blocks` such groups in flight from as many host
        threads, each on its own CUDA stream (the tail of one group overlaps the bulk of another, and the store
        writer of one the sampling of the other).  Blocks are claimed in descending order of a cost proxy (the sum
        over the block of the live-set sizes, which grow with the peak SNR), the same order on every rank: the
        expensive blocks start first and the cheap ones fill the end, which keeps the ranks' finishing times close.
        Returns this rank's list of per-group results (`blocks`: the block numbers of the group)."""
        self._check_partition(world, blocks_per_gpu, list(range(world)))
        barrier = barrier or (lambda: None)
        if rank == 0:
            self._new_store(store_name, world).close()
        barrier()
        from pathlib import Path
        from .store import check_ext
        store_dir = Path(check_ext(str(store_name), ext='store'))
        n_pix = int(np.prod(self.stack.spatial_shape))
        indices = get_block_indices(self.stack.spatial_shape, min(world * int(blocks_per_gpu), n_pix))
        claims = store_dir / 'claims'
        claims.mkdir(exist_ok=True)
        sink = chunk_sink(store_dir, rank, self.store_posteriors)
        if self.utrans is not None and hasattr(self.utrans, 'handle'):
            self.utrans.handle(device)              # the device prior plan exists before the threads start
        # longest-processing-time-first: the same cost-sorted list on every rank, claimed from the top.  (Without a
        # cost proxy -- a stack that cannot give the peak SNR -- every rank starts at its own stretch of the list.)
        if hasattr(self.stack, 'block_max_snr'):
            cost = [float(np.sum(self.mn_kwargs['nlive'] + self.nlive_snr_fact * np.nan_to_num(
                self.stack.block_max_snr(lon, lat), nan=0.0, posinf=0.0))) for lon, lat in indices]
            order = [int(j) for j in np.argsort(-np.asarray(cost), kind='stable')]
        else:
            first = (rank * len(indices)) // world
            order = [(first + k) % len(indices) for k in range(len(indices))]
        n_thr = max(1, min(int(concurrent_blocks), len(indices)))
        per_block = max(1, n_pix // len(indices))
        in_flight = min(float(pixels_in_flight), 0.5 * n_pix / world)
        group = int(max(1, round(in_flight / n_thr / per_block)))
        results, errors, lock = [], [], threading.Lock()
        cursor = [0]

        def claim():
            """Up to `group` blocks nobody has taken yet."""
            mine = []
            while len(mine) < group:
                with lock:
                    if errors or cursor[0] >= len(order):
                        break
                    j = order[cursor[0]]
                    cursor[0] += 1
                try:
                    os.close(os.open(claims / f'block{j}', os.O_CREAT | os.O_EXCL | os.O_WRONLY))
                    mine.append(j)
                except FileExistsError:
                    continue
            return mine

        def worker():
            while True:
                mine = claim()
                if not mine:
                    return
                try:
                    lon = np.concatenate([indices[j][0] for j in mine])
                    lat = np.concatenate([indices[j][1] for j in mine])
                    res = self.fit_block((lon, lat), device=device, group_root=sink)
                    res['blocks'] = mine
                    with lock:
                        results.append(res)
                except BaseException as exc:        # re-raised in the caller's thread
                    with lock:
                        errors.append(exc)
                    return

        t0 = time.perf_counter()
        try:
            if n_thr == 1:
                worker()
            else:
                threads = [threading.Thread(target=worker) for _ in range(n_thr)]
                for th in threads:
                    th.start()
                for th in threads:
                    th.join()
        finally:
            sink.close()
        self.stats['rank_fit_seconds'] = time.perf_counter() - t0
        barrier()           # reached by a failing rank too: the others wait here, and must not wait for ever
        if errors:
            raise errors[0]
        if rank == 0:
            with HdfStore(store_name) as store:
                store.link_files()
        return results


def _block_summary(res, block, worker):
    """What a worker reports back per block: scalars only (the per-pixel arrays are in the store)."""
    keep = ('seconds', 'n_evals', 'n_retried', 'n_rescued', 'n_truncated', 'store_seconds', 'store_wait_seconds',
            'intensity_seconds')
    out = {k: res[k] for k in keep if k in res}
    out.update(block=block, worker=worker, n_pix=int(np.asarray(res.get('nbest', ())).size))
    for k in ('evals_by_ncomp', 'seconds_by_ncomp'):
        if k in res:
            out[k] = np.asarray(res[k]).tolist()
    return out


def _fit_worker(fitter, store_dir, nchunks, i, device, indices, work=None, done=None):
    """Process `i` of fit_cube: fits its block (or blocks taken from the `work` queue) on `device` into chunk `i`."""
    os.environ.setdefault('HDF5_USE_FILE_LOCKING', 'FALSE')
    sink = chunk_sink(store_dir, i, fitter.store_posteriors)
    try:
        if work is None:
            res = fitter.fit_block(indices, device=device, group_root=sink)
            if done is not None:
                done.put(_block_summary(res, i, i))
            return
        while True:
            j = work.get()
            if j is None:
                break
            res = fitter.fit_block(indices[j], device=device, group_root=sink)
            if done is not None:
                done.put(_block_summary(res, j, i))
    finally:
        sink.close()
