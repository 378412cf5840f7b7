"""Batched nested sampling: host wrapper of ``nf_ns_*`` (include/nestfit_b200.h)
and the drop-in ``run_multinest`` / ``Dumper`` pair of the reference
(nestfit/core/core.pyx:564-609,627-687,727-823).

The sampler itself (proposal, prior transform, fused likelihood, accept/replace,
evidence accumulation) runs on the device; this module sizes buffers, launches
the run and packages results in the reference's result contract.
"""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import NsConfig

_VP, _I, _I64 = C.c_void_p, C.c_int, C.c_int64
_lib.register("nf_ns_create", [_VP, _VP, _I, _I, C.POINTER(NsConfig), _I64, _VP, _VP, C.POINTER(_VP)])
_lib.register("nf_ns_run", [_VP])
_lib.register("nf_ns_free", [_VP])
_lib.register("nf_ns_results", [_VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP])
_lib.register("nf_ns_posterior", [_VP, _I64, C.c_int32, _VP, _VP, _VP])
_lib.register("nf_ns_stats", [_VP, C.POINTER(C.c_int32), C.POINTER(_I64)])
_lib.register("nf_ns_products_rows", [_VP, _VP])
_lib.register("nf_ns_products", [_VP, _VP, _I, _VP, _VP])
_lib.register("nf_ns_intensity", [_VP, _VP, _I, _VP, _VP])

from .store import MARG_COLS, MARG_QUANTILES, run_attr_columns  # noqa: E402  (names re-exported)


class NestedSamplingBatch:
    """Lock-step nested sampling of ``n_run`` (pixel, ncomp) fits on one GPU."""

    def __init__(self, block, utrans, ncomp, pix_ids=None, nlive=100, tol=1.0, efr=0.3, n_prop=32, seed=1,
                 max_iter=1_000_000, max_samples=None, cold=False, lte=False, method='auto', walks=0,
                 n_prop_max=None, target_batch=65536, keep_constant_dims=False, mmodal=False):
        """method: 'auto' = ellipsoidal rejection sampling that hands a run over to a
        constrained random walk once its acceptance stalls; 'ellipsoid' / 'rwalk' force one.
        walks: random-walk steps per new point (0 = 20 + number of dimensions the likelihood depends on).
        keep_constant_dims: keep the cube dimensions the priors overwrite (ConstantPrior rows, DuplicatePrior's
        second row) inside the bounding ellipsoid and the walk metric (the round-1 behaviour; default: they are
        drawn uniformly on their own).
        mmodal: MultiNest-style decomposition of the live set into up to 8 ellipsoids for the rejection phase (the
        reference runs MultiNest with mmodal=True, core.pyx:729); default False = one bounding ellipsoid rebuilt every
        lock-step (measured on B200: the decomposition saves 12 % of the likelihood calls of a cube fit but its
        clustering and overlap tests cost more than they save, and it raises ln Z by ~1-3 at 10-15 dimensions;
        DESIGN.md section 4.4).
        n_prop_max / target_batch: once few runs are still active each gets up to n_prop_max
        proposals per lock-step (default 16 n_prop) so that a launch keeps ~target_batch vectors."""
        lib = _lib.load()
        self.block, self.utrans, self.ncomp = block, utrans, int(ncomp)
        if pix_ids is None:
            pix_ids = np.arange(block.n_pix)
        self.pix_ids = np.ascontiguousarray(pix_ids, dtype=np.int32)
        self.n_run = int(self.pix_ids.size)
        self.nlive = np.ascontiguousarray(np.broadcast_to(np.asarray(nlive, dtype=np.int32), (self.n_run,)))
        self.ndim = block.n_model * self.ncomp
        nlive_max = int(self.nlive.max())
        if max_samples is None:
            max_samples = 64 * nlive_max
        if seed is None or seed < 0:       # reference default seed=-1 means "from the clock" (core.pyx:731)
            seed = int(np.random.SeedSequence().generate_state(1)[0])
        self.cfg = NsConfig(nlive_max=nlive_max, n_prop=int(n_prop), max_iter=int(min(max_iter, 2**31 - 1)),
                            max_samples=int(max_samples), bound_update_interval=int(walks),
                            flags={'auto': 0, 'rwalk': 1, 'ellipsoid': 2}[method] | (4 if keep_constant_dims else 0) | (0 if mmodal else 8),
                            tol=float(tol),
                            efr=float(efr), seed=int(seed),
                            n_prop_max=int(16 * n_prop if n_prop_max is None else n_prop_max),
                            target_batch=int(target_batch))
        flags = (_lib.NF_FLAG_COLD if cold else 0) | (_lib.NF_FLAG_LTE if lte else 0)
        out = C.c_void_p()
        _lib.check(lib.nf_ns_create(block.handle, utrans.handle(block.device), self.ncomp, flags,
                                    C.byref(self.cfg), self.n_run, _lib.ptr(self.pix_ids), _lib.ptr(self.nlive),
                                    C.byref(out)), "nf_ns_create")
        self.handle = out
        self._results = None

    def close(self):
        if getattr(self, "handle", None):
            _lib.load().nf_ns_free(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def run(self):
        lib = _lib.load()
        _lib.check(lib.nf_ns_run(self.handle), "nf_ns_run")
        R, D = self.n_run, self.ndim
        res = dict(lnZ=np.empty(R), lnZ_err=np.empty(R), max_loglike=np.empty(R),
                   n_samples=np.empty(R, dtype=np.int32), n_iter=np.empty(R, dtype=np.int32),
                   n_evals=np.empty(R, dtype=np.int64), bestfit=np.empty((R, D)), mapfit=np.empty((R, D)))
        _lib.check(lib.nf_ns_results(self.handle, _lib.ptr(res["lnZ"]), _lib.ptr(res["lnZ_err"]),
                                     _lib.ptr(res["max_loglike"]), _lib.ptr(res["n_samples"]),
                                     _lib.ptr(res["n_iter"]), _lib.ptr(res["n_evals"]), _lib.ptr(res["bestfit"]),
                                     _lib.ptr(res["mapfit"])), "nf_ns_results")
        it, ln = C.c_int32(), C.c_int64()
        lib.nf_ns_stats(self.handle, C.byref(it), C.byref(ln))
        res["lock_iters"], res["launches"] = it.value, ln.value
        # a run that filled its share of the dead-point pool stopped before its evidence converged
        per_live = self.cfg.max_samples // self.cfg.nlive_max
        res["truncated"] = res["n_samples"] >= np.minimum(self.cfg.max_samples, per_live * self.nlive)
        self._results = res
        self._batch = None
        return res

    def products_all(self, marginals=True, posteriors=True):
        """Posterior products of every run with one device pass and one device-to-host copy (instead of one
        `posterior()` round trip per run): dict(row_offsets [n_run + 1], posteriors float32 [rows, ndim + 2] in
        the layout of the reference's `posteriors` dataset (core.pyx:680), marginals [n_run, 15, ndim])."""
        if getattr(self, "_batch", None) is not None:
            return self._batch
        self.results
        lib = _lib.load()
        off = np.empty(self.n_run + 1, dtype=np.int64)
        _lib.check(lib.nf_ns_products_rows(self.handle, _lib.ptr(off)), "nf_ns_products_rows")
        post = np.empty((int(off[-1]), self.ndim + 2), dtype=np.float32) if posteriors else None
        marg = np.empty((self.n_run, MARG_QUANTILES.size, self.ndim)) if marginals else None
        _lib.check(lib.nf_ns_products(self.handle, _lib.ptr(MARG_QUANTILES), MARG_QUANTILES.size if marginals else 0,
                                      _lib.ptr(post), _lib.ptr(marg)), "nf_ns_products")
        self._batch = dict(row_offsets=off, posteriors=post, marginals=marg)
        return self._batch

    def intensity_marginals(self, quantiles=MARG_QUANTILES):
        """Posterior-weighted credible intervals of every component's peak and integrated intensity, computed on
        the device from the run's posterior rows (NH3 and N2H+).  Returns {'peak_intensity_marginals' (K),
        'integrated_intensity_marginals' (K km/s)}, each [n_run, len(quantiles), n_spec, ncomp].  The integrated
        intensity is the model's channel sum times the channel width of the run's spectrum in km/s
        (|dnu| / mean(nu) * c, as DataCube.dv)."""
        if self.block.model == _lib.NF_MODEL_GAUSS:
            raise ValueError("intensity_marginals: the Gaussian model's peak and area are its own parameters")
        q = np.ascontiguousarray(quantiles, dtype=np.float64)
        if q.ndim != 1 or not 1 <= q.size <= 64:
            raise ValueError("intensity_marginals takes 1 to 64 quantiles")
        self.results
        lib = _lib.load()
        if getattr(self, "_batch", None) is None:       # the rows of every run (nf_ns_products_rows)
            off = np.empty(self.n_run + 1, dtype=np.int64)
            _lib.check(lib.nf_ns_products_rows(self.handle, _lib.ptr(off)), "nf_ns_products_rows")
        shape = (self.n_run, q.size, self.block.n_spec, self.ncomp)
        peak, integ = np.empty(shape), np.empty(shape)
        _lib.check(lib.nf_ns_intensity(self.handle, _lib.ptr(q), q.size, _lib.ptr(peak), _lib.ptr(integ)),
                   "nf_ns_intensity")
        kms = np.asarray(self.block.chan_kms, dtype=np.float64)
        kms = kms[self.pix_ids] if kms.ndim == 2 else np.broadcast_to(kms, (self.n_run, kms.size))
        integ *= kms[:, None, :, None]
        return {'peak_intensity_marginals': peak, 'integrated_intensity_marginals': integ}

    @property
    def results(self):
        if self._results is None:
            self.run()
        return self._results

    def posterior(self, run):
        """(n_samples, ndim + 2) float64: physical parameters, lnL, posterior weight
        (MultiNest's `posterior` array convention; weights sum to 1)."""
        res = self.results
        n = int(res["n_samples"][run])
        th = np.empty((n, self.ndim), dtype=np.float32)
        lnl = np.empty(n)
        lnw = np.empty(n)
        _lib.check(_lib.load().nf_ns_posterior(self.handle, run, n, _lib.ptr(th), _lib.ptr(lnl), _lib.ptr(lnw)),
                   "nf_ns_posterior")
        keep = lnl > -np.inf          # logZero points (NaN prior draws among the first live set) carry no weight
        if not keep.all():
            th, lnl, lnw = th[keep], lnl[keep], lnw[keep]
        w = np.exp(lnl + lnw - res["lnZ"][run])
        return np.concatenate([th.astype(np.float64), lnl[:, None], w[:, None]], axis=1)

    def products(self, run, null_lnZ, n_chan_tot):
        """Attributes and datasets the reference's dumper writes for one run
        (core.pyx:645-687), as two dicts."""
        res = self.results
        return run_products(self.ncomp, self.ndim, int(self.nlive[run]), null_lnZ, n_chan_tot, self.posterior(run),
                            res["lnZ"][run], res["lnZ_err"][run], res["max_loglike"][run], res["bestfit"][run],
                            res["mapfit"][run], n_iter=res["n_iter"][run], n_evals=res["n_evals"][run],
                            truncated=res["truncated"][run])


def run_products(ncomp, ndim, nlive, null_lnZ, n_chan_tot, post, lnZ, lnZ_err, max_loglike, bestfit, mapfit,
                 n_iter=0, n_evals=0, truncated=False):
    """What `mn_dump` persists for one run (core.pyx:645-687) from the run's posterior array `post`
    [n_samples, ndim + 2] (theta, lnL, posterior weight) and its summary numbers: (attrs, datasets)."""
    res = dict(lnZ=[lnZ], lnZ_err=[lnZ_err], max_loglike=[max_loglike], n_iter=[n_iter], n_evals=[n_evals],
               truncated=[truncated])
    cols = run_attr_columns(ndim, n_chan_tot, [nlive], [null_lnZ], res, [post.shape[0]])
    attrs = {'ncomp': int(ncomp), 'n_chan_tot': int(n_chan_tot), 'n_params': int(ndim), 'marg_cols': MARG_COLS,
             'marg_quantiles': MARG_QUANTILES}
    attrs.update({k: v[0].item() for k, v in cols.items()})
    dsets = {
        'posteriors': post.astype('float32'),
        # unweighted quantiles over all rows, mirroring core.pyx:596-598
        'marginals': np.quantile(post[:, :-2], MARG_QUANTILES, axis=0),
        'marginals_weighted': weighted_quantiles(post[:, :-2], post[:, -1], MARG_QUANTILES),
        'bestfit_params': np.array(bestfit, dtype=np.float64),
        'map_params': np.array(mapfit, dtype=np.float64),
    }
    return attrs, dsets


def weighted_quantiles(x, w, q):
    """Posterior-weighted quantiles per column (an addition: the reference's
    `marginals` ignores the importance weights)."""
    out = np.empty((len(q), x.shape[1]))
    for j in range(x.shape[1]):
        o = np.argsort(x[:, j])
        cw = np.cumsum(w[o])
        cw /= cw[-1]
        out[:, j] = np.interp(q, cw, x[o, j])
    return out


class Dumper:
    """Result sink with the reference's interface (core.pyx:564-609): writes run
    attributes and datasets into an h5py-like group."""

    def __init__(self, group, no_dump=False):
        self.group = group
        self.no_dump = no_dump
        self.n_calls = 0
        self.n_samples = -1
        self.quantiles = MARG_QUANTILES
        self.marginal_cols = MARG_COLS

    def calc_marginals(self, posteriors):
        return np.quantile(posteriors[:, :-2], self.quantiles, axis=0)

    def flush(self):
        f = getattr(self.group, "file", None)
        if f is not None:
            f.flush()

    def append_attributes(self, **kwargs):
        for name, value in kwargs.items():
            self.group.attrs[name] = value

    def append_datasets(self, **kwargs):
        for name, data in kwargs.items():
            self.group.create_dataset(name, data=data)


def run_multinest(runner, dumper, IS=False, mmodal=True, ceff=False, nlive=400, tol=0.5, efr=0.3, nClsPar=None,
                  maxModes=100, updInt=10, Ztol=-1e90, root='results', seed=-1, pWrap=None, fb=False,
                  resume=False, initMPI=False, outfile=False, logZero=-1e100, maxiter=int(1e6), n_prop=32,
                  intensity_marginals=False):
    """Drop-in for the reference's ``run_multinest`` (core.pyx:727-823): fits the
    runner's pixel with the batched device sampler (one run), sets
    ``runner.run_lnZ`` and writes the reference's products through ``dumper``.
    MultiNest-only switches (IS, mmodal, ceff, nClsPar, maxModes, updInt, Ztol,
    pWrap, fb, resume, initMPI, outfile, logZero, root) are accepted and ignored.
    With ``intensity_marginals`` the dumper also receives 'peak_intensity_marginals' and
    'integrated_intensity_marginals' [15, n_spec, ncomp] (``NestedSamplingBatch.intensity_marginals``)."""
    if intensity_marginals and runner._block.model == _lib.NF_MODEL_GAUSS:
        raise ValueError("intensity_marginals: the Gaussian model's peak and area are its own parameters")
    assert runner.ndim > 0
    assert nlive > 0
    assert tol > 0
    assert 0 < efr <= 1
    assert maxModes > 0
    assert updInt > 0
    assert Ztol is not None and np.isfinite(Ztol)
    assert logZero is not None and np.isfinite(logZero)
    assert maxiter >= 0
    if nClsPar is not None and nClsPar > runner.n_params:
        raise ValueError('Number of clustering parameters must be less than total.')
    ns = NestedSamplingBatch(runner._block, runner.utrans, runner.ncomp, pix_ids=[0], nlive=nlive, tol=tol, efr=efr,
                             n_prop=n_prop, seed=seed, max_iter=maxiter,
                             cold=getattr(runner, "cold", False), lte=getattr(runner, "lte", False))
    res = ns.run()
    runner.run_lnZ = float(res["lnZ"][0])
    if dumper is not None and not dumper.no_dump:
        attrs, dsets = ns.products(0, runner.null_lnZ, runner.n_chan_tot)
        if intensity_marginals:
            dsets.update({k: v[0] for k, v in ns.intensity_marginals().items()})
        dumper.append_attributes(**attrs)
        dumper.append_datasets(**dsets)
    dumper_calls = getattr(dumper, "n_calls", 0)
    if dumper is not None:
        dumper.n_calls = dumper_calls + 1
        dumper.n_samples = int(res["n_samples"][0])
    ns.close()
    return res


def _runner_spectra(runner):
    """The spectra of one runner's pixel (the Gaussian runner holds a single one)."""
    spectra = getattr(runner, "spectra", None)
    return [runner.spectrum] if spectra is None else list(spectra)


def _check_batch(runners, dumpers, nlive, tol, efr, maxiter, max_runs_per_batch, nClsPar, intensity=False):
    """Argument checks of run_multinest_batch; touch no device."""
    if len(runners) == 0:
        raise ValueError("run_multinest_batch needs at least one runner")
    r0 = runners[0]
    if getattr(r0, "model_name", None) is None:
        raise ValueError(f"{type(r0).__name__} is not a runner of this package")
    if intensity and r0.model_name == "gaussian":
        raise ValueError("intensity_marginals: the Gaussian model's peak and area are its own parameters")

    def trans(r):
        return tuple(int(s.trans_id) for s in _runner_spectra(r))

    for i, r in enumerate(runners[1:], start=1):
        for what, a, b in (("class", type(r), type(r0)), ("ncomp", r.ncomp, r0.ncomp),
                           ("number of spectra", r.n_spec, r0.n_spec), ("transition ids", trans(r), trans(r0)),
                           ("cold", bool(getattr(r, "cold", False)), bool(getattr(r0, "cold", False))),
                           ("lte", bool(getattr(r, "lte", False)), bool(getattr(r0, "lte", False)))):
            if a != b:
                raise ValueError(f"runner {i} differs from runner 0 in its {what}: {a!r} != {b!r}")
        if r.utrans is not r0.utrans:
            raise ValueError(f"runner {i} has another prior transformer than runner 0")
    n = len(runners)
    if dumpers is not None and len(dumpers) != n:
        raise ValueError(f"{len(dumpers)} dumpers for {n} runners")
    nl = np.asarray(nlive)
    if nl.ndim > 1 or (nl.ndim == 1 and nl.shape[0] != n):
        raise ValueError(f"nlive must be a scalar or one value per runner ({n}), got shape {nl.shape}")
    if not np.all(nl > 0):
        raise ValueError("nlive must be positive")
    if not tol > 0:
        raise ValueError("tol must be positive")
    if not 0 < efr <= 1:
        raise ValueError("efr must lie in (0, 1]")
    if maxiter < 0:
        raise ValueError("maxiter must not be negative")
    if max_runs_per_batch < 1:
        raise ValueError("max_runs_per_batch must be at least 1")
    if nClsPar is not None and nClsPar > r0.n_params:
        raise ValueError('Number of clustering parameters must be less than total.')


def run_multinest_batch(runners, dumpers=None, nlive=400, tol=0.5, efr=0.3, seed=-1, maxiter=int(1e6), n_prop=32,
                        max_runs_per_batch=16384, intensity_marginals=False, **multinest_switches):
    """Batched form of ``run_multinest``: fits every runner's pixel in lock-step on the device.

    The runners may come from anywhere -- a catalogue of pointed observations, spectra cut from several cubes --
    and each spectrum keeps its own axis and length: their spectra are uploaded as one block with per-pixel axes
    (``PixelBlock.from_spectra``) and fitted by ``NestedSamplingBatch`` in batches of at most
    ``max_runs_per_batch`` runs.  All runners must share class, ``ncomp``, number of spectra, transition ids,
    ``cold`` / ``lte`` and prior transformer (checked, with ``ValueError``, before the device is touched).

    For each runner it sets ``runner.run_lnZ`` and writes into ``dumpers[i]`` (None: no products) what
    ``run_multinest(runners[i], dumpers[i])`` writes, with that runner's own ``null_lnZ`` and ``n_chan_tot``.
    ``nlive`` is a scalar or one value per runner.  Truncated runs are flagged (``truncated``) but not repeated.
    MultiNest-only switches are accepted and ignored, as in ``run_multinest``.  Returns the per-runner result
    arrays (``lnZ``, ``lnZ_err``, ``max_loglike``, ``n_samples``, ``n_iter``, ``n_evals``, ``bestfit``,
    ``mapfit``, ``truncated``) in runner order.  With ``intensity_marginals`` every dumper also receives
    'peak_intensity_marginals' and 'integrated_intensity_marginals' [15, n_spec, ncomp] of its run, computed on the
    device from the batch's posteriors and scaled by that runner's own channel widths.

    Choosing the number of components stays the caller's loop, as with the reference: one call per ncomp over
    the sources that are still improving::

        best = np.zeros(len(catalogue), dtype=int)      # 0: nothing detected
        lnZ_best = np.empty(len(catalogue))
        active = np.arange(len(catalogue))
        for ncomp in (1, 2, 3):
            batch = [AmmoniaRunner(catalogue[i], utrans, ncomp=ncomp) for i in active]
            run_multinest_batch(batch)
            lnZ = np.array([r.run_lnZ for r in batch])
            ref = np.array([r.null_lnZ for r in batch]) if ncomp == 1 else lnZ_best[active]
            better = lnZ - ref > lnZ_thresh                # e.g. lnZ_thresh = 11
            best[active[better]] = ncomp
            lnZ_best[active[better]] = lnZ[better]
            active = active[better]
            if active.size == 0:
                break
    """
    from .pixels import PixelBlock
    runners = list(runners)
    _check_batch(runners, dumpers, nlive, tol, efr, maxiter, max_runs_per_batch, multinest_switches.get("nClsPar"),
                 intensity_marginals)
    n = len(runners)
    r0 = runners[0]
    dumpers = [None] * n if dumpers is None else list(dumpers)
    nlive = np.broadcast_to(np.asarray(nlive, dtype=np.int32), (n,))
    cold, lte = bool(getattr(r0, "cold", False)), bool(getattr(r0, "lte", False))
    block = PixelBlock.from_spectra(r0.model_name, [_runner_spectra(r) for r in runners])
    parts = []
    try:
        for k, b0 in enumerate(range(0, n, max_runs_per_batch)):
            sel = np.arange(b0, min(n, b0 + max_runs_per_batch))
            bseed = seed if seed is None or seed < 0 else seed + k
            ns = NestedSamplingBatch(block, r0.utrans, r0.ncomp, pix_ids=sel, nlive=nlive[sel], tol=tol, efr=efr,
                                     n_prop=n_prop, seed=bseed, max_iter=maxiter, cold=cold, lte=lte)
            try:
                res = ns.run()
                dump = [dumpers[i] is not None and not dumpers[i].no_dump for i in sel]
                if any(dump):          # the posteriors of the whole batch in one device pass and one copy
                    prod = ns.products_all(marginals=False, posteriors=True)
                    off, pool = prod["row_offsets"], prod["posteriors"]
                    inten = ns.intensity_marginals() if intensity_marginals else None
                for j, i in enumerate(sel):
                    runner, dumper = runners[i], dumpers[i]
                    runner.run_lnZ = float(res["lnZ"][j])
                    if dump[j]:
                        post = pool[off[j]:off[j + 1]].astype(np.float64)
                        attrs, dsets = run_products(
                            r0.ncomp, ns.ndim, int(ns.nlive[j]), runner.null_lnZ, runner.n_chan_tot, post,
                            res["lnZ"][j], res["lnZ_err"][j], res["max_loglike"][j], res["bestfit"][j],
                            res["mapfit"][j], n_iter=res["n_iter"][j], n_evals=res["n_evals"][j],
                            truncated=res["truncated"][j])
                        if inten is not None:
                            dsets.update({k: v[j] for k, v in inten.items()})
                        dumper.append_attributes(**attrs)
                        dumper.append_datasets(**dsets)
                    if dumper is not None:
                        dumper.n_calls = getattr(dumper, "n_calls", 0) + 1
                        dumper.n_samples = int(res["n_samples"][j])
                parts.append(res)
            finally:
                ns.close()
    finally:
        block.close()
    out = {key: np.concatenate([p[key] for p in parts]) for key, v in parts[0].items() if isinstance(v, np.ndarray)}
    out["lock_iters"] = sum(p["lock_iters"] for p in parts)
    out["launches"] = sum(p["launches"] for p in parts)
    return out
