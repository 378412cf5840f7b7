"""Store post-processing on the predict kernel: host mirror of the aggregation and
convolution steps the reference runs after a cube fit (nestfit/main.py:529-1061) and, batched
on the GPU, of its two per-pixel ``runner.predict`` loops

    deblend_hf_intensity          nestfit/main.py:1064-1133
    generate_predicted_profiles   nestfit/main.py:1136-1193

The reference walks (lon, lat, component) in Python and calls ``runner.predict``
once per triple (main.py:1106-1113, 1182-1188).  Here the MAP-parameter cube is
flattened to one batch of single-component vectors and scored by one launch of
``nf_nh3_predict`` per chunk of vectors; array shapes, dataset names and axis
orders written to the store are the reference's.
"""
import numpy as np

from .main import nans


# ---------------------------------------------------------------------------
# aggregation of per-pixel run groups into dense arrays (host side, numpy)
# ---------------------------------------------------------------------------
# dense map written to <dpath>/<name>  <-  (attribute of a run group, attribute holding the null-model value or None)
RUN_ATTR_MAPS = {'evidence': ('global_lnZ', 'null_lnZ'), 'evidence_err': ('global_lnZ_err', None),
                 'BIC': ('BIC', 'null_BIC'), 'AIC': ('AIC', 'null_AIC'), 'AICc': ('AICc', 'null_AICc')}


def aggregate_run_attributes(store):
    """The per-run scalars of every pixel gathered into dense maps (main.py:664-721): 'nbest' (b, l) and one
    (m, b, l) map per entry of RUN_ATTR_MAPS, plane 0 holding the null model's value where one exists."""
    hdf = store.hdf
    n_lon, n_lat, n_model = int(hdf.attrs['naxis1']), int(hdf.attrs['naxis2']), int(hdf.attrs['n_max_components']) + 1
    maps = {name: nans((n_model, n_lat, n_lon)) for name in RUN_ATTR_MAPS}
    nbest = np.full((n_lat, n_lon), -1, dtype=np.int32)
    for pix in store.iter_pix_groups():
        lon, lat = int(pix.attrs['i_lon']), int(pix.attrs['i_lat'])
        nbest[lat, lon] = pix.attrs['nbest']
        runs = [pix[key].attrs for key in pix]
        for name, (attr, null_attr) in RUN_ATTR_MAPS.items():
            for a in runs:
                maps[name][int(a['ncomp']), lat, lon] = a[attr]
            if null_attr is not None and runs:
                maps[name][0, lat, lon] = runs[0][null_attr]       # every run of the pixel carries the same null value
    store.create_dataset('nbest', nbest, group=store.dpath)
    for name, arr in maps.items():
        store.create_dataset(name, arr, group=store.dpath)


def gaussian_kernel2d(sigma):
    """Normalised 2-D Gaussian on an odd (8 sigma + 1) grid: astropy's
    ``Gaussian2DKernel(sigma)`` default support."""
    half = max(1, int(np.ceil(4 * sigma)))
    ax = np.arange(-half, half + 1)
    k = np.exp(-0.5 * (ax[:, None]**2 + ax[None, :]**2) / sigma**2)
    return k / k.sum()


def convolve_nan_extend(img, kernel):
    """2-D convolution with edge replication ('extend') in which NaN pixels are
    interpolated over by renormalising the kernel -- the semantics of
    ``astropy.convolution.convolve(img, kernel, boundary='extend')`` that
    `convolve_evidence` relies on (main.py:752-753)."""
    img = np.asarray(img, dtype=np.float64)
    ky, kx = kernel.shape
    py, px = ky // 2, kx // 2
    pad = np.pad(img, ((py, py), (px, px)), mode='edge')
    good = np.isfinite(pad)
    vals = np.where(good, pad, 0.0)
    num = np.zeros_like(img)
    den = np.zeros_like(img)
    for dy in range(ky):
        for dx in range(kx):
            w = kernel[ky - 1 - dy, kx - 1 - dx]
            if w == 0.0:
                continue
            num += w * vals[dy:dy + img.shape[0], dx:dx + img.shape[1]]
            den += w * good[dy:dy + img.shape[0], dx:dx + img.shape[1]]
    with np.errstate(invalid='ignore', divide='ignore'):
        out = num / den          # astropy's default normalize_kernel=True: the kernel's own sum drops out
    out[den == 0] = np.nan
    return out


def convolve_evidence(store, kernel):
    """'conv_evidence' (m, b, l): every evidence plane smoothed with `kernel` (a 2-D array, or the standard deviation
    in pixels of a Gaussian), and 'conv_nbest' (b, l): the model selection redone on the smoothed planes
    (main.py:724-774) -- the number of consecutive models whose smoothed evidence beats the previous one by the store's
    threshold, at most one more than the number actually fitted at that position (no run exists beyond that)."""
    kernel = _as_kernel(kernel)
    hdf, dpath = store.hdf, store.dpath
    evidence = np.asarray(hdf[f'{dpath}/evidence'][...], dtype=np.float64)
    nbest = np.asarray(hdf[f'{dpath}/nbest'][...])
    smooth = np.stack([convolve_nan_extend(plane, kernel) for plane in evidence])
    with np.errstate(invalid='ignore'):
        gains = np.diff(smooth, axis=0) > hdf.attrs['lnZ_threshold']          # NaN compares False
    chain = np.cumprod(gains, axis=0).sum(axis=0).astype(np.int32)          # leading run of passed thresholds
    conv_nbest = np.where(nbest == -1, -1, np.minimum(chain, nbest + 1)).astype(np.int32)
    store.create_dataset('conv_nbest', conv_nbest, group=dpath)
    store.create_dataset('conv_evidence', smooth, group=dpath)


def take_by_components(data, comps, axis=0, incl_zero=True):
    """Pick, per map position, the entry of `data` (..., b, l) along `axis` that belongs to the number of
    components in `comps` (b, l): index `comps - 1`, i.e. 1 component -> entry 0 (main.py:529-562).
    Positions without data (`comps` = -1) and, unless `incl_zero`, noise-only positions (`comps` = 0)
    become NaN."""
    comps = np.asarray(comps)
    idx = np.clip(comps - 1, 0, None)
    idx = idx.reshape((1,) * (data.ndim - idx.ndim) + idx.shape)
    out = np.squeeze(np.take_along_axis(data, idx, axis=axis), axis=axis).astype(float, copy=True)
    out[..., comps < (0 if incl_zero else 1)] = np.nan
    return out


def _circle_rect_area(x0, x1, y0, y1, r):
    """Exact area of the disc x^2 + y^2 <= r^2 inside the rectangle [x0, x1] x [y0, y1]: the chord
    y = +-sqrt(r^2 - x^2) clipped to [y0, y1] is integrated piecewise (Gauss-Legendre on the smooth pieces
    between the abscissae where the chord meets a rectangle edge)."""
    lo, hi = max(x0, -r), min(x1, r)
    if hi <= lo:
        return 0.0
    cuts = {lo, hi}
    for y in (y0, y1):
        if abs(y) < r:
            c = np.sqrt(r * r - y * y)
            cuts.update(v for v in (-c, c) if lo < v < hi)
    cuts = sorted(cuts)
    gx, gw = np.polynomial.legendre.leggauss(48)
    area = 0.0
    for a, b in zip(cuts[:-1], cuts[1:]):
        # substitution x = r sin(t) removes the square-root end-point singularity at |x| = r
        ta, tb = np.arcsin(np.clip(a / r, -1, 1)), np.arcsin(np.clip(b / r, -1, 1))
        t = 0.5 * (tb - ta) * gx + 0.5 * (tb + ta)
        half = r * np.cos(t)
        seg = np.clip(half, y0, y1) - np.clip(-half, y0, y1)
        area += 0.5 * (tb - ta) * np.sum(gw * seg * r * np.cos(t))
    return float(area)


def apply_circular_mask(kernel, radius=None):
    """Weight an odd-shaped kernel by the exact fraction of each pixel inside a circular aperture of
    `radius` pixels about the centre of the middle pixel (main.py:574-610; the reference takes the overlap
    grid from photutils, here it is integrated directly)."""
    kernel = np.asarray(kernel, dtype=float)
    nx, ny = kernel.shape
    if radius is None:
        radius = min(nx, ny) / 2
    if radius > np.sqrt((nx / 2)**2 + (ny / 2)**2):
        return kernel
    if nx % 2 == 0 or ny % 2 == 0:
        raise ValueError(f'Kernel dimensions must be odd: ({nx}, {ny})')
    weights = np.empty((nx, ny))
    for i in range(nx):
        for j in range(ny):
            x0, y0 = i - nx / 2, j - ny / 2
            weights[i, j] = _circle_rect_area(x0, x0 + 1, y0, y0 + 1, radius)
    return weights * kernel


def get_indep_info_kernel(sigma, nrad=1, sigma_taper=None):
    """(2 nrad + 1)^2 kernel of the information that is independent of the centre pixel for a symmetric
    Gaussian beam of standard deviation `sigma` pixels: one minus the beam integrated over each pixel
    relative to its peak, per beam area; optional Gaussian taper; centre = 1 (main.py:613-661)."""
    from math import erf
    assert isinstance(nrad, int) and nrad >= 0
    if nrad == 0:
        return np.array([[1.0]])
    ppbeam = max(1.0, 2 * np.pi * sigma**2)            # a beam smaller than a pixel still counts as one
    ax = np.arange(-nrad, nrad + 1, dtype=float)
    cdf = np.vectorize(lambda z: 0.5 * (1 + erf(z / sigma / np.sqrt(2))))
    frac = cdf(ax + 0.5) - cdf(ax - 0.5)               # beam fraction inside each pixel column / row
    kernel = (1 - np.outer(frac, frac) * (2 * np.pi * sigma**2)) / ppbeam
    if sigma_taper is not None:
        kernel = kernel * np.exp(-0.5 * (ax[:, None]**2 + ax[None, :]**2) / sigma_taper**2)
    kernel[nrad, nrad] = 1
    return kernel


def _as_kernel(kernel):
    if isinstance(kernel, (int, float)):
        kernel = gaussian_kernel2d(float(kernel))
    return np.asarray(kernel, dtype=np.float64)


def extended_masked_evidence(store, kernel, conv=True, lnz_thresh=3):
    """'mext_evidence' (b, l): evidence difference of the one-component model after masking the positions
    already detected above `lnz_thresh` and convolving with `kernel`, to bring out weak extended emission
    (main.py:777-816)."""
    kernel = _as_kernel(kernel)
    hdf, dpath = store.hdf, store.dpath
    data = np.array(hdf[f'{dpath}/evidence'][...], dtype=float)
    mdata = np.asarray(hdf[f"{dpath}/{'conv_evidence' if conv else 'evidence'}"][...])
    mdata = mdata[1] - mdata[0]
    with np.errstate(invalid='ignore'):
        mask = mdata > lnz_thresh
    cdata = nans(data.shape)
    for i in range(data.shape[0]):
        data[i, mask] = np.nan
        cdata[i] = convolve_nan_extend(data[i], kernel)
    mext = cdata[1] - cdata[0]
    mext[np.isnan(mdata) | mask] = np.nan
    store.create_dataset('mext_evidence', mext, group=dpath)


def convolve_fill_interp(data, kernel):
    """Convolution of the last two axes of `data` with zero fill outside the map, NaNs interpolated over by
    renormalising the kernel on the valid pixels, and the kernel's own sum kept (not normalised) -- the
    semantics of ``astropy.convolution.convolve_fft(x, kernel, normalize_kernel=False)`` that
    `convolve_post_pdfs` relies on (main.py:1008-1009)."""
    from scipy import ndimage
    kernel = np.asarray(kernel, dtype=np.float64)
    scale = kernel.sum()
    k = (kernel / scale).reshape((1,) * (data.ndim - 2) + kernel.shape)
    good = np.isfinite(data)
    num = ndimage.convolve(np.where(good, data, 0.0), k, mode='constant', cval=0.0)
    wt = ndimage.convolve(good.astype(np.float64), k, mode='constant', cval=1.0)
    with np.errstate(invalid='ignore', divide='ignore'):
        out = num / wt * scale
    out[wt <= 0] = np.nan
    return out


def convolve_post_pdfs(store, kernel, evid_weight=True):
    """'conv_post_pdfs' (r, m, p, h, b, l): the posterior PDFs multiplied over neighbouring pixels, i.e.
    their logarithms convolved with `kernel`, optionally weighted by each pixel's evidence over the null
    model scaled to [0, 1]; renormalised over the histogram axis (main.py:956-1017)."""
    kernel = _as_kernel(kernel)
    hdf, dpath = store.hdf, store.dpath
    data = np.array(hdf[f'{dpath}/post_pdfs'][...], dtype=np.float64)
    blank = np.isnan(data)
    data[data == 0] = 1e-32                    # keeps the logarithm finite
    ldata = np.log(data)
    if evid_weight:
        evid = np.asarray(hdf[f'{dpath}/evidence'][...])
        nbest = np.asarray(hdf[f'{dpath}/conv_nbest'][...])
        d_evid = take_by_components(evid[1:], nbest) - evid[0]
        d_evid = d_evid - np.nanmin(d_evid)
        d_evid = d_evid / np.nanmax(d_evid)
        ldata = ldata * d_evid.reshape((1, 1, 1, 1) + d_evid.shape)
    cdata = np.zeros_like(data)
    for i_r in range(data.shape[0]):           # components beyond the run's own number stay empty
        cdata[i_r, :i_r + 1] = convolve_fill_interp(ldata[i_r, :i_r + 1], kernel)
    cdata = np.exp(cdata)
    with np.errstate(invalid='ignore', divide='ignore'):
        cdata /= np.nansum(cdata, axis=3, keepdims=True)
    cdata[blank] = np.nan
    store.create_dataset('conv_post_pdfs', cdata.astype('float32'), group=dpath)


def quantize_conv_marginals(store):
    """'conv_marginals' (r, m, p, M, b, l): quantiles of the convolved PDFs, interpolated on their
    cumulative sums at the run quantiles 'marg_quantiles' (main.py:1020-1061)."""
    hdf, dpath = store.hdf, store.dpath
    bins = np.asarray(hdf[f'{dpath}/pdf_bins'][...])                     # (p, h)
    quan = np.asarray(hdf[f'{dpath}/marg_quantiles'][...])
    data = np.asarray(hdf[f'{dpath}/conv_post_pdfs'][...], dtype=np.float64).transpose((0, 1, 2, 4, 5, 3))
    with np.errstate(invalid='ignore', divide='ignore'):
        cdf = np.cumsum(data, axis=5) / np.sum(data, axis=5, keepdims=True)
    margs = nans(cdf.shape[:-1] + (len(quan),))
    flat, out = cdf.reshape(-1, cdf.shape[-1]), margs.reshape(-1, len(quan))
    i_p = np.broadcast_to(np.arange(cdf.shape[2]).reshape(1, 1, -1, 1, 1), cdf.shape[:-1]).reshape(-1)
    for k in np.flatnonzero(np.isfinite(flat[:, -1])):
        out[k] = np.interp(quan, flat[k], bins[i_p[k]])
    store.create_dataset('conv_marginals', margs.transpose((0, 1, 2, 5, 3, 4)).astype('float32'), group=dpath)


def aggregate_run_products(store):
    """'marg_quantiles' (M), 'nbest_MAP' / 'nbest_bestfit' (m, p, b, l) and
    'nbest_marginals' (m, p, M, b, l) (main.py:819-882).  Uses 'conv_nbest' when the
    evidence was convolved, else the per-pixel 'nbest'."""
    hdf, dpath = store.hdf, store.dpath
    n_lon, n_lat = int(hdf.attrs['naxis1']), int(hdf.attrs['naxis2'])
    key = 'conv_nbest' if f'{dpath}/conv_nbest' in hdf else 'nbest'
    nbest_data = np.asarray(hdf[f'{dpath}/{key}'][...]).transpose()
    ncomp_max = int(hdf.attrs['n_max_components'])
    n_params = int(hdf.attrs['n_params'])
    marg_quan = np.asarray(store.find_first_valid_group().attrs['marg_quantiles'])
    n_margs = len(marg_quan)
    mapdata = nans((n_lon, n_lat, n_params, ncomp_max))
    bfdata = nans((n_lon, n_lat, n_params, ncomp_max))
    pardata = nans((n_lon, n_lat, n_margs, n_params, ncomp_max))
    for group in store.iter_pix_groups():
        i_lon, i_lat = int(group.attrs['i_lon']), int(group.attrs['i_lat'])
        nbest = int(nbest_data[i_lon, i_lat])
        if nbest <= 0 or f'{nbest}' not in group:
            continue
        nb_group = group[f'{nbest}']
        p_shape = (n_params, nbest)
        mapdata[i_lon, i_lat, :, :nbest] = np.asarray(nb_group['map_params'][...]).reshape(p_shape)
        bfdata[i_lon, i_lat, :, :nbest] = np.asarray(nb_group['bestfit_params'][...]).reshape(p_shape)
        pardata[i_lon, i_lat, :, :, :nbest] = np.asarray(nb_group['marginals'][...]).reshape((n_margs,) + p_shape)
    store.create_dataset('marg_quantiles', marg_quan, group=dpath)
    store.create_dataset('nbest_MAP', mapdata.transpose(), group=dpath)
    store.create_dataset('nbest_bestfit', bfdata.transpose(), group=dpath)
    store.create_dataset('nbest_marginals', pardata.transpose(), group=dpath)


def aggregate_intensity_marginals(store):
    """'nbest_peak_intensity_marginals' (K) and 'nbest_integrated_intensity_marginals' (K km/s), (t, m, M, b, l):
    the credible intervals of each component's peak and integrated intensity of the preferred model, gathered from
    the runs of a fit made with intensity_marginals=True.  Uses 'conv_nbest' when the evidence was convolved, else
    the per-pixel 'nbest', as aggregate_run_products does; positions and components without a run are NaN."""
    from .store import INTENSITY_DATASETS
    hdf, dpath = store.hdf, store.dpath
    n_lon, n_lat = int(hdf.attrs['naxis1']), int(hdf.attrs['naxis2'])
    key = 'conv_nbest' if f'{dpath}/conv_nbest' in hdf else 'nbest'
    nbest_data = np.asarray(hdf[f'{dpath}/{key}'][...]).transpose()
    ncomp_max = int(hdf.attrs['n_max_components'])
    first = store.find_first_valid_group()
    if INTENSITY_DATASETS[0] not in first:
        raise ValueError('the runs of this store carry no intensity marginals: fit with intensity_marginals=True')
    n_margs, n_spec = np.asarray(first[INTENSITY_DATASETS[0]][...]).shape[:2]
    out = {name: nans((n_lon, n_lat, n_margs, ncomp_max, n_spec)) for name in INTENSITY_DATASETS}
    for group in store.iter_pix_groups():
        i_lon, i_lat = int(group.attrs['i_lon']), int(group.attrs['i_lat'])
        nbest = int(nbest_data[i_lon, i_lat])
        if nbest <= 0 or f'{nbest}' not in group:
            continue
        nb_group = group[f'{nbest}']
        for name in INTENSITY_DATASETS:
            if name not in nb_group:
                raise ValueError(f'run /pix/{i_lon}/{i_lat}/{nbest} carries no {name}')
            out[name][i_lon, i_lat, :, :nbest, :] = np.asarray(nb_group[name][...]).transpose(0, 2, 1)
    for name, arr in out.items():
        store.create_dataset(f'nbest_{name}', arr.transpose(), group=dpath)


def aggregate_run_pdfs(store, par_bins=None):
    """'pdf_bins' (p, h) and 'post_pdfs' (r, m, p, h, b, l) (main.py:885-953)."""
    hdf, dpath = store.hdf, store.dpath
    n_lon, n_lat = int(hdf.attrs['naxis1']), int(hdf.attrs['naxis2'])
    ncomp_max = int(hdf.attrs['n_max_components'])
    n_params = int(hdf.attrs['n_params'])
    if par_bins is None:
        n_bins = 200
        margdata = np.asarray(hdf[f'{dpath}/nbest_marginals'][...])
        vmins = np.nanmin(margdata[:, :, 0, :, :], axis=(0, 2, 3))
        vmaxs = np.nanmax(margdata[:, :, 8, :, :], axis=(0, 2, 3))
        par_bins = np.array([np.linspace(lo, hi, n_bins) for lo, hi in zip(vmins, vmaxs)])
    else:
        par_bins = np.asarray(par_bins)
        n_bins = par_bins.shape[1]
    histdata = nans((n_lon, n_lat, ncomp_max, n_params, ncomp_max, n_bins - 1))
    for group in store.iter_pix_groups():
        i_l, i_b = int(group.attrs['i_lon']), int(group.attrs['i_lat'])
        for i_r in range(ncomp_max):
            n_run = i_r + 1
            if f'{n_run}' not in group or 'posteriors' not in group[f'{n_run}']:
                continue
            post = np.asarray(group[f'{n_run}']['posteriors'][...])
            for i_p, bins in enumerate(par_bins):
                for i_m in range(n_run):
                    hist, _ = np.histogram(post[:, i_p * n_run + i_m], bins=bins)
                    histdata[i_l, i_b, i_r, i_p, i_m, :] = hist
    with np.errstate(invalid='ignore', divide='ignore'):
        histdata /= np.nansum(histdata, axis=5, keepdims=True)
    bin_mids = (par_bins[:, :-1] + par_bins[:, 1:]) / 2
    store.create_dataset('pdf_bins', bin_mids, group=dpath)
    store.create_dataset('post_pdfs', histdata.transpose((2, 4, 3, 5, 1, 0)).astype('float32'), group=dpath)


# ---------------------------------------------------------------------------
# batched predict loops
# ---------------------------------------------------------------------------
def _runner_block(runner):
    blk = getattr(runner, '_block', None)
    if blk is None:
        raise TypeError('runner must be a nestfit_b200 Runner (it owns the device pixel block)')
    return blk


def predict_map_cube(pmap, runner, chunk=32768, want_spectra=False):
    """Model every non-NaN single-component MAP vector of `pmap` (l, b, p, m) with one
    predict launch per `chunk` vectors.  Returns (peak, sum) of shape (l, b, m, t)
    and, if `want_spectra`, the spectra as a list over transitions of (l, b, m, S)."""
    assert runner.ncomp == 1
    blk = _runner_block(runner)
    n_l, n_b, n_p, n_m = pmap.shape
    vec = np.ascontiguousarray(pmap.transpose(0, 1, 3, 2).reshape(-1, n_p))      # (l, b, m) x p
    ok = np.flatnonzero(~np.isnan(vec).any(axis=1))
    n_t = blk.n_spec
    pk = nans((n_l * n_b * n_m, n_t))
    sm = nans((n_l * n_b * n_m, n_t))
    spectra = [nans((n_l * n_b * n_m, blk.n_chan)) for _ in range(n_t)] if want_spectra else None
    kw = {k: getattr(runner, k) for k in ('cold', 'lte') if hasattr(runner, k)}
    for c0 in range(0, ok.size, chunk):
        ix = ok[c0:c0 + chunk]
        pred = blk.predict(np.ascontiguousarray(vec[ix]), 1, **kw)               # [B, t, S]
        pk[ix] = np.nanmax(pred, axis=2)
        sm[ix] = np.nansum(pred, axis=2, dtype=np.float64)
        if want_spectra:
            for t in range(n_t):
                spectra[t][ix] = pred[:, t, :]
    shape = (n_l, n_b, n_m, n_t)
    if want_spectra:
        spectra = [s.reshape(n_l, n_b, n_m, -1) for s in spectra]
    return pk.reshape(shape), sm.reshape(shape), spectra


def deblend_hf_intensity(store, stack, runner):
    """'peak_intensity', 'integrated_intensity' (t, m, b, l) and 'hf_deblended'
    (t, m, S, b, l) from the MAP parameters (main.py:1064-1133)."""
    hdf, dpath = store.hdf, store.dpath
    bins = np.asarray(hdf[f'{dpath}/pdf_bins'][...])
    pmap = np.asarray(hdf[f'{dpath}/nbest_MAP'][...]).transpose()                # (l, b, p, m)
    pkint, intint, _ = predict_map_cube(pmap, runner)
    for i_t, cube in enumerate(stack.cubes):       # K -> K km/s
        intint[:, :, :, i_t] *= cube.dv
    dv_bin = abs(bins[0, 1] - bins[0, 0])
    vaxis = bins[0].reshape(1, 1, 1, 1, -1)
    model = store.model
    if model is None:                  # store opened before the model metadata was inserted
        from .models import MODELS
        model = MODELS[hdf.attrs['model_name']]
    vcen = np.expand_dims(pmap[:, :, model.IX_VCEN, :], (3, 4))
    sigm = np.expand_dims(pmap[:, :, model.IX_SIGM, :], (3, 4))
    norm_fact = dv_bin / (sigm * np.sqrt(2 * np.pi))
    hfdb = norm_fact * intint[..., np.newaxis] * np.exp(-0.5 * ((vaxis - vcen) / sigm)**2)
    store.create_dataset('peak_intensity', pkint.transpose(), group=dpath)
    store.create_dataset('integrated_intensity', intint.transpose(), group=dpath)
    store.create_dataset('hf_deblended', hfdb.transpose((3, 2, 4, 1, 0)).astype('float32'), group=dpath)


def generate_predicted_profiles(store, stack, runner):
    """'model_spec/trans<TRANS_ID>' (m, S, b, l): MAP model profiles per transition
    (main.py:1136-1193)."""
    hdf, dpath = store.hdf, store.dpath
    pmap = np.asarray(hdf[f'{dpath}/nbest_MAP'][...]).transpose()
    _, _, spectra = predict_map_cube(pmap, runner, want_spectra=True)
    for mcube, dcube in zip(spectra, stack):
        store.create_dataset(f'trans{dcube.trans_id}', mcube.transpose((2, 3, 1, 0)).astype('float32'),
                             group=f'{dpath}/model_spec')


def create_fits_from_store(store, prefix='source'):
    """Write the hyperfine-deblended cubes, summed over components, as FITS files
    `<prefix>_hf_deblended_trans<i>.fits` (main.py:1196-1232).  Needs astropy (import-guarded)."""
    try:
        from astropy.io import fits
    except ImportError as exc:                         # pragma: no cover - optional dependency
        raise ImportError('create_fits_from_store needs astropy') from exc
    cube_header = store.read_header(full=True)         # pragma: no cover
    hdf, dpath = store.hdf, store.dpath                # pragma: no cover
    model = store.model                                # pragma: no cover
    vaxis = np.asarray(hdf[f'{dpath}/pdf_bins'][...])[model.IX_VCEN]          # pragma: no cover
    hfdb = np.asarray(hdf[f'{dpath}/hf_deblended'][...])                      # pragma: no cover  (t, m, S, b, l)
    for i_t in range(hfdb.shape[0]):                   # pragma: no cover
        header = cube_header.copy()
        header.update({'BUNIT': 'K', 'NAXIS3': vaxis.size, 'CRPIX3': 1, 'CDELT3': vaxis[1] - vaxis[0],
                       'CUNIT3': 'km/s', 'CTYPE3': 'VRAD', 'CRVAL3': vaxis[0], 'SPECSYS': 'LSRK'})
        fits.PrimaryHDU(np.nansum(hfdb[i_t], axis=0), header).writeto(f'{prefix}_hf_deblended_trans{i_t}.fits',
                                                                      overwrite=True)


def postprocess_run(store, stack, runner, par_bins=None, evid_kernel=None, post_kernel=None, evid_weight=True):
    """The reference's `postprocess_run` sequence (main.py:1240-1272).  The two convolution stages run when
    their kernel is given (the reference requires both)."""
    aggregate_run_attributes(store)
    if evid_kernel is not None:
        convolve_evidence(store, evid_kernel)
    aggregate_run_products(store)
    aggregate_run_pdfs(store, par_bins=par_bins)
    if post_kernel is not None:
        if evid_kernel is None:
            raise ValueError('the posterior convolution needs the convolved evidence: pass evid_kernel too')
        convolve_post_pdfs(store, post_kernel, evid_weight=evid_weight)
        quantize_conv_marginals(store)
    deblend_hf_intensity(store, stack, runner)
    generate_predicted_profiles(store, stack, runner)
