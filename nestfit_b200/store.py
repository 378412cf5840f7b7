"""Result store behind the reference's ``HdfStore`` API (nestfit/main.py:233-377; tree and attribute names of
docs/store_spec.rst:58-150): ``<name>.store/`` with a table file plus one chunk per worker and pixel groups
``/pix/<lon>/<lat>/<ncomp>`` carrying the per-run attributes and datasets of the dumper (core.pyx:645-687).

The reference writes one small HDF5 group per (pixel, ncomp) from inside the MultiNest callback.  The GPU path
finishes thousands of runs at once, so a *wave* (all runs of one ncomp of a pixel block) is the unit that reaches
the store: its posterior rows arrive as one float32 pool with run offsets, its attributes as columns.  Backends:

  slab   (default) a chunk is a directory of per-wave slabs -- ``*.post.npy`` (the pool, memory-mapped on read)
         and ``*.npz`` (attribute columns, marginals, best-fit / MAP vectors, pixel coordinates).  Readers see the
         reference's tree: groups, ``attrs`` and datasets are materialised lazily from the slabs.
  h5py   when h5py is importable the same waves are unrolled into real HDF5 groups, and ``link_files`` makes
         ExternalLinks, exactly like the reference.  (h5py / libhdf5 are absent from this image: the branch is
         exercised only through the h5py-like ``MemGroup``, which `GroupSink` also serves.)
"""
import inspect
import json
import threading
import warnings
from collections.abc import Mapping
from pathlib import Path

import numpy as np

try:  # pragma: no cover - depends on the environment
    import h5py
    HAVE_H5PY = True
except Exception:  # h5py absent in this image
    h5py = None
    HAVE_H5PY = False

# quantiles / labels written per run by the reference (core.pyx:585-594)
MARG_QUANTILES = np.array([
    0.00, 0.01, 0.10, 0.25, 0.50, 0.75, 0.90, 0.99, 1.00,
    1.58655254e-1, 0.84134475,
    2.27501319e-2, 0.97724987,
    1.34989803e-3, 0.99865010,
])
MARG_COLS = ['min', 'p01', 'p10', 'p25', 'p50', 'p75', 'p90', 'p99', 'max',
             '1s_lo', '1s_hi', '2s_lo', '2s_hi', '3s_lo', '3s_hi']

# ---- schema tables ---------------------------------------------------------------------------------
# root attributes of the table file <- attribute of the fitter / constant of the model module (main.py:354-377)
FITTER_ATTRS = {'lnZ_threshold': lambda f: f.lnZ_thresh, 'n_max_components': lambda f: f.ncomp_max,
                'multinest_kwargs': lambda f: str(f.mn_kwargs)}
MODEL_ATTRS = {'n_params': 'N', 'model_name': 'NAME', 'par_names': 'PAR_NAMES', 'par_names_short': 'PAR_NAMES_SHORT',
               'tex_labels': 'TEX_LABELS', 'tex_labels_with_units': 'TEX_LABELS_WITH_UNITS'}
HEADER_GROUPS = {'simple_header': 'simple_header', 'full_header': 'full_header'}
# per-run attributes (core.pyx:645-671) as columns over the runs of a wave; the last two are bookkeeping extras
RUN_ATTR_COLUMNS = ('null_lnZ', 'n_samples', 'n_live', 'global_lnZ', 'global_lnZ_err', 'max_loglike',
                    'BIC', 'AIC', 'AICc', 'null_BIC', 'null_AIC', 'null_AICc', 'n_iter', 'n_evals', 'truncated')
RUN_DATASETS = ('posteriors', 'marginals', 'bestfit_params', 'map_params')
# optional per-run datasets: posterior-weighted quantiles (M, n_spec, ncomp) of each component's peak (K) and
# integrated (K km/s) intensity, written by fits run with intensity_marginals=True
INTENSITY_DATASETS = ('peak_intensity_marginals', 'integrated_intensity_marginals')


def run_attr_columns(ndim, n_chan_tot, nlive, null_lnZ, res, n_samples):
    """The information criteria and bookkeeping the dumper attaches to a run (core.pyx:650-671), for all runs of
    a wave at once.  `res`: arrays of NestedSamplingBatch.run()."""
    k, n = float(ndim), float(n_chan_tot)
    maxL = np.asarray(res['max_loglike'], dtype=np.float64)
    null = np.asarray(null_lnZ, dtype=np.float64)
    small = (2 * k**2 + 2 * k) / (n - k - 1)
    aic, null_aic = 2 * k - 2 * maxL, 2 * k - 2 * null
    cols = {'null_lnZ': null, 'n_samples': np.asarray(n_samples, dtype=np.int64),
            'n_live': np.asarray(nlive, dtype=np.int64), 'global_lnZ': np.asarray(res['lnZ'], dtype=np.float64),
            'global_lnZ_err': np.asarray(res['lnZ_err'], dtype=np.float64), 'max_loglike': maxL,
            'BIC': np.log(n) * k - 2 * maxL, 'AIC': aic, 'AICc': aic + small,
            'null_BIC': np.log(n) * k - 2 * null, 'null_AIC': null_aic, 'null_AICc': null_aic + small,
            'n_iter': np.asarray(res['n_iter'], dtype=np.int64), 'n_evals': np.asarray(res['n_evals'], dtype=np.int64),
            'truncated': np.asarray(res['truncated'], dtype=bool)}
    assert tuple(cols) == RUN_ATTR_COLUMNS
    return cols


class Wave:
    """All runs of one ncomp of a pixel block, as they leave the sampler."""

    def __init__(self, ncomp, ndim, n_chan_tot, i_lon, i_lat, columns, row_offsets, posteriors, marginals,
                 bestfit, mapfit, intensity=None):
        """intensity: None, or {name: [n_run, M, n_spec, ncomp]} for the names of INTENSITY_DATASETS."""
        self.ncomp, self.ndim, self.n_chan_tot = int(ncomp), int(ndim), int(n_chan_tot)
        self.i_lon, self.i_lat = np.asarray(i_lon, dtype=np.int64), np.asarray(i_lat, dtype=np.int64)
        self.columns = columns
        self.row_offsets = np.asarray(row_offsets, dtype=np.int64)
        self.posteriors, self.marginals, self.bestfit, self.mapfit = posteriors, marginals, bestfit, mapfit
        self.intensity = intensity

    def dataset_names(self):
        """The datasets of every run of this wave."""
        names = [n for n in RUN_DATASETS if n != 'posteriors' or self.posteriors is not None]
        return names + (list(INTENSITY_DATASETS) if self.intensity is not None else [])

    @property
    def n_run(self):
        return self.i_lon.size

    def run_attrs(self, r):
        a = {'ncomp': self.ncomp, 'n_chan_tot': self.n_chan_tot, 'n_params': self.ndim, 'marg_cols': MARG_COLS,
             'marg_quantiles': MARG_QUANTILES}
        for name in RUN_ATTR_COLUMNS:
            a[name] = self.columns[name][r].item()
        return a

    def run_dataset(self, r, name):
        if name == 'posteriors':
            return None if self.posteriors is None else self.posteriors[self.row_offsets[r]:self.row_offsets[r + 1]]
        if name == 'marginals':
            return self.marginals[r]
        if name in INTENSITY_DATASETS:
            return self.intensity[name][r]
        return (self.bestfit if name == 'bestfit_params' else self.mapfit)[r]


# ---- h5py look-alike ---------------------------------------------------------------------------------
class _MemFile:
    def __init__(self, root):
        self.root = root

    def flush(self):
        pass


class MemGroup:
    """In-memory stand-in for ``h5py.Group``: ``attrs``, nested groups, datasets as
    numpy arrays, path addressing with '/'."""

    def __init__(self, name="/", parent=None):
        self.name = name
        self.attrs = {}
        self._items = {}
        self._parent = parent

    @property
    def file(self):
        return _MemFile(self._root())

    def _split(self, path):
        return [p for p in str(path).split("/") if p]

    def _root(self):
        g = self
        while g._parent is not None:
            g = g._parent
        return g

    def _resolve(self, path, create=False):
        """(parent group, leaf name) of `path`; absolute paths start at the root."""
        parts = self._split(path)
        g = self._root() if str(path).startswith("/") else self
        for part in parts[:-1]:
            nxt = g._items.get(part)
            if nxt is None:
                if not create:
                    raise KeyError(path)
                nxt = MemGroup(f"{g.name.rstrip('/')}/{part}", g)
                g._items[part] = nxt
            if not isinstance(nxt, MemGroup):
                raise KeyError(path)
            g = nxt
        return g, (parts[-1] if parts else None)

    def create_group(self, path):
        parent, leaf = self._resolve(path, create=True)
        if leaf in parent._items:
            raise ValueError(f"Unable to create group (name already exists): {path}")
        g = MemGroup(f"{parent.name.rstrip('/')}/{leaf}", parent)
        parent._items[leaf] = g
        return g

    def require_group(self, path):
        parent, leaf = self._resolve(path, create=True)
        if leaf is None:
            return parent
        g = parent._items.get(leaf)
        if g is None:
            g = MemGroup(f"{parent.name.rstrip('/')}/{leaf}", parent)
            parent._items[leaf] = g
        return g

    def create_dataset(self, name, data=None):
        parent, leaf = self._resolve(name, create=True)
        if leaf in parent._items:
            raise ValueError(f"Unable to create dataset (name already exists): {name}")
        arr = np.array(data)
        parent._items[leaf] = arr
        return arr

    def __getitem__(self, path):
        parent, leaf = self._resolve(path)
        if leaf is None:
            return parent
        return parent._items[leaf]

    def __setitem__(self, path, value):
        parent, leaf = self._resolve(path, create=True)
        if isinstance(value, MemGroup):
            value._parent = parent
        parent._items[leaf] = value

    def __delitem__(self, path):
        parent, leaf = self._resolve(path)
        del parent._items[leaf]

    def __contains__(self, path):
        try:
            self[path]
            return True
        except KeyError:
            return False

    def __iter__(self):
        return iter(self._items)

    def keys(self):
        return self._items.keys()

    def items(self):
        return self._items.items()

    # ---- persistence --------------------------------------------------------
    def _flatten(self, prefix, out, attrs):
        if self.attrs:
            attrs[prefix or "/"] = {k: _jsonable(v) for k, v in self.attrs.items()}
        for k, v in self._items.items():
            p = f"{prefix}/{k}"
            if isinstance(v, LazyGroup):
                continue                    # a mounted view of other files: not this file's content
            if isinstance(v, MemGroup):
                v._flatten(p, out, attrs)
                if not v._items and not v.attrs:
                    attrs.setdefault(p, {})
            else:
                out[p] = v

    def save(self, path):
        out, attrs = {}, {}
        self._flatten("", out, attrs)
        out["__attrs__"] = np.array(json.dumps(attrs))
        with open(path, "wb") as f:
            np.savez(f, **out)

    @classmethod
    def load(cls, path):
        root = cls("/")
        with np.load(path, allow_pickle=False) as z:
            attrs = json.loads(str(z["__attrs__"]))
            for key in z.files:
                if key == "__attrs__":
                    continue
                root.create_dataset(key, data=z[key])
        for gpath, a in attrs.items():
            g = root.require_group(gpath)
            g.attrs.update({k: _unjson(v) for k, v in a.items()})
        return root


def _jsonable(v):
    if isinstance(v, np.ndarray):
        return {"__nd__": v.tolist()}
    if isinstance(v, (np.integer,)):
        return int(v)
    if isinstance(v, (np.floating,)):
        return float(v)
    if isinstance(v, (np.bool_,)):
        return bool(v)
    if isinstance(v, (list, tuple)):
        return [_jsonable(x) for x in v]
    return v


def _unjson(v):
    if isinstance(v, dict) and "__nd__" in v:
        return np.array(v["__nd__"])
    return v


class _LazyItems(Mapping):
    """Children of a LazyGroup: a key list plus a factory called on first access."""

    def __init__(self, keys, make):
        self._keys, self._make, self._cache = list(keys), make, {}

    def __getitem__(self, k):
        if k not in self._cache:
            if k not in self._keys:
                raise KeyError(k)
            self._cache[k] = self._make(k)
        return self._cache[k]

    def __iter__(self):
        return iter(self._keys)

    def __len__(self):
        return len(self._keys)


class LazyGroup(MemGroup):
    """Read-only group whose children are produced on demand (the slab store's view of the reference tree)."""

    def __init__(self, name, parent, keys, make, attrs=None):
        super().__init__(name, parent)
        self._items = _LazyItems(keys, make)
        if attrs:
            self.attrs.update(attrs)


# ---- sinks: where a finished wave goes ------------------------------------------------------------
class GroupSink:
    """Unrolls waves into an h5py-like group tree (an open ``h5py.File`` or a ``MemGroup``): one group per
    (pixel, ncomp) with the dumper's attributes and datasets, like the reference writes them one run at a time."""

    def __init__(self, root, store_posteriors=True):
        self.root, self.store_posteriors = root, store_posteriors

    def add_wave(self, wave):
        for r in range(wave.n_run):
            sub = self.root.require_group(f'/pix/{wave.i_lon[r]}/{wave.i_lat[r]}').create_group(f'{wave.ncomp}')
            for k, v in wave.run_attrs(r).items():
                sub.attrs[k] = v
            for name in RUN_DATASETS:
                if name == 'posteriors' and not (self.store_posteriors and wave.posteriors is not None):
                    continue
                sub.create_dataset(name, data=wave.run_dataset(r, name))
            if wave.intensity is not None:
                for name in INTENSITY_DATASETS:
                    sub.create_dataset(name, data=wave.run_dataset(r, name))

    def add_pixels(self, i_lon, i_lat, nbest):
        for lon, lat, nb in zip(i_lon, i_lat, nbest):
            g = self.root.require_group(f'/pix/{lon}/{lat}')
            g.attrs['i_lon'], g.attrs['i_lat'], g.attrs['nbest'] = int(lon), int(lat), int(nb)

    def close(self):
        pass


class SlabSink:
    """Writes waves as slabs into a chunk directory: one sequential file write per wave.  Code that writes
    h5py-style instead (``require_group`` / ``create_group`` on the chunk root) lands in a MemGroup that is
    saved beside the slabs and merged into the tree on read."""
    groups_file = 'groups.npz'

    def __init__(self, chunk_dir, store_posteriors=True):
        self.dir = Path(chunk_dir)
        self.dir.mkdir(parents=True, exist_ok=True)
        self.store_posteriors = store_posteriors
        self._seq = len(list(self.dir.glob('w*_n*.npz')))
        self._pseq = len(list(self.dir.glob('pix_*.npz')))
        self._groups = None
        self._lock = threading.Lock()           # several blocks of one rank may write concurrently

    def _group_root(self):
        if self._groups is None:
            p = self.dir / self.groups_file
            self._groups = MemGroup.load(p) if p.exists() else MemGroup("/")
        return self._groups

    def require_group(self, path):
        with self._lock:                        # creation of the intermediate groups is check-then-insert
            return self._group_root().require_group(path)

    def create_group(self, path):
        with self._lock:
            return self._group_root().create_group(path)

    @property
    def attrs(self):
        return self._group_root().attrs

    def add_wave(self, wave):
        with self._lock:
            stem = self.dir / f'w{self._seq:05d}_n{wave.ncomp}'
            self._seq += 1
        have_post = self.store_posteriors and wave.posteriors is not None
        if have_post:
            np.save(f'{stem}.post.npy', wave.posteriors)
        np.savez(f'{stem}.npz', ncomp=wave.ncomp, ndim=wave.ndim, n_chan_tot=wave.n_chan_tot, i_lon=wave.i_lon,
                 i_lat=wave.i_lat, row_offsets=wave.row_offsets, have_post=have_post, marginals=wave.marginals,
                 bestfit=wave.bestfit, mapfit=wave.mapfit, **{f'col_{k}': v for k, v in wave.columns.items()},
                 **(wave.intensity if wave.intensity is not None else {}))

    def add_pixels(self, i_lon, i_lat, nbest):
        with self._lock:
            path = self.dir / f'pix_{self._pseq:05d}.npz'
            self._pseq += 1
        np.savez(path, i_lon=np.asarray(i_lon, dtype=np.int64), i_lat=np.asarray(i_lat, dtype=np.int64),
                 nbest=np.asarray(nbest, dtype=np.int64))

    def close(self):
        if self._groups is not None:
            self._groups.save(self.dir / self.groups_file)


class _SlabWave(Wave):
    """A wave read back from disk; the posterior pool is memory-mapped."""

    def __init__(self, npz_path):
        with np.load(npz_path, allow_pickle=False) as z:
            cols = {k[4:]: z[k] for k in z.files if k.startswith('col_')}
            post = None
            if bool(z['have_post']):
                post = np.load(str(npz_path)[:-4] + '.post.npy', mmap_mode='r')
            inten = {n: z[n] for n in INTENSITY_DATASETS} if INTENSITY_DATASETS[0] in z.files else None
            super().__init__(int(z['ncomp']), int(z['ndim']), int(z['n_chan_tot']), z['i_lon'], z['i_lat'],
                             {k: cols[k] for k in RUN_ATTR_COLUMNS}, z['row_offsets'], post, z['marginals'],
                             z['bestfit'], z['mapfit'], inten)


def read_slab_chunk(chunk_dir):
    """(waves, pix, groups) of a chunk directory: its waves, {(lon, lat): nbest} and the h5py-style side tree."""
    chunk_dir = Path(chunk_dir)
    waves = [_SlabWave(p) for p in sorted(chunk_dir.glob('w*_n*.npz'))]
    pix = {}
    for p in sorted(chunk_dir.glob('pix_*.npz')):
        with np.load(p) as z:
            for lon, lat, nb in zip(z['i_lon'].tolist(), z['i_lat'].tolist(), z['nbest'].tolist()):
                pix[(lon, lat)] = nb
    gp = chunk_dir / SlabSink.groups_file
    return waves, pix, (MemGroup.load(gp) if gp.exists() else None)


def slab_pix_tree(chunk_dirs, parent=None):
    """The ``/pix`` group of the reference tree over the slabs of `chunk_dirs`, materialised lazily."""
    runs, nbest, waves, eager = {}, {}, [], {}
    for d in chunk_dirs:
        w, px, side = read_slab_chunk(d)
        nbest.update(px)
        if side is not None and 'pix' in side:
            for lon_key in side['pix']:
                for lat_key, g in side['pix'][lon_key].items():
                    eager[(int(lon_key), int(lat_key))] = g
        for wave in w:
            wi = len(waves)
            waves.append(wave)
            for r, (lon, lat) in enumerate(zip(wave.i_lon.tolist(), wave.i_lat.tolist())):
                runs.setdefault(lon, {}).setdefault(lat, {})[wave.ncomp] = (wi, r)      # a re-run replaces the run
    for lon, lat in list(nbest) + list(eager):
        runs.setdefault(lon, {}).setdefault(lat, {})

    def make_run(lon, lat, node, ncomp_key):
        wi, r = runs[lon][lat][int(ncomp_key)]
        wave = waves[wi]
        names = wave.dataset_names()
        return LazyGroup(f'/pix/{lon}/{lat}/{ncomp_key}', node, names, lambda n: np.asarray(wave.run_dataset(r, n)),
                         attrs=wave.run_attrs(r))

    def make_pix(lon, node, lat_key):
        lat = int(lat_key)
        attrs = {'i_lon': lon, 'i_lat': lat}
        if (lon, lat) in nbest:
            attrs['nbest'] = nbest[(lon, lat)]
        g = LazyGroup(f'/pix/{lon}/{lat}', node, [str(n) for n in sorted(runs[lon][lat])], None, attrs=attrs)
        g._items._make = lambda k: make_run(lon, lat, g, k)
        side = eager.get((lon, lat))
        if side is not None:                    # written h5py-style: merge attributes and children
            g.attrs.update(side.attrs)
            for k, v in side.items():
                if k not in g._items._keys:
                    g._items._keys.append(k)
                g._items._cache[k] = v
        return g

    def make_lon(lon_key):
        lon = int(lon_key)
        g = LazyGroup(f'/pix/{lon}', root, [str(v) for v in sorted(runs[lon])], None)
        g._items._make = lambda k: make_pix(lon, g, k)
        return g

    root = LazyGroup('/pix', parent, [str(v) for v in sorted(runs)], make_lon)
    return root


def check_ext(store_name, ext='hdf'):
    return store_name if store_name.endswith(f'.{ext}') else f'{store_name}.{ext}'


def chunk_path(store_dir, i):
    return Path(store_dir) / f'{HdfStore.chunk_prefix}{i}.hdf{"" if HAVE_H5PY else ".slab"}'


def chunk_sink(store_dir, i, store_posteriors=True):
    """What worker `i` writes into: takes whole waves (`add_wave`, `add_pixels`) and h5py-style group writes.
    Does not touch the table file (the coordinating process holds it open)."""
    if HAVE_H5PY:  # pragma: no cover - needs h5py
        f = h5py.File(chunk_path(store_dir, i), 'a')
        sink = GroupSink(f, store_posteriors)
        sink.require_group, sink.create_group, sink.attrs = f.require_group, f.create_group, f.attrs
        sink.close = lambda: (f.flush(), f.close())
        return sink
    return SlabSink(chunk_path(store_dir, i), store_posteriors)


class HdfStore:
    """Store directory with the reference's names and methods (main.py:233-377)."""
    linked_table = Path('table.hdf')
    chunk_prefix = 'chunk'
    dpath = '/products'

    def __init__(self, store_name, nchunks=1):
        self.store_name = str(store_name)
        self.store_dir = Path(check_ext(self.store_name, ext='store'))
        self.store_dir.mkdir(parents=True, exist_ok=True)
        self.backend = 'h5py' if HAVE_H5PY else 'slab'
        self._open = True
        if HAVE_H5PY:
            self.hdf = h5py.File(self.store_dir / self.linked_table, 'a')
        else:
            p = self._table_path
            self.hdf = MemGroup.load(p) if p.exists() else MemGroup("/")
        self.nchunks = int(self.hdf.attrs.setdefault('nchunks', nchunks)) if not HAVE_H5PY else self._h5_nchunks(nchunks)
        name = self.hdf.attrs.get('model_name')
        from .models import MODELS
        self.model = MODELS.get(name) if name is not None else None
        if not HAVE_H5PY and self.hdf.attrs.get('linked', False):
            self._mount()

    def _h5_nchunks(self, nchunks):  # pragma: no cover - needs h5py
        if 'nchunks' not in self.hdf.attrs:
            self.hdf.attrs['nchunks'] = nchunks
        return int(self.hdf.attrs['nchunks'])

    @property
    def _table_path(self):
        return self.store_dir / (str(self.linked_table) + ('' if HAVE_H5PY else '.npz'))

    def __enter__(self):
        return self

    def __exit__(self, exc_type, exc_value, traceback):
        self.close()

    @property
    def chunk_paths(self):
        return [chunk_path(self.store_dir, i) for i in range(self.nchunks)]

    @property
    def is_open(self):
        return self._open

    def close(self):
        if not self._open:
            print('Store HDF already closed.')
            return
        if HAVE_H5PY:
            self.hdf.flush()
            self.hdf.close()
        else:
            self.hdf.save(self._table_path)
        self._open = False

    # ---- what a worker writes into ---------------------------------------------------------------
    def open_chunk(self, i):
        """h5py-like root of chunk `i` (an open h5py.File, or the slab chunk's sink, which takes both waves and
        h5py-style writes)."""
        return self.chunk_sink(i)

    def close_chunk(self, i, root):
        root.close()

    def chunk_sink(self, i, store_posteriors=True):
        """Sink of chunk `i` for a worker: add_wave / add_pixels / h5py-style group writes / close."""
        return chunk_sink(self.store_dir, i, store_posteriors)

    # ---- the reference tree -----------------------------------------------------------------------
    def _mount(self):
        self.hdf._items['pix'] = slab_pix_tree([p for p in self.chunk_paths if p.exists()], parent=self.hdf)

    def link_files(self):
        """Make every chunk's pixel groups reachable from the table: ExternalLinks with h5py like the reference
        (main.py:313-322); the slab backend records that the chunks are linked and mounts a view of them."""
        assert self.is_open
        if HAVE_H5PY:  # pragma: no cover - needs h5py
            for chunk_path in self.chunk_paths:
                if not chunk_path.exists():
                    continue
                with h5py.File(chunk_path, 'r') as chunk_hdf:
                    for lon_pix in chunk_hdf.get('/pix', ()):
                        for lat_pix in chunk_hdf[f'/pix/{lon_pix}']:
                            name = f'/pix/{lon_pix}/{lat_pix}'
                            self.hdf[name] = h5py.ExternalLink(chunk_path.name, name)
            self.hdf.flush()
        else:
            self.hdf.attrs['linked'] = True
            self._mount()

    def reset_pix_links(self):
        assert self.is_open
        if '/pix' in self.hdf:
            del self.hdf['/pix']
        if not HAVE_H5PY:
            self.hdf.attrs['linked'] = False

    def iter_pix_groups(self):
        assert self.is_open
        pix = self.hdf['/pix']
        for lon_pix in pix:
            for lat_pix in pix[lon_pix]:
                group = pix[lon_pix][lat_pix]
                if hasattr(group, 'attrs'):
                    yield group

    def find_first_valid_group(self):
        for group in self.iter_pix_groups():
            if '1' in group:
                return group['1']
        raise ValueError('No valid pix groups found.')

    # ---- root attributes, driven by the schema tables ----------------------------------------------
    def insert_header(self, stack):
        if not self.is_open:
            warnings.warn('Could not insert header: the HDF5 file is closed.', category=RuntimeWarning)
            return
        for gname, prop in HEADER_GROUPS.items():
            g = self.hdf.require_group(gname)
            for k, v in getattr(stack, prop).items():
                g.attrs[k] = v
        self.hdf.attrs['naxis1'], self.hdf.attrs['naxis2'] = stack.shape[0], stack.shape[1]

    def read_header(self, full=True):
        """The stored cube header (`full`) or its two-dimensional map part (main.py:345-352): an
        ``astropy.io.fits.Header`` when astropy is importable, else a plain dict with the same cards."""
        assert self.is_open
        cards = dict(self.hdf['full_header' if full else 'simple_header'].attrs.items())
        try:
            from astropy.io import fits
        except ImportError:
            return cards
        header = fits.Header()                  # pragma: no cover - optional dependency
        for k, v in cards.items():              # pragma: no cover
            header[k] = v
        return header                           # pragma: no cover

    def create_dataset(self, dset_name, data, group='', clobber=True):
        assert len(dset_name) > 0
        g = self.hdf.require_group(group) if group else self.hdf
        if dset_name in g and clobber:
            warnings.warn(f'Deleting dataset "{group.rstrip("/")}/{dset_name}"', RuntimeWarning)
            del g[dset_name]
        return g.create_dataset(dset_name, data=data)

    def insert_fitter_pars(self, fitter):
        assert self.is_open
        for name, get in FITTER_ATTRS.items():
            self.hdf.attrs[name] = get(fitter)

    def insert_model_metadata(self, runner_cls):
        assert self.is_open
        module = inspect.getmodule(runner_cls)
        for name, const in MODEL_ATTRS.items():
            self.hdf.attrs[name] = getattr(module, const)
