#!/usr/bin/env python3
"""
TEST INFRASTRUCTURE -- not part of the product path.

Compile the *unmodified* reference likelihood path (Cython + one C file) from
the sources where they lie under ``/root/reference`` into ``oracle/_ref/``.
Only compiled extension modules (``*.so``) and empty package markers are
written there; no reference source text is copied into the repository
(``oracle/_ref/`` is git-ignored but travels to the GPU box with ``gpurun``).

Recipe (SURVEY.md Appendix B):
  * sources are staged in a scratch directory under /tmp (the reference tree
    is read-only and Cython writes its generated C next to the ``.pyx``);
  * ``multinest.h`` is replaced by a stub -- MultiNest (external Fortran, not
    vendored, no Fortran compiler in this image) cannot be built, so
    ``run_multinest`` is a no-op in the oracle build.  The stub forwards to a
    weak hook ``nf_oracle_ns_run`` so a test harness may plug a CPU sampler in;
  * Cython directive ``legacy_implicit_noexcept`` (reference targets Cython
    0.29 callback semantics, core.pyx:622-627,820-821);
  * ``-fopenmp`` dropped (no OpenMP construct exists in the reference);
  * ``-march=x86-64-v3`` instead of ``-march=native`` so the binary built in
    this container also runs on the GPU box's host CPU.

Modules built: nestfit.core.core, nestfit.models.{hyperfine,ammonia,gaussian,
diazenylium}.  Usage: ``python oracle/build_ref.py`` (idempotent).
"""

import os
import shutil
import subprocess
import sys
import tempfile
from pathlib import Path

HERE = Path(__file__).resolve().parent
REF = Path(os.environ.get("NESTFIT_REFERENCE", "/root/reference"))
OUT = HERE / "_ref"

MOD_NAMES = [
    "nestfit.core.core",
    "nestfit.models.hyperfine",
    "nestfit.models.ammonia",
    "nestfit.models.gaussian",
    "nestfit.models.diazenylium",
]

STUB_MULTINEST_H = r"""
/* Stub for the absent MultiNest C interface (cmultinest.pxd:5-33). */
#ifndef NF_STUB_MULTINEST_H
#define NF_STUB_MULTINEST_H
typedef void (*nf_loglike_cb)(double *, int *, int *, double *, void *);
typedef void (*nf_dumper_cb)(int *, int *, int *, double **, double **,
        double **, double *, double *, double *, double *, void *);
typedef void (*nf_ns_run_fn)(int nlive, double tol, double efr, int ndims,
        int nPar, int seed, int maxiter, nf_loglike_cb, nf_dumper_cb, void *);
/* Optional hook a harness can set (through ctypes) to drive a CPU sampler. */
__attribute__((weak)) nf_ns_run_fn nf_oracle_ns_run = 0;
static void run(int IS, int mmodal, int ceff, int nlive, double tol,
        double efr, int ndims, int nPar, int nClsPar, int maxModes,
        int updInt, double Ztol, char root[], int seed, int *pWrap, int fb,
        int resume, int outfile, int initMPI, double logZero, int maxiter,
        nf_loglike_cb LogLike, nf_dumper_cb dumper, void *context)
{
    if (nf_oracle_ns_run)
        nf_oracle_ns_run(nlive, tol, efr, ndims, nPar, seed, maxiter,
                LogLike, dumper, context);
}
#endif
"""

SETUP_PY = r"""
import numpy as np
from setuptools import setup, Extension
from Cython.Build import cythonize

MOD_NAMES = %(mods)r
exts = [
    Extension(
        m, [m.replace('.', '/') + '.pyx', 'nestfit/core/fastexp.c'],
        libraries=['m'],
        include_dirs=[np.get_include(), 'stub', 'nestfit/core', 'includes'],
        extra_compile_args=['-O3', '-march=x86-64-v3', '-mtune=generic',
                            '-ffast-math', '-w'],
    ) for m in MOD_NAMES
]
setup(
    name='nestfit_ref',
    ext_modules=cythonize(
        exts, include_path=['includes', '.'], language_level=3,
        compiler_directives={'legacy_implicit_noexcept': True,
                             'embedsignature': True},
        quiet=True),
    script_args=['build_ext', '--inplace'],
)
"""


def is_built():
    need = [OUT / (m.replace(".", "/")) for m in MOD_NAMES]
    for stem in need:
        if not list(stem.parent.glob(stem.name + ".*.so")):
            return False
    return True


def sources_present():
    """True when the reference's sources can be read at REF; a path the user may not enter counts as absent."""
    try:
        return (REF / "nestfit" / "core" / "core.pyx").is_file() and os.access(REF, os.R_OK | os.X_OK)
    except OSError:
        return False


def build(force=False):
    if is_built() and not force:
        return True
    if not sources_present():
        return False
    work = Path(tempfile.mkdtemp(prefix="nestfit_ref_build_"))
    try:
        shutil.copytree(REF / "nestfit", work / "nestfit")
        shutil.copytree(REF / "includes", work / "includes")
        subprocess.run(["chmod", "-R", "u+w", str(work)], check=True)
        # blank package markers: the real ones import h5py/astropy
        for p in ("nestfit/__init__.py", "nestfit/models/__init__.py",
                  "nestfit/core/__init__.py"):
            (work / p).write_text("")
        (work / "stub").mkdir()
        (work / "stub" / "multinest.h").write_text(STUB_MULTINEST_H)
        (work / "setup_ref.py").write_text(SETUP_PY % {"mods": MOD_NAMES})
        env = dict(os.environ, CC="/usr/bin/gcc", CXX="/usr/bin/g++")
        subprocess.run([sys.executable, "setup_ref.py"], cwd=work, env=env,
                       check=True, stdout=subprocess.DEVNULL)
        if OUT.exists():
            shutil.rmtree(OUT)
        for sub in ("nestfit/core", "nestfit/models"):
            (OUT / sub).mkdir(parents=True)
            (OUT / sub / "__init__.py").write_text("")
            for so in (work / sub).glob("*.so"):
                shutil.copy2(so, OUT / sub / so.name)
        (OUT / "nestfit" / "__init__.py").write_text("")
        (OUT / "README").write_text(
            "Compiled from /root/reference by oracle/build_ref.py; "
            "binaries only, git-ignored.\n")
    finally:
        shutil.rmtree(work, ignore_errors=True)
    return is_built()


if __name__ == "__main__":
    ok = build(force="--force" in sys.argv)
    print("oracle/_ref built" if ok else "oracle/_ref NOT built")
    sys.exit(0 if ok else 1)
