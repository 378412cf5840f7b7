"""ctypes binding of libnestfit_b200.so (the C ABI in include/nestfit_b200.h).

There is no CPU fallback: if the CUDA library is missing or a call fails, an
exception is raised.
"""
import ctypes as C
from pathlib import Path

import numpy as np

_PKG = Path(__file__).resolve().parent
import os as _os
# NESTFIT_B200_LIB lets kernel experiments load an alternative build of the same ABI
LIB_PATH = Path(_os.environ.get("NESTFIT_B200_LIB", _PKG / "libnestfit_b200.so"))

NF_MODEL_NH3, NF_MODEL_GAUSS, NF_MODEL_N2HP = 1, 2, 3
NF_F32, NF_F64 = 0, 1
NF_FLAG_COLD, NF_FLAG_LTE = 1, 2
NF_MAX_SPEC = 6
NF_MAX_NCOMP_NH3 = 4
NF_MAX_NCOMP_GAUSS = 32
NF_MAX_BAND_FRAC = 8e-4      # widest hyperfine spectrum, (nu_last - nu_first) / nu_first


class NfError(RuntimeError):
    pass


class DistDesc(C.Structure):
    _fields_ = [("size", C.c_int32), ("stride", C.c_int32), ("offset", C.c_int32), ("pad_", C.c_int32),
                ("xmin", C.c_double), ("xmax", C.c_double), ("dx", C.c_double), ("du", C.c_double)]


class PriorDesc(C.Structure):
    _fields_ = [("kind", C.c_int32), ("flags", C.c_uint32), ("p_ix", C.c_int32), ("p_ix2", C.c_int32),
                ("dist", C.c_int32), ("dist2", C.c_int32), ("nested", C.c_int32), ("pad_", C.c_int32),
                ("value", C.c_double)]


class NsConfig(C.Structure):
    """Mirror of `nf_ns_config` (include/nestfit_b200.h)."""
    _fields_ = [("nlive_max", C.c_int32), ("n_prop", C.c_int32), ("max_iter", C.c_int32),
                ("max_samples", C.c_int32), ("bound_update_interval", C.c_int32), ("flags", C.c_int32),
                ("tol", C.c_double), ("efr", C.c_double), ("seed", C.c_uint64),
                ("n_prop_max", C.c_int32), ("target_batch", C.c_int32)]


_lib = None

_VP, _I, _I64, _D = C.c_void_p, C.c_int, C.c_int64, C.c_double
_PD, _PI = C.POINTER(C.c_double), C.POINTER(C.c_int)

_SIGNATURES = {
    "nf_abi_version": ([], _I),
    "nf_error_string": ([_I], C.c_char_p),
    "nf_device_count": ([_PI], _I),
    "nf_pixels_create": ([_I, _I, _I64, _I, _I, _VP, _VP, _VP, _VP, _VP, _I, _VP, C.POINTER(_VP)], _I),
    "nf_pixels_create_from_device": ([_I, _I, _I64, _I, _I, _VP, _VP, _VP, _VP, _VP, _VP, C.POINTER(_VP)], _I),
    "nf_pixels_create_axes": ([_I, _I, _I64, _I, _I, _VP, _VP, _VP, _VP, _VP, _VP, _I, _VP, C.POINTER(_VP)], _I),
    "nf_pixels_free": ([_VP], _I),
    "nf_pixels_null_lnz": ([_VP, _VP], _I),
    "nf_nh3_loglike": ([_VP, _VP, _I, _VP, _I64, _I64, _I, _I, _VP, _VP], _I),
    "nf_nh3_predict": ([_VP, _VP, _I, _I64, _I, _I, _VP, _VP], _I),
    "nf_gauss_loglike": ([_VP, _VP, _I, _VP, _I64, _I64, _I, _VP, _VP], _I),
    "nf_gauss_predict": ([_VP, _VP, _I, _I64, _I, _VP, _VP], _I),
    "nf_n2hp_loglike": ([_VP, _VP, _I, _VP, _I64, _I64, _I, _VP, _VP], _I),
    "nf_n2hp_predict": ([_VP, _VP, _I, _I64, _I, _VP, _VP], _I),
    "nf_n2hp_loglike_host": ([_VP, _VP, _I, _VP, _I64, _I64, _I, _VP], _I),
    "nf_n2hp_predict_host": ([_VP, _VP, _I, _I64, _I, _VP], _I),
    "nf_nh3_loglike_host": ([_VP, _VP, _I, _VP, _I64, _I64, _I, _I, _VP], _I),
    "nf_gauss_loglike_host": ([_VP, _VP, _I, _VP, _I64, _I64, _I, _VP], _I),
    "nf_nh3_predict_host": ([_VP, _VP, _I, _I64, _I, _I, _VP], _I),
    "nf_gauss_predict_host": ([_VP, _VP, _I, _I64, _I, _VP], _I),
    "nf_predict_pix": ([_VP, _VP, _I, _VP, _I64, _I, _I, _VP, _VP], _I),
    "nf_predict_pix_host": ([_VP, _VP, _I, _VP, _I64, _I, _I, _VP], _I),
    "nf_predict_moments": ([_VP, _VP, _I, _VP, _I64, _I, _VP, _VP, _VP], _I),
    "nf_predict_moments_host": ([_VP, _VP, _I, _VP, _I64, _I, _VP, _VP], _I),
    "nf_priors_create": ([_I, _VP, _I, _VP, _I, _VP, _I64, _I, C.POINTER(_VP)], _I),
    "nf_priors_free": ([_VP], _I),
    "nf_prior_transform": ([_VP, _VP, _I64, _I, _VP], _I),
    "nf_prior_transform_host": ([_VP, _VP, _I64, _I], _I),
    "nf_last_call_stats": ([_PD, C.POINTER(_I64)], _I),
    "nf_measure_peaks": ([_I, _PD, _PD], _I),
}


def declared_symbols():
    """Names of every function the public headers declare (used by the CPU tests)."""
    import re
    names = []
    for hdr in sorted((_PKG.parent / "include").glob("*.h")):
        text = re.sub(r"/\*.*?\*/", "", hdr.read_text(), flags=re.S)
        names += re.findall(r"\b(nf_[a-z0-9_]+)\s*\(", text)
    return sorted(set(names))


def load():
    """Load the CUDA library, building nothing: a missing library is an error."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise NfError(
            f"{LIB_PATH} not found: build it with `python -m nestfit_b200.build` "
            "(nestfit_b200 has no CPU fallback)")
    lib = C.CDLL(str(LIB_PATH))
    for name, (argtypes, restype) in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = restype
    _lib = lib
    return lib


def register(name, argtypes, restype=_I):
    """Late registration used by optional modules (sampler)."""
    _SIGNATURES[name] = (argtypes, restype)
    if _lib is not None:
        fn = getattr(_lib, name)
        fn.argtypes = argtypes
        fn.restype = restype


def check(code, what=""):
    if code != 0:
        msg = load().nf_error_string(code).decode()
        raise NfError(f"{what or 'nestfit_b200 call'} failed: {msg} (code {code})")


def ptr(arr):
    """void* of a C-contiguous numpy array (or None)."""
    if arr is None:
        return None
    assert arr.flags["C_CONTIGUOUS"]
    return arr.ctypes.data_as(C.c_void_p)


def as_f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)
