"""ctypes binding of libsie_b200.so (declared in include/sie_b200.h).

There is no CPU fallback: if the shared object is missing or a call fails, this raises."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libsie_b200.so")

SIE_JOB_OK, SIE_JOB_NO_NAN_CELL, SIE_JOB_FEW_AREAS, SIE_JOB_CAPACITY = 0, 1, 2, 3
SIE_CORR_AUTO, SIE_CORR_TILES, SIE_CORR_ROWS, SIE_CORR_ROWS_MIRROR, SIE_CORR_TMA = 0, 1, 2, 3, 4
ABI_VERSION = 2
SIE_AREA_WORK = 32   # uint64 profiling counters per job (include/sie_b200.h)

c_i32 = C.c_int32
c_p = C.c_void_p
c_sz = C.c_size_t


class SieGpProblem(C.Structure):
    _fields_ = [("job_sic", c_i32), ("job_sst", c_i32), ("n", c_i32), ("y_off", c_i32), ("rule", c_i32),
                ("zscore", c_i32), ("want_grad", c_i32), ("pad_", c_i32), ("r_sel", C.c_double),
                ("ell", C.c_double), ("sig", C.c_double)]


class SieGpResult(C.Structure):
    _fields_ = [("fmean", C.c_double), ("fvar", C.c_double), ("sigma_f", C.c_double), ("nlml", C.c_double),
                ("g_ell", C.c_double), ("g_sig", C.c_double), ("n_pred", c_i32), ("expm_m", c_i32),
                ("expm_s", c_i32), ("info", c_i32), ("cycles_total", C.c_int64), ("cycles_expm", C.c_int64)]


class SieGpMarginal(C.Structure):
    _fields_ = [("ess", C.c_double), ("w_max", C.c_double), ("n_admissible", c_i32), ("argmax", c_i32)]


_SIGS = {
    "sie_abi_version": (C.c_int, []),
    "sie_last_error": (C.c_char_p, []),
    "sie_device_info": (C.c_int, [C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(c_sz)]),
    "sie_detrend_zscore": (C.c_int, [c_p, c_p, c_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, c_p, c_p, c_p,
                                     c_p, c_p, c_p, c_p, c_p, C.c_int, c_p]),
    "sie_corr_tau": (C.c_int, [c_p, c_p, c_p, c_p, C.c_int, C.c_int, C.c_int, c_p, c_p, c_sz, c_p, c_p, c_p,
                               C.c_int, C.c_int, C.c_int, c_p]),
    "sie_corr_tau_scratch_bytes": (c_sz, [C.c_int, C.c_int]),
    "sie_corr_rows": (C.c_int, [c_p, c_p, C.c_int, C.c_int, C.c_int, C.c_int, c_p, C.c_int, c_p]),
    "sie_corr_stencil": (C.c_int, [c_p, c_p, c_p, C.c_int, c_p, c_p, c_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                   c_p, c_p]),
    "sie_area_level": (C.c_int, [c_p, c_p, c_p, C.c_int, c_p, c_p, c_p, c_p, c_p, c_p, C.c_int, C.c_int, C.c_int,
                                 C.c_int, C.c_int, C.c_int, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_sz, c_p, c_p]),
    "sie_area_level_scratch_bytes": (c_sz, [C.c_int, C.c_int]),
    "sie_intra_links": (C.c_int, [c_p, c_p, c_p, c_p, c_p, c_p, c_p, C.c_int, C.c_int, C.c_int, C.c_int, c_p, c_p,
                                  c_p, c_p, c_p]),
    "sie_gp_forecast": (C.c_int, [c_p, C.c_int, c_p, c_p, c_p, C.c_int, C.c_int, c_p, c_p, C.c_int, C.c_int,
                                  C.c_int, c_p, c_p, c_sz, c_p]),
    "sie_gp_scratch_bytes": (c_sz, [C.c_int, C.c_int, C.c_int]),
    "sie_nsidc_monthly": (C.c_int, [c_p, C.c_int, c_sz, C.c_int, C.c_int, c_p, c_p]),
    "sie_polar_hole_fill": (C.c_int, [c_p, c_p, C.c_double, C.c_int, c_p, c_p, c_p, c_p]),
    "sie_regrid_linear": (C.c_int, [c_p, C.c_int, C.c_int, c_p, c_p, C.c_int, c_p, c_p]),
    "sie_gp_hyper_grid": (C.c_int, [c_p, C.c_int, c_p, C.c_int, c_p, c_p, c_p, C.c_int, C.c_int, c_p, c_p, C.c_int,
                                    C.c_int, C.c_int, c_p, c_p, c_sz, c_p]),
    "sie_gp_grid_select": (C.c_int, [c_p, c_p, C.c_int, c_p, C.c_int, c_p, C.c_int, c_p, c_p, c_p]),
    "sie_gp_grid_marginal": (C.c_int, [c_p, C.c_int, C.c_int, c_p, C.c_int, c_p, c_p, c_p, c_p]),
    "sie_debug_gp_phases": (C.c_int, [C.POINTER(C.c_ulonglong)]),       # profiling aid (tools/gp_phases.py)
}

EXPORTED_SYMBOLS = tuple(_SIGS)
_lib = None


class SieError(RuntimeError):
    pass


def load():
    """Load the shared object (once).  Raises if it has not been built: no fallback path exists."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise SieError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                       "(the CUDA extension is the only implementation; there is no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in _SIGS.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.sie_abi_version() != ABI_VERSION:
        raise SieError(f"{LIB_PATH} has ABI version {lib.sie_abi_version()}, this package needs {ABI_VERSION}: rebuild")
    _lib = lib
    return lib


def check(rc, what):
    if rc != 0:
        msg = load().sie_last_error()
        raise SieError(f"{what} failed (rc={rc}): {msg.decode() if msg else ''}")
