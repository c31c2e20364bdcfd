"""Build + call the host build of the standard-error and T2 interval routines (TEST TOOL ONLY, see pass_shim.cpp)."""
import ctypes as C
import os

import numpy as np

from fetal_t2mapping_b200 import _abi
from tests.hostsim import HERE, compile_so

SO = os.path.join(HERE, "libt2fit_pass_shim.so")
SRC = os.path.join(HERE, "pass_shim.cpp")
CSRC = os.path.join(HERE, "..", "..", "fetal_t2mapping_b200", "csrc")
DEPS = [SRC] + [os.path.join(CSRC, f) for f in ("t2fit_interval.cuh", "t2fit_stderr.cuh", "t2fit_core.cuh", "t2fit_lbfgsb.cuh",
                                                "t2fit_i0e_coeffs.h", "t2fit_i1e_coeffs.h")] + \
    [os.path.join(HERE, "..", "..", "include", "t2fit.h")]


def build(force=False):
    return compile_so(SRC, SO, DEPS, force)


_lib = []


def lib():
    if not _lib:
        l = C.CDLL(build())
        l.stderr_rows.restype = C.c_int
        l.stderr_rows.argtypes = [C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                  C.c_void_p, C.c_void_p]
        l.stderr_i1e.restype = C.c_double
        l.stderr_i1e.argtypes = [C.c_double]
        l.interval_rows.restype = C.c_int
        l.interval_rows.argtypes = [C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int,
                                    C.c_double, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        _lib.append(l)
    return _lib[0]


def stderr_rows(rows, te, fit, norm, k, t2, sigma=None):
    """[M, 3] float64 standard errors (k, T2, sigma; sigma NaN for gaussian) of the rows at the given float32 parameters."""
    rows = np.ascontiguousarray(rows, np.float32)
    te = np.ascontiguousarray(te, np.float64)
    k, t2 = (np.ascontiguousarray(a, np.float32) for a in (k, t2))
    sg = None if sigma is None else np.ascontiguousarray(sigma, np.float32)
    out = np.empty((rows.shape[0], 3), np.float64)
    rc = lib().stderr_rows(rows.ctypes.data, rows.shape[0], rows.shape[1], te.ctypes.data, _abi.MODELS[fit], int(bool(norm)),
                           k.ctypes.data, t2.ctypes.data, None if sg is None else sg.ctypes.data, out.ctypes.data)
    if rc:
        raise ValueError(f"stderr_rows: {rc}")
    return out


def interval_rows(rows, te, fit, norm, box, no_prior, q, n_grid=64, profile=False):
    """(lo, hi, best) float64 [M] each, flags uint8 [M] and, with ``profile``, p at the grid [M, n_grid].  ``box``:
    (k_lo, k_hi, t2_lo, t2_hi, sigma_lo, sigma_hi) in force (k_lo is replaced by y(TE_0) when ``no_prior``)."""
    rows = np.ascontiguousarray(rows, np.float32)
    te = np.ascontiguousarray(te, np.float64)
    b = np.ascontiguousarray(box, np.float64)
    m = rows.shape[0]
    out = np.empty((m, 3), np.float64)
    flags = np.empty(m, np.uint8)
    prof = np.empty((m, n_grid), np.float64) if profile else None
    rc = lib().interval_rows(rows.ctypes.data, m, rows.shape[1], te.ctypes.data, _abi.MODELS[fit], int(bool(norm)),
                             b.ctypes.data, int(bool(no_prior)), float(q), int(n_grid), out.ctypes.data, flags.ctypes.data,
                             None if prof is None else prof.ctypes.data)
    if rc:
        raise ValueError(f"interval_rows: {rc}")
    return out[:, 0], out[:, 1], out[:, 2], flags, prof
