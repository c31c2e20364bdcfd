"""Build + call the host build of the standard-error, T2 interval and parametric-bootstrap routines (TEST TOOL ONLY, see
pass_shim.cpp)."""
import ctypes as C
import os

import numpy as np

from fetal_t2mapping_b200 import _abi
from tests.hostsim import HERE, compile_so

SO = os.path.join(HERE, "libt2fit_pass_shim.so")
SRC = os.path.join(HERE, "pass_shim.cpp")
CSRC = os.path.join(HERE, "..", "..", "fetal_t2mapping_b200", "csrc")
DEPS = [SRC] + [os.path.join(CSRC, f) for f in ("t2fit_interval.cuh", "t2fit_stderr.cuh", "t2fit_bootstrap.cuh", "t2fit_core.cuh",
                                                "t2fit_lbfgsb.cuh", "t2fit_i0e_coeffs.h", "t2fit_i1e_coeffs.h")] + \
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
        l.bootstrap_philox.restype = None
        l.bootstrap_philox.argtypes = [C.c_void_p] * 3
        l.bootstrap_rows.restype = C.c_int
        l.bootstrap_rows.argtypes = [C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_int, C.c_int] + [C.c_void_p] * 5 + \
            [C.c_uint64, C.c_int, C.c_void_p]
        l.bootstrap_stats.restype = C.c_int
        l.bootstrap_stats.argtypes = [C.c_int, C.c_int64, C.c_int] + [C.c_void_p] * 4 + [C.c_double] + [C.c_void_p] * 6
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


def bootstrap_philox(ctr, key):
    """The four Philox4x32-10 words of counter ``ctr`` (4 x uint32) under ``key`` (2 x uint32)."""
    c, k = np.ascontiguousarray(ctr, np.uint32), np.ascontiguousarray(key, np.uint32)
    out = np.empty(4, np.uint32)
    lib().bootstrap_philox(c.ctypes.data, k.ctypes.data, out.ctypes.data)
    return out


def bootstrap_rows(rows, te, fit, norm, k, t2, sigma, noise_sd, voxel_id, seed, n_rep):
    """[M * n_rep, E] float32 replicate rows (row i * n_rep + r) of the host build of csrc/t2fit_bootstrap.cuh."""
    rows = np.ascontiguousarray(rows, np.float32)
    te = np.ascontiguousarray(te, np.float64)
    m = rows.shape[0]
    f32 = [None if a is None else np.ascontiguousarray(a, np.float32) for a in (k, t2, sigma, noise_sd)]
    vid = np.ascontiguousarray(voxel_id, np.int64)
    out = np.empty((m * n_rep, rows.shape[1]), np.float32)
    rc = lib().bootstrap_rows(rows.ctypes.data, m, rows.shape[1], te.ctypes.data, _abi.MODELS[fit], int(bool(norm)),
                              *[None if a is None else a.ctypes.data for a in f32], vid.ctypes.data, int(seed), int(n_rep),
                              out.ctypes.data)
    if rc:
        raise ValueError(f"bootstrap_rows: {rc}")
    return out


def bootstrap_stats(fit, n_rep, k, t2, sigma, status, level):
    """(mean [3, M], sd [3, M], lo [M], hi [M], n_used [M], n_ok [M]) of the replicate results [M * n_rep] (row i * n_rep + r)
    by the host build of the statistics kernel's arithmetic."""
    k, t2 = (np.ascontiguousarray(a, np.float32) for a in (k, t2))
    sg = None if sigma is None else np.ascontiguousarray(sigma, np.float32)
    st = np.ascontiguousarray(status, np.uint8)
    m = k.size // n_rep
    mean, sd = np.empty((3, m), np.float32), np.empty((3, m), np.float32)
    lo, hi = np.empty(m, np.float32), np.empty(m, np.float32)
    nu, no = np.empty(m, np.int32), np.empty(m, np.int32)
    rc = lib().bootstrap_stats(_abi.MODELS[fit], m, int(n_rep), k.ctypes.data, t2.ctypes.data,
                               None if sg is None else sg.ctypes.data, st.ctypes.data, float(level), mean.ctypes.data,
                               sd.ctypes.data, lo.ctypes.data, hi.ctypes.data, nu.ctypes.data, no.ctypes.data)
    if rc:
        raise ValueError(f"bootstrap_stats: {rc}")
    return mean, sd, lo, hi, nu, no
