"""Build + call the host build of the standard-error routine (TEST TOOL ONLY, see stderr_shim.cpp)."""
import ctypes as C
import os
import subprocess

import numpy as np

from fetal_t2mapping_b200 import _abi

HERE = os.path.dirname(os.path.abspath(__file__))
SO = os.path.join(HERE, "libt2fit_stderr_shim.so")
SRC = os.path.join(HERE, "stderr_shim.cpp")
CSRC = os.path.join(HERE, "..", "..", "fetal_t2mapping_b200", "csrc")
DEPS = [SRC] + [os.path.join(CSRC, f) for f in ("t2fit_stderr.cuh", "t2fit_core.cuh", "t2fit_lbfgsb.cuh", "t2fit_i0e_coeffs.h",
                                                "t2fit_i1e_coeffs.h")] + [os.path.join(HERE, "..", "..", "include", "t2fit.h")]


def build(force=False):
    """-ffp-contract=fast with FMA, as nvcc contracts a*b+c on the device."""
    if not force and os.path.isfile(SO) and all(os.path.getmtime(SO) >= os.path.getmtime(d) for d in DEPS):
        return SO
    cmd = ["g++", "-O2", "-std=c++17", "-mfma", "-ffp-contract=fast", "-shared", "-fPIC", "-x", "c++", SRC, "-o", SO, "-lm"]
    subprocess.run(cmd, check=True, cwd=HERE)
    return SO


_lib = []


def lib():
    if not _lib:
        l = C.CDLL(build())
        l.stderr_rows.restype = C.c_int
        l.stderr_rows.argtypes = [C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                  C.c_void_p, C.c_void_p]
        l.stderr_i1e.restype = C.c_double
        l.stderr_i1e.argtypes = [C.c_double]
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
