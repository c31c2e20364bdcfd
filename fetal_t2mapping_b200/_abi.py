"""ctypes view of ``include/t2fit.h`` and the loader of the in-tree ``libt2fit.so``.

The library is the product: if it is missing or fails to load this module raises,
there is no Python / CPU substitute for the fit.
"""
from __future__ import annotations

import ctypes as C
import os

ABI_VERSION = 5
MAX_ECHO = 32
MAX_DUP = 7

MODEL_GAUSSIAN = 0
MODEL_GAUSSIAN_RICIAN = 1
MODEL_RICIAN = 2
MODELS = {"gaussian": MODEL_GAUSSIAN, "gaussian_rician": MODEL_GAUSSIAN_RICIAN, "rician": MODEL_RICIAN}
SOLVER_FAST, SOLVER_LBFGSB, SOLVER_LBFGSB_DENSE = 0, 1, 2
SOLVERS = {"fast": SOLVER_FAST, "lbfgsb": SOLVER_LBFGSB, "lbfgsb_dense": SOLVER_LBFGSB_DENSE}

LAYOUT_AOS = 0
LAYOUT_SOA = 1
LAYOUT_PLANES = 2
DTYPES = {"uint8": 0, "int16": 1, "uint16": 2, "int32": 3, "float32": 4, "float64": 5, "bool": 0}
# element types a HOST echo array may have (t2fit_problem.echo_dtype; 0 = float32)
ECHO_DTYPES = {"float32": 0, "int16": 1, "uint16": 2, "int32": 3, "float64": 5}
IDX_I64, IDX_I32 = 0, 1
MEM_HOST = 0
MEM_DEVICE = 1

ST_OK, ST_NONFINITE, ST_NOTCONVERGED, ST_BADBOUNDS = 0, 1, 2, 3
INIT_LOGLINEAR, INIT_PRESET, INIT_BEST = 0, 1, 2

ERRORS = {0: "OK", -1: "EINVAL", -2: "ENODEVICE", -3: "ENOTINIT", -4: "ECUDA", -5: "ENOMEM"}


class Problem(C.Structure):
    """``t2fit_problem`` (include/t2fit.h)."""
    _fields_ = [
        ("echoes", C.c_void_p),
        ("layout", C.c_int32),
        ("memory", C.c_int32),
        ("ld", C.c_int64),
        ("mask_idx", C.c_void_p),
        ("n_vox", C.c_int64),
        ("n_fit", C.c_int64),
        ("n_echo", C.c_int32),
        ("model", C.c_int32),
        ("te_ms", C.POINTER(C.c_double)),
        ("x0", C.c_double * 3),
        ("lb", C.c_double * 3),
        ("ub", C.c_double * 3),
        ("no_prior", C.c_int32),
        ("no_prior_k_ub", C.c_double),
        ("no_prior_t2_lb", C.c_double),
        ("no_prior_t2_ub", C.c_double),
        ("norm", C.c_int32),
        ("max_iter", C.c_int32),
        ("tol", C.c_float),
        ("init", C.c_int32),
        ("solver", C.c_int32),
        ("lbfgsb_ftol", C.c_double),
        ("lbfgsb_gtol", C.c_double),
        ("lbfgsb_maxls", C.c_int32),
        ("lbfgsb_maxiter", C.c_int32),
        ("lbfgsb_maxfun", C.c_int32),
        ("echo_dtype", C.c_int32),
        ("idx_dtype", C.c_int32),
    ]


class Outputs(C.Structure):
    """``t2fit_outputs`` (include/t2fit.h)."""
    _fields_ = [
        ("t2", C.c_void_p),
        ("k", C.c_void_p),
        ("sigma", C.c_void_p),
        ("res", C.c_void_p),
        ("status", C.c_void_p),
        ("nit", C.c_void_p),
        ("fun", C.c_void_p),
        ("dense", C.c_int32),
        ("status_count", C.c_int64 * 4),
        ("trace_f", C.c_void_p),
        ("trace_step", C.c_void_p),
        ("trace_len", C.c_void_p),
        ("trace_cap", C.c_int32),
        ("zero_fill_mask", C.c_void_p),
        ("n_dup", C.c_int32),
        ("dup_t2", C.c_void_p * MAX_DUP),
        ("dup_k", C.c_void_p * MAX_DUP),
        ("dup_sigma", C.c_void_p * MAX_DUP),
        ("dup_res", C.c_void_p * MAX_DUP),
        ("dup_status", C.c_void_p * MAX_DUP),
        ("counts_dev", C.c_void_p),
    ]


# every symbol include/t2fit.h declares: (name, restype, argtypes)
SYMBOLS = [
    ("t2fit_init", C.c_int, [C.c_int]),
    ("t2fit_shutdown", None, []),
    ("t2fit_last_error", C.c_char_p, []),
    ("t2fit_abi_version", C.c_int, []),
    ("t2fit_device_info", C.c_int, [C.c_char_p, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    ("t2fit_run", C.c_int, [C.POINTER(Problem), C.POINTER(Outputs), C.c_void_p]),
    ("t2fit_status_counts", C.c_int, [C.c_void_p, C.POINTER(C.c_int64)]),
    ("t2fit_mask_indices", C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.POINTER(C.c_int64), C.c_void_p]),
    ("t2fit_mask_union", C.c_int, [C.POINTER(C.c_void_p), C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_int64, C.c_void_p,
                                   C.c_void_p]),
    ("t2fit_host_mask_union_indices", C.c_int, [C.POINTER(C.c_void_p), C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_int64,
                                                C.c_void_p, C.c_void_p, C.POINTER(C.c_int64)]),
    ("t2fit_host_gather_planes", C.c_int, [C.POINTER(C.c_void_p), C.c_int32, C.c_int32, C.c_void_p, C.c_int64, C.c_int64,
                                           C.c_void_p, C.c_int64]),
    ("t2fit_roi_stats", C.c_int, [C.POINTER(C.c_void_p), C.c_int32, C.c_void_p, C.c_int64, C.c_int32, C.POINTER(C.c_double),
                                  C.POINTER(C.c_double), C.POINTER(C.c_int64), C.c_void_p]),
    ("t2fit_shared_alloc", C.c_int, [C.c_int64, C.POINTER(C.c_void_p), C.c_char_p]),
    ("t2fit_shared_free", C.c_int, [C.c_void_p]),
    ("t2fit_shared_open", C.c_int, [C.c_char_p, C.POINTER(C.c_void_p)]),
    ("t2fit_shared_close", C.c_int, [C.c_void_p]),
    ("t2fit_pack_soa", C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64,
                                 C.c_void_p]),
    ("t2fit_scatter", C.c_int, [C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_int32, C.c_void_p, C.c_int64,
                                C.c_void_p]),
    ("t2fit_residuals", C.c_int, [C.POINTER(Problem), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    ("t2fit_stderr", C.c_int, [C.POINTER(Problem), C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p,
                               C.c_void_p, C.c_void_p]),
    ("t2fit_t2_interval", C.c_int, [C.POINTER(Problem), C.c_double, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    ("t2fit_bootstrap_replicates", C.c_int, [C.POINTER(Problem), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                             C.c_uint64, C.c_int32, C.c_void_p, C.c_void_p]),
    ("t2fit_bootstrap_stats", C.c_int, [C.c_int32, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_double] + [C.c_void_p] * 7),
    ("t2fit_work_model", C.c_int, [C.c_int32, C.c_int32] + [C.POINTER(C.c_double)] * 5),
]

# T2FIT_LIB: developer knob, another build of the same library (e.g. an occupancy variant under measurement)
LIB_PATH = os.environ.get("T2FIT_LIB") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "csrc", "libt2fit.so")

_lib = None


class T2FitError(RuntimeError):
    pass


def load_library(path: str | None = None):
    """dlopen libt2fit.so and bind every declared symbol.  Raises if the library is not built."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or LIB_PATH
    if not os.path.isfile(p):
        raise T2FitError(f"{p} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                         "(nvcc, sm_100a).  There is no CPU fallback for the fit.")
    lib = C.CDLL(p)
    for name, restype, argtypes in SYMBOLS:
        fn = getattr(lib, name)            # AttributeError if the export is missing
        fn.restype = restype
        fn.argtypes = argtypes
    if lib.t2fit_abi_version() != ABI_VERSION:
        raise T2FitError("libt2fit ABI version mismatch")
    if path is None:
        _lib = lib
    return lib


def check(lib, rc: int, what: str):
    if rc != 0:
        msg = lib.t2fit_last_error()
        raise T2FitError(f"{what}: {ERRORS.get(rc, rc)}: {msg.decode() if msg else ''}")
