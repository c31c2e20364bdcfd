"""Build + call the host simulation of the solver core (TEST TOOL ONLY, see hostsim.cpp)."""
import ctypes as C
import os
import subprocess

import numpy as np

from fetal_t2mapping_b200 import _abi

HERE = os.path.dirname(os.path.abspath(__file__))
SO = os.path.join(HERE, "libt2fit_hostsim.so")
SRC = os.path.join(HERE, "hostsim.cpp")
DEPS = [SRC] + [os.path.join(HERE, "..", "..", "fetal_t2mapping_b200", "csrc", f)
                for f in ("t2fit_core.cuh", "t2fit_consts.h", "t2fit_lbfgsb.cuh", "t2fit_lbfgsb_coop.cuh", "t2fit_lbfgsb_dense.cuh", "t2fit_i0e_coeffs.h")] + \
    [os.path.join(HERE, "lane_emu.h")] + [os.path.join(HERE, "..", "..", "include", "t2fit.h")]


SO_STRICT = os.path.join(HERE, "libt2fit_hostsim_strict.so")


def compile_so(src, so, deps, force=False, strict=False):
    """g++ ``src`` into the shared library ``so`` unless it is newer than every file of ``deps``.
    strict=False: -mfma + contraction, as the device fuses a*b+c (cancellation noise, e.g. D - k*C at a converged point,
    is then as small on the host simulation as on the GPU).  strict=True: no contraction at all -- every product and sum
    rounds separately whatever the expression shape, so two implementations that perform the same operations in the same
    order agree BIT FOR BIT (the serial and the cooperative L-BFGS-B solver, tests/test_hostsim_coop.py)."""
    if not force and os.path.isfile(so) and all(os.path.getmtime(so) >= os.path.getmtime(d) for d in deps):
        return so
    fp = ["-ffp-contract=off"] if strict else ["-mfma", "-ffp-contract=fast"]
    tmp = f"{so[:-3]}.{os.getpid()}.tmp.so"
    cmd = ["g++", "-O2", "-std=c++17"] + fp + ["-shared", "-fPIC", "-x", "c++", src, "-o", tmp, "-lm"]
    subprocess.run(cmd, check=True, cwd=HERE)
    os.replace(tmp, so)    # test processes that build at once (the ranks of a distributed test) never load a partial file
    return so


def build(force=False, strict=False):
    return compile_so(SRC, SO_STRICT if strict else SO, DEPS, force, strict)


_libs = {}


def lib(strict=False):
    if strict not in _libs:
        l = C.CDLL(build(strict=strict))
        l.hostsim_fit.restype = C.c_int
        l.hostsim_last_error.restype = C.c_char_p
        l.hostsim_lbfgsb.restype = C.c_int
        l.hostsim_lbfgsb_coop.restype = C.c_int
        l.hostsim_lbfgsb_dense.restype = C.c_int
        l.hostsim_i0e.restype = C.c_double
        l.hostsim_i0e.argtypes = [C.c_double]
        _libs[strict] = l
    return _libs[strict]


def make_problem(rows, te, fit, x0, bounds, prior, norm, max_iter=0, tol=0.0, init=0, options=None):
    rows = np.ascontiguousarray(rows, np.float32)
    te = np.ascontiguousarray(te, np.float64)
    p = _abi.Problem()
    p.echoes = rows.ctypes.data
    p.layout = _abi.LAYOUT_AOS
    p.memory = _abi.MEM_HOST
    p.n_vox = rows.shape[0]
    p.n_fit = rows.shape[0]
    p.n_echo = rows.shape[1]
    p.model = _abi.MODELS[fit]
    p.te_ms = te.ctypes.data_as(C.POINTER(C.c_double))
    for i in range(len(x0)):
        p.x0[i] = float(x0[i])
        p.lb[i] = float(bounds[i][0])
        p.ub[i] = float(bounds[i][1])
    p.no_prior = 0 if prior else 1
    p.no_prior_k_ub, p.no_prior_t2_lb, p.no_prior_t2_ub = 10000.0, 10.0, 2000.0
    p.norm = int(bool(norm))
    p.max_iter = max_iter
    p.tol = tol
    p.init = init
    if options is not None:
        p.solver = _abi.SOLVER_LBFGSB
        p.lbfgsb_ftol = float(options.get("ftol", 0.0))
        p.lbfgsb_gtol = float(options.get("gtol", 0.0))
        p.lbfgsb_maxls = int(options.get("maxls", 0))
        p.lbfgsb_maxiter = int(options.get("maxiter", 0))
        p.lbfgsb_maxfun = int(options.get("maxfun", 0))
    return p, (rows, te)


def fit(rows, te, fit, x0, bounds, prior, norm=False, use_double=False, **kw):
    p, keep = make_problem(rows, te, fit, x0, bounds, prior, norm, **kw)
    m = keep[0].shape[0]
    out = {n: np.zeros(m, np.float32) for n in ("k", "t2", "sigma", "res", "fun")}
    out["nit"] = np.zeros(m, np.int32)
    out["status"] = np.zeros(m, np.uint8)
    rc = lib().hostsim_fit(C.byref(p), int(use_double), *[out[n].ctypes.data_as(C.c_void_p) for n in
                                                         ("k", "t2", "sigma", "res", "fun", "nit", "status")])
    if rc:
        raise ValueError(lib().hostsim_last_error().decode())
    return out


def lbfgsb(rows, te, fit, x0, bounds, prior, norm=False, options=None, trace_cap=0, tol=0.0, strict=False, coop_lanes=0,
           reverse=False, dense=False):
    """The reference-faithful solver compiled for the host: the serial form (csrc/t2fit_lbfgsb.cuh) or, with
    ``coop_lanes`` = 4 / 8 / 16 / 32, the cooperative form (csrc/t2fit_lbfgsb_coop.cuh) on the lane emulator."""
    p, keep = make_problem(rows, te, fit, x0, bounds, prior, norm, options=options or {}, tol=tol)
    m = keep[0].shape[0]
    out = {"x": np.zeros((m, 3), np.float64), "fun": np.zeros(m, np.float64), "nit": np.zeros(m, np.int32),
           "nfev": np.zeros(m, np.int32), "status": np.zeros(m, np.uint8), "result": np.zeros(m, np.int32)}
    tf = np.full((m, max(trace_cap, 1)), np.nan, np.float32)
    ts = np.full((m, max(trace_cap, 1)), np.nan, np.float32)
    tl = np.zeros(m, np.int32)
    vp = lambda a: a.ctypes.data_as(C.c_void_p)
    args = (vp(out["x"]), vp(out["fun"]), vp(out["nit"]), vp(out["nfev"]), vp(out["status"]), vp(out["result"]),
            vp(tf) if trace_cap else None, vp(ts) if trace_cap else None, vp(tl), C.c_int(trace_cap))
    L = lib(strict)
    if dense:
        rc = L.hostsim_lbfgsb_dense(C.byref(p), *args)
    elif coop_lanes:
        rc = L.hostsim_lbfgsb_coop(C.byref(p), C.c_int(coop_lanes), C.c_int(int(reverse)), *args)
    else:
        rc = L.hostsim_lbfgsb(C.byref(p), *args)
    if rc:
        raise ValueError(L.hostsim_last_error().decode())
    out["trace_f"], out["trace_step"], out["trace_len"] = tf, ts, tl
    return out
