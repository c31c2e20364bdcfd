"""Host-side mirror of the reference's fit block, over the libt2fit C ABI.

Drop-in for the call pair inside ``process_t2maps`` (run_t2mapping.py:430-461)::

    all_results = pool.map(partial(fit_voxel, fit=, fit_params=, TEeffs=, reshaped_t2w=, prior=, norm=), mask_indices)
    res_map     = compute_residuals(reshaped_t2w, TEeffs, fit, norm, k_map, t2_map, sigma_map, res_map, mask_indices, mask)

``fit_voxels_batch`` takes exactly those arguments (same names, same meaning) and returns the
same information for every masked voxel at once; ``t2map_volume`` wraps the whole hot block
(mask union, flatten, fit, scatter, residual map; :383-386, :411-461, :471-473).

numpy arrays are treated as host memory (the library stages them through pinned buffers);
torch CUDA tensors are treated as device memory (zero-copy, asynchronous on the current torch
stream).  The fit itself only exists as sm_100a CUDA kernels: without the built library or
without a GPU these functions raise.
"""
from __future__ import annotations

import ctypes as C
import os
from collections import namedtuple
from dataclasses import dataclass

import numpy as np

from . import _abi
from .presets import NO_PRIOR_K_UB, NO_PRIOR_T2_BOUNDS

__all__ = ["fit_voxels_batch", "fit_voxels_into", "check_counts", "t2map_volume", "compute_residuals", "parameter_stderr", "t2_interval", "FitResult", "init",
           "parametric_bootstrap", "BootstrapResult", "BootstrapMaps", "shutdown", "device_info", "mask_indices_device",
           "work_model", "pinned_array", "BOUNDS_ERROR"]

BOUNDS_ERROR = "An upper bound is less than the corresponding lower bound."   # scipy's text

_state = {"device": None}


def init(device: int | None = None):
    """Bind this process to one GPU (default: LOCAL_RANK, else torch's current device, else 0)."""
    lib = _abi.load_library()
    if device is None:
        if _state["device"] is not None:
            return lib
        device = int(os.environ.get("LOCAL_RANK", "0"))
    if _state["device"] == device:
        return lib
    # one process per GPU: share the host cores between the ranks of this node for the staging threads of the host path
    lws = int(os.environ.get("LOCAL_WORLD_SIZE", "1") or 1)
    if lws > 1 and "T2FIT_HOST_THREADS" not in os.environ:
        ncpu = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
        os.environ["T2FIT_HOST_THREADS"] = str(max(2, min(16, ncpu // lws)))
    _abi.check(lib, lib.t2fit_init(int(device)), "t2fit_init")
    _state["device"] = int(device)
    return lib


def shutdown():
    if _state["device"] is not None:
        _abi.load_library().t2fit_shutdown()
        _state["device"] = None


def device_info():
    lib = init()
    name = C.create_string_buffer(256)
    sm, maj, mnr = C.c_int(), C.c_int(), C.c_int()
    _abi.check(lib, lib.t2fit_device_info(name, 256, C.byref(sm), C.byref(maj), C.byref(mnr)), "t2fit_device_info")
    return {"name": name.value.decode(), "sm_count": sm.value, "cc": (maj.value, mnr.value), "device": _state["device"]}


def work_model(fit: str, n_echo: int):
    """Algorithmic work of the shipped kernel per voxel (roofline accounting, DESIGN.md)."""
    lib = _abi.load_library()
    v = [C.c_double() for _ in range(5)]
    _abi.check(lib, lib.t2fit_work_model(_abi.MODELS[fit], n_echo, *[C.byref(x) for x in v]), "t2fit_work_model")
    keys = ("flop_per_pass", "mufu_per_pass", "flop_fixed", "mufu_fixed", "bytes_per_voxel")
    return {k: x.value for k, x in zip(keys, v)}


def _host_echoes(y, p):
    """The host echo array as the library takes it.  The reference casts the whole volume (`.astype(np.float32)`,
    run_t2mapping.py:411); a C-contiguous int16 / uint16 / int32 / float64 array -- what the NIfTI reader returns -- is
    passed as it is instead and cast by the library while it gathers the masked rows (t2fit_problem.echo_dtype)."""
    code = _abi.ECHO_DTYPES.get(y.dtype.name)
    if code is None or not y.flags.c_contiguous:
        y = np.ascontiguousarray(y, dtype=np.float32)
        code = 0
    p.echo_dtype = code
    return y


def _is_torch(x):
    return type(x).__module__.startswith("torch")


def pinned_array(shape, dtype=np.float32, like=None):
    """A numpy array in page-locked host memory (backed by a torch pinned tensor that lives as long as the array).
    ``like``: copy this array into it.  When ``reshaped_t2w`` (and optionally ``mask_indices``) handed to
    :func:`fit_voxels_batch` are page-locked, the call needs no staging: the kernel gathers the masked rows straight
    from host memory over PCIe and stores the results straight back (``run_host_mapped`` in csrc/t2fit_kernels.cu)."""
    import torch
    if like is not None:
        like = np.asarray(like)
        shape, dtype = like.shape, like.dtype
    t = torch.empty(tuple(np.atleast_1d(shape)) if not isinstance(shape, tuple) else shape,
                    dtype=getattr(torch, np.dtype(dtype).name), pin_memory=True)
    a = t.numpy()
    if like is not None:
        np.copyto(a, like)
    return a


def _host_block(m, fields):
    """All result arrays of one call as views into ONE page-locked block (one pinned allocation / DMA mapping instead
    of one per field).  ``fields``: list of (name, dtype).  Falls back to plain numpy without torch."""
    offs, total = {}, 0
    for name, dt in fields:
        total = (total + 255) // 256 * 256                       # 256-byte aligned views (vector stores, cache lines)
        offs[name] = total
        total += m * np.dtype(dt).itemsize
    try:
        import torch
        base = torch.empty(max(total, 1), dtype=torch.uint8, pin_memory=True).numpy()
    except Exception:
        base = np.empty(max(total, 1), np.uint8)
    return {name: base[offs[name]:offs[name] + m * np.dtype(dt).itemsize].view(dt) for name, dt in fields}


@dataclass
class FitResult:
    """Everything ``pool.map(fit_voxel)`` + ``compute_residuals`` produce, for all masked voxels.

    ``results``            f64[M,P] in the reference order (k, T2[, sigma])       (:449)
    ``convergence_flags``  bool[M]   == ``result.success``                        (:450)
    ``num_iterations``     int32[M]  passes of the CUDA solver (not L-BFGS-B's)   (:451)
    ``final_errors``       f64[M]    mean squared error at the solution           (:452)
    ``res``                f32[M]    signed mean residual (compute_residuals)     (:461)
    ``status``             uint8[M]  0 ok / 1 non-finite input / 2 iteration cap / 3 bad bounds
    ``iteration_infos``    the callback traces (:180-234) when the call asked for them (``trace_cap``,
                           L-BFGS-B solver), else ``[]`` per voxel
    ``se_k``, ``se_t2``, ``se_sigma``  f32[M] standard errors of the parameters (``want`` with "se"; see
                           :func:`parameter_stderr`), else None; ``standard_errors`` stacks them as ``results`` does
    For device calls the float fields are torch CUDA tensors (float32).
    """
    t2: object
    k: object
    _sigma: object
    res: object
    fun: object
    nit: object
    status: object
    fit: str
    status_count: tuple = (0, 0, 0, 0)
    solver: str = "fast"
    trace_f: object = None       # float32[M, trace_cap]  f_val per L-BFGS-B iteration
    trace_step: object = None    # float32[M, trace_cap]  step_size (NaN for the first iteration)
    trace_len: object = None     # int32[M]               entries used = min(nit, trace_cap)
    se_k: object = None          # float32[M]             standard errors (want "se"); se_sigma None for gaussian
    se_t2: object = None
    se_sigma: object = None

    @property
    def sigma(self):
        """sigma_map values; all zeros for the 2-parameter fit (run_t2mapping.py:417,457-458), created on first use."""
        if self._sigma is None:
            self._sigma = np.zeros(self.t2.shape[0], np.float32)
        return self._sigma

    @property
    def iteration_infos(self):
        """``iteration_info`` of every voxel as the reference's callbacks build it (run_t2mapping.py:180-234):
        a list of ``{'f_val', 'grad_norm': None, 'step_size'}`` per L-BFGS-B iteration."""
        m = int(self.nit.shape[0]) if self.nit is not None else int(self.t2.shape[0])
        if self.trace_len is None:
            return [[] for _ in range(m)]
        tn = np.asarray(self.trace_len.cpu() if _is_torch(self.trace_len) else self.trace_len)
        tf = np.asarray(self.trace_f.cpu() if _is_torch(self.trace_f) else self.trace_f)
        ts = np.asarray(self.trace_step.cpu() if _is_torch(self.trace_step) else self.trace_step)
        return [[{"f_val": float(tf[i, j]), "grad_norm": None, "step_size": float(ts[i, j])} for j in range(tn[i])]
                for i in range(m)]

    @property
    def results(self):
        cols = [self.k, self.t2] + ([self.sigma] if self.fit != "gaussian" else [])
        if _is_torch(self.k):
            import torch
            return torch.stack(cols, dim=1).double()
        return np.stack(cols, axis=1).astype(np.float64)

    @property
    def standard_errors(self):
        """f64[M,P] standard errors in the order of ``results`` (k, T2[, sigma]); None unless the call asked for "se"."""
        if self.se_t2 is None:
            return None
        cols = [self.se_k, self.se_t2] + ([self.se_sigma] if self.fit != "gaussian" else [])
        if _is_torch(self.se_t2):
            import torch
            return torch.stack(cols, dim=1).double()
        return np.stack(cols, axis=1).astype(np.float64)

    @property
    def convergence_flags(self):
        return self.status == 0

    @property
    def num_iterations(self):
        return self.nit

    @property
    def final_errors(self):
        return self.fun.double() if _is_torch(self.fun) else self.fun.astype(np.float64)

    def as_all_results(self):
        """The list ``pool.map`` returned: one ``(params, success, nit, fun, iteration_info)`` per voxel."""
        r = self.results.cpu().numpy() if _is_torch(self.k) else self.results
        ok = np.asarray(self.convergence_flags.cpu() if _is_torch(self.status) else self.convergence_flags)
        nit = np.asarray(self.nit.cpu() if _is_torch(self.nit) else self.nit)
        fun = np.asarray(self.final_errors.cpu() if _is_torch(self.fun) else self.final_errors)
        infos = self.iteration_infos
        return [(r[i], bool(ok[i]), int(nit[i]), float(fun[i]), infos[i]) for i in range(r.shape[0])]


def _device_counts(torch, device):
    """[4] zeroed int64 device counters for ONE device-memory call (t2fit_outputs.counts_dev): slot 0 = mask indices out
    of range, 1..3 = voxels per non-OK status.  Every call of the mirror owns its counters, so nothing leaks between calls
    or streams."""
    return torch.zeros(4, dtype=torch.int64, device=device)


def _raise_for_counts(cnt):
    """What the reference does for such voxels: numpy's fancy indexing raises IndexError for an index outside the array,
    scipy raises ValueError for lb > ub inside the first such voxel and pool.map aborts the whole map."""
    if cnt[0] > 0:
        raise IndexError("mask_indices out of range")
    if cnt[3] > 0:
        raise ValueError(BOUNDS_ERROR)


def resolve_solver(fit, solver):
    """``auto``: the float32 Newton/LM kernels for 'gaussian' (they reach the bounded minimiser the reference's
    ftol=1e-6 run approaches); the reference's own optimiser (L-BFGS-B restated in FP64) for 'gaussian_rician' and
    'rician', whose presets stop at ftol=gtol=1e-2, far from any minimiser -- only the same trajectory gives the
    same maps there.  Of its two forms 'auto' takes 'lbfgsb_dense' (the limited-memory matrix as the n x n matrix it
    represents: same parity with the reference on every golden fixture, 5-15x the throughput); 'lbfgsb' is scipy's
    compact 2m x 2m form restated operation by operation."""
    if solver == "auto":
        return "fast" if fit == "gaussian" else "lbfgsb_dense"
    if solver not in _abi.SOLVERS:
        raise ValueError(f"unknown solver {solver!r}")
    if solver == "fast" and fit == "rician":
        raise ValueError("fit='rician' is a negative log-likelihood, not least squares: use solver='lbfgsb_dense' or 'lbfgsb'")
    return solver


def _fill_problem(p, fit, fit_params, TEeffs, prior, norm, max_iter, tol, init_mode, solver="fast"):
    if fit not in _abi.MODELS:
        raise ValueError(f"unknown fit {fit!r}")
    p.solver = _abi.SOLVERS[solver]
    if solver in ("lbfgsb", "lbfgsb_dense"):   # fit_params['options'] as handed to scipy.optimize.minimize (:260-286)
        opt = dict(fit_params.get("options") or {})
        p.lbfgsb_ftol = float(opt.get("ftol", 0.0))
        p.lbfgsb_gtol = float(opt.get("gtol", 0.0))
        p.lbfgsb_maxls = int(opt.get("maxls", 0))
        p.lbfgsb_maxiter = int(opt.get("maxiter", 0))
        p.lbfgsb_maxfun = int(opt.get("maxfun", 0))
    x0 = list(fit_params["initial_guess"])
    bounds = list(fit_params["param_bounds"])
    npar = 2 if fit == "gaussian" else 3
    if len(x0) != npar:
        raise ValueError(f"fit {fit!r} takes {npar} parameters, initial_guess has {len(x0)}")
    if len(bounds) != len(x0):
        raise ValueError("The number of bounds is not compatible with the length of `x0`.")   # scipy's text
    te = np.ascontiguousarray(np.asarray(TEeffs, dtype=np.float64).reshape(-1))
    p.n_echo = te.size
    p.te_ms = te.ctypes.data_as(C.POINTER(C.c_double))
    p.model = _abi.MODELS[fit]
    for i in range(npar):
        lo, hi = bounds[i]
        p.x0[i] = float(x0[i])
        p.lb[i] = -np.inf if lo is None else float(lo)
        p.ub[i] = np.inf if hi is None else float(hi)
    p.no_prior = 0 if prior else 1
    p.no_prior_k_ub = NO_PRIOR_K_UB
    p.no_prior_t2_lb, p.no_prior_t2_ub = NO_PRIOR_T2_BOUNDS
    p.norm = int(bool(norm))
    p.max_iter = int(max_iter)
    p.tol = float(tol)
    if init_mode == "auto":                # 3-parameter fast solver: multi-start (several local minima); 2-parameter: log-linear
        init_mode = "best" if fit != "gaussian" else "loglinear"
    p.init = {"loglinear": _abi.INIT_LOGLINEAR, "preset": _abi.INIT_PRESET, "best": _abi.INIT_BEST}[init_mode]
    return te      # keep alive


def _run(lib, p, o, stream):
    rc = lib.t2fit_run(C.byref(p), C.byref(o), stream)
    if rc != 0:
        msg = (lib.t2fit_last_error() or b"").decode()
        if rc == -1 and "upper bound" in msg:
            raise ValueError(msg)
        if rc == -1 and "mask_idx out of range" in msg:
            raise IndexError("mask_indices out of range")
        raise _abi.T2FitError(f"t2fit_run: {_abi.ERRORS.get(rc, rc)}: {msg}")


def _stderr_launch(lib, p, fit, params, dense, se, stream):
    """t2fit_stderr on the echoes / indices / sizes already in ``p`` (device AoS): ``params`` (k, t2, sigma) and ``se``
    (se_k, se_t2, se_sigma) are device addresses or None."""
    k, t2, sg = params
    _abi.check(lib, lib.t2fit_stderr(C.byref(p), k, t2, sg if fit != "gaussian" else None, int(dense), *se, stream),
               "t2fit_stderr")


def _stderr_pass(lib, p, fit, k, t2, sigma, dense):
    """t2fit_stderr on the device rows of ``p`` at the float32 device parameters ``k``, ``t2``, ``sigma`` (None for
    'gaussian'), on the current stream of their GPU.  Returns float32 [3, n] (se_k, se_t2, se_sigma): n = p.n_vox, zeros
    off the index, when ``dense``, else n = p.n_fit with se_sigma unset for 'gaussian'."""
    import torch
    se = (torch.zeros if dense else torch.empty)((3, p.n_vox if dense else p.n_fit), dtype=torch.float32, device=k.device)
    _stderr_launch(lib, p, fit, [k.data_ptr(), t2.data_ptr(), sigma.data_ptr() if sigma is not None else None], dense,
                   [se[i].data_ptr() for i in range(3)], torch.cuda.current_stream(k.device).cuda_stream)
    return se


def _staged(p, rows, *params):
    """Host input for a device pass: a copy of ``p`` that reads ``rows`` [M, E], copied to the bound GPU, without an
    index (rows 0..M-1, so dense and compact output slots coincide), and the device tensors [rows, *params], each per-row
    array of ``params`` copied as float32 (None stays None).  The tensors must stay alive for the pass."""
    import torch
    dev = torch.device("cuda", _state["device"])
    y = torch.from_numpy(np.ascontiguousarray(rows, dtype=np.float32)).to(dev)
    q = _abi.Problem.from_buffer_copy(p)
    q.echoes, q.memory, q.layout, q.mask_idx, q.idx_dtype = y.data_ptr(), _abi.MEM_DEVICE, _abi.LAYOUT_AOS, None, _abi.IDX_I64
    q.n_vox, q.n_fit, q.ld = y.shape[0], y.shape[0], 0
    return q, [y] + [torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(dev) if a is not None else None
                     for a in params]


def _interval_q(fit, n_echo, level):
    """The quantile q of t2fit_t2_interval for a confidence level: t^2_{E-P}(1 - alpha/2) for the least-squares fits (the
    profile-t interval), chi^2_1(level) for 'rician' (the likelihood ratio).  E <= P leaves no residual degrees of freedom:
    every voxel is invalid then, and q is only a placeholder."""
    from scipy import stats
    if not 0.0 < float(level) < 1.0:
        raise ValueError("level must lie in (0, 1)")
    if fit == "rician":
        return float(stats.chi2.ppf(level, 1))
    dof = n_echo - (2 if fit == "gaussian" else 3)
    return float(stats.t.ppf(0.5 + 0.5 * level, dof) ** 2) if dof > 0 else 0.0


def interval_grid(t2_lo, t2_hi, n_grid=64):
    """The T2 grid of the interval pass: ``T2_g = t2_lo (t2_hi / t2_lo)^(g / (n_grid - 1))``, both bounds included."""
    t = t2_lo * np.power(t2_hi / t2_lo, np.arange(n_grid, dtype=np.float64) / (n_grid - 1))
    t[-1] = t2_hi
    return t


def _interval_launch(lib, p, q, n_grid, dense, outs, profile, stream):
    """t2fit_t2_interval on the echoes / indices / sizes already in ``p`` (device AoS): ``outs`` (lo, hi, best, flags) and
    ``profile`` are device addresses or None."""
    _abi.check(lib, lib.t2fit_t2_interval(C.byref(p), q, int(n_grid), int(dense), *outs, profile, stream), "t2fit_t2_interval")


def _interval_pass(lib, p, q, n_grid, profile):
    """t2fit_t2_interval on the device rows of ``p`` on the current stream of the bound GPU, compact.  Returns (f, flags,
    prof): f float32 [3, p.n_fit] (lo, hi, best), flags uint8 [p.n_fit] and with ``profile`` p at the grid, float64
    [p.n_fit, n_grid], else None."""
    import torch
    device = torch.device("cuda", _state["device"])
    f = torch.empty((3, p.n_fit), dtype=torch.float32, device=device)
    fl = torch.empty(p.n_fit, dtype=torch.uint8, device=device)
    pr = torch.empty((p.n_fit, n_grid), dtype=torch.float64, device=device) if profile else None
    _interval_launch(lib, p, q, n_grid, 0, [f[0].data_ptr(), f[1].data_ptr(), f[2].data_ptr(), fl.data_ptr()],
                     pr.data_ptr() if pr is not None else None, torch.cuda.current_stream(device).cuda_stream)
    return f, fl, pr


def _device_rows(p, reshaped_t2w, mask_indices):
    """Points ``p`` at device echo rows: ``reshaped_t2w`` must be a contiguous float32 CUDA tensor [N, p.n_echo] on the
    bound GPU.  ``mask_indices`` (numpy or torch on any device; None = every row) is brought to that GPU, int32 kept as
    int32 (half the index bytes), anything else as contiguous int64.  Returns the index tensor, which must stay alive for
    the call."""
    import torch
    y = reshaped_t2w
    if not (_is_torch(y) and y.is_cuda and y.dtype == torch.float32 and y.is_contiguous() and y.dim() == 2):
        raise ValueError("device input must be a contiguous float32 CUDA tensor [N, E]")
    if y.device.index != _state["device"]:
        raise ValueError(f"tensor on cuda:{y.device.index}, library bound to cuda:{_state['device']}")
    if y.shape[1] != p.n_echo:
        raise ValueError(f"reshaped_t2w has {y.shape[1]} echoes, TEeffs has {p.n_echo}")
    idx = mask_indices
    if idx is not None:
        if not _is_torch(idx):
            idx = np.asarray(idx)
            idx = torch.as_tensor(np.ascontiguousarray(idx, dtype=np.int32 if idx.dtype == np.int32 else np.int64), device=y.device)
        idx = idx.to(device=y.device, dtype=torch.int32 if idx.dtype == torch.int32 else torch.int64).contiguous()
        p.idx_dtype = _abi.IDX_I32 if idx.dtype == torch.int32 else _abi.IDX_I64
    p.echoes, p.memory, p.layout, p.ld = y.data_ptr(), _abi.MEM_DEVICE, _abi.LAYOUT_AOS, 0
    p.mask_idx = idx.data_ptr() if idx is not None else None
    p.n_vox, p.n_fit = y.shape[0], (y.shape[0] if idx is None else idx.numel())
    return idx


def _pass_input(p, reshaped_t2w, mask_indices, *params):
    """The input of a pass over the voxels ``mask_indices`` (None = every row) of ``reshaped_t2w`` [N, E] for a problem ``p``
    that :func:`_fill_problem` filled.  Returns (q, params, ids, fin, keep): ``q`` the device problem the pass entries read;
    each per-voxel array of ``params`` as a contiguous float32 CUDA tensor [M] (None stays None); ``ids`` the int64 flat
    voxel ids of q's rows (numpy) when q reads staged rows, None when it reads the echoes through the index; ``fin`` turns a
    device result into what the caller returns (numpy for host input); ``keep`` must stay alive for the pass.  A CUDA tensor
    is taken as :func:`_device_rows` takes it.  Host input: an index outside [0, N) raises IndexError, as in the fit; the
    masked rows and the params are staged once (:func:`_staged`)."""
    import torch
    if _is_torch(reshaped_t2w):
        idx = _device_rows(p, reshaped_t2w, mask_indices)
        dev = reshaped_t2w.device
        to_dev = lambda a: (a if _is_torch(a) else torch.from_numpy(np.ascontiguousarray(a))).to(
            device=dev, dtype=torch.float32).reshape(-1).contiguous()
        return p, [to_dev(a) if a is not None else None for a in params], None, (lambda t: t), [idx]
    y = np.asarray(reshaped_t2w)
    if y.ndim != 2 or y.shape[1] != p.n_echo:
        raise ValueError(f"reshaped_t2w must be [N, {p.n_echo}]")
    ids = np.arange(y.shape[0], dtype=np.int64) if mask_indices is None else np.asarray(mask_indices).astype(np.int64)
    if ids.size and (ids.min() < 0 or ids.max() >= y.shape[0]):
        raise IndexError("mask_indices out of range")
    host = lambda a: a.cpu().numpy() if _is_torch(a) else a
    q, (ys, *par) = _staged(p, y if mask_indices is None else y[ids], *[host(a) if a is not None else None for a in params])
    return q, par, ids, (lambda t: t.cpu().numpy() if t is not None else None), [ys]


def _scatter(vals, idx, n_vox):
    """Compact values [..., M] of a pass (a CUDA tensor) for the flat voxels ``idx`` as [..., n_vox] of their dtype, zeros
    elsewhere: a CUDA tensor for a CUDA ``idx``, else a numpy array."""
    if _is_torch(idx):
        import torch
        return torch.zeros(tuple(vals.shape[:-1]) + (n_vox,), dtype=vals.dtype, device=vals.device).index_copy_(
            vals.dim() - 1, idx, vals)
    v = vals.cpu().numpy()
    a = np.zeros(v.shape[:-1] + (n_vox,), dtype=v.dtype)
    a[..., idx] = v
    return a


def fit_voxels_batch(reshaped_t2w, mask_indices, TEeffs, fit, fit_params, prior=True, norm=False, *,
                     solver="auto", trace_cap=0, max_iter=0, tol=0.0, init_mode="auto", check_bounds=True,
                     dense_out=None, want=("nit", "fun", "status")) -> FitResult:
    """Fit every voxel ``mask_indices[i]`` of ``reshaped_t2w`` (float32 ``[N, E]``, run_t2mapping.py:411).

    Arguments as ``fit_voxel`` (run_t2mapping.py:120): ``fit`` in {'gaussian','gaussian_rician','rician'},
    ``fit_params`` the preset dict (``initial_guess``, ``param_bounds``, ``options``), ``prior`` False =
    ``--no_prior`` per-voxel bounds (:243-245), ``norm`` row-max normalisation (:237-240).
    ``mask_indices`` None fits all rows.  Raises ``ValueError`` where scipy would (bounds with
    lb > ub, including any masked voxel with S(TE0) > 10000 under ``--no_prior``).
    ``solver``: 'fast' | 'lbfgsb_dense' | 'lbfgsb' | 'auto' (see :func:`resolve_solver`).  ``trace_cap`` > 0 (L-BFGS-B solver)
    also returns the callback trace of every fitted voxel (``FitResult.iteration_infos``) -- meant for the
    sampled voxels of the convergence plots (utils/t2map_utils.py:115-292), pass their indices only.
    ``want`` with "se": also the standard errors of the fitted parameters (``FitResult.se_*``, :func:`parameter_stderr`),
    computed by a second kernel on the same stream from the compact results; asynchronous for device inputs.
    """
    lib = init()
    solver = resolve_solver(fit, solver)
    p, o = _abi.Problem(), _abi.Outputs()
    keep = [_fill_problem(p, fit, fit_params, TEeffs, prior, norm, max_iter, tol, init_mode, solver)]
    tracing = solver in ("lbfgsb", "lbfgsb_dense") and trace_cap > 0
    dev = _is_torch(reshaped_t2w)
    if dev:
        import torch
        y = reshaped_t2w
        idx = _device_rows(p, y, mask_indices)
        m = p.n_fit

        def alloc(dt=torch.float32):
            return torch.empty(m, dtype=dt, device=y.device)
        out = {"t2": alloc(), "k": alloc(), "res": alloc(),
               "sigma": alloc() if fit != "gaussian" else torch.zeros(m, dtype=torch.float32, device=y.device),
               "fun": alloc() if "fun" in want else None,
               "nit": alloc(torch.int32) if "nit" in want else None,
               "status": alloc(torch.uint8) if "status" in want else None}
        if tracing:
            out["trace_f"] = torch.full((m, trace_cap), float("nan"), dtype=torch.float32, device=y.device)
            out["trace_step"] = torch.full((m, trace_cap), float("nan"), dtype=torch.float32, device=y.device)
            out["trace_len"] = torch.zeros(m, dtype=torch.int32, device=y.device)
        ptr = lambda t: t.data_ptr() if t is not None else None
        stream = torch.cuda.current_stream(y.device).cuda_stream
        dcnt = _device_counts(torch, y.device)
        o.counts_dev = dcnt.data_ptr()
        keep += [y, idx, dcnt]
    else:
        y = _host_echoes(np.asarray(reshaped_t2w), p)
        if y.ndim != 2:
            raise ValueError("reshaped_t2w must be [N, E]")
        n_vox, n_echo = y.shape
        if n_echo != p.n_echo:
            raise ValueError(f"reshaped_t2w has {n_echo} echoes, TEeffs has {p.n_echo}")
        idx = None
        if mask_indices is not None:               # int32 indices are taken as they are (half the index bytes over PCIe)
            idx = np.asarray(mask_indices)
            idx = np.ascontiguousarray(idx, dtype=np.int32 if idx.dtype == np.int32 else np.int64)
            p.idx_dtype = _abi.IDX_I32 if idx.dtype == np.int32 else _abi.IDX_I64
        m = n_vox if idx is None else idx.size
        fields = [("t2", np.float32), ("k", np.float32), ("res", np.float32)]
        fields += [("sigma", np.float32)] if fit != "gaussian" else []                  # 2-parameter fit: zeros, made on first access
        fields += [(n, dt) for n, dt in (("fun", np.float32), ("nit", np.int32), ("status", np.uint8)) if n in want]
        out = {"sigma": None, "fun": None, "nit": None, "status": None}
        out.update(_host_block(m, fields))
        if tracing:
            out["trace_f"] = np.full((m, trace_cap), np.nan, np.float32)
            out["trace_step"] = np.full((m, trace_cap), np.nan, np.float32)
            out["trace_len"] = np.zeros(m, np.int32)
        p.echoes, p.memory = y.ctypes.data, _abi.MEM_HOST
        p.mask_idx = idx.ctypes.data if idx is not None else None
        p.layout, p.ld, p.n_vox, p.n_fit = _abi.LAYOUT_AOS, 0, n_vox, m
        ptr = lambda a: a.ctypes.data if a is not None else None
        stream = None
        keep += [y, idx]
    if tracing:
        o.trace_f, o.trace_step, o.trace_len = ptr(out["trace_f"]), ptr(out["trace_step"]), ptr(out["trace_len"])
        o.trace_cap = int(trace_cap)
    o.t2, o.k, o.res = ptr(out["t2"]), ptr(out["k"]), ptr(out["res"])
    o.sigma = ptr(out["sigma"]) if fit != "gaussian" else None
    o.fun, o.nit, o.status = ptr(out["fun"]), ptr(out["nit"]), ptr(out["status"])
    o.dense = 0
    _run(lib, p, o, stream)
    se = (None, None, None)
    if "se" in want:
        ps, (k, t2, sg), _, fin, pin = _pass_input(p, y, idx, out["k"], out["t2"], out["sigma"])
        keep += pin
        se = fin(_stderr_pass(lib, ps, fit, k, t2, sg, False))
        se = (se[0], se[1], se[2] if fit != "gaussian" else None)
    if dev:
        counts = None
        if check_bounds:                           # one small D2H: waits for the call (check_bounds=False stays asynchronous)
            cnt = [int(v) for v in dcnt.cpu()]
            _raise_for_counts(cnt)
            counts = (m - cnt[1] - cnt[2] - cnt[3], cnt[1], cnt[2], cnt[3])
    else:
        counts = tuple(o.status_count)
        if counts[3] > 0:
            # scipy raises inside the first such voxel and the reference's pool.map aborts the whole map
            raise ValueError(BOUNDS_ERROR)
    return FitResult(out["t2"], out["k"], out["sigma"], out["res"], out["fun"], out["nit"], out["status"], fit,
                     counts if counts is not None else (0, 0, 0, 0), solver, out.get("trace_f"), out.get("trace_step"),
                     out.get("trace_len"), *se)


def fit_voxels_into(reshaped_t2w, mask_indices, TEeffs, fit, fit_params, prior, norm, out, *, solver="auto", counts=None,
                    init_mode="auto", max_iter=0, tol=0.0):
    """Device-memory fit whose compact results go to caller-given raw device pointers: ``out`` maps 't2', 'k', 'res'
    (and 'sigma' for the 3-parameter fits; optionally 'status', 'nit', 'fun') to integer addresses of arrays with room
    for ``len(mask_indices)`` elements -- local memory or a peer GPU's buffer mapped with ``t2fit_shared_open`` (the
    fused gather of ``distributed.fit_voxels_sharded``); an address may be None (that output is skipped).  Asynchronous on
    the current torch stream.  ``counts``: a zeroed int64 CUDA tensor [4] the call adds its histogram to (slot 0 indices
    out of range, 1..3 voxels per non-OK status); the caller reads it when it synchronises and raises as
    :func:`fit_voxels_batch` does (``check_counts``).  ``init_mode``, ``max_iter``, ``tol`` as in :func:`fit_voxels_batch`."""
    import torch
    lib = init()
    solver = resolve_solver(fit, solver)
    p, o = _abi.Problem(), _abi.Outputs()
    keep = [_fill_problem(p, fit, fit_params, TEeffs, prior, norm, max_iter, tol, init_mode, solver)]
    y = reshaped_t2w
    idx = _device_rows(p, y, mask_indices)
    if counts is None:
        counts = _device_counts(torch, y.device)           # never the per-process counters: nothing leaks into later calls
    o.counts_dev = counts.data_ptr()
    o.t2, o.k, o.res = out["t2"], out["k"], out["res"]
    o.sigma = out.get("sigma") if fit != "gaussian" else None
    o.status, o.nit, o.fun = out.get("status"), out.get("nit"), out.get("fun")
    o.dense = 0
    _run(lib, p, o, torch.cuda.current_stream(y.device).cuda_stream)
    keep += [y, idx, counts]
    return p.n_fit


def check_counts(counts):
    """Raise what the reference raises for the histogram of a device call (synchronises on the tensor)."""
    _raise_for_counts([int(v) for v in counts.cpu()])


def mask_indices_device(mask, n_masks=None):
    """``mask_indices`` of a device mask: union over the per-TE axis (``np.sum(mask, axis=3) > 0``,
    run_t2mapping.py:383-384) and ascending C-order compaction (:412,:421).  ``mask`` is a uint8/bool
    CUDA tensor ``[z,y,x]`` or ``[z,y,x,n_masks]``; returns an int64 CUDA tensor."""
    import torch
    lib = init()
    mk = mask
    if mk.dtype == torch.bool:
        mk = mk.view(torch.uint8)
    if mk.dtype != torch.uint8:
        mk = (mk > 0).view(torch.uint8)
    mk = mk.contiguous()
    nm = 1 if mk.dim() == 3 else mk.shape[-1]
    n_vox = mk.numel() // nm
    idx = torch.empty(n_vox, dtype=torch.int64, device=mk.device)
    n = C.c_int64()
    stream = torch.cuda.current_stream(mk.device).cuda_stream
    _abi.check(lib, lib.t2fit_mask_indices(mk.data_ptr(), n_vox, nm, idx.data_ptr(), C.byref(n), stream),
               "t2fit_mask_indices")
    return idx[:n.value]


def t2map_volume(t2w, mask, TEeffs, fit, fit_params, prior=True, norm=False, stderr=False, t2_interval=None, bootstrap=None,
                 **kw):
    """Stacked per-TE volumes ``t2w[z,y,x,E]``, mask ``[z,y,x]`` or per-TE masks ``[z,y,x,E]`` and the
    TE vector in; ``(t2_map, k_map, sigma_map, res_map)`` float32 ``[z,y,x]`` out, zeros off-mask --
    the whole hot block of ``process_t2maps`` (run_t2mapping.py:383-386, :411-461, :471-473).
    ``stderr=True`` adds a fifth element ``(se_t2_map, se_k_map, se_sigma_map)``: the standard errors of the fitted
    parameters (:func:`parameter_stderr`), float32 ``[z,y,x]``, zeros off-mask (se_sigma all zeros for 'gaussian').
    ``t2_interval=level`` (e.g. 0.95) appends ``(t2_lo_map, t2_hi_map, t2_best_map, flags_map)`` as the last element: the
    profile-likelihood confidence interval for T2 at that level (:func:`t2_interval`, default grid), float32 / uint8
    ``[z,y,x]``, zeros off-mask.  ``bootstrap=n_rep`` appends, after those, a :data:`BootstrapMaps` ``(t2_mean, t2_sd, t2_lo,
    t2_hi, k_sd, sigma_sd, n_used, n_ok)`` of ``[z,y,x]`` maps, zeros off-mask: the parametric bootstrap of the fitted maps
    (:func:`parametric_bootstrap` with level 0.95, seed 0 and the estimated noise level)."""
    lib = init()
    shape3 = tuple(t2w.shape[:3])
    n_echo = t2w.shape[-1]
    p, o = _abi.Problem(), _abi.Outputs()
    solver = resolve_solver(fit, kw.get("solver", "auto"))
    keep = [_fill_problem(p, fit, fit_params, TEeffs, prior, norm, kw.get("max_iter", 0), kw.get("tol", 0.0),
                          kw.get("init_mode", "auto"), solver)]
    q = _interval_q(fit, p.n_echo, t2_interval) if t2_interval is not None else None
    if bootstrap is not None:
        _bootstrap_args(bootstrap, 0.95)
    fused_mask = None
    if _is_torch(t2w):
        import torch
        y = t2w.reshape(-1, n_echo)
        if y.dtype != torch.float32:
            y = y.float()
        y = y.contiguous()
        mk = mask if mask.dim() == 3 else (mask != 0).any(dim=3)                       # :383-384
        mk = (mk if mk.dtype in (torch.bool, torch.uint8) else (mk != 0)).contiguous()
        mk = mk.view(torch.uint8) if mk.dtype == torch.bool else mk
        idx = mask_indices_device(mk)                                                   # :412,:421
        n_vox, m = y.shape[0], idx.numel()
        # the four maps are zero-filled by the fit launch itself (or zero_fill_kernel on a side stream), see t2fit.h (:415-418)
        maps = torch.empty((4, n_vox), dtype=torch.float32, device=y.device)
        fused_mask = mk.reshape(-1)
        p.echoes, p.memory, p.mask_idx = y.data_ptr(), _abi.MEM_DEVICE, idx.data_ptr()
        stream = torch.cuda.current_stream(y.device).cuda_stream
        mp = [maps[i].data_ptr() for i in range(4)]
        dcnt = _device_counts(torch, y.device)
        o.counts_dev = dcnt.data_ptr()
        keep += [y, idx, mk, dcnt]
    else:
        y = _host_echoes(np.reshape(np.asarray(t2w), (-1, n_echo)), p)                  # :411
        mk = np.asarray(mask)
        mk = (np.sum(mk, axis=3) > 0) if mk.ndim == 4 else (mk if mk.dtype == np.bool_ else mk > 0)    # :383-384
        idx = np.flatnonzero(mk.reshape(-1)).astype(np.int64, copy=False)               # :412,:421
        n_vox, m = y.shape[0], idx.size
        maps = np.zeros((4, n_vox), np.float32)                                         # :415-418
        p.echoes, p.memory, p.mask_idx = y.ctypes.data, _abi.MEM_HOST, idx.ctypes.data
        stream = None
        mp = [maps[i].ctypes.data for i in range(4)]
        keep += [y, idx]
    if n_echo != p.n_echo:
        raise ValueError(f"t2w has {n_echo} echoes, TEeffs has {p.n_echo}")
    p.layout, p.ld, p.n_vox, p.n_fit = _abi.LAYOUT_AOS, 0, n_vox, m
    o.t2, o.k, o.res = mp[0], mp[1], mp[3]
    o.sigma = mp[2] if (fit != "gaussian" or fused_mask is not None) else None
    o.dense = 1
    if fused_mask is not None:
        o.zero_fill_mask = fused_mask.data_ptr()
    _run(lib, p, o, stream)
    if stream is not None:
        _raise_for_counts([int(v) for v in dcnt.cpu()])
    elif o.status_count[3] > 0:
        raise ValueError(BOUNDS_ERROR)
    out = tuple(maps[i].reshape(shape3) for i in range(4))
    if not stderr and t2_interval is None and bootstrap is None:
        return out
    import torch
    # every pass runs compact over the masked voxels, on the fitted problem (device input) or on the masked rows staged once
    if stream is not None:
        ps, (t2, k, sg) = p, maps[:3].index_select(1, idx)
    else:
        ps, (ys, t2, k, sg) = _staged(p, y[idx], *maps[:3, idx])
        keep.append(ys)
    put = lambda t: _scatter(t, idx, n_vox)
    if stderr:                                     # (k, t2, sigma) rows of the pass, (t2, k, sigma) maps out
        se = _stderr_pass(lib, ps, fit, k, t2, sg, False)
        if fit == "gaussian":
            se[2].zero_()                          # left unset by the compact pass
        se = put(se)
        out = out + (tuple(se[i].reshape(shape3) for i in (1, 0, 2)),)
    if t2_interval is not None:
        f, fl, _ = _interval_pass(lib, ps, q, 64, False)
        f = put(f)
        out = out + (tuple(f[i].reshape(shape3) for i in range(3)) + (put(fl).reshape(shape3),),)
    if bootstrap is not None:                      # the noise keyed by the flat voxel index
        vid = torch.from_numpy(idx).to(k.device) if stream is None else None
        mean, sd, lo, hi, nu, no = _bootstrap_pass(
            lib, ps, fit, fit_params, TEeffs, prior, norm, solver, kw.get("init_mode", "auto"), kw.get("max_iter", 0),
            kw.get("tol", 0.0), [k, t2, sg if fit != "gaussian" else None], None, vid, bootstrap, 0.95, 0, None)
        if fit == "gaussian":
            sd[2].zero_()
        out = out + (BootstrapMaps(*[put(c).reshape(shape3) for c in (mean[1], sd[1], lo, hi, sd[0], sd[2], nu, no)]),)
    return out


def _map_problem(reshaped_t2w, TEeffs, fit, norm, mask_indices, *maps):
    """The device problem of a pass over existing maps: ``reshaped_t2w`` (float32), ``mask_indices`` (int64) and the
    ``maps`` (float32, flattened) moved to the bound GPU, contiguous; TE, model and norm from the arguments, placeholder
    fit parameters (these passes take none).  Returns (p, y, maps, keep); ``keep`` must stay alive for the call."""
    import torch
    dev = torch.device("cuda", _state["device"])

    def to_dev(a, dt):
        t = a if _is_torch(a) else torch.from_numpy(np.ascontiguousarray(a))
        return t.to(device=dev, dtype=dt).contiguous()
    y = to_dev(reshaped_t2w, torch.float32)
    idx = to_dev(mask_indices, torch.int64)
    maps = [to_dev(a, torch.float32).reshape(-1) for a in maps]
    p = _abi.Problem()
    dummy = {"initial_guess": [1.0, 100.0] + ([1.0] if fit != "gaussian" else []),
             "param_bounds": [(0.0, 1e9), (1e-3, 1e9)] + ([(0.0, 1e9)] if fit != "gaussian" else [])}
    te = _fill_problem(p, fit, dummy, TEeffs, True, norm, 0, 0.0, "loglinear")
    p.echoes, p.memory, p.layout, p.mask_idx = y.data_ptr(), _abi.MEM_DEVICE, _abi.LAYOUT_AOS, idx.data_ptr()
    p.n_vox, p.n_fit = y.shape[0], idx.numel()
    return p, y, maps, (te, idx)


def compute_residuals(reshaped_t2w, TEeffs, fit, norm, k_map, t2_map, sigma_map, res_map, mask_indices, mask):
    """Signature of the reference's ``compute_residuals`` (utils/t2map_utils.py:62-89) for callers that
    keep the two-step structure (``fit_voxels_batch`` already returns the same residuals).  Runs the
    stand-alone CUDA residual pass (``t2fit_residuals``); numpy inputs are staged through torch."""
    import torch
    lib = init()
    p, y, (k, t2, sg, res), keep = _map_problem(reshaped_t2w, TEeffs, fit, norm, mask_indices, k_map, t2_map, sigma_map,
                                                res_map)
    res = res.clone()
    stream = torch.cuda.current_stream(y.device).cuda_stream
    _abi.check(lib, lib.t2fit_residuals(C.byref(p), k.data_ptr(), t2.data_ptr(), sg.data_ptr(), res.data_ptr(), stream),
               "t2fit_residuals")
    del keep
    shape3 = tuple(mask.shape[:3])
    if not _is_torch(reshaped_t2w):
        return res.cpu().numpy().reshape(shape3)
    return res.reshape(shape3)


def parameter_stderr(reshaped_t2w, TEeffs, fit, norm, k_map, t2_map, sigma_map, mask_indices, mask):
    """Standard errors of the fitted parameters for maps that already exist (e.g. read back from NIfTI), with the
    argument conventions of :func:`compute_residuals`; returns ``(se_t2_map, se_k_map, se_sigma_map)`` float32 shaped like
    ``mask``, zeros off-mask (se_sigma all zeros for 'gaussian').  Runs the CUDA pass ``t2fit_stderr``; numpy inputs are
    staged through torch and numpy maps come back.

    Per voxel, in FP64, at the given parameters theta = (k, T2[, sigma]) with bounds ignored: for 'gaussian' and
    'gaussian_rician' ``sqrt(diag(s^2 (J'J)^-1))`` with ``s^2 = sum_e r_e^2 / (E - P)`` (scipy ``curve_fit``'s ``pcov``);
    for 'rician' ``sqrt(diag(H^-1))``, H the Hessian of the summed negative log-likelihood.  NaN where the voxel's input
    is not finite (rician: an echo <= 0), T2 <= 0, E <= P, or the matrix is not positive definite (DESIGN.md section 11)."""
    lib = init()
    p, y, (k, t2, sg), keep = _map_problem(reshaped_t2w, TEeffs, fit, norm, mask_indices, k_map, t2_map, sigma_map)
    if y.dim() != 2 or y.shape[1] != p.n_echo:
        raise ValueError(f"reshaped_t2w must be [N, {p.n_echo}]")
    se = _stderr_pass(lib, p, fit, k, t2, sg, True)
    del keep
    shape3 = tuple(mask.shape[:3])
    if not _is_torch(reshaped_t2w):
        se = se.cpu().numpy()
    return tuple(se[i].reshape(shape3) for i in (1, 0, 2))


def t2_interval(reshaped_t2w, mask_indices, TEeffs, fit, fit_params, prior=True, norm=False, *, level=0.95, n_grid=64,
                profile=False):
    """Profile-likelihood confidence interval for T2 of every voxel ``mask_indices[i]`` of ``reshaped_t2w`` (float32
    ``[N, E]``; ``mask_indices`` None = all rows), with the arguments of :func:`fit_voxels_batch`.  Runs the CUDA pass
    ``t2fit_t2_interval`` (FP64 per voxel).  Returns compact ``(t2_lo, t2_hi, t2_best, flags)`` -- float32, float32,
    float32, uint8 ``[M]`` -- and with ``profile=True`` also ``profile`` float64 ``[M, n_grid]`` (p at the grid) and
    ``grid`` float64 ``[n_grid]`` (the T2 values).  numpy input gives numpy output (the masked rows are staged through
    torch); a CUDA tensor gives CUDA tensors, asynchronously on the current stream.

    Definition (DESIGN.md section 12): with the fit's objective f (mean squared error for 'gaussian' / 'gaussian_rician',
    summed negative log-likelihood for 'rician') and the fit's box, ``p(T2) = min over (k[, sigma]) of f``; the interval
    is the hull of ``{T2 : p(T2) <= thr}``, ``thr = p* (1 + q / (E - P))`` with ``q = t^2_{E-P}((1 + level) / 2)`` for the
    least-squares fits, ``thr = p* + q / 2`` with ``q = chi^2_1(level)`` for 'rician'; ``t2_best`` is the T2 of the
    bounded minimiser.  ``flags``: 1 t2_lo is the lower T2 bound, 2 t2_hi is the upper T2 bound (upper end not
    determined), 4 the set is not one interval at grid resolution, 8 invalid (NaN; non-finite echoes, rician echoes <= 0,
    E <= P, the --no_prior voxel with S(TE0) above the k bound).  The interval does not depend on the fit's point, so it is
    the same whichever solver fits the maps.  ``n_grid``: 16..256 grid points (default 64)."""
    lib = init()
    p = _abi.Problem()
    keep = [_fill_problem(p, fit, fit_params, TEeffs, prior, norm, 0, 0.0, "auto")]
    q = _interval_q(fit, p.n_echo, level)
    if not 16 <= int(n_grid) <= 256:
        raise ValueError("n_grid must lie in 16..256")
    t_lo, t_hi = (NO_PRIOR_T2_BOUNDS if not prior else (p.lb[1], p.ub[1]))
    ps, _, _, fin, pin = _pass_input(p, reshaped_t2w, mask_indices)
    keep += pin
    f, fl, pr = (fin(t) for t in _interval_pass(lib, ps, q, n_grid, profile))
    lo, hi, best = f[0], f[1], f[2]
    del keep
    if not profile:
        return lo, hi, best, fl
    return lo, hi, best, fl, pr, interval_grid(t_lo, t_hi, n_grid)


@dataclass
class BootstrapResult:
    """Per-voxel parametric bootstrap (:func:`parametric_bootstrap`), compact over the fitted voxels.

    ``mean``, ``sd``      float32 [M, P]  mean and standard deviation (ddof 1) of the refitted parameters, in the order of
                                          ``FitResult.results`` (k, T2[, sigma])
    ``t2_lo``, ``t2_hi``  float32 [M]     T2 quantiles at (1 - level) / 2 and (1 + level) / 2 of the refits
    ``n_used``            int32 [M]       replicates whose refit has status 0 or 2 and finite parameters
    ``n_ok``              int32 [M]       replicates whose refit has status 0
    mean, sd, t2_lo and t2_hi are NaN where n_used < 2.  numpy for numpy input, CUDA tensors for CUDA input.
    """
    mean: object
    sd: object
    t2_lo: object
    t2_hi: object
    n_used: object
    n_ok: object


# the bootstrap maps t2map_volume(..., bootstrap=n_rep) appends: float32 [z,y,x] (n_used / n_ok int32), zeros off-mask
BootstrapMaps = namedtuple("BootstrapMaps", "t2_mean t2_sd t2_lo t2_hi k_sd sigma_sd n_used n_ok")

BOOTSTRAP_BUDGET = 1 << 30       # bytes of replicate rows plus refit results one chunk of voxels may hold


def _bootstrap_chunk(n_echo, n_rep, fit):
    """Voxels per chunk of the bootstrap: the replicate rows (float32 [n_rep, E]) and refit results (k, T2[, sigma] float32,
    status uint8) of one voxel, within BOOTSTRAP_BUDGET."""
    per_voxel = n_rep * (4 * n_echo + 4 * (2 if fit == "gaussian" else 3) + 1)
    return max(1, BOOTSTRAP_BUDGET // per_voxel)


def _bootstrap_pass(lib, p, fit, fit_params, TEeffs, prior, norm, solver, init_mode, max_iter, tol, params, noise, vid,
                    n_rep, level, seed, chunk):
    """The bootstrap of the device rows of ``p`` (AoS, compact): ``params`` (k, t2, sigma) float32 CUDA [M] (sigma None for
    'gaussian'), ``noise`` float32 CUDA [M] or None, ``vid`` int64 CUDA [M] flat voxel ids or None (= the row read).  Per
    chunk of voxels: t2fit_bootstrap_replicates into one replicate buffer, the refit by fit_voxels_into (same solver, preset,
    prior and norm; status 3 is excluded by the statistics, never raised), t2fit_bootstrap_stats.  Asynchronous on the
    current stream.  Returns float32 mean [3, M], sd [3, M], lo [M], hi [M] and int32 n_used [M], n_ok [M]."""
    import torch
    dev = params[0].device
    M, E = p.n_fit, p.n_echo
    P = 2 if fit == "gaussian" else 3
    if p.mask_idx is None and vid is None:       # chunks read rows a.. of the echoes: key the noise by the row itself
        vid = torch.arange(M, dtype=torch.int64, device=dev)
    chunk = max(1, min(int(chunk) if chunk is not None else _bootstrap_chunk(E, n_rep, fit), M or 1))
    mean, sd = torch.empty((3, M), dtype=torch.float32, device=dev), torch.empty((3, M), dtype=torch.float32, device=dev)
    lo, hi = torch.empty(M, dtype=torch.float32, device=dev), torch.empty(M, dtype=torch.float32, device=dev)
    nu, no = torch.empty(M, dtype=torch.int32, device=dev), torch.empty(M, dtype=torch.int32, device=dev)
    rows = torch.empty((chunk * n_rep, E), dtype=torch.float32, device=dev)
    rep = torch.empty((P, chunk * n_rep), dtype=torch.float32, device=dev)
    rst = torch.empty(chunk * n_rep, dtype=torch.uint8, device=dev)
    cm, cs = torch.empty(3 * chunk, dtype=torch.float32, device=dev), torch.empty(3 * chunk, dtype=torch.float32, device=dev)
    counts = _device_counts(torch, dev)                      # the refit's histogram: status 3 is a replicate outcome here
    stream = torch.cuda.current_stream(dev).cuda_stream
    isz = 4 if p.idx_dtype == _abi.IDX_I32 else 8
    ptr = lambda t, a: t[a:].data_ptr() if t is not None else None
    out = {"t2": rep[1].data_ptr(), "k": rep[0].data_ptr(), "sigma": rep[2].data_ptr() if P == 3 else None, "res": None,
           "status": rst.data_ptr()}
    for a in range(0, M, chunk):
        n = min(chunk, M - a)
        q = _abi.Problem.from_buffer_copy(p)
        q.n_fit = n
        if p.mask_idx is not None:
            q.mask_idx = p.mask_idx + a * isz
        else:
            q.echoes, q.n_vox = p.echoes + a * E * 4, p.n_vox - a
        _abi.check(lib, lib.t2fit_bootstrap_replicates(C.byref(q), ptr(params[0], a), ptr(params[1], a), ptr(params[2], a),
                                                       ptr(noise, a), ptr(vid, a), int(seed) & 0xFFFFFFFFFFFFFFFF,
                                                       int(n_rep), rows.data_ptr(), stream), "t2fit_bootstrap_replicates")
        fit_voxels_into(rows[:n * n_rep], None, TEeffs, fit, fit_params, prior, norm, out, solver=solver, counts=counts,
                        init_mode=init_mode, max_iter=max_iter, tol=tol)
        _abi.check(lib, lib.t2fit_bootstrap_stats(p.model, n, int(n_rep), rep[0].data_ptr(), rep[1].data_ptr(),
                                                  rep[2].data_ptr() if P == 3 else None, rst.data_ptr(), float(level),
                                                  cm.data_ptr(), cs.data_ptr(), ptr(lo, a), ptr(hi, a), ptr(nu, a), ptr(no, a),
                                                  stream), "t2fit_bootstrap_stats")
        mean[:, a:a + n] = cm[:3 * n].view(3, n)
        sd[:, a:a + n] = cs[:3 * n].view(3, n)
    return mean, sd, lo, hi, nu, no


def _bootstrap_args(n_rep, level):
    if not 16 <= int(n_rep) <= 4096:
        raise ValueError("n_rep must lie in 16..4096")
    if not 0.0 < float(level) < 1.0:
        raise ValueError("level must lie in (0, 1)")


def parametric_bootstrap(reshaped_t2w, mask_indices, TEeffs, fit, fit_params, prior=True, norm=False, *, n_rep=200,
                         level=0.95, seed=0, noise_sd=None, params=None, solver="auto", init_mode="auto", chunk=None):
    """Parametric bootstrap of the fit of every voxel ``mask_indices[i]`` of ``reshaped_t2w`` (float32 ``[N, E]``;
    ``mask_indices`` None = all rows), with the arguments of :func:`fit_voxels_batch`: the sampling distribution of the
    estimator as it is run -- solver, preset, bounds, early stopping, ``prior`` and ``norm`` included.

    Per voxel: ``n_rep`` (16..4096) replicates are simulated from the fitted curve (DESIGN.md section 13) --
    'gaussian' ``k u + s z``, 'gaussian_rician' ``sqrt((k u)^2 + sigma^2) + s z``, 'rician' the modulus of ``k u`` plus
    complex noise of sd sigma_n, ``u = exp(-TE / T2)`` -- and refitted with the same solver.  ``s`` is ``noise_sd`` if
    given (a float or an [M] array, in the units of the stored echoes) else ``sqrt(sum r^2 / (E - P))`` at the fit;
    sigma_n is ``noise_sd`` if given else the fitted sigma.  The normals come from Philox4x32-10 keyed by ``seed`` and the
    flat voxel index, so a voxel's replicates do not depend on which other voxels are bootstrapped or how they are chunked.
    ``params``: the fit ``(k, t2, sigma)`` compact over the voxels (e.g. maps read back from NIfTI; sigma None for
    'gaussian'); None fits first with ``solver`` / ``init_mode`` (raising what :func:`fit_voxels_batch` raises).  ``chunk``:
    voxels per replicate buffer (default: 1 GiB of replicate rows plus refit results).

    Returns a :class:`BootstrapResult`.  Replicates whose refit has status 1 or 3 are not used (an invalid voxel -- echoes
    not finite, T2 <= 0, E <= P with s estimated -- gets NaN rows, so none of its replicates is used).  numpy input gives
    numpy output (the masked rows are staged through torch); a CUDA tensor gives CUDA tensors, asynchronously on the
    current stream when ``params`` is given."""
    import torch
    lib = init()
    _bootstrap_args(n_rep, level)
    solver = resolve_solver(fit, solver)
    p = _abi.Problem()
    keep = [_fill_problem(p, fit, fit_params, TEeffs, prior, norm, 0, 0.0, init_mode, solver)]
    if params is None:
        r = fit_voxels_batch(reshaped_t2w, mask_indices, TEeffs, fit, fit_params, prior, norm, solver=solver,
                             init_mode=init_mode, want=("status",))
        params = (r.k, r.t2, r.sigma if fit != "gaussian" else None)
    if len(params) != 3:
        raise ValueError("params must be (k, t2, sigma)")
    scalar_noise = noise_sd is not None and np.ndim(noise_sd) == 0 and not _is_torch(noise_sd)
    q, (*par, noise), ids, fin, pin = _pass_input(p, reshaped_t2w, mask_indices, *params,
                                                  None if scalar_noise else noise_sd)
    keep += pin
    M = q.n_fit
    if fit == "gaussian":
        par[2] = None
    elif par[2] is None:
        raise ValueError(f"fit {fit!r} needs sigma in params")
    if any(a is not None and a.numel() != M for a in par):
        raise ValueError(f"params must hold {M} values each")
    dev = torch.device("cuda", _state["device"])
    if scalar_noise:
        noise = torch.full((M,), float(noise_sd), dtype=torch.float32, device=dev)
    elif noise is not None and noise.numel() != M:
        raise ValueError(f"noise_sd must be a float or hold {M} values")
    vid = torch.from_numpy(ids).to(dev) if ids is not None else None
    res = _bootstrap_pass(lib, q, fit, fit_params, TEeffs, prior, norm, solver, init_mode, 0, 0.0, par, noise, vid, n_rep,
                          level, seed, chunk)
    del keep
    P = 2 if fit == "gaussian" else 3
    mean, sd, lo, hi, nu, no = res
    mean, sd = mean[:P].t().contiguous(), sd[:P].t().contiguous()
    return BootstrapResult(*(fin(t) for t in (mean, sd, lo, hi, nu, no)))
