"""numpy/scipy float64 statement of the per-voxel profile-likelihood interval for T2 (DESIGN.md section 12).

TEST INFRASTRUCTURE ONLY (see ``oracle/__init__.py``): the checker for ``t2fit_t2_interval`` /
``csrc/t2fit_interval.cuh``; never imported by the product.

For one voxel, with the fit's objective f (the mean squared error for ``gaussian`` / ``gaussian_rician``, the summed NLL of
:func:`oracle.fit_oracle.objective_rician_nll` for ``rician``, in float64 on the float32 echoes) and the fit's box:

* ``p(T2) = min over (k[, sigma]) in the box of f``; ``p* = min over T2`` at ``t2_best``;
* the set ``{T2 : p(T2) <= thr}``, ``thr = p* (1 + q / (E - P))`` (least squares, ``q = t^2_{E-P}(1 - alpha/2)``) or
  ``p* + q / 2`` (rician, ``q = chi^2_1(1 - alpha)``); ``lo`` / ``hi`` its smallest / largest member;
* ``flags``: 1 lo on the lower T2 bound, 2 hi on the upper T2 bound, 4 a grid point strictly between lo and hi outside
  the set, 8 invalid (NaN lo / hi / best).

The procedure is the kernel's: p on the geometric grid ``T2_g = lb (ub/lb)^(g/(G-1))``, golden-section search in log T2
around the grid minimum, bisection in log T2 of the two crossings that bound the hull.  ``gaussian`` uses the closed-form
inner problem; ``gaussian_rician`` and ``rician`` a bounded scipy minimisation (L-BFGS-B, analytic gradient) from the same
starts as the kernel: the fixed start, an ascending and a descending sweep warm-started from the neighbouring grid point,
and off the grid the solutions at the two enclosing grid points.  The lowest value wins.
"""
from __future__ import annotations

import numpy as np
from scipy.optimize import minimize
from scipy.special import i0e

from .stderr_oracle import bessel_ratio, signal

NPAR = {"gaussian": 2, "gaussian_rician": 3, "rician": 3}
TOL_MIN = 1e-8        # log T2 width of the final golden-section bracket
TOL_CROSS = 1e-7      # log T2 width of the final bisection bracket
GOLD = 0.6180339887498949


def voxel_box(fit, fit_params, prior, rows_raw, no_prior_k_ub=10000.0, no_prior_t2=(10.0, 2000.0)):
    """(box [M, 6] = (k_lo, k_hi, t2_lo, t2_hi, sigma_lo, sigma_hi), empty [M]) the fit uses for each row
    (run_t2mapping.py:243-245): under ``--no_prior`` k in [y(TE_0), no_prior_k_ub] -- the raw echo, as the fit --, T2 in
    ``no_prior_t2``; an empty k box is the fit's status 3."""
    b = [tuple(map(float, x)) for x in fit_params["param_bounds"]]
    s = b[2] if len(b) == 3 else (1.0, 1.0)
    m = rows_raw.shape[0]
    box = np.tile(np.array([b[0][0], b[0][1], b[1][0], b[1][1], s[0], s[1]], np.float64), (m, 1))
    empty = box[:, 0] > box[:, 1]
    if not prior:
        y0 = np.asarray(rows_raw, np.float32)[:, 0]
        box[:, 0], box[:, 1] = y0.astype(np.float64), no_prior_k_ub
        box[:, 2], box[:, 3] = no_prior_t2
        with np.errstate(invalid="ignore"):
            empty = y0 > np.float32(no_prior_k_ub)
    return box, empty


def grid(t_lo, t_hi, G):
    g = np.arange(G, dtype=np.float64)
    t = t_lo * np.power(t_hi / t_lo, g / (G - 1))
    t[-1] = t_hi
    return t


def _value(fit, y, u, k, s):
    if fit == "gaussian_rician":
        r = y - np.sqrt((k * u) ** 2 + s * s)
        return float(np.sum(r * r) / y.size)
    s2 = s * s
    m = k * u
    x = m * y / s2
    return float(-np.sum((np.log(y) - np.log(s2)) - (y * y + m * m) / (2.0 * s2) + (np.abs(x) + np.log(i0e(x)))))


def _value_grad(fit, y, u, k, s):
    if fit == "gaussian_rician":
        ku = k * u
        m = np.sqrt(ku * ku + s * s)
        r = m - y
        g = 2.0 / y.size * np.array([np.sum(r * ku * u / m), np.sum(r * s / m)])
        return float(np.sum(r * r) / y.size), g
    s2 = s * s
    m = k * u
    x = m * y / s2
    a, _ = bessel_ratio(x)
    f = -np.sum((np.log(y) - np.log(s2)) - (y * y + m * m) / (2.0 * s2) + (np.abs(x) + np.log(i0e(x))))
    tm = (m - y * a) / s2
    ts = 2.0 / s - (y * y + m * m) / (s2 * s) + 2.0 * x * a / s
    return float(f), np.array([np.sum(tm * u), np.sum(ts)])


def _inner(fit, y, u, box, x0):
    """Bounded minimisation over (k, sigma) from x0 (scaled to O(1) variables): (f, x)."""
    lo, hi = np.array([box[0], box[4]]), np.array([box[1], box[5]])
    x0 = np.clip(np.asarray(x0, np.float64), lo, hi)
    sc = np.maximum(np.abs(x0), 1e-300)

    def fun(z):
        f, g = _value_grad(fit, y, u, *(z * sc))
        return f, g * sc
    r = minimize(fun, x0 / sc, jac=True, method="L-BFGS-B", bounds=list(zip(lo / sc, hi / sc)),
                 options={"ftol": 1e-16, "gtol": 1e-14, "maxiter": 2000, "maxls": 50})
    x = np.clip(r.x * sc, lo, hi)
    f = _value(fit, y, u, *x)
    f0 = _value(fit, y, u, *x0)
    return (f, x) if f <= f0 else (f0, x0)


def _fixed_start(y, u, box):
    k = np.clip(np.sum(y * u) / np.sum(u * u), box[0], box[1])
    s = np.sqrt(np.sum((y - k * u) ** 2) / y.size)
    return np.array([k, np.clip(s, box[4], box[5]) if np.isfinite(s) else box[4]])


class _Profile:
    """p(T2) of one voxel with the kernel's start rules."""

    def __init__(self, fit, y, te, box, G):
        self.fit, self.y, self.te, self.box, self.G = fit, y, te, box, G
        self.t = grid(box[2], box[3], G)
        self.p = np.empty(G)
        self.x = np.zeros((G, 2))

    def _u(self, t2):
        return np.exp(-self.te / t2)

    def at(self, t2, starts, use_fixed=True):
        u = self._u(t2)
        if self.fit == "gaussian":
            k = np.clip(np.sum(self.y * u) / np.sum(u * u), self.box[0], self.box[1])
            return float(np.sum((self.y - k * u) ** 2) / self.y.size), np.array([k, 0.0])
        cand = ([_fixed_start(self.y, u, self.box)] if use_fixed else []) + list(starts)
        best = None
        for x0 in cand:
            f, x = _inner(self.fit, self.y, u, self.box, x0)
            if best is None or f < best[0] or not np.isfinite(best[0]):
                best = (f, x)
        return best

    def run_grid(self):
        G = self.G
        if self.fit == "gaussian":
            U = np.exp(-self.te[None, :] / self.t[:, None])
            k = np.clip((U @ self.y) / np.sum(U * U, axis=1), self.box[0], self.box[1])
            self.p[:] = np.sum((self.y[None, :] - k[:, None] * U) ** 2, axis=1) / self.y.size
            return
        for g in range(G):
            self.p[g], self.x[g] = self.at(self.t[g], [self.x[g - 1]] if g > 0 else [])
        for g in range(G - 2, -1, -1):
            f, x = self.at(self.t[g], [self.x[g + 1]], use_fixed=False)
            if f < self.p[g]:
                self.p[g], self.x[g] = f, x

    def off_grid(self, s):
        s0, s1 = np.log(self.box[2]), np.log(self.box[3])
        g = int(np.floor((s - s0) / (s1 - s0) * (self.G - 1)))
        g = min(max(g, 0), self.G - 2)
        return self.at(np.exp(s), [self.x[g], self.x[g + 1]])[0]


def voxel_interval(fit, y, te, box, q, G=64):
    """(lo, hi, best, flags, profile [G], p*) of one voxel whose NaN rule has passed (y float64 of the float32 echoes)."""
    P = NPAR[fit]
    pr = _Profile(fit, y, te, box, G)
    pr.run_grid()
    fin = np.isfinite(pr.p)
    if not fin.any():
        return np.nan, np.nan, np.nan, 8, pr.p, np.nan
    gm = int(np.argmin(np.where(fin, pr.p, np.inf)))
    pstar, tbest = pr.p[gm], pr.t[gm]
    a, b = np.log(pr.t[max(gm - 1, 0)]), np.log(pr.t[min(gm + 1, G - 1)])
    c, d = b - GOLD * (b - a), a + GOLD * (b - a)
    fc, fd = pr.off_grid(c), pr.off_grid(d)
    if fc < pstar:
        pstar, tbest = fc, np.exp(c)
    if fd < pstar:
        pstar, tbest = fd, np.exp(d)
    while b - a > TOL_MIN:
        if fc < fd:
            b, d, fd = d, c, fc
            c = b - GOLD * (b - a)
            fc = pr.off_grid(c)
            if fc < pstar:
                pstar, tbest = fc, np.exp(c)
        else:
            a, c, fc = c, d, fd
            d = a + GOLD * (b - a)
            fd = pr.off_grid(d)
            if fd < pstar:
                pstar, tbest = fd, np.exp(d)
    if not np.isfinite(pstar):
        return np.nan, np.nan, np.nan, 8, pr.p, np.nan
    thr = pstar + 0.5 * q if fit == "rician" else pstar * (1.0 + q / (y.size - P))

    def crossing(s_out, s_in):
        while abs(s_in - s_out) > TOL_CROSS:
            mid = 0.5 * (s_out + s_in)
            if pr.off_grid(mid) <= thr:
                s_in = mid
            else:
                s_out = mid
        return np.exp(s_in)
    inside = pr.p <= thr
    sg = np.log(pr.t)
    sb = np.log(tbest)
    fl = 0
    idx = np.flatnonzero(inside)
    first_in, last_in = (idx[0], idx[-1]) if idx.size else (G, -1)
    if first_in == 0:
        lo, fl = box[2], fl | 1
    elif first_in == G or sb < sg[first_in]:
        below = np.flatnonzero(sg < sb)
        if below.size == 0:
            lo, fl = box[2], fl | 1
        else:
            lo = crossing(sg[below[-1]], sb)
    else:
        lo = crossing(sg[first_in - 1], sg[first_in])
    if last_in == G - 1:
        hi, fl = box[3], fl | 2
    elif last_in < 0 or sb > sg[last_in]:
        above = np.flatnonzero(sg > sb)
        if above.size == 0:
            hi, fl = box[3], fl | 2
        else:
            hi = crossing(sg[above[0]], sb)
    else:
        hi = crossing(sg[last_in + 1], sg[last_in])
    if np.any((pr.t > lo) & (pr.t < hi) & ~inside):
        fl |= 4
    return lo, hi, tbest, fl, pr.p, pstar


def interval_rows(rows, te, fit, norm, box, empty, q, G=64, voxels=None):
    """(lo, hi, best [M] float64, flags [M] uint8, profile [M, G], p* [M]) for the rows (all, or the indices ``voxels``);
    ``box`` / ``empty`` from :func:`voxel_box`."""
    y = signal(rows, norm)
    te = np.asarray(te, np.float64)
    E, P = y.shape[1], NPAR[fit]
    sel = np.arange(y.shape[0]) if voxels is None else np.asarray(voxels)
    n = sel.size
    lo, hi, best = np.full(n, np.nan), np.full(n, np.nan), np.full(n, np.nan)
    flags = np.full(n, 8, np.uint8)
    prof = np.full((n, G), np.nan)
    pstar = np.full(n, np.nan)
    for j, i in enumerate(sel):
        yi = y[i]
        ok = np.all(np.isfinite(np.asarray(rows, np.float32)[i])) and np.all(np.isfinite(yi)) and E > P and not empty[i]
        ok = ok and box[i, 0] <= box[i, 1]
        if fit == "rician":
            ok = ok and np.all(yi > 0)
        if not ok:
            continue
        lo[j], hi[j], best[j], flags[j], prof[j], pstar[j] = voxel_interval(fit, yi.astype(np.float64), te, box[i], q, G)
    return lo, hi, best, flags, prof, pstar
