"""numpy/scipy float64 statement of the per-voxel standard errors (DESIGN.md section 11).

TEST INFRASTRUCTURE ONLY (see ``oracle/__init__.py``): the checker for ``t2fit_stderr`` /
``csrc/t2fit_stderr.cuh``; never imported by the product.

At the given float32 parameters theta = (k, T2[, sigma]) of a voxel, bounds ignored:

* ``gaussian`` / ``gaussian_rician``: ``Cov = s^2 (J'J)^-1`` with ``J[e, j] = d m_e / d theta_j`` and
  ``s^2 = sum_e r_e^2 / (E - P)`` -- ``scipy.optimize.curve_fit``'s ``pcov`` (``absolute_sigma=False``).
* ``rician``: ``Cov = H^-1``, ``H`` the analytic Hessian of the summed negative log-likelihood
  (:func:`oracle.fit_oracle.objective_rician_nll`), with ``A(x) = i1e(x) / i0e(x)`` and
  ``A'(x) = 1 - A/x - A^2`` (series below ``x = 1e-4``).

``se_j = sqrt(Cov_jj)``, obtained from a Cholesky factorisation of ``D A D``, ``D = diag(A_jj^-1/2)``.
All standard errors of a voxel are NaN when an echo is not finite (rician: or <= 0), a parameter is
not finite or T2 <= 0, E <= P, a diagonal entry of A is <= 0 or the factorisation fails.
"""
from __future__ import annotations

import numpy as np
from scipy.special import i0e, i1e

NPAR = {"gaussian": 2, "gaussian_rician": 3, "rician": 3}


def signal(rows, norm):
    """The echoes as the fit sees them: float32, scaled by ``y / max(y)`` in float32 when ``norm`` (run_t2mapping.py:237-240)."""
    y = np.asarray(rows, np.float32)
    if norm:
        with np.errstate(all="ignore"):
            y = y / np.max(y, axis=1, keepdims=True)
    return y


def bessel_ratio(x):
    """A(x) = I1(x) / I0(x) and A'(x) = 1 - A(x)/x - A(x)^2 (float64 arrays)."""
    x = np.asarray(x, np.float64)
    z = np.abs(x)
    a = i1e(z) / i0e(z)
    small = z < 1e-4
    with np.errstate(all="ignore"):
        da = np.where(small, 0.5 - 3.0 * z ** 2 / 16.0 + 5.0 * z ** 4 / 96.0, 1.0 - a / z - a * a)
    return np.sign(x) * a, da


def jacobian(fit, te, k, t2, sigma=None):
    """J [M, E, P] of the least-squares model at float64 parameters [M]."""
    te = np.asarray(te, np.float64)[None, :]
    k, t2 = k[:, None], t2[:, None]
    u = np.exp(-te / t2)
    if fit == "gaussian":
        m = k * u
        return np.stack([u, m * te / t2 ** 2], axis=2), m
    s = sigma[:, None]
    m = np.sqrt(k ** 2 * u ** 2 + s ** 2)
    return np.stack([k * u ** 2 / m, k ** 2 * u ** 2 * te / (t2 ** 2 * m), s / m], axis=2), m


def rician_hessian(y, te, k, t2, sigma):
    """H [M, 3, 3]: analytic Hessian of the summed Rician NLL in (k, T2, sigma) at float64 parameters [M]."""
    y = np.asarray(y, np.float64)
    te = np.asarray(te, np.float64)[None, :]
    k, t2, s = k[:, None], t2[:, None], sigma[:, None]
    s2 = s * s
    u = np.exp(-te / t2)
    m = k * u
    x = y * m / s2
    a, da = bessel_ratio(x)
    tm = (m - y * a) / s2
    tmm = 1.0 / s2 - da * y ** 2 / s2 ** 2
    tms = 2.0 * (y * a - m + x * y * da) / (s2 * s)
    tss = (-2.0 + 3.0 * (y ** 2 + m ** 2) / s2 - 6.0 * x * a - 4.0 * x ** 2 * da) / s2
    mk, mt = u, m * te / t2 ** 2
    mkt, mtt = u * te / t2 ** 2, mt * (te - 2.0 * t2) / t2 ** 2
    H = np.empty((y.shape[0], 3, 3))
    H[:, 0, 0] = np.sum(tmm * mk * mk, axis=1)
    H[:, 0, 1] = H[:, 1, 0] = np.sum(tmm * mk * mt + tm * mkt, axis=1)
    H[:, 1, 1] = np.sum(tmm * mt * mt + tm * mtt, axis=1)
    H[:, 0, 2] = H[:, 2, 0] = np.sum(tms * mk, axis=1)
    H[:, 1, 2] = H[:, 2, 1] = np.sum(tms * mt, axis=1)
    H[:, 2, 2] = np.sum(tss, axis=1)
    return H


def information(rows, te, fit, norm, k, t2, sigma=None, param_dtype=np.float32):
    """(A [M, P, P], scale [M], valid [M]): Cov = scale * A^-1 on the voxels the NaN rule lets through.  The parameters
    are taken as float32 (what the fit returns) unless ``param_dtype`` says otherwise."""
    y = signal(rows, norm)
    E, P = y.shape[1], NPAR[fit]
    k, t2 = np.asarray(k, param_dtype).astype(np.float64), np.asarray(t2, param_dtype).astype(np.float64)
    s = None if P == 2 else np.asarray(sigma, param_dtype).astype(np.float64)
    valid = np.all(np.isfinite(y), axis=1) & np.isfinite(k) & np.isfinite(t2) & (t2 > 0) & (E > P)
    if s is not None:
        valid &= np.isfinite(s)
    if fit == "rician":
        valid &= np.all(y > 0, axis=1)
    with np.errstate(all="ignore"):
        if fit == "rician":
            A = rician_hessian(y, te, k, t2, s)
            scale = np.ones(y.shape[0])
        else:
            J, m = jacobian(fit, te, k, t2, s)
            A = np.einsum("mei,mej->mij", J, J)
            scale = np.sum((y.astype(np.float64) - m) ** 2, axis=1) / max(E - P, 1)
    return A, scale, valid


def stderr_rows(rows, te, fit, norm, k, t2, sigma=None, param_dtype=np.float32):
    """(se [M, 3] float64 in (k, T2, sigma) order -- sigma NaN for gaussian --, rcond [M]): the standard errors and the
    reciprocal 2-norm condition number min|lambda| / max|lambda| of D A D (NaN where the input part of the NaN rule applies;
    finite for an indefinite matrix, whose standard errors are NaN)."""
    A, scale, valid = information(rows, te, fit, norm, k, t2, sigma, param_dtype)
    M, P = A.shape[0], A.shape[1]
    se = np.full((M, 3), np.nan)
    rcond = np.full(M, np.nan)
    with np.errstate(all="ignore"):
        d = np.diagonal(A, axis1=1, axis2=2)
        valid &= np.all(np.isfinite(A.reshape(M, -1)), axis=1) & np.all(d > 0, axis=1)
        for i in np.flatnonzero(valid):
            D = 1.0 / np.sqrt(d[i])
            B = A[i] * D[:, None] * D[None, :]
            ev = np.linalg.eigvalsh(B)
            rcond[i] = np.min(np.abs(ev)) / np.max(np.abs(ev))
            try:
                L = np.linalg.cholesky(B)
            except np.linalg.LinAlgError:
                continue
            if not np.all(np.isfinite(L)):
                continue
            Li = np.linalg.inv(L)
            v = np.sum(Li * Li, axis=0)                    # diag((D A D)^-1) = diag(L^-T L^-1)
            se[i, :P] = np.sqrt(scale[i] * v) * D
    return se, rcond
