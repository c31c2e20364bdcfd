"""Per-voxel standard errors without a GPU: the oracle against scipy, i1e against scipy.special, and the header the
stderr_kernel runs (csrc/t2fit_stderr.cuh, compiled by g++) against the oracle."""
import ctypes as C

import numpy as np
import pytest
from scipy.optimize import curve_fit
from scipy.special import i1e

from oracle import stderr_oracle as so
from oracle.fit_oracle import model_floor, model_mono, objective_rician_nll
from tests.conftest import load_golden
from tests.hostsim import pass_shim as stderr_shim

FIXTURES = ["c1_gaussian_noprior", "c1_gaussian_prior", "c2_gaussian_noprior", "c2_gaussian_hf_prior", "c4_gaussian_noprior",
            "c3_floor_noprior", "c3_floor_prior", "c5_floor_noprior", "c3_rician_prior", "norm_gaussian",
            "cli3_gaussian_lf_noprior", "cli3_floor_hf_prior", "cli3_rician_hf_prior", "cli3_rician_lf_noprior"]


def _rician_rows(rng, n, te, k, t2, sigma):
    s = k * np.exp(-te[None, :] / t2)
    return np.sqrt((s + rng.normal(0, sigma, (n, te.size))) ** 2 + rng.normal(0, sigma, (n, te.size)) ** 2)


@pytest.mark.parametrize("fit", ["gaussian", "gaussian_rician"])
def test_least_squares_covariance_is_curve_fit_pcov(fit):
    """At the exact (unbounded) minimiser the oracle's s^2 (J'J)^-1 is scipy's curve_fit pcov (absolute_sigma=False)."""
    rng = np.random.default_rng(3)
    te = np.array([113, 133, 152, 176, 203, 230, 254, 296, 340, 400, 480, 600], float)
    rows = _rician_rows(rng, 8, te, 800.0, 90.0, 25.0).astype(np.float32)      # the echoes as the library stores them
    model = (lambda t, k, t2: model_mono(t, k, t2)) if fit == "gaussian" else (lambda t, k, t2, s: model_floor(t, k, t2, s))

    def jac(t, *p):
        J, _ = so.jacobian(fit, t, *[np.array([v]) for v in p])
        return J[0]
    p0 = [800.0, 90.0] + ([25.0] if fit != "gaussian" else [])
    for y in rows:
        popt, pcov = curve_fit(model, te, y.astype(np.float64), p0=p0, jac=jac, absolute_sigma=False, method="trf",
                               xtol=1e-15, ftol=1e-15, gtol=1e-15)
        se, _ = so.stderr_rows(y[None, :], te, fit, False, *[np.array([v]) for v in popt], param_dtype=np.float64)
        assert np.allclose(se[0, :len(popt)], np.sqrt(np.diag(pcov)), rtol=1e-8, atol=0)


def test_rician_hessian_is_second_difference_of_nll():
    """The oracle's analytic H equals central second differences of objective_rician_nll (the summed NLL)."""
    rng = np.random.default_rng(5)
    te = np.array([113, 133, 152, 176, 203, 230, 254, 296, 340, 400, 480, 600], float)
    for k, t2, s in ((800.0, 90.0, 25.0), (300.0, 60.0, 40.0), (2000.0, 900.0, 15.0), (60.0, 200.0, 50.0)):
        y = _rician_rows(rng, 3, te, k, t2, s)
        th = np.array([k * 1.03, t2 * 0.97, s * 1.05])
        H = so.rician_hessian(y, te, *[np.full(3, v) for v in th])
        for n in range(3):
            f = lambda p: objective_rician_nll(p, te, y[n])

            def second_differences(h):
                Hfd = np.empty((3, 3))
                for i in range(3):
                    for j in range(3):
                        ei, ej = np.eye(3)[i] * h[i], np.eye(3)[j] * h[j]
                        Hfd[i, j] = (f(th + ei + ej) - f(th + ei - ej) - f(th - ei + ej) + f(th - ei - ej)) / (4 * h[i] * h[j])
                return Hfd
            h = 1e-3 * th
            Hfd = (4.0 * second_differences(h / 2) - second_differences(h)) / 3.0      # Richardson: O(h^4) truncation
            scale = np.sqrt(np.outer(np.abs(np.diag(H[n])), np.abs(np.diag(H[n]))))
            assert np.all(np.abs(Hfd - H[n]) <= 1e-6 * scale), (k, t2, s, H[n], Hfd)


def test_i1e_matches_scipy():
    x = np.concatenate([np.linspace(0.0, 20.0, 100001), np.geomspace(1e-12, 1e4, 100001), [8.0, np.nextafter(8.0, 9.0)]])
    f = stderr_shim.lib().stderr_i1e
    got = np.array([f(v) for v in x])
    ref = i1e(x)
    rel = np.abs(got - ref) / np.maximum(np.abs(ref), np.finfo(float).tiny)
    assert rel.max() <= 2e-15, (rel.max(), x[rel.argmax()])
    assert f(-3.5) == -f(3.5) and f(0.0) == 0.0


def _params(g):
    p = g["ref_params"].astype(np.float32)
    return p[:, 0], p[:, 1], (p[:, 2] if p.shape[1] == 3 else None)


@pytest.mark.parametrize("name", FIXTURES)
def test_host_build_matches_oracle_on_fixtures(name):
    """g++ build of the device header vs the numpy oracle at the fixtures' reference parameters: the same NaN set, 1e-12
    relative where D A D is reasonably conditioned (rcond >= 1e-4), rounding-limited (rel * rcond <= 1e-13) elsewhere."""
    g = load_golden(name)
    k, t2, s = _params(g)
    P = 2 if g["fit"] == "gaussian" else 3
    ref, rcond = so.stderr_rows(g["rows"], g["te"], g["fit"], g["norm"], k, t2, s)
    got = stderr_shim.stderr_rows(g["rows"], g["te"], g["fit"], g["norm"], k, t2, s)
    ref, got = ref[:, :P], got[:, :P]
    assert np.array_equal(np.isnan(ref), np.isnan(got))
    assert np.array_equal(np.isnan(ref).any(axis=1), np.isnan(ref).all(axis=1))       # all of a voxel or none
    fin = np.isfinite(ref).all(axis=1)
    assert np.all(got[fin] > 0)
    rel = np.abs(got - ref) / ref
    well = fin & (rcond >= 1e-4)
    assert np.all(rel[well] <= 1e-12), rel[well].max()
    assert np.all(rel[fin] * rcond[fin, None] <= 1e-13)
    if g["te"].size <= P:                                            # no residual degrees of freedom
        assert not fin.any()


@pytest.mark.parametrize("fit", ["gaussian", "gaussian_rician", "rician"])
def test_nan_rule_on_hand_made_rows(fit):
    te = np.array([114.0, 150.0, 202.0, 299.0, 350.0])
    good = [900.0, 750.0, 570.0, 350.0, 270.0]          # ~ 1600 exp(-te / 195) + noise: near the minimiser of every model
    rows = np.array([good, [np.nan] + good[1:], good[:2] + [np.inf] + good[3:], good[:4] + [-np.inf], good,
                     good[:3] + [0.0] + good[4:], good[:1] + [-5.0] + good[2:]], np.float32)
    k = np.full(7, 1613.0, np.float32)
    t2 = np.array([195.4, 195.4, 195.4, 195.4, 0, 195.4, 195.4], np.float32)
    s = np.full(7, 1.85 if fit == "rician" else 20.0, np.float32)       # the rician NLL's minimiser has sigma ~ 1.85 here
    P = 2 if fit == "gaussian" else 3
    for norm in (False, True):
        c = np.float32(1 / 900 if norm else 1)                # the normalised signal's minimiser: k and sigma scaled by 1 / max
        ref, _ = so.stderr_rows(rows, te, fit, norm, k * c, t2, s * c)
        got = stderr_shim.stderr_rows(rows, te, fit, norm, k * c, t2, s * c)
        expect_nan = [False, True, True, True, True, fit == "rician", fit == "rician"]
        assert list(np.isnan(got[:, :P]).all(axis=1)) == expect_nan, (fit, norm, got)
        assert list(np.isnan(ref[:, :P]).all(axis=1)) == expect_nan, (fit, norm, ref)
        ok = ~np.array(expect_nan)
        assert np.all(np.isfinite(got[ok, :P])) and np.all(got[ok, :P] > 0)
    # a non-finite parameter
    for j, bad in ((0, np.nan), (1, np.inf), (1, -10.0)):
        p = [k[:1].copy(), t2[:1].copy(), s[:1].copy()]
        p[j][0] = bad
        assert np.isnan(stderr_shim.stderr_rows(rows[:1], te, fit, False, *p)[0, :P]).all()
    # E <= P: no residual degrees of freedom
    got = stderr_shim.stderr_rows(rows[:1, :P], te[:P], fit, False, k[:1], t2[:1], s[:1])
    assert np.isnan(got[0, :P]).all()


def test_stderr_entry_needs_a_device():
    """There is no CPU path behind the C entry: without a device it reports ENOTINIT."""
    try:
        import torch
        if torch.cuda.is_available():
            pytest.skip("GPU present")
    except ImportError:
        pass
    from fetal_t2mapping_b200 import _abi, build
    build.build_lib()
    lib = _abi.load_library()
    assert lib.t2fit_abi_version() == 5
    p = _abi.Problem()
    assert lib.t2fit_stderr(C.byref(p), None, None, None, 0, None, None, None, None) == -3
