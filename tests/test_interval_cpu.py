"""Profile-likelihood T2 intervals without a GPU: the oracle against an independent inner solve, the fixtures' exact
minimisers, a fine grid and noise realisations, and the header the interval_kernel runs (csrc/t2fit_interval.cuh, compiled
by g++) against the oracle."""
import ctypes as C

import numpy as np
import pytest
from scipy.optimize import least_squares
from scipy.stats import chi2, t as tdist

from oracle import interval_oracle as io
from oracle import stderr_oracle as so
from tests.conftest import fit_params_of, load_golden
from tests.hostsim import pass_shim as interval_shim

FIXTURES = ["c1_gaussian_noprior", "c1_gaussian_prior", "c2_gaussian_noprior", "c2_gaussian_hf_prior", "c4_gaussian_noprior",
            "c3_floor_noprior", "c3_floor_prior", "c5_floor_noprior", "c3_rician_prior", "norm_gaussian",
            "cli3_gaussian_lf_noprior", "cli3_floor_hf_prior", "cli3_rician_hf_prior", "cli3_rician_lf_noprior"]
EDGE = ["edge_gaussian_noprior", "edge_gaussian_prior", "edge_gaussian_rician_noprior", "edge_gaussian_rician_prior"]
# The oracle's 3-parameter inner problem is a scipy minimisation per start and grid point (~0.5 s per voxel at G = 64):
# those fixtures are checked on a fixed sample of their voxels; the 2-parameter ones on every voxel.
SAMPLE_3P = 12


def q_of(fit, n_echo, level=0.95):
    if fit == "rician":
        return chi2.ppf(level, 1)
    dof = n_echo - io.NPAR[fit]
    return tdist.ppf(0.5 + 0.5 * level, dof) ** 2 if dof > 0 else 0.0


def sample(g, n3=SAMPLE_3P):
    m = g["rows"].shape[0]
    if g["fit"] == "gaussian" or g["te"].size <= 3:
        return np.arange(m)
    return np.unique(np.linspace(0, m - 1, n3).astype(int))


def run_oracle(g, G=64, voxels=None):
    box, empty = io.voxel_box(g["fit"], fit_params_of(g), g["prior"], g["rows"])
    return io.interval_rows(g["rows"], g["te"], g["fit"], g["norm"], box, empty, q_of(g["fit"], g["te"].size), G, voxels)


def run_host(g, G=64, voxels=None):
    rows = g["rows"] if voxels is None else g["rows"][voxels]
    box, _ = io.voxel_box(g["fit"], fit_params_of(g), g["prior"], rows[:1])
    return interval_shim.interval_rows(rows, g["te"], g["fit"], g["norm"], box[0], not g["prior"],
                                       q_of(g["fit"], g["te"].size), G, profile=True)


def compare(ref, got, name):
    """The thresholds of the kernel checks: profile <= oracle (1 + 1e-9) everywhere and >= oracle (1 - 1e-9) on 99.9 % of
    grid points (relative to |p|: the rician NLL can be negative); lo / hi / best within 1e-6 relative where the flags
    agree; flags equal on 99.9 % of voxels."""
    pr, pg = ref[4], got[4]
    assert np.array_equal(np.isnan(pr), np.isnan(pg)), name
    fin = np.isfinite(pr)
    d = (pg[fin] - pr[fin]) / np.maximum(np.abs(pr[fin]), 1e-300)
    assert d.size == 0 or d.max() <= 1e-9, (name, d.max())
    assert d.size == 0 or np.mean(d >= -1e-9) >= 0.999, (name, np.mean(d >= -1e-9))
    fr, fg = ref[3], got[3]
    same = fr == fg
    for i in np.flatnonzero(~same):
        print(f"[interval] {name} voxel {i}: flags oracle {fr[i]} kernel {fg[i]}, lo {ref[0][i]} / {got[0][i]}, "
              f"hi {ref[1][i]} / {got[1][i]}")
    assert same.mean() >= 0.999, (name, same.mean())
    ok = same & (fr & 8 == 0)
    for j, what in enumerate(("lo", "hi", "best")):
        r = np.abs(got[j][ok] - ref[j][ok]) / ref[j][ok]
        assert r.size == 0 or r.max() <= 1e-6, (name, what, r.max())
    assert np.all(np.isnan(got[0][fg == 8])) and np.all(np.isnan(got[2][fg == 8]))
    return ok


def test_gaussian_closed_form_profile_is_the_inner_minimum():
    """The closed-form inner problem (k = clamp(sum y u / sum u^2)) equals a bounded least_squares solve over k."""
    g = load_golden("c2_gaussian_noprior")
    box, _ = io.voxel_box("gaussian", fit_params_of(g), False, g["rows"])
    y = io.signal(g["rows"], False).astype(np.float64)
    for i in range(0, y.shape[0], 150):
        pr = io._Profile("gaussian", y[i], g["te"], box[i], 64)
        pr.run_grid()
        for t2, p in zip(pr.t[::7], pr.p[::7]):
            u = np.exp(-g["te"] / t2)
            r = least_squares(lambda k: y[i] - k[0] * u, [0.5 * (box[i, 0] + min(box[i, 1], 4 * box[i, 0]))],
                              bounds=([box[i, 0]], [box[i, 1]]), xtol=1e-15, ftol=1e-15, gtol=1e-15)
            ls = 2.0 * r.cost / y.shape[1]
            assert abs(p - ls) <= 1e-10 * ls, (i, t2, p, ls)


@pytest.mark.parametrize("name", [n for n in FIXTURES if "exact" in " ".join(load_golden(n).keys())])
def test_oracle_minimum_is_the_exact_minimiser(name):
    """p* <= exact_fun (1 + 1e-9) on every voxel; t2_best within 1e-4 of exact T2 on >= 99 % (the rest are flat valleys)."""
    g = load_golden(name)
    vox = sample(g)
    lo, hi, best, flags, _, pstar = run_oracle(g, voxels=vox)
    ok = flags & 8 == 0
    if g["te"].size <= io.NPAR[g["fit"]]:
        assert not ok.any()
        return
    ef, et = g["exact_fun"][vox], g["exact_params"][vox, 1]
    assert np.all(pstar[ok] <= ef[ok] * (1 + 1e-9) + 1e-300), name
    rel = np.abs(best - et) / et
    within = rel[ok] <= 1e-4
    for i in np.flatnonzero(ok)[~within]:
        print(f"[interval] {name} voxel {vox[i]}: t2_best {best[i]:.6g} exact {et[i]:.6g} p* {pstar[i]:.9g} "
              f"exact_fun {ef[i]:.9g} (flat valley)")
    assert within.mean() >= 0.99, (name, within.mean())


@pytest.mark.parametrize("name", FIXTURES)
def test_grid_resolution_effect(name):
    """lo / hi at G = 64 against G = 2048: the share of voxels whose ends move by more than 1e-4 relative (DESIGN §12)."""
    g = load_golden(name)
    vox = sample(g, n3=4)
    a = run_oracle(g, 64, vox)
    b = run_oracle(g, 2048, vox)
    ok = (a[3] & 8 == 0) & (b[3] & 8 == 0)
    assert np.array_equal(a[3] & 8, b[3] & 8)
    moved = (np.abs(a[0] - b[0]) > 1e-4 * b[0]) | (np.abs(a[1] - b[1]) > 1e-4 * b[1])
    share = moved[ok].mean() if ok.any() else 0.0
    print(f"[interval grid] {name}: {moved[ok].sum()} of {ok.sum()} voxels move by > 1e-4 between G = 64 and 2048 "
          f"(share {share:.4f})")
    assert share <= 0.01, (name, share)


# The scenarios of the numpy check in DESIGN §12: c2's five echoes under the --no_prior box (k in [y(TE_0), 10000],
# T2 in [10, 2000]), Gaussian noise sd 12; and a well-determined 32-echo voxel.
TE5 = np.array([114.0, 132.0, 150.0, 176.0, 202.0])
TE32 = np.linspace(10.0, 320.0, 32)
FP_GAUSS = {"initial_guess": [650.0, 165.0], "param_bounds": [(600.0, 10000.0), (10.0, 600.0)]}
FP_WIDE = {"initial_guess": [650.0, 165.0], "param_bounds": [(0.0, 10000.0), (10.0, 600.0)]}
SCENARIOS = [("wm", TE5, 450.0, 118.0, 12.0, False), ("gm", TE5, 300.0, 165.0, 12.0, False),
             ("csf", TE5, 450.0, 1500.0, 12.0, False), ("e32", TE32, 2000.0, 100.0, 20.0, True)]


def _realisations(te, k, t2, sd, prior, n=4000, seed=11):
    rng = np.random.default_rng(seed)
    rows = (k * np.exp(-te / t2))[None, :] + rng.normal(0, sd, (n, te.size))
    g = {"rows": rows.astype(np.float32), "te": te, "fit": "gaussian", "norm": False, "prior": prior}
    box, empty = io.voxel_box("gaussian", FP_WIDE if prior else FP_GAUSS, prior, g["rows"])
    return g, box, empty


@pytest.mark.parametrize("scen", SCENARIOS, ids=[s[0] for s in SCENARIOS])
def test_gaussian_interval_is_calibrated(scen):
    """Coverage of the true T2 over 4000 seeded realisations: [0.93, 0.965] for the interior scenarios; for CSF >= 0.93
    with the upper end on the bound (bit 1) in >= 90 %."""
    label, te, k, t2, sd, prior = scen
    g, box, empty = _realisations(te, k, t2, sd, prior)
    lo, hi, best, flags, _, _ = io.interval_rows(g["rows"], te, "gaussian", False, box, empty, q_of("gaussian", te.size))
    ok = flags & 8 == 0
    assert ok.mean() >= 0.99
    cov = np.mean((lo[ok] <= t2) & (t2 <= hi[ok]))
    at_ub = np.mean(flags[ok] & 2 != 0)
    print(f"[interval calibration] {label}: coverage {cov:.4f}, median width {np.median(hi[ok] - lo[ok]):.1f} ms, "
          f"upper end on the bound {at_ub:.3f}")
    if label == "csf":
        assert cov >= 0.93 and at_ub >= 0.90
    else:
        assert 0.93 <= cov <= 0.965
    if label == "e32":
        se, _ = so.stderr_rows(g["rows"][ok], te, "gaussian", False, *_best_k_t2(g["rows"][ok], te, best[ok]),
                               param_dtype=np.float64)
        ratio = 0.5 * (hi[ok] - lo[ok]) / (np.sqrt(q_of("gaussian", te.size)) * se[:, 1])
        print(f"[interval calibration] e32: half-width / (t se_T2) median {np.median(ratio):.4f}, "
              f"p5-p95 {np.percentile(ratio, 5):.4f}-{np.percentile(ratio, 95):.4f}")
        assert 0.98 <= np.median(ratio) <= 1.02


def _best_k_t2(rows, te, t2):
    y = rows.astype(np.float64)
    u = np.exp(-te[None, :] / t2[:, None])
    return np.sum(y * u, axis=1) / np.sum(u * u, axis=1), t2


@pytest.mark.parametrize("name", FIXTURES + EDGE)
def test_host_build_matches_oracle_on_fixtures(name):
    g = load_golden(name)
    vox = sample(g)
    ref = run_oracle(g, voxels=vox)
    got = run_host(g, voxels=vox)
    ok = compare(ref, got, name)
    if g["te"].size <= io.NPAR[g["fit"]]:
        assert not ok.any()
    print(f"[interval] {name}: {len(vox)} voxels, flag histogram {np.bincount(got[3], minlength=9)[[0, 1, 2, 3, 4, 8]]}")


@pytest.mark.parametrize("fit", ["gaussian", "gaussian_rician", "rician"])
def test_nan_rule_on_hand_made_rows(fit):
    te = np.array([114.0, 150.0, 202.0, 299.0, 350.0])
    good = [900.0, 750.0, 570.0, 350.0, 270.0]
    rows = np.array([good, [np.nan] + good[1:], good[:2] + [np.inf] + good[3:], good[:4] + [-np.inf], good,
                     good[:3] + [0.0] + good[4:], good[:1] + [-5.0] + good[2:], [20000.0] + good[1:]], np.float32)
    fp = {"initial_guess": [650.0, 165.0] + ([40.0] if fit != "gaussian" else []),
          "param_bounds": [(0.0, 10000.0), (10.0, 2000.0)] + ([(1e-3, 1000.0)] if fit != "gaussian" else [])}
    q = q_of(fit, te.size)
    for norm in (False, True):
        for prior in (True, False):
            g = {"rows": rows, "te": te, "fit": fit, "norm": norm, "prior": prior}
            box, empty = io.voxel_box(fit, fp, prior, rows)
            ref = io.interval_rows(rows, te, fit, norm, box, empty, q)
            got = interval_shim.interval_rows(rows, te, fit, norm, box[0], not prior, q, profile=True)
            expect = [False, True, True, True, False, fit == "rician", fit == "rician", not prior]
            assert list(got[3] == 8) == expect, (fit, norm, prior, got[3])
            assert list(ref[3] == 8) == expect, (fit, norm, prior, ref[3])
            compare(ref, got, f"{fit}/norm={norm}/prior={prior}")
            assert np.all(np.isfinite(got[0][~np.array(expect)]))
    # E <= P: no residual degrees of freedom
    P = io.NPAR[fit]
    got = interval_shim.interval_rows(rows[:1, :P], te[:P], fit, False, box[0], False, 1.0)
    assert got[3][0] == 8 and np.isnan(got[0][0])


def test_exact_fit_is_valid():
    """A least-squares voxel the model fits exactly (p* = 0) is valid: its set is where p = 0."""
    te = np.array([10.0, 20.0, 40.0, 80.0])
    rows = np.zeros((1, 4), np.float32)                          # k = 0 on the box fits every T2 exactly
    got = interval_shim.interval_rows(rows, te, "gaussian", False, (0.0, 100.0, 10.0, 600.0, 1.0, 1.0), False, 9.0,
                                      profile=True)
    assert got[3][0] == 3 and got[0][0] == 10.0 and got[1][0] == 600.0 and np.all(got[4] == 0.0)


def test_interval_entry_needs_a_device():
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
    p = _abi.Problem()
    assert lib.t2fit_t2_interval(C.byref(p), 1.0, 64, 0, None, None, None, None, None, None) == -3
