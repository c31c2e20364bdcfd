"""Per-voxel standard errors on the GPU (t2fit_stderr / stderr_kernel): against the float64 oracle at the GPU's own fitted
parameters on every fit fixture, through every public entry, without moving any existing output, and calibrated against
the spread of the fits over noise realisations."""
import ctypes as C

import numpy as np
import pytest

from oracle import stderr_oracle as so
from oracle.fit_oracle import model_floor, model_mono
from tests.conftest import fit_params_of, load_golden

pytestmark = pytest.mark.gpu

FIXTURES = ["c1_gaussian_noprior", "c1_gaussian_prior", "c2_gaussian_noprior", "c2_gaussian_hf_prior", "c4_gaussian_noprior",
            "c3_floor_noprior", "c3_floor_prior", "c5_floor_noprior", "c3_rician_prior", "norm_gaussian",
            "cli3_gaussian_lf_noprior", "cli3_floor_hf_prior", "cli3_rician_hf_prior", "cli3_rician_lf_noprior"]
FIELDS = ("t2", "k", "sigma", "res", "fun", "nit", "status")


def _np(a):
    return None if a is None else (a.cpu().numpy() if hasattr(a, "cpu") else np.asarray(a))


def _check_against_oracle(g, r, name):
    P = 2 if g["fit"] == "gaussian" else 3
    k, t2, s = _np(r.k), _np(r.t2), (_np(r.sigma) if P == 3 else None)
    ref, rcond = so.stderr_rows(g["rows"], g["te"], g["fit"], g["norm"], k, t2, s)
    got = np.stack([_np(r.se_k), _np(r.se_t2)] + ([_np(r.se_sigma)] if P == 3 else []), axis=1).astype(np.float64)
    assert np.array_equal(got, _np(r.standard_errors), equal_nan=True)
    ref = ref[:, :P]
    assert np.array_equal(np.isnan(got).any(axis=1), np.isnan(got).all(axis=1)), name      # all of a voxel or none
    well = rcond >= 1e-10
    nan_r, nan_g = np.isnan(ref).any(axis=1), np.isnan(got).any(axis=1)
    assert np.array_equal(nan_r[well], nan_g[well]), name
    both = well & ~nan_r
    rel = np.abs(got[both] - ref[both]) / ref[both]
    assert rel.size == 0 or rel.max() <= 1e-6, (name, rel.max())
    rest = ~well & ~nan_g
    assert np.all(np.isfinite(got[rest])) and np.all(got[rest] > 0), name
    st1 = _np(r.status) == 1
    assert np.array_equal(nan_r[st1], nan_g[st1]) and nan_g[st1].all(), name
    return nan_g.mean()


@pytest.mark.parametrize("name", FIXTURES)
def test_stderr_matches_oracle_at_the_gpu_parameters(gpu_lib, name):
    """Default solver and the fast solver where it applies; host input without indices, device input with int64 and with
    int32 indices (norm=True: the norm fixture).  Host and device give the same standard errors bit for bit."""
    import torch
    g = load_golden(name)
    fp = fit_params_of(g)
    rows = np.ascontiguousarray(g["rows"])
    m = rows.shape[0]
    want = ("nit", "fun", "status", "se")
    for solver in ["auto"] + (["fast"] if g["fit"] != "rician" else []):
        kw = dict(prior=g["prior"], norm=g["norm"], solver=solver, want=want)
        r_host = gpu_lib.fit_voxels_batch(rows, None, g["te"], g["fit"], fp, **kw)
        share = _check_against_oracle(g, r_host, f"{name}/{solver}/host")
        yd = torch.from_numpy(rows).cuda()
        for idt in (torch.int64, torch.int32):
            idx = torch.arange(m, dtype=idt, device="cuda")
            r_dev = gpu_lib.fit_voxels_batch(yd, idx, g["te"], g["fit"], fp, **kw)
            torch.cuda.synchronize()
            _check_against_oracle(g, r_dev, f"{name}/{solver}/device/{idt}")
            for f in ("se_k", "se_t2") + (("se_sigma",) if g["fit"] != "gaussian" else ()):
                assert np.array_equal(_np(getattr(r_dev, f)), _np(getattr(r_host, f)), equal_nan=True), (name, solver, f)
        print(f"[stderr] {name} solver={solver}: NaN share {share:.4f}")


def _volume(fit):
    from fetal_t2mapping_b200 import synth
    y, mask, te, _ = synth.make_volume("c1", scale=0.25)
    return y, mask, te


@pytest.mark.parametrize("fit,solver", [("gaussian", "auto"), ("gaussian_rician", "fast"), ("gaussian_rician", "auto"),
                                        ("rician", "auto")])
@pytest.mark.parametrize("device", [True, False], ids=["device", "host"])
def test_entries_agree_and_nothing_else_moves(gpu_lib, fit, solver, device):
    """parameter_stderr on the maps of t2map_volume == t2map_volume(stderr=True) == fit_voxels_batch's compact results, bit
    for bit; zeros off-mask.  The outputs of fit_voxels_batch with and without "se", and the four maps of t2map_volume with
    stderr on and off, are bit-identical."""
    import torch
    y, mask, te = _volume(fit)
    _, fp = gpu_lib.preset(fit, True)
    flat = np.ascontiguousarray(y.reshape(-1, te.size))
    idx = np.flatnonzero(mask.reshape(-1))
    cv = (lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()) if device else (lambda a: a)
    kw = dict(prior=False, norm=False, solver=solver)
    maps0 = gpu_lib.t2map_volume(cv(y), cv(mask), te, fit, fp, **kw)
    maps1 = gpu_lib.t2map_volume(cv(y), cv(mask), te, fit, fp, stderr=True, **kw)
    assert len(maps0) == 4 and len(maps1) == 5
    for a, b in zip(maps0, maps1[:4]):
        assert np.array_equal(_np(a), _np(b), equal_nan=True)
    se_vol = [_np(a) for a in maps1[4]]
    se_par = gpu_lib.parameter_stderr(cv(flat), te, fit, False, maps1[1], maps1[0], maps1[2], cv(idx), cv(mask))
    for a, b in zip(se_vol, se_par):
        assert np.array_equal(a, _np(b), equal_nan=True)
        assert a.shape == mask.shape and a.dtype == np.float32 and np.all(a[~mask] == 0)
    if fit == "gaussian":
        assert np.all(se_vol[2] == 0)
    r0 = gpu_lib.fit_voxels_batch(cv(flat), cv(idx), te, fit, fp, **kw)
    r1 = gpu_lib.fit_voxels_batch(cv(flat), cv(idx), te, fit, fp, want=("nit", "fun", "status", "se"), **kw)
    assert r0.se_t2 is None and r0.standard_errors is None
    for f in FIELDS:
        assert np.array_equal(_np(getattr(r0, f)), _np(getattr(r1, f)), equal_nan=True), f
    sel = mask.reshape(-1)
    assert np.array_equal(_np(r1.se_t2), se_vol[0].reshape(-1)[sel], equal_nan=True)
    assert np.array_equal(_np(r1.se_k), se_vol[1].reshape(-1)[sel], equal_nan=True)
    if fit != "gaussian":
        assert np.array_equal(_np(r1.se_sigma), se_vol[2].reshape(-1)[sel], equal_nan=True)
    assert np.isfinite(se_vol[0][mask]).mean() > (0.9 if fit != "rician" else 0.0)
    if device:                                     # an index tensor in host memory is moved to the echoes' GPU
        for dt in (torch.int64, torch.int32):
            r2 = gpu_lib.fit_voxels_batch(cv(flat), torch.from_numpy(idx).to(dt), te, fit, fp,
                                          want=("nit", "fun", "status", "se"), **kw)
            for f in FIELDS + ("se_k", "se_t2") + (("se_sigma",) if fit != "gaussian" else ()):
                assert np.array_equal(_np(getattr(r1, f)), _np(getattr(r2, f)), equal_nan=True), f


# Calibration: 2^16 seeded noise realisations of one voxel per fit, 32 echoes at TE = 10..320 ms, bounds far from the
# answer (no bound hits).  The empirical std of the fitted T2 against the median se_T2 of the same fits.
#   gaussian         k = 2000, T2 = 100 ms, Gaussian noise sd 20 (SNR 100 at TE = 0), fast solver
#   gaussian_rician  k = 1500, T2 = 60 ms, floor sigma = 50, Gaussian noise sd 10 around sqrt(k^2 u^2 + sigma^2) (SNR 150),
#                    fast solver, init_mode="best"
#   rician           k = 1500, T2 = 60 ms, Rician noise sigma = 20 (SNR 75), lbfgsb_dense with ftol=1e-12, gtol=1e-8
CALIBRATION = [("gaussian", (2000.0, 100.0), 20.0, "fast", 0.05),
               ("gaussian_rician", (1500.0, 60.0, 50.0), 10.0, "fast", 0.10),
               ("rician", (1500.0, 60.0), 20.0, "lbfgsb_dense", 0.10)]


@pytest.mark.parametrize("fit,theta,noise,solver,tol", CALIBRATION, ids=[c[0] for c in CALIBRATION])
def test_standard_error_is_calibrated(gpu_lib, fit, theta, noise, solver, tol):
    import torch
    n = 1 << 16
    te = np.linspace(10.0, 320.0, 32)
    rng = np.random.default_rng(2024)
    if fit == "gaussian":
        y = model_mono(te, *theta)[None] + rng.normal(0, noise, (n, te.size))
    elif fit == "gaussian_rician":
        y = model_floor(te, *theta)[None] + rng.normal(0, noise, (n, te.size))
    else:
        s = model_mono(te, *theta)[None]
        y = np.sqrt((s + rng.normal(0, noise, (n, te.size))) ** 2 + rng.normal(0, noise, (n, te.size)) ** 2)
    x0 = list(theta) + ([noise] if fit == "rician" else [])
    bounds = [(1.0, 1e5), (1.0, 5000.0)] + ([(0.1, 1e4)] if fit != "gaussian" else [])
    fp = {"initial_guess": x0, "param_bounds": bounds, "solver": "L-BFGS-B",
          "options": {"ftol": 1e-12, "gtol": 1e-8, "maxls": 50}}
    r = gpu_lib.fit_voxels_batch(torch.from_numpy(y.astype(np.float32)).cuda(), None, te, fit, fp, prior=True, solver=solver,
                                 init_mode="best" if fit == "gaussian_rician" else "auto", want=("nit", "fun", "status", "se"))
    t2, se = _np(r.t2).astype(np.float64), _np(r.se_t2).astype(np.float64)
    lo, hi = np.array([b[0] for b in bounds]), np.array([b[1] for b in bounds])
    par = _np(r.results)
    assert not np.any(np.isclose(par, lo) | np.isclose(par, hi)), "a fit reached a bound"
    assert np.isfinite(se).mean() >= 0.999
    ratio = t2.std() / np.median(se[np.isfinite(se)])
    print(f"[stderr calibration] {fit}: std(T2) {t2.std():.4f} ms, median se_T2 {np.median(se[np.isfinite(se)]):.4f} ms, "
          f"ratio {ratio:.4f}, status != 0: {(_np(r.status) != 0).mean():.4f}")
    assert abs(ratio - 1.0) <= tol


def test_empty_call_and_argument_errors(gpu_lib):
    import torch
    from fetal_t2mapping_b200 import _abi
    lib = _abi.load_library()
    y = torch.ones((8, 4), dtype=torch.float32, device="cuda")
    par = torch.ones(8, dtype=torch.float32, device="cuda")
    out = torch.zeros(8, dtype=torch.float32, device="cuda")
    te = np.array([10.0, 20.0, 30.0, 40.0])

    def problem(**kw):
        p = _abi.Problem()
        p.echoes, p.layout, p.memory, p.n_vox, p.n_fit, p.n_echo = y.data_ptr(), _abi.LAYOUT_AOS, _abi.MEM_DEVICE, 8, 8, 4
        p.model, p.te_ms = _abi.MODEL_GAUSSIAN_RICIAN, te.ctypes.data_as(C.POINTER(C.c_double))
        for f, v in kw.items():
            setattr(p, f, v)
        return p

    def call(p, k=par.data_ptr(), t2=par.data_ptr(), s=par.data_ptr()):
        return lib.t2fit_stderr(C.byref(p), k, t2, s, 0, out.data_ptr(), out.data_ptr(), out.data_ptr(), None)
    assert call(problem(n_fit=0), None, None, None) == 0                               # a no-op, NULL pointers and all
    torch.cuda.synchronize()
    assert float(out.abs().sum()) == 0.0
    assert call(problem()) == 0
    torch.cuda.synchronize()
    assert call(problem(layout=_abi.LAYOUT_SOA)) == -1
    assert call(problem(layout=_abi.LAYOUT_PLANES)) == -1
    assert call(problem(memory=_abi.MEM_HOST)) == -1
    assert call(problem(n_echo=1)) == -1 and call(problem(n_echo=33)) == -1
    assert call(problem(), k=None) == -1 and call(problem(), t2=None) == -1 and call(problem(), s=None) == -1
    assert call(problem(model=_abi.MODEL_GAUSSIAN), s=None) == 0                       # sigma is not needed for 2 parameters
    assert call(problem(echoes=None)) == -1
    torch.cuda.synchronize()
