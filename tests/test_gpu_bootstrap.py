"""Parametric bootstrap on the GPU (t2fit_bootstrap_replicates / replicate_kernel, the refit through fit_voxels_into,
t2fit_bootstrap_stats / bootstrap_stats_kernel): the generator against the numpy oracle through every input path, the
statistics against the host build, zero noise, agreement with a Monte Carlo of the estimator, calibration, invariance
to chunking / indices / input memory, and no effect on any existing output."""
import ctypes as C

import numpy as np
import pytest

from oracle import bootstrap_oracle as bo
from oracle.fit_oracle import model_floor, model_mono
from tests.conftest import fit_params_of, load_golden
from tests.hostsim import pass_shim as bootstrap_shim

pytestmark = pytest.mark.gpu

GEN_FIXTURES = ["c2_gaussian_hf_prior", "norm_gaussian", "c3_floor_prior", "c3_rician_prior", "cli3_rician_hf_prior"]
FIELDS = ("mean", "sd", "t2_lo", "t2_hi", "n_used", "n_ok")


def _np(a):
    return None if a is None else (a.cpu().numpy() if hasattr(a, "cpu") else np.asarray(a))


def _ulps(a, b):
    return np.abs(a.view(np.int32).astype(np.int64) - b.view(np.int32).astype(np.int64))


def _scatter(g, seed=0):
    """The fixture's rows at ascending scattered positions of a larger array (faint rows elsewhere) and their index."""
    rows = np.ascontiguousarray(g["rows"], np.float32)
    m, E = rows.shape
    rng = np.random.default_rng(seed)
    idx = np.sort(rng.choice(3 * m, m, replace=False)).astype(np.int64)
    big = np.abs(rng.normal(5.0, 1.0, (3 * m, E))).astype(np.float32)
    big[idx] = rows
    return big, idx


def _replicates(gpu_lib, y, idx, te, fit, norm, k, t2, s, noise, vid, seed, n_rep):
    """t2fit_bootstrap_replicates on device rows ``y`` (index ``idx`` torch int32 / int64 or None)."""
    import torch
    from fetal_t2mapping_b200 import _abi
    api = gpu_lib.api
    lib = _abi.load_library()
    p = _abi.Problem()
    keep = [api._fill_problem(p, fit, gpu_lib.preset(fit, True)[1], te, True, norm, 0, 0.0, "auto")]
    keep.append(api._device_rows(p, y, idx))
    dev = lambda a, dt=torch.float32: None if a is None else torch.as_tensor(np.asarray(a)).to("cuda", dt).contiguous()
    par = [dev(k), dev(t2), dev(s), dev(noise), dev(vid, torch.int64)]
    out = torch.full((p.n_fit * n_rep, p.n_echo), -1.0, dtype=torch.float32, device="cuda")
    ptr = lambda t: None if t is None else t.data_ptr()
    rc = lib.t2fit_bootstrap_replicates(C.byref(p), *[ptr(t) for t in par], seed, n_rep, out.data_ptr(),
                                        torch.cuda.current_stream().cuda_stream)
    assert rc == 0, lib.t2fit_last_error()
    torch.cuda.synchronize()
    return out.cpu().numpy()


@pytest.mark.parametrize("name", GEN_FIXTURES)
def test_generator_matches_oracle(gpu_lib, name):
    """Rows within 1 float32 ulp of the oracle and bit-equal on >= 99.9 % of the echoes: every model, int64 / int32 / no
    index, an explicit voxel_id, with and without noise_sd and norm."""
    import torch
    g = load_golden(name)
    fit, te = g["fit"], g["te"]
    p = g["ref_params"].astype(np.float32)
    k, t2, s = p[:, 0], p[:, 1], (p[:, 2] if fit != "gaussian" else None)
    big, idx = _scatter(g)
    m = idx.size
    noise = np.random.default_rng(1).uniform(0.0, 30.0, m).astype(np.float32)
    yd = torch.from_numpy(big).cuda()
    B, seed = 32, 0xFEDCBA9876543210
    cases = [("i64", torch.from_numpy(idx).cuda(), None, idx), ("i32", torch.from_numpy(idx.astype(np.int32)).cuda(), None, idx),
             ("vid", torch.from_numpy(idx).cuda(), idx * 7 + (1 << 35), idx * 7 + (1 << 35))]
    exact, total = 0, 0
    for norm in (False, True):
        for ns in (None, noise):
            for tag, ti, vid, key in cases:
                got = _replicates(gpu_lib, yd, ti, te, fit, norm, k, t2, s, ns, vid, seed, B)
                want = bo.replicate_rows(big[idx], te, fit, norm, k, t2, s, ns, voxel_id=key, seed=seed, n_rep=B)
                assert np.array_equal(np.isnan(got), np.isnan(want)), (tag, norm)
                f = np.isfinite(want)
                if f.any():
                    assert _ulps(got[f], want[f]).max() <= 1, (tag, norm)
                exact += int((_ulps(got[f], want[f]) == 0).sum())
                total += int(f.sum())
            # no index: rows 0..m-1, keyed by the row
            got = _replicates(gpu_lib, yd[:m].contiguous(), None, te, fit, norm, k, t2, s, ns, None, seed, B)
            want = bo.replicate_rows(big[:m], te, fit, norm, k, t2, s, ns, seed=seed, n_rep=B)
            assert np.array_equal(np.isnan(got), np.isnan(want))
            f = np.isfinite(want)
            if f.any():
                assert _ulps(got[f], want[f]).max() <= 1
    print(f"[bootstrap generator] {name}: bit-equal {exact / max(total, 1):.6f} of {total} echoes")
    assert total == 0 or exact / total >= 0.999


def test_index_out_of_range_gives_nan_rows(gpu_lib):
    import torch
    g = load_golden("c2_gaussian_hf_prior")
    p = g["ref_params"].astype(np.float32)
    y = torch.from_numpy(np.ascontiguousarray(g["rows"][:4])).cuda()
    idx = torch.tensor([0, 7, -1, 3], dtype=torch.int64, device="cuda")
    got = _replicates(gpu_lib, y, idx, g["te"], "gaussian", False, p[:4, 0], p[:4, 1], None, None, None, 5, 16).reshape(4, 16, -1)
    assert np.isnan(got[1]).all() and np.isnan(got[2]).all()
    assert np.isfinite(got[0]).all() and np.isfinite(got[3]).all()


@pytest.mark.parametrize("fit", ["gaussian", "gaussian_rician", "rician"])
def test_stats_kernel_matches_host_build(gpu_lib, fit):
    """Bit for bit the host build of the same arithmetic (fixed summation order), and numpy within 1 ulp."""
    import torch
    from fetal_t2mapping_b200 import _abi
    lib = _abi.load_library()
    rng = np.random.default_rng(3)
    for B in (16, 200, 333, 4096):
        m = 64 if B < 4096 else 4
        P = 2 if fit == "gaussian" else 3
        k = rng.normal(1000.0, 40.0, m * B).astype(np.float32)
        t2 = rng.normal(80.0, 6.0, m * B).astype(np.float32)
        t2[:B] = np.round(t2[:B])
        s = rng.normal(20.0, 2.0, m * B).astype(np.float32) if P == 3 else None
        st = rng.choice(np.array([0, 1, 2, 3], np.uint8), m * B, p=[0.7, 0.1, 0.15, 0.05])
        st[B:2 * B] = 1
        st[2 * B:3 * B] = 3
        st[2 * B + 4] = 0
        k[3 * B + 1] = np.nan
        d = lambda a: None if a is None else torch.from_numpy(a).cuda()
        outs = [torch.empty(3 * m, device="cuda"), torch.empty(3 * m, device="cuda"), torch.empty(m, device="cuda"),
                torch.empty(m, device="cuda"), torch.empty(m, dtype=torch.int32, device="cuda"),
                torch.empty(m, dtype=torch.int32, device="cuda")]
        ins = [d(k), d(t2), d(s), d(st)]
        rc = lib.t2fit_bootstrap_stats(_abi.MODELS[fit], m, B, *[None if t is None else t.data_ptr() for t in ins], 0.9,
                                       *[t.data_ptr() for t in outs], None)
        assert rc == 0
        torch.cuda.synchronize()
        got = [o.cpu().numpy() for o in outs]
        got[0], got[1] = got[0].reshape(3, m), got[1].reshape(3, m)
        host = bootstrap_shim.bootstrap_stats(fit, B, k, t2, s, st, 0.9)
        ref = bo.bootstrap_stats(fit, B, k, t2, s, st, 0.9)
        for a, h, r in zip(got, host, ref):
            assert np.array_equal(a, h, equal_nan=True), B
            if a.dtype.kind == "f":
                r = r.astype(np.float32)
                f = np.isfinite(r)
                assert np.array_equal(np.isnan(a), np.isnan(r)) and _ulps(a[f], r[f]).max() <= 1
            else:
                assert np.array_equal(a, r)


@pytest.mark.parametrize("fit,solver", [("gaussian", "fast"), ("gaussian_rician", "lbfgsb_dense"), ("gaussian_rician", "fast"),
                                        ("rician", "lbfgsb_dense")])
def test_zero_noise(gpu_lib, fit, solver):
    """noise_sd = 0: every replicate row is the model row, every refit is the fit of that row, SD = 0, lo = hi = mean."""
    import torch
    te = np.linspace(20.0, 320.0, 10)
    rng = np.random.default_rng(4)
    m = 64
    k = rng.uniform(600.0, 2000.0, m).astype(np.float32)
    t2 = rng.uniform(40.0, 300.0, m).astype(np.float32)
    s = rng.uniform(5.0, 40.0, m).astype(np.float32) if fit != "gaussian" else None
    mu, _, _ = bo.source(np.ones((m, te.size), np.float32), te, fit, False, k, t2, s, np.zeros(m, np.float32))
    rows = mu.astype(np.float32)
    fp = gpu_lib.preset(fit, True)[1]
    yd = torch.from_numpy(rows).cuda()
    gen = _replicates(gpu_lib, yd, None, te, fit, False, k, t2, s, np.zeros(m, np.float32), None, 0, 16)
    assert np.array_equal(gen, np.repeat(rows, 16, axis=0))
    r = gpu_lib.fit_voxels_batch(yd, None, te, fit, fp, prior=True, solver=solver)
    b = gpu_lib.parametric_bootstrap(yd, None, te, fit, fp, prior=True, n_rep=16, noise_sd=0.0, params=(k, t2, s),
                                     solver=solver)
    torch.cuda.synchronize()
    st = _np(r.status)
    used = (st == 0) | (st == 2)
    assert np.array_equal(_np(b.n_used), np.where(used, 16, 0)) and np.array_equal(_np(b.n_ok), np.where(st == 0, 16, 0))
    P = 2 if fit == "gaussian" else 3
    fitted = _np(r.results).astype(np.float32)[:, :P]
    mean, sd = _np(b.mean), _np(b.sd)
    assert np.array_equal(mean[used], fitted[used])
    assert np.all(sd[used] == 0)
    assert np.array_equal(_np(b.t2_lo)[used], fitted[used, 1]) and np.array_equal(_np(b.t2_hi)[used], fitted[used, 1])
    assert used.mean() >= 0.9


TE32 = np.linspace(10.0, 320.0, 32)
TE_C3 = np.array([113, 133, 152, 176, 203, 230, 254, 296, 340, 400, 480, 600], float)
_WIDE = {"initial_guess": None, "param_bounds": None, "solver": "L-BFGS-B", "options": {"ftol": 1e-12, "gtol": 1e-8, "maxls": 50}}
# (id, fit, truth (k, T2[, sigma]), noise, TE, solver, init_mode, fit_params or None = wide bounds around the truth)
MONTE_CARLO = [("gaussian", "gaussian", (2000.0, 100.0), 20.0, TE32, "fast", "auto", None),
               ("gaussian_rician", "gaussian_rician", (1500.0, 60.0, 50.0), 10.0, TE32, "fast", "best", None),
               ("rician", "rician", (1500.0, 60.0, 20.0), 20.0, TE32, "lbfgsb_dense", "auto", None),
               ("c3_gaussian_rician_lf", "gaussian_rician", (1500.0, 90.0, 20.0), 20.0, TE_C3, "lbfgsb_dense", "auto", "lf")]


def _mc_rows(rng, fit, theta, noise, te, n):
    if fit == "gaussian":
        return model_mono(te, *theta)[None] + rng.normal(0, noise, (n, te.size))
    if fit == "gaussian_rician":
        return model_floor(te, *theta)[None] + rng.normal(0, noise, (n, te.size))
    s = model_mono(te, *theta[:2])[None]
    return np.sqrt((s + rng.normal(0, noise, (n, te.size))) ** 2 + rng.normal(0, noise, (n, te.size)) ** 2)


@pytest.mark.parametrize("case", MONTE_CARLO, ids=[c[0] for c in MONTE_CARLO])
def test_bootstrap_is_the_estimators_monte_carlo(gpu_lib, case):
    """One voxel with params = the truth and noise_sd = the true noise, B = 4096, against 2^16 independent numpy-noise rows
    fitted by fit_voxels_batch: SD within 5 %, mean within 3 Monte Carlo standard errors, lo / hi within 5 %."""
    import torch
    _, fit, theta, noise, te, solver, init_mode, preset = case
    if preset is None:
        fp = dict(_WIDE, initial_guess=list(theta), param_bounds=[(1.0, 1e5), (1.0, 5000.0)] + ([(0.1, 1e4)] if fit != "gaussian" else []))
    else:
        fp = gpu_lib.preset(fit, preset == "lf")[1]
    rng = np.random.default_rng(2025)
    y_obs = _mc_rows(rng, fit, theta, noise, te, 1).astype(np.float32)
    th = np.asarray(theta + ((0.0,) if fit == "gaussian" else ()), np.float32)
    b = gpu_lib.parametric_bootstrap(torch.from_numpy(y_obs).cuda(), None, te, fit, fp, prior=True, n_rep=4096, seed=11,
                                     noise_sd=noise, params=(th[:1], th[1:2], th[2:3] if fit != "gaussian" else None),
                                     solver=solver, init_mode=init_mode)
    mc = _mc_rows(rng, fit, theta, noise, te, 1 << 16).astype(np.float32)
    r = gpu_lib.fit_voxels_batch(torch.from_numpy(mc).cuda(), None, te, fit, fp, prior=True, solver=solver, init_mode=init_mode)
    torch.cuda.synchronize()
    st, t2 = _np(r.status), _np(r.t2).astype(np.float64)
    t2 = t2[((st == 0) | (st == 2)) & np.isfinite(t2)]
    m_mc, s_mc = t2.mean(), t2.std(ddof=1)
    q_lo, q_hi = np.quantile(t2, [0.025, 0.975])
    mean, sd = float(_np(b.mean)[0, 1]), float(_np(b.sd)[0, 1])
    lo, hi = float(_np(b.t2_lo)[0]), float(_np(b.t2_hi)[0])
    n_used = int(_np(b.n_used)[0])
    se = s_mc * np.sqrt(1.0 / n_used + 1.0 / t2.size)
    print(f"[bootstrap MC] {case[0]}: sd {sd:.4f} vs {s_mc:.4f}, mean {mean:.4f} vs {m_mc:.4f} ({abs(mean - m_mc) / se:.2f} se), "
          f"lo {lo:.3f} vs {q_lo:.3f}, hi {hi:.3f} vs {q_hi:.3f}, n_used {n_used}, n_ok {int(_np(b.n_ok)[0])}")
    assert n_used >= 4000
    assert abs(sd / s_mc - 1.0) <= 0.05
    assert abs(mean - m_mc) <= 3.0 * se
    assert abs(lo / q_lo - 1.0) <= 0.05 and abs(hi / q_hi - 1.0) <= 0.05


def test_calibration_gaussian_32_echoes(gpu_lib):
    """4096 noisy voxels (k = 2000, T2 = 100 ms, sd 20, 32 echoes), B = 400, s estimated: the 95 % percentile interval covers
    the true T2 in [0.93, 0.97] of the voxels, and the median t2_sd / se_T2 lies in [0.95, 1.05]."""
    import torch
    theta, noise, n = (2000.0, 100.0), 20.0, 4096
    rng = np.random.default_rng(77)
    y = torch.from_numpy(_mc_rows(rng, "gaussian", theta, noise, TE32, n).astype(np.float32)).cuda()
    fp = dict(_WIDE, initial_guess=list(theta), param_bounds=[(1.0, 1e5), (1.0, 5000.0)])
    r = gpu_lib.fit_voxels_batch(y, None, TE32, "gaussian", fp, prior=True, solver="fast", want=("status", "se"))
    b = gpu_lib.parametric_bootstrap(y, None, TE32, "gaussian", fp, prior=True, n_rep=400, seed=3,
                                     params=(r.k, r.t2, None), solver="fast")
    torch.cuda.synchronize()
    lo, hi = _np(b.t2_lo), _np(b.t2_hi)
    cover = float(np.mean((lo <= theta[1]) & (theta[1] <= hi)))
    ratio = float(np.median(_np(b.sd)[:, 1] / _np(r.se_t2)))
    print(f"[bootstrap calibration] coverage {cover:.4f}, median t2_sd / se_T2 {ratio:.4f}")
    assert 0.93 <= cover <= 0.97
    assert 0.95 <= ratio <= 1.05


def test_finite_where_stderr_is_nan(gpu_lib):
    """c3_rician_prior fitted with its preset: section 11 is NaN on most voxels; t2_sd is finite on every voxel with valid
    echoes."""
    import torch
    g = load_golden("c3_rician_prior")
    fp = fit_params_of(g)
    rows = np.ascontiguousarray(g["rows"])
    r = gpu_lib.fit_voxels_batch(rows, None, g["te"], g["fit"], fp, prior=g["prior"], want=("status", "se"))
    b = gpu_lib.parametric_bootstrap(rows, None, g["te"], g["fit"], fp, prior=g["prior"], n_rep=200,
                                     params=(r.k, r.t2, r.sigma))
    valid = np.isfinite(rows).all(axis=1) & (rows > 0).all(axis=1)
    sd = b.sd[:, 1]
    print(f"[bootstrap c3_rician_prior] stderr NaN share {np.isnan(r.se_t2).mean():.4f}, t2_sd finite on "
          f"{np.isfinite(sd[valid]).mean():.4f} of valid voxels, n_ok share {b.n_ok.sum() / (200 * rows.shape[0]):.4f}, "
          f"n_used share {b.n_used.sum() / (200 * rows.shape[0]):.4f}")
    assert np.isfinite(sd[valid]).all()
    assert isinstance(b.sd, np.ndarray) and b.mean.shape == (rows.shape[0], 3)


INVARIANCE = [("c2_gaussian_hf_prior", "auto"), ("c3_floor_prior", "auto"), ("c3_floor_prior", "fast"), ("c3_rician_prior", "auto")]


@pytest.mark.parametrize("name,solver", INVARIANCE, ids=[f"{n}-{s}" for n, s in INVARIANCE])
def test_invariance(gpu_lib, name, solver):
    """Bit-identical results for chunk = 1, 7 and the default; a subset of mask_indices against the whole; int32 against
    int64 indices; host against device input; two runs with the same seed.  Another seed changes the result."""
    import torch
    g = load_golden(name)
    fp = fit_params_of(g)
    big, idx = _scatter(g, 9)
    kw = dict(prior=g["prior"], norm=g["norm"], n_rep=16, seed=1234, solver=solver)
    fit, te = g["fit"], g["te"]

    def run(y, ix, **extra):
        res = gpu_lib.parametric_bootstrap(y, ix, te, fit, fp, **dict(kw, **extra))
        torch.cuda.synchronize()
        return [_np(getattr(res, f)) for f in FIELDS]

    def same(a, b, what):
        for f, x, z in zip(FIELDS, a, b):
            assert np.array_equal(x, z, equal_nan=True), (what, f)

    yd, id64 = torch.from_numpy(big).cuda(), torch.from_numpy(idx).cuda()
    ref = run(yd, id64)
    same(ref, run(yd, id64, chunk=1), "chunk=1")
    same(ref, run(yd, id64, chunk=7), "chunk=7")
    same(ref, run(yd, id64.to(torch.int32)), "int32")
    same(ref, run(big, idx), "host")
    same(ref, run(big, idx.astype(np.int32), chunk=7), "host int32")
    same(ref, run(yd, id64), "repeat")
    sub = np.arange(3, idx.size, 5)
    part = run(yd, id64[torch.from_numpy(sub).cuda()])
    same([a[sub] for a in ref], part, "subset")
    other = run(yd, id64, seed=1235)
    assert not np.array_equal(other[1], ref[1], equal_nan=True)
    assert np.isfinite(ref[1][:, 1]).mean() >= 0.9


@pytest.mark.parametrize("fit,solver", [("gaussian", "auto"), ("gaussian_rician", "auto"), ("rician", "auto")])
@pytest.mark.parametrize("device", [True, False], ids=["device", "host"])
def test_volume_maps_and_nothing_else_moves(gpu_lib, fit, solver, device):
    """t2map_volume maps, standard errors and interval are bit-identical with bootstrap on and off; the bootstrap maps are
    those of parametric_bootstrap at the fitted maps, zeros off-mask."""
    import torch
    from fetal_t2mapping_b200 import synth
    y, mask, te, _ = synth.make_volume("c1", scale=0.25)
    _, fp = gpu_lib.preset(fit, True)
    cv = (lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()) if device else (lambda a: a)
    kw = dict(prior=False, norm=False, solver=solver, stderr=True, t2_interval=0.95)
    off = gpu_lib.t2map_volume(cv(y), cv(mask), te, fit, fp, **kw)
    on = gpu_lib.t2map_volume(cv(y), cv(mask), te, fit, fp, bootstrap=32, **kw)
    assert len(off) == 6 and len(on) == 7
    for a, b in zip(off, on[:6]):
        a, b = (a,) if not isinstance(a, tuple) else a, (b,) if not isinstance(b, tuple) else b
        for x, z in zip(a, b):
            assert np.array_equal(_np(x), _np(z), equal_nan=True)
    bm = on[6]
    assert isinstance(bm, gpu_lib.BootstrapMaps)
    idx = np.flatnonzero(mask.reshape(-1))
    flat = np.ascontiguousarray(y.reshape(-1, te.size))
    t2m, km, sm = (_np(on[i]).reshape(-1)[idx] for i in (0, 1, 2))
    ref = gpu_lib.parametric_bootstrap(flat, idx, te, fit, fp, prior=False, n_rep=32, solver=solver,
                                       params=(km, t2m, sm if fit != "gaussian" else None))
    want = {"t2_mean": ref.mean[:, 1], "t2_sd": ref.sd[:, 1], "t2_lo": ref.t2_lo, "t2_hi": ref.t2_hi, "k_sd": ref.sd[:, 0],
            "sigma_sd": ref.sd[:, 2] if fit != "gaussian" else np.zeros(idx.size, np.float32), "n_used": ref.n_used,
            "n_ok": ref.n_ok}
    for f, w in want.items():
        a = _np(getattr(bm, f))
        assert a.shape == mask.shape and np.all(a[~mask] == 0), f
        assert np.array_equal(a.reshape(-1)[idx], w, equal_nan=True), f
    assert np.isfinite(_np(bm.t2_sd)[mask]).mean() >= 0.9


def test_argument_errors(gpu_lib):
    import torch
    from fetal_t2mapping_b200 import _abi
    lib = _abi.load_library()
    te = np.array([10.0, 20.0, 30.0, 40.0])
    y = np.abs(np.random.default_rng(0).normal(100, 10, (8, 4))).astype(np.float32)
    fp = gpu_lib.preset("gaussian", True)[1]
    for bad in (dict(n_rep=15), dict(n_rep=4097), dict(level=0.0), dict(level=1.0)):
        with pytest.raises(ValueError):
            gpu_lib.parametric_bootstrap(y, None, te, "gaussian", fp, **bad)
    with pytest.raises(ValueError):
        gpu_lib.parametric_bootstrap(y, None, te, "gaussian", fp, noise_sd=np.ones(3))
    with pytest.raises(ValueError):
        gpu_lib.parametric_bootstrap(y, None, te, "gaussian_rician", gpu_lib.preset("gaussian_rician", True)[1],
                                     params=(np.ones(8), np.ones(8), None))
    with pytest.raises(ValueError):
        gpu_lib.t2map_volume(y.reshape(2, 2, 2, 4), np.ones((2, 2, 2), bool), te, "gaussian", fp, bootstrap=8)
    yd = torch.from_numpy(y).cuda()
    par = torch.ones(8, dtype=torch.float32, device="cuda")
    rows = torch.empty((8 * 16, 4), dtype=torch.float32, device="cuda")
    p = _abi.Problem()
    p.echoes, p.layout, p.memory, p.n_vox, p.n_fit, p.n_echo = yd.data_ptr(), _abi.LAYOUT_AOS, _abi.MEM_DEVICE, 8, 8, 4
    p.model, p.te_ms = _abi.MODEL_GAUSSIAN_RICIAN, te.ctypes.data_as(C.POINTER(C.c_double))
    rep = lambda q, n_rep=16, s=par.data_ptr(), out=rows.data_ptr(): lib.t2fit_bootstrap_replicates(
        C.byref(q), par.data_ptr(), par.data_ptr(), s, None, None, 0, n_rep, out, None)
    assert rep(p) == 0
    assert rep(p, n_rep=15) == -1 and rep(p, n_rep=4097) == -1
    assert rep(p, s=None) == -1 and rep(p, out=None) == -1
    for f, v in (("layout", _abi.LAYOUT_SOA), ("memory", _abi.MEM_HOST), ("n_echo", 1), ("model", 7)):
        q = _abi.Problem.from_buffer_copy(p)
        setattr(q, f, v)
        assert rep(q) == -1, f
    st = torch.zeros(8 * 16, dtype=torch.uint8, device="cuda")
    stats = lambda model=1, n_rep=16, level=0.95, s=par.data_ptr(): lib.t2fit_bootstrap_stats(
        model, 8 if n_rep == 16 else 1, n_rep, rows.data_ptr(), rows.data_ptr(), s, st.data_ptr(), level,
        *([None] * 6), None)
    assert stats() == 0
    assert stats(level=0.0) == -1 and stats(level=1.0) == -1 and stats(level=float("nan")) == -1
    assert stats(n_rep=15) == -1 and stats(n_rep=4097) == -1 and stats(model=3) == -1 and stats(s=None) == -1
    assert stats(model=0, s=None) == 0
    torch.cuda.synchronize()
