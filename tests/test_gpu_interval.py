"""Profile-likelihood T2 intervals on the GPU (t2fit_t2_interval / interval_kernel): against the float64 oracle on every
fit fixture and the edge fixtures through every input path, the public entries agreeing bit for bit, nothing else moving,
and the coverage of the true T2 over noise realisations."""
import ctypes as C

import numpy as np
import pytest

from oracle import interval_oracle as io
from oracle.fit_oracle import model_floor, model_mono
from tests.conftest import fit_params_of, load_golden
from tests.test_interval_cpu import EDGE, FIXTURES, compare, q_of, sample

pytestmark = pytest.mark.gpu

_ORACLE = {}


def _np(a):
    return None if a is None else (a.cpu().numpy() if hasattr(a, "cpu") else np.asarray(a))


def _oracle(name, G, vox):
    key = (name, G)
    if key not in _ORACLE:
        g = load_golden(name)
        box, empty = io.voxel_box(g["fit"], fit_params_of(g), g["prior"], g["rows"])
        _ORACLE[key] = io.interval_rows(g["rows"], g["te"], g["fit"], g["norm"], box, empty, q_of(g["fit"], g["te"].size), G,
                                        vox)
    return _ORACLE[key]


@pytest.mark.parametrize("G", [16, 64, 256])
@pytest.mark.parametrize("name", FIXTURES + EDGE)
def test_interval_matches_oracle(gpu_lib, name, G):
    """Host input, device input with int64 and int32 indices, compact and dense outputs: the same bits, and the oracle's
    thresholds (tests/test_interval_cpu.py::compare).  The 3-parameter fixtures on a fixed voxel sample (fewer at G = 256)."""
    import torch
    from fetal_t2mapping_b200 import _abi
    g = load_golden(name)
    fp = fit_params_of(g)
    vox = sample(g, n3=12 if G < 256 else 4)
    rows = np.ascontiguousarray(g["rows"])
    kw = dict(prior=g["prior"], norm=g["norm"], n_grid=G, profile=True)
    host = gpu_lib.t2_interval(rows, vox, g["te"], g["fit"], fp, **kw)
    ref = _oracle(name, G, vox)
    got = tuple(np.asarray(a, np.float64) if j < 3 else a for j, a in enumerate(host[:5]))
    compare(ref[:5], got, f"{name}/G={G}")
    assert np.allclose(host[5], io.grid(*io.voxel_box(g["fit"], fp, g["prior"], rows[:1])[0][0, 2:4], G), rtol=1e-15)
    yd = torch.from_numpy(rows).cuda()
    for idt in (torch.int64, torch.int32):
        idx = torch.from_numpy(vox).to(device="cuda", dtype=idt)
        dev = gpu_lib.t2_interval(yd, idx, g["te"], g["fit"], fp, **kw)
        torch.cuda.synchronize()
        for a, b in zip(host[:5], dev[:5]):
            assert np.array_equal(_np(a), _np(b), equal_nan=True), (name, G, idt)
        # dense outputs indexed by row, through the C entry
        p = _abi.Problem()
        keep = gpu_lib.api._fill_problem(p, g["fit"], fp, g["te"], g["prior"], g["norm"], 0, 0.0, "auto")
        p.echoes, p.memory, p.layout, p.mask_idx = yd.data_ptr(), _abi.MEM_DEVICE, _abi.LAYOUT_AOS, idx.data_ptr()
        p.idx_dtype = _abi.IDX_I32 if idt == torch.int32 else _abi.IDX_I64
        p.n_vox, p.n_fit = rows.shape[0], vox.size
        d = torch.zeros((3, rows.shape[0]), dtype=torch.float32, device="cuda")
        df = torch.zeros(rows.shape[0], dtype=torch.uint8, device="cuda")
        gpu_lib.api._interval_launch(_abi.load_library(), p, q_of(g["fit"], g["te"].size), G, 1,
                                     [d[0].data_ptr(), d[1].data_ptr(), d[2].data_ptr(), df.data_ptr()], None,
                                     torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        del keep
        for j in range(3):
            assert np.array_equal(_np(d[j])[vox], _np(host[j]), equal_nan=True), (name, G, idt, j)
        assert np.array_equal(_np(df)[vox], _np(host[3]))
        rest = np.setdiff1d(np.arange(rows.shape[0]), vox)
        assert np.all(_np(d)[:, rest] == 0) and np.all(_np(df)[rest] == 0)


def _volume():
    from fetal_t2mapping_b200 import synth
    y, mask, te, _ = synth.make_volume("c1", scale=0.25)
    return y, mask, te


@pytest.mark.parametrize("fit,solver", [("gaussian", "auto"), ("gaussian_rician", "fast"), ("rician", "auto")])
@pytest.mark.parametrize("device", [True, False], ids=["device", "host"])
def test_entries_agree_and_nothing_else_moves(gpu_lib, fit, solver, device):
    """t2map_volume(t2_interval=0.95) == t2_interval on the masked rows, bit for bit, zeros off-mask; the four maps and the
    standard errors are bit-identical with the interval requested or not."""
    import torch
    y, mask, te = _volume()
    _, fp = gpu_lib.preset(fit, True)
    flat = np.ascontiguousarray(y.reshape(-1, te.size))
    idx = np.flatnonzero(mask.reshape(-1))
    cv = (lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()) if device else (lambda a: a)
    kw = dict(prior=False, norm=False, solver=solver)
    maps0 = gpu_lib.t2map_volume(cv(y), cv(mask), te, fit, fp, stderr=True, **kw)
    maps1 = gpu_lib.t2map_volume(cv(y), cv(mask), te, fit, fp, stderr=True, t2_interval=0.95, **kw)
    maps2 = gpu_lib.t2map_volume(cv(y), cv(mask), te, fit, fp, t2_interval=0.95, **kw)
    assert len(maps0) == 5 and len(maps1) == 6 and len(maps2) == 5
    for a, b, c in zip(maps0[:4], maps1[:4], maps2[:4]):
        assert np.array_equal(_np(a), _np(b), equal_nan=True) and np.array_equal(_np(a), _np(c), equal_nan=True)
    for a, b in zip(maps0[4], maps1[4]):
        assert np.array_equal(_np(a), _np(b), equal_nan=True)
    for a, b in zip(maps1[5], maps2[4]):
        assert np.array_equal(_np(a), _np(b), equal_nan=True)
    iv = [_np(a) for a in maps1[5]]
    lo, hi, best, fl = (_np(a) for a in gpu_lib.t2_interval(cv(flat), cv(idx), te, fit, fp, prior=False, norm=False))
    sel = mask.reshape(-1)
    for a, b in zip(iv, (lo, hi, best, fl)):
        assert a.shape == mask.shape and np.array_equal(a.reshape(-1)[sel], b, equal_nan=True)
        assert np.all(a[~mask] == 0)
    assert iv[0].dtype == np.float32 and iv[3].dtype == np.uint8
    valid = (fl & 8) == 0
    assert valid.mean() > (0.9 if fit != "rician" else 0.0)
    assert np.all(lo[valid] <= best[valid]) and np.all(best[valid] <= hi[valid])
    if device:                                     # an index tensor in host memory is moved to the echoes' GPU
        for dt in (torch.int64, torch.int32):
            got = gpu_lib.t2_interval(cv(flat), torch.from_numpy(idx).to(dt), te, fit, fp, prior=False, norm=False)
            for a, b in zip(got, (lo, hi, best, fl)):
                assert np.array_equal(_np(a), b, equal_nan=True)


# The three scenarios of test_gpu_stderr.py::test_standard_error_is_calibrated (32 echoes at TE = 10..320 ms, bounds far
# from the answer), 2^16 seeded realisations each: coverage of the true T2 by the 95 % interval.
CALIBRATION = [("gaussian", (2000.0, 100.0), 20.0), ("gaussian_rician", (1500.0, 60.0, 50.0), 10.0),
               ("rician", (1500.0, 60.0), 20.0)]


@pytest.mark.parametrize("fit,theta,noise", CALIBRATION, ids=[c[0] for c in CALIBRATION])
def test_interval_is_calibrated(gpu_lib, fit, theta, noise):
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
    fp = {"initial_guess": x0, "param_bounds": bounds, "solver": "L-BFGS-B", "options": {}}
    lo, hi, best, fl = (_np(a) for a in gpu_lib.t2_interval(torch.from_numpy(y.astype(np.float32)).cuda(), None, te, fit,
                                                            fp, prior=True))
    valid = (fl & 8) == 0
    assert valid.mean() >= 0.999
    cov = np.mean((lo[valid] <= theta[1]) & (theta[1] <= hi[valid]))
    print(f"[interval calibration] {fit}: coverage {cov:.4f}, median width {np.median(hi[valid] - lo[valid]):.3f} ms, "
          f"flags {np.bincount(fl, minlength=9)[[0, 1, 2, 3, 4, 8]]}")
    assert 0.93 <= cov <= 0.97


def test_empty_call_and_argument_errors(gpu_lib):
    import torch
    from fetal_t2mapping_b200 import _abi
    lib = _abi.load_library()
    y = torch.ones((8, 4), dtype=torch.float32, device="cuda")
    out = torch.zeros(8, dtype=torch.float32, device="cuda")
    te = np.array([10.0, 20.0, 30.0, 40.0])

    def problem(**kw):
        p = _abi.Problem()
        p.echoes, p.layout, p.memory, p.n_vox, p.n_fit, p.n_echo = y.data_ptr(), _abi.LAYOUT_AOS, _abi.MEM_DEVICE, 8, 8, 4
        p.model, p.te_ms = _abi.MODEL_GAUSSIAN_RICIAN, te.ctypes.data_as(C.POINTER(C.c_double))
        p.lb[0], p.ub[0], p.lb[1], p.ub[1], p.lb[2], p.ub[2] = 0.0, 10.0, 10.0, 600.0, 0.1, 10.0
        for f, v in kw.items():
            setattr(p, f, v)
        return p

    def call(p, q=3.0, G=64):
        return lib.t2fit_t2_interval(C.byref(p), q, G, 0, out.data_ptr(), out.data_ptr(), out.data_ptr(), None, None, None)
    assert call(problem(n_fit=0)) == 0
    torch.cuda.synchronize()
    assert float(out.abs().sum()) == 0.0
    assert call(problem()) == 0
    torch.cuda.synchronize()
    assert call(problem(layout=_abi.LAYOUT_SOA)) == -1
    assert call(problem(memory=_abi.MEM_HOST)) == -1
    assert call(problem(n_echo=1)) == -1 and call(problem(n_echo=33)) == -1
    assert call(problem(), G=15) == -1 and call(problem(), G=257) == -1
    assert call(problem(), q=float("nan")) == -1 and call(problem(), q=-1.0) == -1
    p = problem()
    p.lb[1] = 0.0
    assert call(p) == -1
    p = problem()
    p.ub[1] = float("inf")
    assert call(p) == -1
    p = problem()
    p.lb[2] = 0.0
    assert call(p) == -1
    p = problem(model=_abi.MODEL_GAUSSIAN)
    p.lb[2] = 0.0
    assert call(p) == 0                                   # sigma bounds do not matter for 2 parameters
    assert call(problem(echoes=None)) == -1
    torch.cuda.synchronize()
    # an index outside [0, N): host input raises what the fit raises, device input gives an invalid (NaN, flag 8) slot
    fp = gpu_lib.preset("gaussian_rician", True)[1]
    rows = np.abs(np.random.default_rng(0).normal(100.0, 10.0, (8, 4))).astype(np.float32)
    par = (np.full(1, 600.0), np.full(1, 50.0), np.full(1, 5.0))
    for bad in ([-1], [8]):
        with pytest.raises(IndexError, match="mask_indices out of range"):
            gpu_lib.t2_interval(rows, np.array(bad), te, "gaussian_rician", fp)
        with pytest.raises(IndexError, match="mask_indices out of range"):
            gpu_lib.parametric_bootstrap(rows, np.array(bad), te, "gaussian_rician", fp, n_rep=16, params=par)
        with pytest.raises(IndexError, match="mask_indices out of range"):
            gpu_lib.fit_voxels_batch(rows, np.array(bad), te, "gaussian_rician", fp, want=("se",))
        lo, hi, best, fl = gpu_lib.t2_interval(torch.from_numpy(rows).cuda(), torch.tensor(bad, device="cuda"), te,
                                               "gaussian_rician", fp)
        torch.cuda.synchronize()
        assert all(np.isnan(_np(a)).all() for a in (lo, hi, best)) and _np(fl).tolist() == [8], bad
