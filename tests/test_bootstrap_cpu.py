"""Parametric bootstrap without a GPU: the oracle's Philox against the Random123 known answers, and the header the
replicate and statistics kernels run (csrc/t2fit_bootstrap.cuh, compiled by g++) against the oracle."""
import numpy as np
import pytest

from oracle import bootstrap_oracle as bo
from tests.conftest import load_golden
from tests.hostsim import pass_shim as bootstrap_shim

FIXTURES = ["c1_gaussian_noprior", "c2_gaussian_hf_prior", "c3_floor_prior", "c3_rician_prior", "norm_gaussian",
            "cli3_gaussian_lf_noprior", "cli3_floor_hf_prior", "cli3_rician_hf_prior", "cli3_rician_lf_noprior",
            "edge_gaussian_rician_noprior"]

# Random123's kat_vectors for philox4x32_10: (counter, key, output)
KAT = [((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
       ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
       ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
        (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1))]


@pytest.mark.parametrize("ctr,key,want", KAT)
def test_philox_known_answers(ctr, key, want):
    got = [int(w) for w in bo.philox4x32_10(*ctr, *key)]
    assert got == list(want)
    assert [int(w) for w in bootstrap_shim.bootstrap_philox(ctr, key)] == list(want)


def test_philox_words_agree_on_many_counters():
    rng = np.random.default_rng(11)
    c = rng.integers(0, 2 ** 32, (256, 4), dtype=np.uint64)
    k = rng.integers(0, 2 ** 32, (256, 2), dtype=np.uint64)
    want = np.stack(bo.philox4x32_10(c[:, 0], c[:, 1], c[:, 2], c[:, 3], k[:, 0], k[:, 1]), axis=1)
    got = np.stack([bootstrap_shim.bootstrap_philox(c[i], k[i]) for i in range(256)]).astype(np.uint64)
    assert np.array_equal(got, want)


def test_normals_are_standard_normal():
    z = bo.normals(7, np.arange(4096, dtype=np.uint64)[:, None], np.arange(16)[None, :], 8).reshape(-1)
    assert abs(z.mean()) < 0.01 and abs(z.std() - 1.0) < 0.01
    assert abs(np.mean(np.abs(z) < 1.959964) - 0.95) < 0.003


def _ulps(a, b):
    return np.abs(a.view(np.int32).astype(np.int64) - b.view(np.int32).astype(np.int64))


def _params(g):
    p = g["ref_params"].astype(np.float32)
    return p[:, 0], p[:, 1], (p[:, 2] if g["fit"] != "gaussian" else None)


@pytest.mark.parametrize("name", FIXTURES)
@pytest.mark.parametrize("norm", [False, True], ids=["raw", "norm"])
@pytest.mark.parametrize("given", [False, True], ids=["estimated", "noise_sd"])
def test_host_rows_match_oracle(name, norm, given):
    """Every model, with and without norm and noise_sd, at the reference's parameters of the golden fixtures: the g++ build
    gives the oracle's float32 rows within 1 ulp (in practice bit for bit); invalid voxels are NaN in both."""
    g = load_golden(name)
    k, t2, s = _params(g)
    m = g["rows"].shape[0]
    rng = np.random.default_rng(5)
    noise = rng.uniform(0.0, 40.0, m).astype(np.float32) if given else None
    vid = rng.integers(0, 2 ** 40, m)
    args = (g["rows"], g["te"], g["fit"], norm, k, t2, s, noise, vid, 0x123456789ABCDEF, 16)
    got = bootstrap_shim.bootstrap_rows(*args)
    want = bo.replicate_rows(*args[:8], voxel_id=vid, seed=args[9], n_rep=16)
    assert np.array_equal(np.isnan(got), np.isnan(want))
    fin = np.isfinite(want)
    if fin.any():                                   # cli3: E = P, so every voxel is invalid while s is estimated
        assert _ulps(got[fin], want[fin]).max() <= 1
        assert (_ulps(got[fin], want[fin]) == 0).mean() >= 0.999
    nan_vox = np.isnan(got).reshape(m, 16, -1).all(axis=(1, 2))
    assert np.array_equal(nan_vox, np.isnan(got).reshape(m, 16, -1).any(axis=(1, 2)))    # all of a voxel or none
    _, _, ok = bo.source(g["rows"], g["te"], g["fit"], norm, k, t2, s, noise)
    assert np.array_equal(nan_vox, ~ok)


def test_invalid_voxels_get_nan_rows():
    te = np.array([10.0, 20.0, 40.0, 80.0])
    base = (1000.0 * np.exp(-te / 60.0)).astype(np.float32)
    rows = np.tile(base, (9, 1))
    k = np.full(9, 1000.0, np.float32)
    t2 = np.full(9, 60.0, np.float32)
    s = np.full(9, 10.0, np.float32)
    noise = np.full(9, 5.0, np.float32)
    rows[1, 2] = np.nan                 # echo not finite
    rows[2, 0] = np.inf
    t2[3] = 0.0                         # T2 <= 0
    k[4] = np.nan                       # parameter not finite
    s[5] = np.inf                       # sigma not finite (3-parameter models)
    noise[6] = -1.0                     # noise level < 0
    noise[7] = np.nan
    rows[8, 3] = -2.0                   # rician: echo <= 0
    vid = np.arange(9)
    expect = {"gaussian": [1, 2, 3, 4, 6, 7], "gaussian_rician": [1, 2, 3, 4, 5, 6, 7], "rician": [1, 2, 3, 4, 5, 6, 7, 8]}
    for fit, bad in expect.items():
        sg = s if fit != "gaussian" else None
        got = bootstrap_shim.bootstrap_rows(rows, te, fit, False, k, t2, sg, noise, vid, 3, 16).reshape(9, 16, 4)
        want = bo.replicate_rows(rows, te, fit, False, k, t2, sg, noise, vid, 3, 16).reshape(9, 16, 4)
        assert np.array_equal(np.isnan(got), np.isnan(want))
        nan_vox = np.isnan(got).all(axis=(1, 2))
        assert sorted(np.flatnonzero(nan_vox)) == bad, fit
        assert not np.isnan(got[~nan_vox]).any()
    # E <= P with s to estimate: a 3-parameter fit of 3 echoes, a 2-parameter fit of 2; a given noise_sd is fine there
    for fit, E in (("gaussian_rician", 3), ("gaussian", 2)):
        sg = s[:1] if fit != "gaussian" else None
        r = rows[:1, :E]
        assert np.isnan(bootstrap_shim.bootstrap_rows(r, te[:E], fit, False, k[:1], t2[:1], sg, None, vid[:1], 3, 16)).all()
        assert np.isfinite(bootstrap_shim.bootstrap_rows(r, te[:E], fit, False, k[:1], t2[:1], sg, noise[:1], vid[:1], 3, 16)).all()


def test_zero_noise_rows_are_the_model_rows():
    te = np.linspace(10.0, 320.0, 9)
    k, t2, s = np.float32(900.0), np.float32(75.0), np.float32(30.0)
    u = np.exp(-te / np.float64(t2))
    for fit, model in (("gaussian", np.float64(k) * u), ("gaussian_rician", np.sqrt((np.float64(k) * u) ** 2 + np.float64(s) ** 2)),
                       ("rician", np.float64(k) * u)):
        rows = model.astype(np.float32)[None]
        got = bootstrap_shim.bootstrap_rows(rows, te, fit, False, [k], [t2], None if fit == "gaussian" else [s], [0.0], [0], 9, 16)
        assert np.array_equal(got, np.tile(model.astype(np.float32), (16, 1))), fit


def test_noise_is_keyed_by_voxel_id_and_seed():
    g = load_golden("c2_gaussian_hf_prior")
    k, t2, _ = _params(g)
    rows = g["rows"][:4]
    a = bootstrap_shim.bootstrap_rows(rows, g["te"], "gaussian", False, k[:4], t2[:4], None, None, [10, 11, 12, 13], 1, 16)
    b = bootstrap_shim.bootstrap_rows(rows[2:3], g["te"], "gaussian", False, k[2:3], t2[2:3], None, None, [12], 1, 16)
    assert np.array_equal(a[32:48], b)                                      # the same voxel id: the same replicates
    c = bootstrap_shim.bootstrap_rows(rows[2:3], g["te"], "gaussian", False, k[2:3], t2[2:3], None, None, [12], 2, 16)
    d = bootstrap_shim.bootstrap_rows(rows[2:3], g["te"], "gaussian", False, k[2:3], t2[2:3], None, None, [1 << 33 | 12], 1, 16)
    assert not np.array_equal(b, c) and not np.array_equal(b, d)


def _replicate_set(rng, fit, n_rep, m):
    P = 2 if fit == "gaussian" else 3
    k = rng.normal(1000.0, 40.0, m * n_rep).astype(np.float32)
    t2 = rng.normal(80.0, 6.0, m * n_rep).astype(np.float32)
    s = rng.normal(20.0, 2.0, m * n_rep).astype(np.float32) if P == 3 else None
    st = rng.choice(np.array([0, 1, 2, 3], np.uint8), m * n_rep, p=[0.7, 0.1, 0.15, 0.05])
    t2[: n_rep // 2] = np.round(t2[: n_rep // 2])                            # ties in voxel 0
    t2[n_rep: 2 * n_rep] = 77.0                                              # voxel 1: every used value equal
    st[2 * n_rep: 3 * n_rep] = 1                                             # voxel 2: none used
    st[3 * n_rep: 4 * n_rep] = 3                                             # voxel 3: one used
    st[3 * n_rep + 5] = 2
    st[4 * n_rep: 5 * n_rep] = 1                                             # voxel 4: two used
    st[4 * n_rep + 1] = 0
    st[4 * n_rep + 9] = 2
    k[5 * n_rep + 3] = np.nan                                                # voxel 5: NaN parameters are not used
    t2[5 * n_rep + 4] = np.inf
    if P == 3:
        s[5 * n_rep + 6] = np.nan
    return k, t2, s, st


@pytest.mark.parametrize("fit", ["gaussian", "gaussian_rician", "rician"])
@pytest.mark.parametrize("n_rep", [16, 200, 4096])
def test_host_stats_match_numpy(fit, n_rep):
    """mean / std(ddof=1) / quantile of the used replicates; excluded statuses, NaN parameters, n_used of 0, 1 and 2, ties."""
    rng = np.random.default_rng(n_rep)
    k, t2, s, st = _replicate_set(rng, fit, n_rep, 8)
    for level in (0.95, 0.5, 0.8):
        got = bootstrap_shim.bootstrap_stats(fit, n_rep, k, t2, s, st, level)
        want = bo.bootstrap_stats(fit, n_rep, k, t2, s, st, level)
        for name, a, b in zip(("mean", "sd", "lo", "hi", "n_used", "n_ok"), got, want):
            if a.dtype.kind == "i":
                assert np.array_equal(a, b), name
                continue
            b32 = b.astype(np.float32)
            assert np.array_equal(np.isnan(a), np.isnan(b32)), name
            f = np.isfinite(b32)
            assert _ulps(a[f], b32[f]).max() <= 1, name
        nu = got[4]
        assert nu[2] == 0 and nu[3] == 1 and nu[4] == 2
        assert np.isnan(got[0][:, 2:4]).all() and np.isfinite(got[0][:2 if fit == "gaussian" else 3, 4]).all()
        assert got[1][1, 1] == 0.0 and got[2][1] == got[3][1] == 77.0        # all used values equal
        if fit == "gaussian":
            assert np.isnan(got[0][2]).all() and np.isnan(got[1][2]).all()
