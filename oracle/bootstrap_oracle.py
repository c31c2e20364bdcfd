"""numpy restatement of the per-voxel parametric bootstrap (DESIGN.md section 13; csrc/t2fit_bootstrap.cuh).

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

``philox4x32_10``  Philox4x32-10 on uint64 arrays (Salmon et al., SC'11; the Random123 / cuRAND constants)
``normals``        the standard normals z[..., 0..n) of replicate r of voxel v: counter (j, r, v lo32, v hi32), key (seed lo32,
                   seed hi32), u = (w + 0.5) 2^-32, Box-Muller on (w0, w1) and (w2, w3) of block j
``replicate_rows`` the replicate rows of every voxel: source (mean curve, noise level, validity) and the model's noise
``bootstrap_stats`` the statistics of replicate results: used = status 0 or 2 with finite parameters; mean, SD (ddof 1),
                   the T2 quantiles (np.quantile, linear), n_used, n_ok
"""
from __future__ import annotations

import numpy as np

M0, M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
W0, W1 = np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)
MASK = np.uint64(0xFFFFFFFF)
S32 = np.uint64(32)


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """The four output words (uint64 arrays holding 32-bit values) of counters (c0..c3) under keys (k0, k1), broadcast."""
    c = [np.asarray(x, np.uint64) & MASK for x in (c0, c1, c2, c3)]
    k = [np.asarray(x, np.uint64) & MASK for x in (k0, k1)]
    for _ in range(10):
        p0, p1 = M0 * c[0], M1 * c[2]                       # < 2^64: exact in uint64
        c = [(p1 >> S32) ^ c[1] ^ k[0], p1 & MASK, (p0 >> S32) ^ c[3] ^ k[1], p0 & MASK]
        k = [(k[0] + W0) & MASK, (k[1] + W1) & MASK]
    return c


def normals(seed, r, v, n):
    """z[..., 0..n): normals of replicate(s) ``r`` of voxel id(s) ``v`` (broadcast), float64."""
    seed = int(seed)
    r, v = np.asarray(r, np.uint64), np.asarray(v, np.int64).astype(np.uint64)
    out = []
    for j in range((n + 3) // 4):
        w = philox4x32_10(np.uint64(j), r, v & MASK, v >> S32, seed & 0xFFFFFFFF, seed >> 32)
        u = [(x.astype(np.float64) + 0.5) * 2.0 ** -32 for x in w]
        for a, b in ((u[0], u[1]), (u[2], u[3])):
            rho = np.sqrt(-2.0 * np.log(a))
            ang = 6.283185307179586 * b
            out += [rho * np.cos(ang), rho * np.sin(ang)]
    return np.stack(out[:n], axis=-1)


def source(rows, te, fit, norm, k, t2, sigma=None, noise_sd=None):
    """(mu [M, E] float64, level [M] float64, ok [M] bool): the mean curve (the amplitude k u_e for rician), the noise level
    and the validity of every voxel.  ``rows``: the float32 echoes as stored; parameters float32 [M]; ``noise_sd`` [M] or
    None (estimated / the fitted sigma)."""
    P = 2 if fit == "gaussian" else 3
    y32 = np.asarray(rows, np.float32)
    E = y32.shape[1]
    ok = np.isfinite(y32).all(axis=1)
    ymax = y32.max(axis=1)
    with np.errstate(all="ignore"):
        y = (y32 / ymax[:, None]).astype(np.float32) if norm else y32
        ok &= np.isfinite(y).all(axis=1)
        if fit == "rician":
            ok &= (y > 0).all(axis=1)
        y = y.astype(np.float64)
        k, t2 = np.asarray(k, np.float32).astype(np.float64), np.asarray(t2, np.float32).astype(np.float64)
        sg = np.asarray(sigma, np.float32).astype(np.float64) if P == 3 else np.zeros_like(k)
        ok &= np.isfinite(k) & np.isfinite(t2) & (t2 > 0) & np.isfinite(sg)
        a = k[:, None] * np.exp(-np.asarray(te, np.float64)[None, :] / t2[:, None])
        mu = np.sqrt(a * a + sg[:, None] ** 2) if fit == "gaussian_rician" else a
        if noise_sd is not None:
            level = np.asarray(noise_sd, np.float32).astype(np.float64)
            if norm:
                level = level / ymax.astype(np.float64)
        elif fit == "rician":
            level = sg
        else:
            level = np.sqrt(((y - mu) ** 2).sum(axis=1) / (E - P)) if E > P else np.full(k.shape, np.nan)
        ok &= np.isfinite(level) & (level >= 0)
    return mu, level, ok


def replicate_rows(rows, te, fit, norm, k, t2, sigma=None, noise_sd=None, voxel_id=None, seed=0, n_rep=200):
    """[M * n_rep, E] float32 replicate rows, row i * n_rep + r.  ``voxel_id``: the flat voxel ids [M] (default 0..M-1)."""
    mu, level, ok = source(rows, te, fit, norm, k, t2, sigma, noise_sd)
    m, E = mu.shape
    vid = np.arange(m, dtype=np.int64) if voxel_id is None else np.asarray(voxel_id, np.int64)
    rr = np.arange(n_rep, dtype=np.uint64)
    z = normals(seed, rr[None, :], vid[:, None], 2 * E if fit == "rician" else E)       # [M, n_rep, n]
    mu3, lv = mu[:, None, :], level[:, None, None]
    with np.errstate(all="ignore"):
        if fit == "rician":
            out = np.sqrt((mu3 + lv * z[..., 0::2]) ** 2 + (lv * z[..., 1::2]) ** 2)
        else:
            out = mu3 + lv * z
        out = out.astype(np.float32)
    out[~ok] = np.nan
    return out.reshape(m * n_rep, E)


def bootstrap_stats(fit, n_rep, k, t2, sigma, status, level):
    """(mean [3, M], sd [3, M], lo [M], hi [M], n_used [M], n_ok [M]) of replicate results [M * n_rep] (row i * n_rep + r):
    float64 mean / SD (ddof 1) and np.quantile of the used values, NaN with fewer than 2 used (and for sigma of gaussian)."""
    P = 2 if fit == "gaussian" else 3
    cols = [np.asarray(k, np.float32), np.asarray(t2, np.float32)] + ([np.asarray(sigma, np.float32)] if P == 3 else [])
    st = np.asarray(status, np.uint8).reshape(-1, n_rep)
    vals = [c.astype(np.float64).reshape(-1, n_rep) for c in cols]
    m = st.shape[0]
    used = (st == 0) | (st == 2)
    for v in vals:
        used &= np.isfinite(v)
    mean, sd = np.full((3, m), np.nan), np.full((3, m), np.nan)
    lo, hi = np.full(m, np.nan), np.full(m, np.nan)
    nu, no = used.sum(axis=1).astype(np.int32), (st == 0).sum(axis=1).astype(np.int32)
    q = [(1.0 - level) / 2.0, (1.0 + level) / 2.0]
    for i in range(m):
        if nu[i] < 2:
            continue
        for j in range(P):
            x = vals[j][i][used[i]]
            mean[j, i], sd[j, i] = np.mean(x), np.std(x, ddof=1)
        lo[i], hi[i] = np.quantile(vals[1][i][used[i]], q)
    return mean, sd, lo, hi, nu, no
