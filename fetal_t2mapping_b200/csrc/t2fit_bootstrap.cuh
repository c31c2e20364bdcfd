// Per-voxel parametric bootstrap (DESIGN.md section 13): the replicate rows a voxel's fitted curve and noise level give, and
// the statistics of the parameters the fit returns for them.  The refits themselves are ordinary t2fit_run calls.
//
//   noise level   gaussian, gaussian_rician: s = noise_sd if given, else sqrt(sum_e r_e^2 / (E - P)) at theta (FP64, as in
//                 section 11); rician: sigma_n = noise_sd if given, else the fitted sigma.  A given noise_sd is in the units
//                 of the stored echoes and is divided by max(y) under norm.
//   normals       Philox4x32-10, key (seed lo32, seed hi32), counter (j, r, v lo32, v hi32): r the replicate, v the flat voxel
//                 id.  Word w -> u = (w + 0.5) 2^-32 in FP64; block j gives normals 4j..4j+3 by Box-Muller on (w0, w1) and
//                 (w2, w3): rho = sqrt(-2 ln u_a), (rho cos 2 pi u_b, rho sin 2 pi u_b).
//   rows (FP64, stored as float32), u_e = exp(-te_e / T2):
//                 gaussian         k u_e + s z_e
//                 gaussian_rician  sqrt((k u_e)^2 + sigma^2) + s z_e
//                 rician           sqrt((k u_e + sigma_n z_2e)^2 + (sigma_n z_2e+1)^2)
//   invalid voxel (every row NaN): an observed echo not finite (rician: or <= 0), a parameter not finite or T2 <= 0, a noise
//                 level not finite or < 0, or E <= P with s to estimate.  The echoes are those of the fit: float32, scaled by
//                 y / max(y) in float32 under norm.
//   statistics    a replicate is used when its status is 0 or 2 and its parameters are finite; FP64 mean and SD (ddof 1) per
//                 parameter and the T2 quantiles at (1 -+ level) / 2 by numpy's default (linear) method over the used
//                 values; NaN with fewer than 2 used.  Sums run in a fixed order (kStatThreads partial sums, then a halving
//                 tree), so the result does not depend on anything but the replicate values.
//
// Plain C++ when T2FIT_HOSTSIM is defined (tests/hostsim/pass_shim.cpp checks it against oracle/bootstrap_oracle.py).
#pragma once
#include "../../include/t2fit.h"
#include "t2fit_lbfgsb.cuh"
#ifdef T2FIT_HOSTSIM
#include <algorithm>
#endif

namespace t2fit {
namespace bs {

constexpr int kMinRep = 16, kMaxRep = 4096;
constexpr int kStatThreads = 128;            // threads of one voxel's statistics = partial sums of the fixed summation order

// Philox4x32-10 (Salmon et al., SC'11; the Random123 / cuRAND constants).
T2_HD void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t (&w)[4]) {
#pragma unroll
    for (int round = 0; round < 10; ++round) {
        const uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
        const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
        c1 = (uint32_t)p1;
        c3 = (uint32_t)p0;
        c0 = n0;
        c2 = n2;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    w[0] = c0; w[1] = c1; w[2] = c2; w[3] = c3;
}

T2_HD double uniform(uint32_t w) { return ((double)w + 0.5) * 2.3283064365386963e-10; }   // (w + 0.5) 2^-32, in (0, 1)

// normals 4j .. 4j+3 of replicate r of voxel v
T2_HD void normals4(uint64_t seed, int r, uint64_t v, int j, double (&z)[4]) {
    uint32_t w[4];
    philox4x32_10((uint32_t)j, (uint32_t)r, (uint32_t)v, (uint32_t)(v >> 32), (uint32_t)seed, (uint32_t)(seed >> 32), w);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const double rho = sqrt(-2.0 * log(uniform(w[2 * h]))), a = 6.283185307179586 * uniform(w[2 * h + 1]);
        z[2 * h] = rho * cos(a);
        z[2 * h + 1] = rho * sin(a);
    }
}

// What a voxel's replicates are drawn from: the mean curve (the amplitude k u_e for rician) and the noise level.
template <int E>
struct Source {
    double mu[E];
    double level;
    bool ok;
};

// yraw: the float32 echoes as stored; (kf, t2f, sf): the float32 parameters (sf unused for gaussian); noise: the given
// noise_sd when has_noise, else the level is estimated (least squares) or the fitted sigma (rician).
template <int E>
T2_HD void load_source(const float (&yraw)[E], const double* te, int model, bool norm, float kf, float t2f, float sf,
                       bool has_noise, float noise, Source<E>& src) {
    const int P = model == T2FIT_MODEL_GAUSSIAN ? 2 : 3;
    bool ok = true;
    float ymax = yraw[0];
#pragma unroll
    for (int e = 0; e < E; ++e) {
        ok = ok && finite_r(yraw[e]);
        ymax = yraw[e] > ymax ? yraw[e] : ymax;
    }
    double y[E];
#pragma unroll
    for (int e = 0; e < E; ++e) {
        const float v = norm ? yraw[e] / ymax : yraw[e];
        ok = ok && finite_r(v) && (model != T2FIT_MODEL_RICIAN || v > 0.0f);
        y[e] = (double)v;
    }
    const double k = kf, t2 = t2f, sg = sf;
    ok = ok && finite_r(k) && finite_r(t2) && t2 > 0.0 && (P == 2 || finite_r(sg));
    double ssr = 0.0;
#pragma unroll
    for (int e = 0; e < E; ++e) {
        const double a = k * exp(-te[e] / t2);
        src.mu[e] = model == T2FIT_MODEL_GAUSSIAN_RICIAN ? sqrt(a * a + sg * sg) : a;
        ssr += (y[e] - src.mu[e]) * (y[e] - src.mu[e]);
    }
    double level;
    if (has_noise) level = norm ? (double)noise / (double)ymax : (double)noise;
    else if (model == T2FIT_MODEL_RICIAN) level = sg;
    else {
        ok = ok && E > P;
        level = sqrt(ssr / (double)(E - P));
    }
    src.level = level;
    src.ok = ok && finite_r(level) && level >= 0.0;
}

// Replicate r of voxel v (flat id) from its source, as float32.
template <int E>
T2_HD void replicate_row(const Source<E>& src, int model, uint64_t seed, int r, uint64_t v, float (&row)[E]) {
    if (!src.ok) {
#pragma unroll
        for (int e = 0; e < E; ++e) row[e] = NAN;
        return;
    }
    if (model != T2FIT_MODEL_RICIAN) {
#pragma unroll
        for (int j = 0; j < (E + 3) / 4; ++j) {
            double z[4];
            normals4(seed, r, v, j, z);
#pragma unroll
            for (int h = 0; h < 4; ++h)
                if (4 * j + h < E) row[4 * j + h] = (float)(src.mu[4 * j + h] + src.level * z[h]);
        }
    } else {
#pragma unroll
        for (int j = 0; j < (E + 1) / 2; ++j) {
            double z[4];
            normals4(seed, r, v, j, z);
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int e = 2 * j + h;
                if (e < E) {
                    const double a = src.mu[e] + src.level * z[2 * h], b = src.level * z[2 * h + 1];
                    row[e] = (float)sqrt(a * a + b * b);
                }
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// statistics
// ---------------------------------------------------------------------------------------------
T2_HD bool rep_used(uint8_t st, float k, float t2, float s, int P) {
    return (st == T2FIT_ST_OK || st == T2FIT_ST_NOTCONVERGED) && finite_r(k) && finite_r(t2) && (P == 2 || finite_r(s));
}

// The fixed summation order: kStatThreads partial sums p[t] over the used replicates t, t + kStatThreads, ... in ascending
// order, then p[t] += p[t + h] for h = kStatThreads / 2, ..., 1; every sum and product rounded separately.

// numpy.quantile(x, q) of the ascending values x[0..n) (n >= 1), the default 'linear' method: virtual index (n - 1) q,
// lerp as numpy's _lerp (from the nearer end, no fused multiply-add).
T2_HD double quantile_sorted(const float* x, int n, double q) {
    const double vi = lb::mul((double)(n - 1), q);
    const double below = floor(vi);
    const double g = lb::sub(vi, below);
    const int i0 = (int)below, i1 = i0 + 1 < n ? i0 + 1 : n - 1;
    const double a = x[i0], b = x[i1], d = lb::sub(b, a);
    return g >= 0.5 ? lb::sub(b, lb::mul(d, lb::sub(1.0, g))) : lb::add(a, lb::mul(d, g));
}

#ifdef T2FIT_HOSTSIM
// The statistics kernel's arithmetic for one voxel, serially: the same partial sums, tree and quantiles, so the host build
// gives the device's bits.  rk / rt / rs / st: the voxel's n_rep replicate results (rs NULL for gaussian); out: mean[3],
// sd[3], lo, hi (float32 as stored); counts: n_used, n_ok.
inline void voxel_stats_host(int model, int n_rep, const float* rk, const float* rt, const float* rs, const uint8_t* st,
                             double level, float* mean, float* sd, float* lo, float* hi, int32_t* n_used, int32_t* n_ok) {
    const int P = model == T2FIT_MODEL_GAUSSIAN ? 2 : 3;
    const int T = kStatThreads;
    double p[3][T], q[3][T];
    int nu = 0, no = 0;
    float sorted[kMaxRep];
    auto val = [&](int j, int r) { return j == 0 ? rk[r] : j == 1 ? rt[r] : rs[r]; };
    auto used = [&](int r) { return rep_used(st[r], rk[r], rt[r], rs ? rs[r] : 0.0f, P); };
    for (int t = 0; t < T; ++t)
        for (int j = 0; j < 3; ++j) p[j][t] = q[j][t] = 0.0;
    for (int r = 0; r < n_rep; ++r) {
        no += st[r] == T2FIT_ST_OK;
        if (!used(r)) continue;
        sorted[nu++] = rt[r];
        for (int j = 0; j < P; ++j) p[j][r % T] = lb::add(p[j][r % T], (double)val(j, r));
    }
    for (int h = T / 2; h >= 1; h /= 2)
        for (int t = 0; t < h; ++t)
            for (int j = 0; j < 3; ++j) p[j][t] = lb::add(p[j][t], p[j][t + h]);
    double m[3];
    for (int j = 0; j < 3; ++j) m[j] = p[j][0] / (double)nu;
    for (int r = 0; r < n_rep; ++r) {
        if (!used(r)) continue;
        for (int j = 0; j < P; ++j) {
            const double d = lb::sub((double)val(j, r), m[j]);
            q[j][r % T] = lb::add(q[j][r % T], lb::mul(d, d));
        }
    }
    for (int h = T / 2; h >= 1; h /= 2)
        for (int t = 0; t < h; ++t)
            for (int j = 0; j < 3; ++j) q[j][t] = lb::add(q[j][t], q[j][t + h]);
    std::sort(sorted, sorted + nu);
    const bool enough = nu >= 2;
    for (int j = 0; j < 3; ++j) {
        mean[j] = enough && j < P ? (float)m[j] : NAN;
        sd[j] = enough && j < P ? (float)sqrt(q[j][0] / (double)(nu - 1)) : NAN;
    }
    *lo = enough ? (float)quantile_sorted(sorted, nu, lb::mul(0.5, lb::sub(1.0, level))) : NAN;
    *hi = enough ? (float)quantile_sorted(sorted, nu, lb::mul(0.5, lb::add(1.0, level))) : NAN;
    *n_used = nu;
    *n_ok = no;
}
#endif

}  // namespace bs
}  // namespace t2fit
