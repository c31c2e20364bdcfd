// Per-voxel standard errors of the fitted parameters (k, T2[, sigma]): the unconstrained local linearisation of the fit's
// objective at the parameters the fit returned (DESIGN.md section 11).  One voxel per thread, FP64 throughout.
//
//   gaussian, gaussian_rician (least squares):  J[e][j] = d m_e / d theta_j,   s^2 = sum_e r_e^2 / (E - P),
//                                               Cov = s^2 (J'J)^-1             (scipy curve_fit's pcov, absolute_sigma=False)
//   rician (negative log-likelihood):           Cov = H^-1, H the analytic Hessian of the SUMMED NLL (rician_obj,
//                                               run_t2mapping.py:157-177) -- the observed information
//
// with theta = (k, T2[, sigma]) in the units of the maps and bounds ignored.  The P x P matrix A (J'J or H) is inverted by a
// Cholesky factorisation of D A D, D = diag(A_jj^-1/2), and se_j = sqrt(scale (D A D)^-1_jj) D_j.  All standard errors of a
// voxel are NaN when an echo is not finite (rician: or <= 0), a parameter is not finite or T2 <= 0, E <= P, a diagonal entry
// of A is <= 0, or a Cholesky pivot is <= 0 or not finite; otherwise they are finite and >= 0 (0 only for a least-squares
// fit with every residual exactly zero), however ill-determined the voxel.
//
// Plain C++ when T2FIT_HOSTSIM is defined (tests/hostsim/pass_shim.cpp checks it against oracle/stderr_oracle.py).
#pragma once
#include "../../include/t2fit.h"
#include "t2fit_lbfgsb.cuh"
#include "t2fit_i1e_coeffs.h"

namespace t2fit {
namespace se {

// Clenshaw's recurrence as lb::chebev, every product and sum rounded separately (no FMA contraction): with the 29 / 25
// coefficients of tools/make_i1e_coeffs.py this is the published Cephes evaluation scipy.special.i1e performs, so the two
// agree to the last bit instead of differing by the ~2e-15 that two independently rounded evaluations near |x| = 8 reach.
template <int NC>
T2_HD double chebev_rn(double y, const double (&c)[NC]) {
    double b0 = c[0], b1 = 0.0, b2 = 0.0;
#pragma unroll
    for (int i = 1; i < NC; ++i) { b2 = b1; b1 = b0; b0 = lb::add(lb::sub(lb::mul(y, b1), b2), c[i]); }
    return lb::mul(0.5, lb::sub(b0, b2));
}

// exp(-|x|) I1(x) (scipy.special.i1e), odd in x: the Chebyshev expansions of tools/make_i1e_coeffs.py on the intervals of i0e.
// For |x| <= 8 the expansion is of i1e(x) / x itself, which bessel_ratio uses directly.
T2_HD double i1e_over_x_small(double z) {                     // |x| <= 8
    const double a[T2FIT_I1E_NA] = {T2FIT_I1E_A_LIST};
    return chebev_rn<T2FIT_I1E_NA>(lb::sub(lb::mul(0.5, z), 2.0), a);
}
T2_NI double i1e(double x) {
    const double z = fabs(x);
    double r;
    if (z <= 8.0) {
        r = lb::mul(i1e_over_x_small(z), z);
    } else {
        const double b[T2FIT_I1E_NB] = {T2FIT_I1E_B_LIST};
        r = chebev_rn<T2FIT_I1E_NB>(lb::sub(32.0 / z, 2.0), b) / sqrt(z);
    }
    return x < 0 ? -r : r;
}

// A(z) = I1(z) / I0(z) and A(z) / z for z >= 0.  Below 8 the quotient A / z comes from the expansion of i1e(z) / z, so it is
// exact at z = 0 (limit 1/2) where the textbook form 1 - A/z - A^2 of A' would divide 0 by 0.
T2_HD void bessel_ratio(double z, double& a, double& a_over_z) {
    const double i0 = lb::i0e(z);
    if (z <= 8.0) {
        a_over_z = i1e_over_x_small(z) / i0;
        a = a_over_z * z;
    } else {
        a = i1e(z) / i0;
        a_over_z = a / z;
    }
}

// Standard errors of one voxel.  MODEL: T2FIT_MODEL_*; yraw: the float32 echoes as stored; te: echo times [ms];
// norm: scale the echoes by y / max(y) in float32 first, as the fit does (run_t2mapping.py:237-240); (k, t2, sigma): the
// fitted float32 parameters (sigma unused for gaussian).  se[0..P-1] = (se_k, se_T2[, se_sigma]).
template <int MODEL, int E>
T2_HD void voxel_stderr(const float (&yraw)[E], const double* te, bool norm, float kf, float t2f, float sf, double (&se)[3]) {
    constexpr int P = MODEL == T2FIT_MODEL_GAUSSIAN ? 2 : 3;
    se[0] = se[1] = se[2] = NAN;
    float y[E];
    bool ok = E > P;
    float ymax = yraw[0];
#pragma unroll
    for (int e = 0; e < E; ++e) {
        y[e] = yraw[e];
        ok = ok && finite_r(yraw[e]);
        ymax = yraw[e] > ymax ? yraw[e] : ymax;
    }
    if (norm) {
#pragma unroll
        for (int e = 0; e < E; ++e) { y[e] = yraw[e] / ymax; ok = ok && finite_r(y[e]); }
    }
    if (MODEL == T2FIT_MODEL_RICIAN) {
#pragma unroll
        for (int e = 0; e < E; ++e) ok = ok && y[e] > 0.0f;
    }
    const double k = kf, t2 = t2f, s = sf;
    ok = ok && finite_r(k) && finite_r(t2) && t2 > 0.0 && (P == 2 || finite_r(s));
    if (!ok) return;

    // A = J'J (least squares) or the Hessian H of the summed NLL (rician); upper triangle a[i][j], i <= j
    double a[3][3] = {{0.0, 0.0, 0.0}, {0.0, 0.0, 0.0}, {0.0, 0.0, 0.0}};
    double ssr = 0.0;
    const double r2 = 1.0 / (t2 * t2);
#pragma unroll
    for (int e = 0; e < E; ++e) {
        const double u = exp(-te[e] / t2);
        const double yd = (double)y[e];
        if (MODEL == T2FIT_MODEL_GAUSSIAN) {                     // m = k u
            const double m = k * u;
            const double jk = u, jt = m * te[e] * r2;
            a[0][0] += jk * jk; a[0][1] += jk * jt; a[1][1] += jt * jt;
            ssr += (yd - m) * (yd - m);
        } else if (MODEL == T2FIT_MODEL_GAUSSIAN_RICIAN) {       // m = sqrt(k^2 u^2 + sigma^2)
            const double ku2 = k * u * u;
            const double m = sqrt(k * ku2 + s * s);
            const double jk = ku2 / m, jt = k * ku2 * te[e] * r2 / m, js = s / m;
            a[0][0] += jk * jk; a[0][1] += jk * jt; a[0][2] += jk * js;
            a[1][1] += jt * jt; a[1][2] += jt * js; a[2][2] += js * js;
            ssr += (yd - m) * (yd - m);
        } else {                                                 // NLL term of m = k u, x = y m / sigma^2
            const double s2 = s * s;
            const double m = k * u;
            const double x = yd * m / s2;
            double az, az_over_z;
            bessel_ratio(fabs(x), az, az_over_z);
            const double ax = x < 0 ? -az : az;                  // A(x), odd
            const double dax = 1.0 - az_over_z - az * az;        // A'(x) = 1 - A/x - A^2, even
            const double tm = (m - yd * ax) / s2;                                             // d t / d m
            const double tmm = 1.0 / s2 - dax * yd * yd / (s2 * s2);                          // d2 t / d m2
            const double tms = 2.0 * (yd * ax - m + x * yd * dax) / (s2 * s);                 // d2 t / d m d sigma
            const double tss = (-2.0 + 3.0 * (yd * yd + m * m) / s2 - 6.0 * x * ax - 4.0 * x * x * dax) / s2;
            const double mk = u, mt = m * te[e] * r2;                                         // dm/dk, dm/dT2
            const double mkt = u * te[e] * r2, mtt = mt * (te[e] - 2.0 * t2) * r2;            // d2m/dk dT2, d2m/dT2^2
            a[0][0] += tmm * mk * mk;
            a[0][1] += tmm * mk * mt + tm * mkt;
            a[1][1] += tmm * mt * mt + tm * mtt;
            a[0][2] += tms * mk;
            a[1][2] += tms * mt;
            a[2][2] += tss;
        }
    }
    const double scale = MODEL == T2FIT_MODEL_RICIAN ? 1.0 : ssr / (double)(E - P);

    // Cholesky factorisation of B = D A D (unit diagonal), then the diagonal of B^-1 = L^-T L^-1
    double d[3];
#pragma unroll
    for (int j = 0; j < P; ++j) {
        if (!(a[j][j] > 0.0) || !finite_r(a[j][j])) return;
        d[j] = 1.0 / sqrt(a[j][j]);
    }
    const double b01 = a[0][1] * d[0] * d[1];
    const double p1 = 1.0 - b01 * b01;                           // second pivot (the first is 1)
    if (!(p1 > 0.0) || !finite_r(p1)) return;
    const double l11 = sqrt(p1);
    double v0, v1, v2;                                           // diagonal of B^-1
    if (P == 2) {
        v0 = 1.0 / p1;                                           // (1 + l10^2 / l11^2) with l10 = b01
        v1 = 1.0 / p1;
        v2 = 0.0;
    } else {
        const double b02 = a[0][2] * d[0] * d[2], b12 = a[1][2] * d[1] * d[2];
        const double l20 = b02, l21 = (b12 - l20 * b01) / l11;
        const double p2 = 1.0 - l20 * l20 - l21 * l21;           // third pivot
        if (!(p2 > 0.0) || !finite_r(p2)) return;
        const double l22 = sqrt(p2);
        // L^-1 (lower triangular, unit first diagonal entry)
        const double i11 = 1.0 / l11, i22 = 1.0 / l22;
        const double i10 = -b01 * i11;
        const double i21 = -l21 * i11 * i22;
        const double i20 = -(l20 + l21 * i10) * i22;
        v0 = 1.0 + i10 * i10 + i20 * i20;
        v1 = i11 * i11 + i21 * i21;
        v2 = i22 * i22;
    }
    se[0] = sqrt(scale * v0) * d[0];
    se[1] = sqrt(scale * v1) * d[1];
    if (P == 3) se[2] = sqrt(scale * v2) * d[2];
}

}  // namespace se
}  // namespace t2fit
