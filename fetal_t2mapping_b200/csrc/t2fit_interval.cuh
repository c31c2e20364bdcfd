// Per-voxel profile-likelihood confidence interval for T2 (DESIGN.md section 12).  One voxel per thread, FP64 throughout.
//
// For one voxel, with the fit's objective f and the fit's box:
//   f:       gaussian, gaussian_rician: the mean squared error; rician: the summed NLL (rician_obj, run_t2mapping.py:157-177);
//            FP64 on the float32 echoes (scaled by y / max(y) in float32 first when norm is set, as the fit does)
//   box:     the preset bounds, or under --no_prior k in [y(TE_0), no_prior_k_ub], T2 in [no_prior_t2_lb, no_prior_t2_ub]
//            (sigma keeps its preset bounds)
//   profile: p(T2) = min over (k[, sigma]) in the box of f(k, T2[, sigma])
//   minimum: p* = min over T2 in [lb, ub] of p(T2), reached at t2_best
//   set:     {T2 in the box : p(T2) <= thr},  least squares thr = p* (1 + q / (E - P))  (q = t^2_{E-P}(1 - alpha/2)),
//                                             rician        thr = p* + q / 2           (q = chi^2_1(1 - alpha))
//   t2_lo / t2_hi = the smallest / largest member of the set (its hull when the set is not connected)
//   flags:   bit 0 t2_lo is the lower T2 bound, bit 1 t2_hi is the upper T2 bound, bit 2 a grid point strictly between
//            t2_lo and t2_hi lies outside the set, bit 3 invalid (lo, hi, best NaN): a non-finite echo (rician: or an
//            echo <= 0), E <= P, an empty box (the fit's status 3) or a non-finite p*.
//
// Numerical procedure (oracle/interval_oracle.py restates it step by step):
//   1. p on G points T2_g = lb (ub/lb)^(g/(G-1)), both bounds included.  For the 3-parameter models the inner problem is a
//      projected damped Newton iteration over (k, sigma) (iv::newton2); an ascending sweep takes the better of a fixed start
//      (iv::fixed_start) and the solution at g-1, a descending sweep then retries each point from the solution at g+1.
//   2. Golden-section search in log T2 over the grid minimum's neighbours to a width of kTolMin; p* and t2_best are the
//      lowest point evaluated (grid points included).
//   3. Bisection in log T2 of the two threshold crossings that bound the hull, to a width of kTolCross (the inside end is
//      returned).  Off-grid points start from the fixed start and the solutions at the two enclosing grid points.
//
// Plain C++ when T2FIT_HOSTSIM is defined (tests/hostsim/pass_shim.cpp checks it against oracle/interval_oracle.py).
#pragma once
#include "t2fit_stderr.cuh"

namespace t2fit {
namespace iv {

constexpr int kMaxGrid = 256;
constexpr int kMinGrid = 16;
constexpr double kTolMin = 1e-8;       // log T2 width of the final golden-section bracket (relative T2 tolerance <= 1e-7)
constexpr double kTolCross = 1e-7;     // log T2 width of the final bisection bracket (relative T2 tolerance <= 1e-6)
constexpr int kNewtonIter = 100;

enum Flag : int { kLoAtBound = 1, kHiAtBound = 2, kGap = 4, kInvalid = 8 };

struct Box {
    double k_lo, k_hi, t_lo, t_hi, s_lo, s_hi;
};

T2_HD double clampd(double v, double lo, double hi) { return v < lo ? lo : (v > hi ? hi : v); }

// The echoes of one voxel and the decay u_e = exp(-TE_e / T2) at the T2 being profiled.
struct Voxel {
    double y[kMaxEcho];
    double te[kMaxEcho];
    double u[kMaxEcho];
    int n;
    int model;
    Box b;
};

T2_HD void set_t2(Voxel& v, double t2) {
    for (int e = 0; e < v.n; ++e) v.u[e] = exp(-v.te[e] / t2);
}

// exp(-|x|) I0(x), A(x) = I1(x) / I0(x) and A(x) / x for x >= 0 (se::bessel_ratio with the i0e kept)
T2_HD void bessel3(double z, double& i0, double& a, double& a_over_z) {
    i0 = lb::i0e(z);
    if (z <= 8.0) {
        a_over_z = se::i1e_over_x_small(z) / i0;
        a = a_over_z * z;
    } else {
        a = se::i1e(z) / i0;
        a_over_z = a / z;
    }
}

// f(k, sigma) at the current u: the mean squared error (gaussian_rician) or the summed NLL (rician)
T2_NI double value3(const Voxel& v, double k, double s) {
    double f = 0.0;
    if (v.model == T2FIT_MODEL_GAUSSIAN_RICIAN) {
        for (int e = 0; e < v.n; ++e) {
            const double ku = k * v.u[e];
            const double r = v.y[e] - sqrt(ku * ku + s * s);
            f += r * r;
        }
        return f / v.n;
    }
    const double s2 = s * s;
    for (int e = 0; e < v.n; ++e) {
        const double y = v.y[e], m = k * v.u[e];
        const double x = m * y / s2;
        f -= (log(y) - log(s2)) - (y * y + m * m) / (2.0 * s2) + (fabs(x) + log(lb::i0e(x)));
    }
    return f;
}

// f, its gradient g = (df/dk, df/dsigma) and Hessian h = (kk, ks, ss) at the current u
T2_NI double value_grad_hess3(const Voxel& v, double k, double s, double (&g)[2], double (&h)[3]) {
    double f = 0.0;
    g[0] = g[1] = h[0] = h[1] = h[2] = 0.0;
    if (v.model == T2FIT_MODEL_GAUSSIAN_RICIAN) {        // m = sqrt(k^2 u^2 + s^2), f = sum (y - m)^2 / E
        for (int e = 0; e < v.n; ++e) {
            const double u = v.u[e], ku = k * u;
            const double m = sqrt(ku * ku + s * s);
            const double r = m - v.y[e];
            const double mk = ku * u / m, ms = s / m;
            const double m3 = m * m * m;
            const double mkk = u * u * s * s / m3, mks = -ku * u * s / m3, mss = ku * ku / m3;
            f += r * r;
            g[0] += r * mk; g[1] += r * ms;
            h[0] += mk * mk + r * mkk; h[1] += mk * ms + r * mks; h[2] += ms * ms + r * mss;
        }
        const double c = 2.0 / v.n;
        g[0] *= c; g[1] *= c; h[0] *= c; h[1] *= c; h[2] *= c;
        return f / v.n;
    }
    const double s2 = s * s;                            // rician: the terms of se::voxel_stderr, summed NLL
    for (int e = 0; e < v.n; ++e) {
        const double y = v.y[e], u = v.u[e], m = k * u;
        const double x = m * y / s2;
        double i0, az, az_over_z;
        bessel3(fabs(x), i0, az, az_over_z);
        const double ax = x < 0 ? -az : az;
        const double dax = 1.0 - az_over_z - az * az;
        f -= (log(y) - log(s2)) - (y * y + m * m) / (2.0 * s2) + (fabs(x) + log(i0));
        const double tm = (m - y * ax) / s2;
        const double ts = 2.0 / s - (y * y + m * m) / (s2 * s) + 2.0 * x * ax / s;
        const double tmm = 1.0 / s2 - dax * y * y / (s2 * s2);
        const double tms = 2.0 * (y * ax - m + x * y * dax) / (s2 * s);
        const double tss = (-2.0 + 3.0 * (y * y + m * m) / s2 - 6.0 * x * ax - 4.0 * x * x * dax) / s2;
        g[0] += tm * u; g[1] += ts;
        h[0] += tmm * u * u; h[1] += tms * u; h[2] += tss;
    }
    return f;
}

// Projected damped Newton over (k, sigma) in the box from x: a variable at a bound whose gradient points out of the box is
// held; the free block is solved with Levenberg-Marquardt damping lam |H_jj| until the projected step lowers f.  Stops
// when no step lowers f or the decrease falls below 1e-15 |f|.  Returns f(x) at the final x.
T2_NI double newton2(const Voxel& v, double (&x)[2]) {
    const double lo[2] = {v.b.k_lo, v.b.s_lo}, hi[2] = {v.b.k_hi, v.b.s_hi};
    x[0] = clampd(x[0], lo[0], hi[0]);
    x[1] = clampd(x[1], lo[1], hi[1]);
    double g[2], h[3];
    double f = value_grad_hess3(v, x[0], x[1], g, h);
    double lam = 0.0;
    for (int it = 0; it < kNewtonIter; ++it) {
        bool fr[2];
        for (int j = 0; j < 2; ++j) fr[j] = !((x[j] <= lo[j] && g[j] > 0.0) || (x[j] >= hi[j] && g[j] < 0.0));
        if (!fr[0] && !fr[1]) break;
        bool accepted = false, moved = true;
        double xn[2], fn = f;
        for (int tr = 0; tr < 40; ++tr) {
            const double a00 = h[0] + lam * fmax(fabs(h[0]), 1e-300), a11 = h[2] + lam * fmax(fabs(h[2]), 1e-300);
            double d0 = 0.0, d1 = 0.0;
            bool pd;
            if (fr[0] && fr[1]) {
                const double det = a00 * a11 - h[1] * h[1];
                pd = a00 > 0.0 && det > 0.0;
                if (pd) { d0 = -(a11 * g[0] - h[1] * g[1]) / det; d1 = -(a00 * g[1] - h[1] * g[0]) / det; }
            } else if (fr[0]) {
                pd = a00 > 0.0;
                if (pd) d0 = -g[0] / a00;
            } else {
                pd = a11 > 0.0;
                if (pd) d1 = -g[1] / a11;
            }
            if (pd) {
                xn[0] = clampd(x[0] + d0, lo[0], hi[0]);
                xn[1] = clampd(x[1] + d1, lo[1], hi[1]);
                if (xn[0] == x[0] && xn[1] == x[1]) { moved = false; break; }
                fn = value3(v, xn[0], xn[1]);
                if (fn < f) { accepted = true; break; }
            }
            lam = lam == 0.0 ? 1e-3 : lam * 10.0;
        }
        if (!accepted || !moved) break;
        const double df = f - fn;
        x[0] = xn[0]; x[1] = xn[1];
        f = value_grad_hess3(v, x[0], x[1], g, h);
        lam = lam < 1e-9 ? 0.0 : lam * 0.1;
        if (df <= 1e-15 * fabs(f)) break;
    }
    return f;
}

// The start that does not depend on a neighbour: k the closed-form least-squares amplitude at this T2, sigma the rms of
// its residuals, both clipped to the box.
T2_HD void fixed_start(const Voxel& v, double (&x)[2]) {
    double syu = 0.0, suu = 0.0;
    for (int e = 0; e < v.n; ++e) { syu += v.y[e] * v.u[e]; suu += v.u[e] * v.u[e]; }
    const double k = clampd(syu / suu, v.b.k_lo, v.b.k_hi);
    double r2 = 0.0;
    for (int e = 0; e < v.n; ++e) { const double r = v.y[e] - k * v.u[e]; r2 += r * r; }
    const double s = sqrt(r2 / v.n);
    x[0] = finite_r(k) ? k : v.b.k_lo;
    x[1] = finite_r(s) ? clampd(s, v.b.s_lo, v.b.s_hi) : v.b.s_lo;
}

// p(T2) at the T2 set_t2 was last called with.  gaussian: the closed form, k = clamp(sum y u / sum u^2).  3-parameter
// models: the lowest newton2 result over the fixed start (when use_fixed) and the n_warm warm starts, in that order (the
// first of equal values wins); its point is returned in xbest.
T2_NI double profile_here(const Voxel& v, bool use_fixed, const double* warm, int n_warm, double (&xbest)[2]) {
    if (v.model == T2FIT_MODEL_GAUSSIAN) {
        double syu = 0.0, suu = 0.0;
        for (int e = 0; e < v.n; ++e) { syu += v.y[e] * v.u[e]; suu += v.u[e] * v.u[e]; }
        const double k = clampd(syu / suu, v.b.k_lo, v.b.k_hi);
        double f = 0.0;
        for (int e = 0; e < v.n; ++e) { const double r = v.y[e] - k * v.u[e]; f += r * r; }
        xbest[0] = k; xbest[1] = 0.0;
        return f / v.n;
    }
    double best = NAN;
    for (int j = use_fixed ? -1 : 0; j < n_warm; ++j) {
        double x[2];
        if (j < 0) fixed_start(v, x);
        else { x[0] = warm[2 * j]; x[1] = warm[2 * j + 1]; }
        const double f = newton2(v, x);
        if (f < best || !(best == best)) { best = f; xbest[0] = x[0]; xbest[1] = x[1]; }
    }
    return best;
}

T2_HD double grid_t2(const Box& b, int g, int G) {
    return g == G - 1 ? b.t_hi : b.t_lo * pow(b.t_hi / b.t_lo, (double)g / (double)(G - 1));
}

// Work space of one voxel: the profile at the grid and (3-parameter models) the inner minimiser there.
struct Grid {
    double p[kMaxGrid];
    double x[kMaxGrid][2];
};

// p at an off-grid log T2 s: fixed start plus the solutions at the two enclosing grid points
T2_HD double profile_off_grid(Voxel& v, const Grid& w, int G, double s) {
    set_t2(v, exp(s));
    const double s0 = log(v.b.t_lo), s1 = log(v.b.t_hi);
    int g = (int)floor((s - s0) / (s1 - s0) * (G - 1));
    g = g < 0 ? 0 : (g > G - 2 ? G - 2 : g);
    double xb[2];
    return profile_here(v, true, &w.x[g][0], 2, xb);
}

// Bisection in log T2 between an outside point s_out (p > thr) and an inside point s_in (p <= thr); returns the inside end.
T2_HD double crossing(Voxel& v, const Grid& w, int G, double thr, double s_out, double s_in) {
    while (fabs(s_in - s_out) > kTolCross) {
        const double mid = 0.5 * (s_out + s_in);
        if (profile_off_grid(v, w, G, mid) <= thr) s_in = mid;
        else s_out = mid;
    }
    return exp(s_in);
}

// The interval of one voxel.  v.y / v.te / v.n / v.model / v.b set by the caller (the box after the --no_prior override);
// q the quantile; G in [kMinGrid, kMaxGrid].  prof (may be NULL): the G grid values of p.
T2_NI void voxel_interval(Voxel& v, bool valid, double q, int G, Grid& w, double& lo, double& hi, double& best,
                          int& flags, double* prof) {
    lo = hi = best = NAN;
    flags = kInvalid;
    const int P = v.model == T2FIT_MODEL_GAUSSIAN ? 2 : 3;
    valid = valid && v.n > P && v.b.k_lo <= v.b.k_hi;
    if (!valid) {
        if (prof) for (int g = 0; g < G; ++g) prof[g] = NAN;
        return;
    }
    // 1. the grid: ascending sweep (fixed start + previous point), descending sweep (next point)
    for (int g = 0; g < G; ++g) {
        set_t2(v, grid_t2(v.b, g, G));
        w.p[g] = profile_here(v, true, g > 0 ? &w.x[g - 1][0] : nullptr, g > 0 ? 1 : 0, w.x[g]);
    }
    if (P == 3) {
        for (int g = G - 2; g >= 0; --g) {
            set_t2(v, grid_t2(v.b, g, G));
            double xb[2];
            const double f = profile_here(v, false, &w.x[g + 1][0], 1, xb);
            if (f < w.p[g]) { w.p[g] = f; w.x[g][0] = xb[0]; w.x[g][1] = xb[1]; }
        }
    }
    if (prof) for (int g = 0; g < G; ++g) prof[g] = w.p[g];
    int gm = -1;
    for (int g = 0; g < G; ++g)
        if (finite_r(w.p[g]) && (gm < 0 || w.p[g] < w.p[gm])) gm = g;
    if (gm < 0) return;
    // 2. golden section around the grid minimum
    double pstar = w.p[gm], tbest = grid_t2(v.b, gm, G);
    {
        const double r = 0.6180339887498949;
        double a = log(grid_t2(v.b, gm > 0 ? gm - 1 : 0, G)), b = log(grid_t2(v.b, gm < G - 1 ? gm + 1 : G - 1, G));
        double c = b - r * (b - a), d = a + r * (b - a);
        double fc = profile_off_grid(v, w, G, c), fd = profile_off_grid(v, w, G, d);
        if (fc < pstar) { pstar = fc; tbest = exp(c); }
        if (fd < pstar) { pstar = fd; tbest = exp(d); }
        while (b - a > kTolMin) {
            if (fc < fd) {
                b = d; d = c; fd = fc; c = b - r * (b - a);
                fc = profile_off_grid(v, w, G, c);
                if (fc < pstar) { pstar = fc; tbest = exp(c); }
            } else {
                a = c; c = d; fc = fd; d = a + r * (b - a);
                fd = profile_off_grid(v, w, G, d);
                if (fd < pstar) { pstar = fd; tbest = exp(d); }
            }
        }
    }
    if (!finite_r(pstar)) return;
    const double thr = v.model == T2FIT_MODEL_RICIAN ? pstar + 0.5 * q : pstar * (1.0 + q / (double)(v.n - P));
    // 3. the hull's two ends
    int first_in = G, last_in = -1;
    for (int g = 0; g < G; ++g)
        if (w.p[g] <= thr) { if (first_in == G) first_in = g; last_in = g; }
    const double sb = log(tbest);
    int fl = 0;
    if (first_in == 0) {
        lo = v.b.t_lo; fl |= kLoAtBound;
    } else if (first_in == G || sb < log(grid_t2(v.b, first_in, G))) {    // only t2_best inside below the first grid member
        int gb = -1;
        for (int g = 0; g < G; ++g) if (log(grid_t2(v.b, g, G)) < sb) gb = g;
        if (gb < 0) { lo = v.b.t_lo; fl |= kLoAtBound; }
        else lo = crossing(v, w, G, thr, log(grid_t2(v.b, gb, G)), sb);
    } else {
        lo = crossing(v, w, G, thr, log(grid_t2(v.b, first_in - 1, G)), log(grid_t2(v.b, first_in, G)));
    }
    if (last_in == G - 1) {
        hi = v.b.t_hi; fl |= kHiAtBound;
    } else if (last_in < 0 || sb > log(grid_t2(v.b, last_in, G))) {
        int ga = G;
        for (int g = G - 1; g >= 0; --g) if (log(grid_t2(v.b, g, G)) > sb) ga = g;
        if (ga >= G) { hi = v.b.t_hi; fl |= kHiAtBound; }
        else hi = crossing(v, w, G, thr, log(grid_t2(v.b, ga, G)), sb);
    } else {
        hi = crossing(v, w, G, thr, log(grid_t2(v.b, last_in + 1, G)), log(grid_t2(v.b, last_in, G)));
    }
    for (int g = 0; g < G; ++g) {
        const double t = grid_t2(v.b, g, G);
        if (t > lo && t < hi && !(w.p[g] <= thr)) fl |= kGap;
    }
    best = tbest;
    flags = fl;
}

// Load one voxel: the float32 echoes (scaled by y / max(y) in float32 when norm), the validity part of the NaN rule that
// depends on the echoes, and the box (k lower bound y(TE_0) under --no_prior; empty box = the fit's status 3).
template <int E>
T2_HD bool load_voxel(const float (&yraw)[E], const double* te, int model, bool norm, const Box& box, bool no_prior,
                      Voxel& v) {
    bool ok = true;
    float ymax = yraw[0];
#pragma unroll
    for (int e = 0; e < E; ++e) {
        ok = ok && finite_r(yraw[e]);
        ymax = yraw[e] > ymax ? yraw[e] : ymax;
    }
#pragma unroll
    for (int e = 0; e < E; ++e) {
        const float y = norm ? yraw[e] / ymax : yraw[e];
        ok = ok && finite_r(y) && (model != T2FIT_MODEL_RICIAN || y > 0.0f);
        v.y[e] = (double)y;
        v.te[e] = te[e];
    }
    v.n = E;
    v.model = model;
    v.b = box;
    if (no_prior) {
        if (yraw[0] > (float)box.k_hi) ok = false;                 // scipy: "An upper bound is less than ..." (status 3)
        v.b.k_lo = (double)yraw[0];
    }
    return ok;
}

}  // namespace iv
}  // namespace t2fit
