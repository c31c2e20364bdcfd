// Per-voxel T2 relaxation fit: the solver core (one voxel per thread, everything in registers).
//
// Replaces the arithmetic of the reference's fit_voxel (run_t2mapping.py:120-312), i.e. the
// bounded minimisation of
//     gaussian         :  sum_e (y_e - k exp(-te_e/T2))^2 / E                      (:129-131,141-147)
//     gaussian_rician  :  sum_e (y_e - sqrt(k^2 exp(-2 te_e/T2) + sigma^2))^2 / E  (:133-138,149-155)
// over the box the preset / --no_prior gives (:36-106,243-245).  The reference hands these to
// scipy's L-BFGS-B with finite-difference gradients; here the bounded minimiser is reached with a
// register-resident projected Gauss-Newton / Levenberg-Marquardt iteration on closed-form 2x2 / 3x3
// normal equations.  Decay-rate parametrisation r = 1/T2 (same box, same minimiser, no divisions in
// the echo loop).
//
// This header is plain C++ when T2FIT_HOSTSIM is defined (tests/hostsim builds it with g++ to unit
// test the solver logic on GPU-less CI).  The product library only ever compiles it with nvcc for
// sm_100a; there is no CPU path in libt2fit.
#pragma once
#include <stdint.h>
#include <math.h>
#include <type_traits>
#include <utility>

#if defined(__CUDACC__) && !defined(T2FIT_HOSTSIM)
#define T2_HD __device__ __forceinline__
#define T2_DEVICE_BUILD 1
#else
#define T2_HD inline
#define T2_DEVICE_BUILD 0
#endif

namespace t2fit {

constexpr int kMaxEcho = 32;

// Host-side echo-count dispatch: f(std::integral_constant<int, E>{}) for the run-time n_echo == E in 2..kMaxEcho, a
// value-initialised result (nullptr for a kernel pointer) for any other count.  Every per-echo-count template table goes
// through it, so this is the one place that decides which E are instantiated.
template <class F, int... I>
auto with_echo_count(int n_echo, F&& f, std::integer_sequence<int, I...>) {
    decltype(f(std::integral_constant<int, 2>{})) r{};
    ((n_echo == I + 2 ? (void)(r = f(std::integral_constant<int, I + 2>{})) : (void)0), ...);
    return r;
}
template <class F>
auto with_echo_count(int n_echo, F&& f) {
    return with_echo_count(n_echo, f, std::make_integer_sequence<int, kMaxEcho - 1>{});
}

enum Model : int { kMono2 = 0, kFloor3 = 1 };
enum Status : int { kOk = 0, kNonFinite = 1, kNotConverged = 2, kBadBounds = 3 };
enum InitMode : int { kInitLogLinear = 0, kInitPreset = 1, kInitBest = 2 };

// Launch-invariant constants.  Passed BY VALUE as a kernel parameter, so they live in the constant
// bank (c[0x0][...]) without a __constant__ symbol: launches on different streams never race.
struct FitConsts {
    float te[kMaxEcho];     // TE_e [ms]
    float nte2[kMaxEcho];   // -TE_e * log2(e):   exp(-TE_e r) = ex2(nte2_e * r)
    float tec[kMaxEcho];    // TE_e - mean(TE)   (centred abscissa of the log-linear initial guess)
    float x0[3];            // preset initial_guess (k, T2, sigma)          run_t2mapping.py:38,49,...
    float lb[3], ub[3];     // box actually in force for (k, T2, sigma); lb[0] is per voxel if no_prior
    float r_lo, r_hi;       // 1/ub[1], 1/lb[1]
    float r_x0;             // clamp(1/x0[1])
    float tol;              // relative step at which the iteration switches to its final pass
    int n_echo;
    int max_iter;
    int no_prior;           // lb[0] := y(TE_0) per voxel                   run_t2mapping.py:243-245
    int norm;               // y := y / max_e y                             run_t2mapping.py:237-240
    int init_mode;
};

struct VoxelFit {
    float k, t2, sigma;     // reference parameter order (k, T2, sigma)
    float res;              // signed mean residual                         utils/t2map_utils.py:81-84
    float fun;              // mean squared error at the solution           run_t2mapping.py:147,155
    int nit;
    int status;
};

// ---------------------------------------------------------------------------------------------
// math: MUFU approximations on the device, libm on the host simulation
// ---------------------------------------------------------------------------------------------
#if T2_DEVICE_BUILD
T2_HD float fast_ex2(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
T2_HD float fast_lg2(float x) { float y; asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
T2_HD float fast_rcp(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
T2_HD float fast_rsqrt(float x) { float y; asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
T2_HD bool warp_any(bool p) { return __any_sync(0xffffffffu, p); }
#else
T2_HD float fast_ex2(float x) { return exp2f(x); }
T2_HD float fast_lg2(float x) { return log2f(x); }
T2_HD float fast_rcp(float x) { return 1.0f / x; }
T2_HD float fast_rsqrt(float x) { return 1.0f / sqrtf(x); }
T2_HD bool warp_any(bool p) { return p; }
#endif
T2_HD double fast_ex2(double x) { return exp2(x); }
T2_HD double fast_lg2(double x) { return log2(x); }
T2_HD double fast_rcp(double x) { return 1.0 / x; }
T2_HD double fast_rsqrt(double x) { return 1.0 / sqrt(x); }

template <typename R> T2_HD R fdiv(R a, R b) { return a * fast_rcp(b); }
template <typename R> T2_HD R rmin(R a, R b) { return a < b ? a : b; }
template <typename R> T2_HD R rmax(R a, R b) { return a > b ? a : b; }
template <typename R> T2_HD R clampr(R x, R lo, R hi) { return rmin(rmax(x, lo), hi); }
template <typename R> T2_HD bool finite_r(R x) { return (x - x) == R(0); }
template <typename R> T2_HD R absr(R x) { return x < R(0) ? -x : x; }

// ---------------------------------------------------------------------------------------------
// log-linear initial guess of the decay rate:  weighted least squares of log2 y_e on TE_e with
// weights y_e^2, echoes with y_e <= 0 skipped.  Falls back to the preset T2 when fewer than two
// echoes are usable.
// ---------------------------------------------------------------------------------------------
template <typename R, int E>
T2_HD R loglinear_rate(const R (&y)[E], const FitConsts& c) {
    R sw = 0, swt = 0, swtt = 0, swl = 0, swtl = 0;
#pragma unroll
    for (int e = 0; e < E; ++e) {
        const R ye = y[e];
        const bool ok = ye > R(0);
        const R l = fast_lg2(ok ? ye : R(1));
        const R w = ok ? ye * ye : R(0);
        const R wt = w * R(c.tec[e]);
        sw += w;
        swt += wt;
        swtt += wt * R(c.tec[e]);
        swl += w * l;
        swtl += wt * l;
    }
    const R den = sw * swtt - swt * swt;
    const R num = sw * swtl - swt * swl;
    R r = -R(0.69314718055994531) * num * fast_rcp(den);      // slope is in log2 units per ms
    if (!(den > R(0)) || !finite_r(r)) r = R(c.r_x0);
    return clampr(r, R(c.r_lo), R(c.r_hi));
}

// ---------------------------------------------------------------------------------------------
// mono-exponential, 2 parameters (k, r).  k enters linearly, so one pass over the echoes yields the
// 2x2 normal equations for ANY k:
//     A = sum u^2   B = sum y u   C = sum te u^2   D = sum te y u   F = sum te^2 u^2 ,  u = exp(-te r)
//     J^T J = [[A, -kC], [-kC, k^2 F]]      J^T res = [B - kA,  -k (D - kC)]
// The k-row is solved exactly, k*(r) = clamp(B/A, kl, ku); what remains is the 1-D root of the reduced
// gradient g(r) = k (D - kC) on [r_lo, r_hi].  Its Gauss-Newton slope is the Schur complement
// k^2 (F - C^2/A) (k free) or k^2 F (k on a bound); with one more sum H = sum te^2 y u the exact slope
//     g'(r) = k (2kF - H) - (D - 2kC)^2 / A      (second term only while k is free)
// is available, so the iteration is a safeguarded Newton method (quadratic convergence): sign
// bracket of g, regime-aware step across the kink where k*(r) meets a bound, geometric expansion
// towards an unevaluated box bound, bisection when steps stop shrinking.  One MUFU.EX2 per echo per
// pass.  The iteration stops WITHOUT a verifying pass once a genuine Newton step is below `tol`
// (the error after the step is O(tol^2)); the epilogue evaluates k at the final r.
// ---------------------------------------------------------------------------------------------
template <typename R>
struct MonoSums { R A, B, C, D, F, H; };

template <typename R, int E>
T2_HD MonoSums<R> mono_pass(const R (&y)[E], const R (&ty)[E], const FitConsts& c, R r) {
    MonoSums<R> s{0, 0, 0, 0, 0, 0};
#pragma unroll
    for (int e = 0; e < E; ++e) {                 // per echo: FMUL, MUFU.EX2, FMUL, 6 FFMA
        const R u = fast_ex2(R(c.nte2[e]) * r);
        const R tu = R(c.te[e]) * u;
        s.A += u * u;
        s.B += y[e] * u;
        s.C += tu * u;
        s.D += ty[e] * u;
        s.F += tu * tu;
        s.H += ty[e] * tu;
    }
    return s;
}

template <typename R, int E>
T2_HD void solve_mono2(const R (&y)[E], const FitConsts& c, R kl, R ku, R r0, R& r_out, int& nit_out, int& status_out,
                       bool lane_valid) {
    const R r_lo = R(c.r_lo), r_hi = R(c.r_hi), tol = R(c.tol);
    R ty[E];
#pragma unroll
    for (int e = 0; e < E; ++e) ty[e] = R(c.te[e]) * y[e];
    R a = r_lo, b = r_hi;             // sign bracket of g:  g(a) < 0 < g(b) once evaluated
    bool ha = false, hb = false;      // bracket end has been evaluated (otherwise it is the box bound)
    R r = r0;
    int run_len = 0;                  // consecutive steps towards a bracket end that is still the box bound
    R dx1 = r_hi, dx2 = r_hi;         // magnitudes of the last two steps (stagnation guard)
    bool prev_small = false;
    int nit = 0;
    bool done = !lane_valid;
    int status = kOk;
    const int max_pass = c.max_iter;
    for (int it = 0; it < max_pass; ++it) {
        if (!warp_any(!done)) break;                      // convergence vote: whole warp leaves together
        const MonoSums<R> s = mono_pass<R, E>(y, ty, c, r);
        if (!done) {
            ++nit;
            const R inv_a = fast_rcp(s.A);
            const R kf = s.B * inv_a;                               // unconstrained linear parameter k*(r)
            const R k = clampr(kf, kl, ku);
            const bool free = (kf > kl) && (kf < ku);               // regime: k free / on a bound
            const R schur = free ? inv_a : R(0);
            const R kc = k * s.C;
            const R w = s.D - kc;
            const R g = k * w;                                      // 1/2 d cost/dr at k*(r)
            const R w2 = w - kc;                                    // D - 2kC
            const R h_gn = (k * k) * (s.F - s.C * (s.C * schur));   // Gauss-Newton slope (>= 0)
            const R h_ex = k * ((k + k) * s.F - s.H) - (w2 * w2) * schur;   // exact slope g'(r)
            const bool newton = h_ex > R(0.25) * h_gn;
            const R h = newton ? h_ex : h_gn;
            const R dr = (h > R(0)) ? -(g * fast_rcp(h)) : R(0);
            const R dkf = -(w2 * inv_a);                            // d k*/dr
            const R kf_new = kf + dkf * dr;
            const bool free_new = (kf_new > kl) && (kf_new < ku);
            const R adr = absr(dr);
            const bool brk = ha && hb;
            // the plain case: interior point, genuine Newton step, same regime after the step, step inside the
            // bracket and shrinking -- everything else goes through the guarded path below
            const bool interior = (r > r_lo) && (r < r_hi);
            const R a_n = (g > R(0)) ? a : r, b_n = (g > R(0)) ? r : b;
            const R rn_p = r + dr;
            const bool small_p = adr <= tol * r;
            // a Newton step below tol ends the iteration whatever the bracket says (at a converged point the
            // step can round to zero, rn_p == r); larger steps must stay inside the bracket and keep shrinking
            const bool plain = newton && interior && (free == free_new) && (it < max_pass - 1) &&
                               (small_p || ((rn_p > a_n) && (rn_p < b_n) &&
                                            (brk ? !(adr > R(0.5) * dx2) : !(it > 0 && adr > R(0.5) * dx1))));
#ifdef T2FIT_TRACE
            printf("it %d r %.9g T2 %.6f k %.6f free %d g %.6g hgn %.6g hex %.6g a %.6g b %.6g plain %d rn %.9g\n", it,
                   (double)r, 1.0 / (double)r, (double)k, (int)free, (double)g, (double)h_gn, (double)h_ex, (double)a,
                   (double)b, (int)plain, (double)rn_p);
#endif
            if (plain) {
                a = a_n; b = b_n;
                if (g > R(0)) hb = true; else ha = true;
                run_len = 0;
                done = small_p;           // Newton step below tol: the error after it is O(tol^2)
                prev_small = small_p;
                dx2 = dx1; dx1 = adr;
                r = rn_p;
            } else {
                const bool at_lo = (r <= r_lo) && (g >= R(0));      // T2 on its upper bound, gradient outward
                const bool at_hi = (r >= r_hi) && (g <= R(0));      // T2 on its lower bound
                if (at_lo || at_hi || g == R(0)) {
                    done = true;                                    // r is final
                } else if (it == max_pass - 1) {
                    done = true;
                    status = kNotConverged;
                } else {
                    // does the step cross the kink where k*(r) meets a bound?  then minimise the piecewise
                    // quadratic model: other regime's step if it lands beyond the kink, else the kink itself
                    R rn = rn_p;
                    const int q = (kf <= kl) ? -1 : ((kf >= ku) ? 1 : 0);
                    const int q_new = (kf_new <= kl) ? -1 : ((kf_new >= ku) ? 1 : 0);
                    const bool cross = (q_new != q) && (dkf != R(0));
                    if (cross) {
                        const int qb = (q != 0) ? q : q_new;        // the bound involved
                        const R kb = qb < 0 ? kl : ku;
                        const R r_kink = r + fdiv(kb - kf, dkf);
                        const bool to_free = (q != 0);
                        const R k2 = to_free ? kf : kb;
                        const R g2 = k2 * (s.D - k2 * s.C);
                        const R h2 = k2 * k2 * (s.F - (to_free ? s.C * s.C * inv_a : R(0)));
                        const R r2 = (h2 > R(0)) ? r - fdiv(g2, h2) : r_kink;
                        const bool beyond = (dr > R(0)) ? (r2 > r_kink) : (r2 < r_kink);
                        rn = beyond ? r2 : r_kink;
                    }
                    a = a_n; b = b_n;
                    if (g > R(0)) hb = true; else ha = true;
                    bool guarded = cross;
                    if (ha && hb) {
                        run_len = 0;
                        if (absr(rn - r) > R(0.5) * dx2) { rn = R(0.5) * (a + b); guarded = true; }   // steps not shrinking
                    } else if (it > 0 && !cross && absr(rn - r) > R(0.5) * dx1) {   // walking towards an unevaluated bound:
                        run_len = run_len < 4 ? run_len + 1 : 4;                    // expand the step geometrically
                        rn = r + (rn - r) * R(1 << run_len);
                        guarded = true;
                    }
                    if (!(rn > a && rn < b)) {                      // leave the bracket: bound or bisection
                        if (rn <= a) rn = ha ? R(0.5) * (a + b) : a;
                        else if (rn >= b) rn = hb ? R(0.5) * (a + b) : b;
                        else rn = R(0.5) * (a + b);
                        guarded = true;
                    }
                    const R step = absr(rn - r);
                    const bool small = step <= tol * r;
                    // guarded / Gauss-Newton steps converge linearly at best: stop on a step 16x below tol,
                    // or on two consecutive steps below tol
                    if (step <= R(0.0625) * tol * r || (small && prev_small)) done = true;
                    prev_small = small;
                    dx2 = dx1; dx1 = absr(rn - r);
                    r = rn;
                }
            }
        }
    }
    r_out = r; nit_out = nit; status_out = status;
}

// ---------------------------------------------------------------------------------------------
// noise-floor model, 3 parameters (k, r, s):  m_e = sqrt(k^2 u_e^2 + s^2).  Projected
// Levenberg-Marquardt on the 3x3 normal equations (Marquardt-scaled), active set from the sign of
// J^T res at the bounds, trial point clamped to the box, accept / reject on the true cost.  One
// MUFU.EX2 + one MUFU.RSQ per echo per pass.
// ---------------------------------------------------------------------------------------------
template <typename R>
struct FloorSums {
    R cost;
    R gk, gr, gs;                 // J^T res
    R hkk, hkr, hks, hrr, hrs, hss;
};

template <typename R, int E>
T2_HD FloorSums<R> floor_pass(const R (&y)[E], const FitConsts& c, R k, R r, R s2) {
    // third parameter is s2 = sigma^2: dm/ds2 = 1/(2m) does not vanish as sigma -> 0, so the
    // Gauss-Newton model stays valid when the floor is far below the signal
    FloorSums<R> a{0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
#pragma unroll
    for (int e = 0; e < E; ++e) {
        const R u = fast_ex2(R(c.nte2[e]) * r);
        const R ku = k * u;
        const R w = ku * ku + s2;
        const R inv = w > R(0) ? fast_rsqrt(w) : R(0);
        const R m = w * inv;
        const R res = y[e] - m;
        const R jk = ku * u * inv;                 // dm/dk
        const R jr = -R(c.te[e]) * ku * ku * inv;  // dm/dr
        const R js = R(0.5) * inv;                 // dm/d(sigma^2)
        a.cost += res * res;
        a.gk += jk * res; a.gr += jr * res; a.gs += js * res;
        a.hkk += jk * jk; a.hkr += jk * jr; a.hks += jk * js;
        a.hrr += jr * jr; a.hrs += jr * js; a.hss += js * js;
    }
    return a;
}

// The optimiser as a resumable run: start() = clipped start point, step() = one pass over the echoes at the trial point
// followed by the reaction to it (accept / reject, new trial point or stop).  The one-shot kernel steps all lanes of a
// warp until the last one has stopped; the queue kernel hands a lane that has stopped the next voxel instead.
constexpr int kFloorStarts = 4;   // kInitBest: log-linear, preset x0, T2 on its lower bound, T2 mid-box

template <typename R>
struct FloorRun {
    R kl, ku;                    // per-voxel bounds of k (the others are launch constants)
    R x[3], xt[3];               // accepted point and trial point, x = (k, r, sigma^2)
    FloorSums<R> cur;
    R lambda;
    int nit, status, it;
    bool have_cur, active;
    // kInitBest (multi-start): the objective has several local minima on noise-floor voxels (T2 on its lower bound with
    // sigma carrying the signal, T2 on its upper bound with k carrying it, the decaying solution in between); the run is
    // restarted from kFloorStarts start points and the lowest cost is kept
    int phase;                   // start point in use
    R bx[3], bcost;              // best finished run so far
    int bstatus, nit_sum;

    // the sigma box maps monotonically (sigma bounds are clamped to >= 0 on the host)
    T2_HD R lo(const FitConsts& c, int i) const { return i == 0 ? kl : i == 1 ? R(c.r_lo) : R(c.lb[2]) * R(c.lb[2]); }
    T2_HD R hi(const FitConsts& c, int i) const { return i == 0 ? ku : i == 1 ? R(c.r_hi) : R(c.ub[2]) * R(c.ub[2]); }

    T2_HD void start(const FitConsts& c, R kl_, R ku_, R k0, R r0, R s0, bool run) {
        kl = kl_; ku = ku_;
        x[0] = clampr(k0, lo(c, 0), hi(c, 0)); x[1] = clampr(r0, lo(c, 1), hi(c, 1)); x[2] = clampr(s0 * s0, lo(c, 2), hi(c, 2));
        xt[0] = x[0]; xt[1] = x[1]; xt[2] = x[2];
        cur = FloorSums<R>{};
        lambda = R(1e-3);
        nit = 0; status = kOk; it = 0;
        have_cur = false;
        active = run;
        phase = 0; bcost = R(INFINITY); bstatus = kOk; nit_sum = 0;
        bx[0] = x[0]; bx[1] = x[1]; bx[2] = x[2];
    }

    // kInitBest: the run from start `phase` has stopped.  Keep it if it is the best so far, then either restart from the
    // next start point (returns with active = true) or hand back the best run.
    template <int E>
    T2_HD void next_start(const R (&y)[E], const FitConsts& c) {
        nit_sum += nit;
        const R cost = have_cur ? cur.cost : R(INFINITY);
        // a run that hit the pass cap only wins against other capped runs
        const bool better = (status == kOk && (bstatus != kOk || cost < bcost)) || (status != kOk && bstatus != kOk && cost < bcost) ||
                            phase == 0;
        if (better) { bx[0] = x[0]; bx[1] = x[1]; bx[2] = x[2]; bcost = cost; bstatus = status; }
        ++phase;
        if (phase >= kFloorStarts) {
            x[0] = bx[0]; x[1] = bx[1]; x[2] = bx[2]; cur.cost = bcost; status = bstatus; nit = nit_sum;
            active = false;
            return;
        }
        R k0, r0, s0;
        if (phase == 1) { k0 = R(c.x0[0]); r0 = R(c.r_x0); s0 = R(c.x0[2]); }           // the reference's start: clipped preset x0
        else {
            r0 = phase == 2 ? R(c.r_hi) : sqrt(R(c.r_lo) * R(c.r_hi));                   // T2 on its lower bound / mid-box (geometric)
            R sa = 0, sb = 0, sy = 0;
#pragma unroll
            for (int e = 0; e < E; ++e) {
                const R u = fast_ex2(R(c.nte2[e]) * r0);
                sa += u * u; sb += y[e] * u; sy += y[e] * y[e];
            }
            k0 = sa > R(0) ? fdiv(sb, sa) : kl;
            if (!finite_r(k0)) k0 = kl;
            s0 = phase == 2 ? sqrt(sy * (R(1) / R(E))) : R(c.x0[2]);                     // the floor carries the signal / preset sigma
        }
        x[0] = clampr(k0, lo(c, 0), hi(c, 0)); x[1] = clampr(r0, lo(c, 1), hi(c, 1)); x[2] = clampr(s0 * s0, lo(c, 2), hi(c, 2));
        xt[0] = x[0]; xt[1] = x[1]; xt[2] = x[2];
        lambda = R(1e-3);
        nit = 0; status = kOk; it = 0;
        have_cur = false;
        active = true;
    }

    template <int E>
    T2_HD void step(const R (&y)[E], const FitConsts& c) {
        const R tol = R(c.tol);
        const int max_pass = c.max_iter;
        const FloorSums<R> t = floor_pass<R, E>(y, c, xt[0], xt[1], xt[2]);
        if (active) {
            bool accepted = false;
            R step_rel = 0, dec_rel = 1;
            if (!have_cur || t.cost <= cur.cost) {          // accept (the first pass always)
                if (have_cur) {
                    dec_rel = (cur.cost - t.cost) * fast_rcp(rmax(t.cost, R(1e-30)));
#pragma unroll
                    for (int i = 0; i < 3; ++i)
                        step_rel = rmax(step_rel, absr(xt[i] - x[i]) * fast_rcp(rmax(absr(x[i]), R(1e-12))));
                    lambda = rmax(lambda * R(0.2), R(1e-9));
                    ++nit;
                }
                cur = t; x[0] = xt[0]; x[1] = xt[1]; x[2] = xt[2];
                accepted = have_cur;
                have_cur = true;
            } else {
                lambda = rmin(lambda * R(8), R(1e12));
            }
            const bool last = (it == max_pass - 1);
            if (accepted && (step_rel <= tol || dec_rel <= R(1e-6))) {
                active = false;
            } else if (last) {
                active = false; status = kNotConverged;
            } else {
                // active set: on a bound with the (descent) direction J^T res pointing outward
                const R g[3] = {cur.gk, cur.gr, cur.gs};
                bool fixed[3];
#pragma unroll
                for (int i = 0; i < 3; ++i)
                    fixed[i] = (x[i] <= lo(c, i) && g[i] <= R(0)) || (x[i] >= hi(c, i) && g[i] >= R(0)) || !(lo(c, i) < hi(c, i));
                // Marquardt scaling: d_i = 1/sqrt(H_ii)
                const R dk = cur.hkk > R(0) ? fast_rsqrt(cur.hkk) : R(0);
                const R dr = cur.hrr > R(0) ? fast_rsqrt(cur.hrr) : R(0);
                const R ds = cur.hss > R(0) ? fast_rsqrt(cur.hss) : R(0);
                const bool f0 = fixed[0] || !(dk > R(0)), f1 = fixed[1] || !(dr > R(0)), f2 = fixed[2] || !(ds > R(0));
                const R one = R(1) + lambda;
                // scaled symmetric system  M z = b,  fixed rows/cols replaced by identity / zero rhs
                const R m01 = (f0 || f1) ? R(0) : cur.hkr * dk * dr;
                const R m02 = (f0 || f2) ? R(0) : cur.hks * dk * ds;
                const R m12 = (f1 || f2) ? R(0) : cur.hrs * dr * ds;
                const R b0 = f0 ? R(0) : cur.gk * dk;
                const R b1 = f1 ? R(0) : cur.gr * dr;
                const R b2 = f2 ? R(0) : cur.gs * ds;
                // closed-form inverse of [[one,m01,m02],[m01,one,m12],[m02,m12,one]] (cofactors)
                const R c00 = one * one - m12 * m12;
                const R c01 = m02 * m12 - m01 * one;
                const R c02 = m01 * m12 - m02 * one;
                const R c11 = one * one - m02 * m02;
                const R c12 = m01 * m02 - m12 * one;
                const R c22 = one * one - m01 * m01;
                const R det = one * c00 + m01 * c01 + m02 * c02;
                const R idet = fast_rcp(det);
                const R z0 = (c00 * b0 + c01 * b1 + c02 * b2) * idet;
                const R z1 = (c01 * b0 + c11 * b1 + c12 * b2) * idet;
                const R z2 = (c02 * b0 + c12 * b1 + c22 * b2) * idet;
                const R d[3] = {z0 * dk, z1 * dr, z2 * ds};
                R prop = 0;
                const bool all_fixed = f0 && f1 && f2;
#pragma unroll
                for (int i = 0; i < 3; ++i) {
                    R xn = clampr(x[i] + d[i], lo(c, i), hi(c, i));
                    if (!finite_r(xn)) xn = x[i];
                    prop = rmax(prop, absr(xn - x[i]) * fast_rcp(rmax(absr(x[i]), R(1e-12))));
                    xt[i] = xn;
                }
                if (all_fixed || prop <= tol * R(0.01)) {
                    active = false;                     // KKT point (or the step has vanished)
                    xt[0] = x[0]; xt[1] = x[1]; xt[2] = x[2];
                }
            }
            ++it;
            if (!active && c.init_mode == kInitBest) next_start<E>(y, c);
        }
    }

    T2_HD R sigma(const FitConsts& c) const {
        R sig = sqrt(x[2]);
        if (x[2] <= lo(c, 2)) sig = R(c.lb[2]);
        if (x[2] >= hi(c, 2)) sig = R(c.ub[2]);
        return sig;
    }
};

template <typename R, int E>
T2_HD void solve_floor3(const R (&y)[E], const FitConsts& c, R kl, R ku, R k0, R r0, R s0, R& k_out, R& r_out,
                        R& s_out, R& cost_out, int& nit_out, int& status_out, bool lane_valid) {
    FloorRun<R> run;
    run.start(c, kl, ku, k0, r0, s0, lane_valid);
    const int max_pass = c.max_iter * (c.init_mode == kInitBest ? kFloorStarts : 1);
    for (int it = 0; it < max_pass; ++it) {
        if (!warp_any(run.active)) break;
        run.template step<E>(y, c);
    }
    k_out = run.x[0]; r_out = run.x[1]; s_out = run.sigma(c); cost_out = run.cur.cost; nit_out = run.nit; status_out = run.status;
}

// ---------------------------------------------------------------------------------------------
// One voxel end to end: validity, normalisation, per-voxel bounds, initial guess, solve, residual
// epilogue.  Mirrors the contract of fit_voxel + compute_residuals:
//   * non-finite echo      -> status kNonFinite, params = clip(x0, bounds), nit 0, fun NaN
//                             (scipy: ABNORMAL, success False, x = clipped x0; SURVEY.md 8(a))
//   * no_prior & y0 > ub_k -> status kBadBounds (scipy raises ValueError; the host shim re-raises)
//   * res  = sum_e (y_e - pred_e) / E   signed                (utils/t2map_utils.py:81-84)
//   * fun  = sum_e (y_e - pred_e)^2 / E                       (run_t2mapping.py:147,155)
// ---------------------------------------------------------------------------------------------
// what the preamble of fit_voxel decides per voxel: bounds of k, validity, and the start point
template <typename R>
struct VoxelPre {
    R kl, ku;
    R k0, r0, s0;
    int status;              // kOk, kNonFinite or kBadBounds
};

// validity, normalisation (in place), per-voxel bounds, initial guess
template <typename R, int MODEL, int E>
T2_HD VoxelPre<R> voxel_prepare(R (&y)[E], const FitConsts& c) {
    VoxelPre<R> p;
    const R y0_raw = y[0];
    R fin = 0;                                              // 0 if every echo is finite, NaN otherwise
#pragma unroll
    for (int e = 0; e < E; ++e) fin += y[e] * R(0);
    if (c.norm) {                                           // run_t2mapping.py:237-240
        R ymax = y[0];
#pragma unroll
        for (int e = 1; e < E; ++e) ymax = rmax(ymax, y[e]);
        const R inv = fast_rcp(ymax);
        fin = 0;
#pragma unroll
        for (int e = 0; e < E; ++e) { y[e] *= inv; fin += y[e] * R(0); }
    }
    p.kl = c.no_prior ? y0_raw : R(c.lb[0]);                // run_t2mapping.py:243-245
    p.ku = R(c.ub[0]);
    p.status = kOk;
    if (c.no_prior && (y0_raw > p.ku)) p.status = kBadBounds;   // scipy: "An upper bound is less than ..."
    else if (!(fin == R(0))) p.status = kNonFinite;
    p.r0 = R(c.r_x0); p.k0 = R(c.x0[0]); p.s0 = R(c.x0[2]);
    if (c.init_mode != kInitPreset) {
        p.r0 = loglinear_rate<R, E>(y, c);
        if (MODEL != kMono2) {
            R sa = 0, sb = 0;
#pragma unroll
            for (int e = 0; e < E; ++e) {
                const R u = fast_ex2(R(c.nte2[e]) * p.r0);
                sa += u * u;
                sb += y[e] * u;
            }
            p.k0 = sa > R(0) ? fdiv(sb, sa) : p.k0;
        }
    }
    return p;
}

// what fit_voxel returns + the residual epilogue, from the solver's (k, r, s) -- ignored when pre.status != kOk
template <typename R, int MODEL, int E>
T2_HD VoxelFit voxel_finish(const R (&y)[E], const FitConsts& c, const VoxelPre<R>& pre, R k, R r, R s, int nit, int st) {
    VoxelFit out;
    const R kl = pre.kl, ku = pre.ku;
    int status = pre.status;
    R t2;
    const bool solved = (status == kOk);
    if (solved) {
        status = st;
        t2 = fast_rcp(r);
        if (r <= R(c.r_lo)) t2 = R(c.ub[1]);
        if (r >= R(c.r_hi)) t2 = R(c.lb[1]);
    } else {
        // clipped x0, NaN bounds ignored (np.clip semantics seen in the reference run, SURVEY 8(a))
        k = R(c.x0[0]);
        if (kl == kl) k = rmax(k, kl);
        k = rmin(k, ku);
        t2 = clampr(R(c.x0[1]), R(c.lb[1]), R(c.ub[1]));
        s = (MODEL == kMono2) ? R(0) : clampr(R(c.x0[2]), R(c.lb[2]), R(c.ub[2]));
        nit = 0;
        if (status == kBadBounds) { k = t2 = R(NAN); if (MODEL != kMono2) s = R(NAN); }
    }
    // epilogue on the stored (float32) T2, as compute_residuals does: decay factors once, then (mono)
    // the linear parameter k = clamp(B/A) at exactly this T2, then the residual sums
    const float t2f = float(t2), sf = float(s);
    const R rr = fast_rcp(R(t2f));
    R u[E];
    R sa = 0, sb = 0;
#pragma unroll
    for (int e = 0; e < E; ++e) {
        u[e] = fast_ex2(R(c.nte2[e]) * rr);
        sa += u[e] * u[e];
        sb += y[e] * u[e];
    }
    if (MODEL == kMono2 && solved) k = clampr(sa > R(0) ? fdiv(sb, sa) : R(0), kl, ku);
    const float kf = float(k);
    R rsum = 0, csum = 0;
#pragma unroll
    for (int e = 0; e < E; ++e) {
        R pred = R(kf) * u[e];
        if (MODEL != kMono2) {
            const R w = pred * pred + R(sf) * R(sf);
            pred = w > R(0) ? w * fast_rsqrt(w) : R(0);
        }
        const R d = y[e] - pred;
        rsum += d;
        csum += d * d;
    }
    const R inv_e = R(1) / R(E);
    out.k = kf; out.t2 = t2f; out.sigma = sf;
    out.res = float(rsum * inv_e);
    out.fun = (status == kNonFinite || status == kBadBounds) ? NAN : float(csum * inv_e);
    out.nit = nit;
    out.status = status;
    return out;
}

template <typename R, int MODEL, int E>
T2_HD VoxelFit fit_voxel(R (&y)[E], const FitConsts& c, bool lane_valid) {
    const VoxelPre<R> pre = voxel_prepare<R, MODEL, E>(y, c);
    const bool run = lane_valid && pre.status == kOk;       // lanes that do not run start as `done`
    R k = 0, r = R(c.r_x0), s = 0;
    int nit = 0, st = kOk;
    if (MODEL == kMono2) {
        solve_mono2<R, E>(y, c, pre.kl, pre.ku, pre.r0, r, nit, st, run);
    } else {
        R cost = 0;
        solve_floor3<R, E>(y, c, pre.kl, pre.ku, pre.k0, pre.r0, pre.s0, k, r, s, cost, nit, st, run);
    }
    return voxel_finish<R, MODEL, E>(y, c, pre, k, r, s, nit, st);
}

}  // namespace t2fit
