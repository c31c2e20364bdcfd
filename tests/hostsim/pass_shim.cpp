// Host build of the per-voxel analysis routines (fetal_t2mapping_b200/csrc/t2fit_stderr.cuh, t2fit_interval.cuh,
// t2fit_bootstrap.cuh) -- TEST TOOL ONLY.
//
// g++ compiles the same headers stderr_kernel, interval_kernel, replicate_kernel and bootstrap_stats_kernel run
// (T2FIT_HOSTSIM), so the `-m "not gpu"` suite can check the arithmetic against oracle/stderr_oracle.py,
// oracle/interval_oracle.py and oracle/bootstrap_oracle.py without a device.  Never linked into libt2fit; not a fallback.
#define T2FIT_HOSTSIM 1
#include "../../fetal_t2mapping_b200/csrc/t2fit_interval.cuh"
#include "../../fetal_t2mapping_b200/csrc/t2fit_bootstrap.cuh"

#include <stdint.h>
#include <vector>

using namespace t2fit;

template <int MODEL, int E>
static void stderr_rows_e(const float* rows, int64_t m, const double* te, int norm, const float* k, const float* t2,
                          const float* s, double* out) {
    for (int64_t i = 0; i < m; ++i) {
        float y[E];
        for (int e = 0; e < E; ++e) y[e] = rows[i * E + e];
        double v[3];
        se::voxel_stderr<MODEL, E>(y, te, norm != 0, k[i], t2[i], s ? s[i] : 0.0f, v);
        for (int j = 0; j < 3; ++j) out[3 * i + j] = v[j];
    }
}

// rows: [m, n_echo] float32; k / t2 / sigma: [m] float32 (sigma may be NULL for gaussian); out: [m, 3] float64 (k, T2, sigma)
extern "C" int stderr_rows(const float* rows, int64_t m, int n_echo, const double* te, int model, int norm, const float* k,
                           const float* t2, const float* sigma, double* out) {
    const bool ran = with_echo_count(n_echo, [&](auto e) {
        constexpr int E = decltype(e)::value;
        if (model == T2FIT_MODEL_GAUSSIAN) stderr_rows_e<T2FIT_MODEL_GAUSSIAN, E>(rows, m, te, norm, k, t2, sigma, out);
        else if (model == T2FIT_MODEL_GAUSSIAN_RICIAN) stderr_rows_e<T2FIT_MODEL_GAUSSIAN_RICIAN, E>(rows, m, te, norm, k, t2, sigma, out);
        else if (model == T2FIT_MODEL_RICIAN) stderr_rows_e<T2FIT_MODEL_RICIAN, E>(rows, m, te, norm, k, t2, sigma, out);
        else return false;
        return true;
    });
    return ran ? 0 : T2FIT_EINVAL;
}

extern "C" double stderr_i1e(double x) { return se::i1e(x); }

template <int E>
static void interval_rows_e(const float* rows, int64_t m, const double* te, int model, int norm, const double* box,
                            int no_prior, double q, int G, double* out, uint8_t* flags, double* prof) {
    const iv::Box b{box[0], box[1], box[2], box[3], box[4], box[5]};
    std::vector<iv::Grid> w(1);
    for (int64_t i = 0; i < m; ++i) {
        float y[E];
        for (int e = 0; e < E; ++e) y[e] = rows[i * E + e];
        iv::Voxel v;
        const bool ok = iv::load_voxel<E>(y, te, model, norm != 0, b, no_prior != 0, v);
        int fl;
        iv::voxel_interval(v, ok, q, G, w[0], out[3 * i], out[3 * i + 1], out[3 * i + 2], fl, prof ? prof + i * G : nullptr);
        flags[i] = (uint8_t)fl;
    }
}

// rows: [m, n_echo] float32; box: (k_lo, k_hi, t2_lo, t2_hi, sigma_lo, sigma_hi) as in t2fit_problem (k_lo replaced by
// y(TE_0) when no_prior); out: [m, 3] float64 (lo, hi, best); flags: [m]; prof: [m, G] float64 or NULL
extern "C" int interval_rows(const float* rows, int64_t m, int n_echo, const double* te, int model, int norm,
                             const double* box, int no_prior, double q, int G, double* out, uint8_t* flags, double* prof) {
    if (G < iv::kMinGrid || G > iv::kMaxGrid) return T2FIT_EINVAL;
    if (model != T2FIT_MODEL_GAUSSIAN && model != T2FIT_MODEL_GAUSSIAN_RICIAN && model != T2FIT_MODEL_RICIAN) return T2FIT_EINVAL;
    const bool ran = with_echo_count(n_echo, [&](auto e) {
        interval_rows_e<decltype(e)::value>(rows, m, te, model, norm, box, no_prior, q, G, out, flags, prof);
        return true;
    });
    return ran ? 0 : T2FIT_EINVAL;
}

extern "C" void bootstrap_philox(const uint32_t* ctr, const uint32_t* key, uint32_t* out) {
    uint32_t w[4];
    bs::philox4x32_10(ctr[0], ctr[1], ctr[2], ctr[3], key[0], key[1], w);
    for (int j = 0; j < 4; ++j) out[j] = w[j];
}

template <int E>
static void bootstrap_rows_e(const float* rows, int64_t m, const double* te, int model, int norm, const float* k,
                             const float* t2, const float* s, const float* noise, const int64_t* vid, uint64_t seed, int n_rep,
                             float* out) {
    for (int64_t i = 0; i < m; ++i) {
        float y[E];
        for (int e = 0; e < E; ++e) y[e] = rows[i * E + e];
        bs::Source<E> src;
        bs::load_source<E>(y, te, model, norm != 0, k[i], t2[i], s ? s[i] : 0.0f, noise != nullptr, noise ? noise[i] : 0.0f, src);
        for (int r = 0; r < n_rep; ++r) {
            float row[E];
            bs::replicate_row<E>(src, model, seed, r, (uint64_t)vid[i], row);
            for (int e = 0; e < E; ++e) out[((i * n_rep) + r) * E + e] = row[e];
        }
    }
}

// rows: [m, n_echo] float32 (the voxels' echoes); k / t2 / sigma / noise: [m] float32 (sigma NULL for gaussian, noise NULL =
// estimated); vid: [m] flat voxel ids; out: [m * n_rep, n_echo] float32, row i * n_rep + r
extern "C" int bootstrap_rows(const float* rows, int64_t m, int n_echo, const double* te, int model, int norm, const float* k,
                              const float* t2, const float* sigma, const float* noise, const int64_t* vid, uint64_t seed,
                              int n_rep, float* out) {
    if (model != T2FIT_MODEL_GAUSSIAN && model != T2FIT_MODEL_GAUSSIAN_RICIAN && model != T2FIT_MODEL_RICIAN) return T2FIT_EINVAL;
    const bool ran = with_echo_count(n_echo, [&](auto e) {
        bootstrap_rows_e<decltype(e)::value>(rows, m, te, model, norm, k, t2, sigma, noise, vid, seed, n_rep, out);
        return true;
    });
    return ran ? 0 : T2FIT_EINVAL;
}

// rep_*: [m * n_rep] replicate results (row i * n_rep + r; sigma NULL for gaussian); mean / sd: [3, m]; lo / hi / n_used /
// n_ok: [m]
extern "C" int bootstrap_stats(int model, int64_t m, int n_rep, const float* rk, const float* rt, const float* rs,
                               const uint8_t* st, double level, float* mean, float* sd, float* lo, float* hi, int32_t* n_used,
                               int32_t* n_ok) {
    if (n_rep < bs::kMinRep || n_rep > bs::kMaxRep) return T2FIT_EINVAL;
    for (int64_t i = 0; i < m; ++i) {
        const int64_t b = i * n_rep;
        float mu[3], s[3];
        bs::voxel_stats_host(model, n_rep, rk + b, rt + b, rs ? rs + b : nullptr, st + b, level, mu, s, lo + i, hi + i,
                             n_used + i, n_ok + i);
        for (int j = 0; j < 3; ++j) { mean[j * m + i] = mu[j]; sd[j * m + i] = s[j]; }
    }
    return 0;
}
