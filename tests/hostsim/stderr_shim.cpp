// Host build of the per-voxel standard-error routine (fetal_t2mapping_b200/csrc/t2fit_stderr.cuh) -- TEST TOOL ONLY.
//
// g++ compiles the same header the stderr_kernel runs (T2FIT_HOSTSIM), so the `-m "not gpu"` suite can check the
// arithmetic against oracle/stderr_oracle.py without a device.  Never linked into libt2fit; not a fallback.
#define T2FIT_HOSTSIM 1
#include "../../fetal_t2mapping_b200/csrc/t2fit_stderr.cuh"

#include <stdint.h>

using namespace t2fit;

template <int MODEL, int E>
static void rows_e(const float* rows, int64_t m, const double* te, int norm, const float* k, const float* t2, const float* s,
                   double* out) {
    for (int64_t i = 0; i < m; ++i) {
        float y[E];
        for (int e = 0; e < E; ++e) y[e] = rows[i * E + e];
        double v[3];
        se::voxel_stderr<MODEL, E>(y, te, norm != 0, k[i], t2[i], s ? s[i] : 0.0f, v);
        for (int j = 0; j < 3; ++j) out[3 * i + j] = v[j];
    }
}

template <int MODEL>
static int rows_model(int n_echo, const float* rows, int64_t m, const double* te, int norm, const float* k, const float* t2,
                      const float* s, double* out) {
    switch (n_echo) {
#define CASE(E) case E: rows_e<MODEL, E>(rows, m, te, norm, k, t2, s, out); return 0;
        CASE(2) CASE(3) CASE(4) CASE(5) CASE(6) CASE(7) CASE(8) CASE(9) CASE(10) CASE(11) CASE(12) CASE(13) CASE(14) CASE(15)
        CASE(16) CASE(17) CASE(18) CASE(19) CASE(20) CASE(21) CASE(22) CASE(23) CASE(24) CASE(25) CASE(26) CASE(27) CASE(28)
        CASE(29) CASE(30) CASE(31) CASE(32)
#undef CASE
        default: return T2FIT_EINVAL;
    }
}

// rows: [m, n_echo] float32; k / t2 / sigma: [m] float32 (sigma may be NULL for gaussian); out: [m, 3] float64 (k, T2, sigma)
extern "C" int stderr_rows(const float* rows, int64_t m, int n_echo, const double* te, int model, int norm, const float* k,
                           const float* t2, const float* sigma, double* out) {
    if (model == T2FIT_MODEL_GAUSSIAN) return rows_model<T2FIT_MODEL_GAUSSIAN>(n_echo, rows, m, te, norm, k, t2, sigma, out);
    if (model == T2FIT_MODEL_GAUSSIAN_RICIAN)
        return rows_model<T2FIT_MODEL_GAUSSIAN_RICIAN>(n_echo, rows, m, te, norm, k, t2, sigma, out);
    if (model == T2FIT_MODEL_RICIAN) return rows_model<T2FIT_MODEL_RICIAN>(n_echo, rows, m, te, norm, k, t2, sigma, out);
    return T2FIT_EINVAL;
}

extern "C" double stderr_i1e(double x) { return se::i1e(x); }
