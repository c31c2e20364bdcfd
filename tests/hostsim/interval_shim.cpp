// Host build of the per-voxel T2 interval routine (fetal_t2mapping_b200/csrc/t2fit_interval.cuh) -- TEST TOOL ONLY.
//
// g++ compiles the same header the interval_kernel runs (T2FIT_HOSTSIM), so the `-m "not gpu"` suite can check it
// against oracle/interval_oracle.py without a device.  Never linked into libt2fit; not a fallback.
#define T2FIT_HOSTSIM 1
#include "../../fetal_t2mapping_b200/csrc/t2fit_interval.cuh"

#include <stdint.h>
#include <vector>

using namespace t2fit;

template <int E>
static void rows_e(const float* rows, int64_t m, const double* te, int model, int norm, const double* box, int no_prior,
                   double q, int G, double* out, uint8_t* flags, double* prof) {
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
    switch (n_echo) {
#define CASE(E) case E: rows_e<E>(rows, m, te, model, norm, box, no_prior, q, G, out, flags, prof); return 0;
        CASE(2) CASE(3) CASE(4) CASE(5) CASE(6) CASE(7) CASE(8) CASE(9) CASE(10) CASE(11) CASE(12) CASE(13) CASE(14) CASE(15)
        CASE(16) CASE(17) CASE(18) CASE(19) CASE(20) CASE(21) CASE(22) CASE(23) CASE(24) CASE(25) CASE(26) CASE(27) CASE(28)
        CASE(29) CASE(30) CASE(31) CASE(32)
#undef CASE
        default: return T2FIT_EINVAL;
    }
}
