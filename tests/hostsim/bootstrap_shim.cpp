// Host build of the parametric-bootstrap routines (fetal_t2mapping_b200/csrc/t2fit_bootstrap.cuh) -- TEST TOOL ONLY.
//
// g++ compiles the same header replicate_kernel and bootstrap_stats_kernel run (T2FIT_HOSTSIM), so the `-m "not gpu"` suite
// can check the Philox words, the replicate rows and the statistics against oracle/bootstrap_oracle.py without a device.
// Never linked into libt2fit; not a fallback.
#define T2FIT_HOSTSIM 1
#include "../../fetal_t2mapping_b200/csrc/t2fit_bootstrap.cuh"

#include <stdint.h>

using namespace t2fit;

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
