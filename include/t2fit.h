/* t2fit.h - C ABI of libt2fit: the B200 (sm_100a) per-voxel T2 relaxation fit.
 *
 * Drop-in boundary.  The reference (Medical-Image-Analysis-Laboratory/fetal_t2mapping) has no
 * FFI; its hot path is the call pair inside process_t2maps:
 *
 *     all_results = pool.map(partial(fit_voxel, fit, fit_params, TEeffs, reshaped_t2w, prior, norm),
 *                            mask_indices)                                 run_t2mapping.py:430-443
 *     res_map     = compute_residuals(reshaped_t2w, TEeffs, fit, norm, k_map, t2_map, sigma_map,
 *                                     res_map, mask_indices, mask)         run_t2mapping.py:461
 *
 * plus the glue around it (mask union :383-384, flatten :411-412, np.where :421, zero maps :415-418,
 * scatter :455-458).  Each entry point below names the reference lines it replaces.  Plain
 * pointers and sizes only; the caller owns every buffer; nothing here throws; every function
 * returns 0 on success or a negative T2FIT_E* code, with text in t2fit_last_error().
 * Per-voxel problems are reported in status[], never in the return code.
 *
 * There is NO CPU implementation of the fit behind this ABI: without a CUDA device
 * t2fit_init() fails with T2FIT_ENODEVICE and every compute call fails with T2FIT_ENOTINIT.
 */
#ifndef T2FIT_H
#define T2FIT_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define T2FIT_ABI_VERSION 5
#define T2FIT_MAX_ECHO 32
#define T2FIT_MAX_DUP 7 /* peer destinations of the fused all-gather: the other GPUs of an 8-GPU node */

/* return codes */
#define T2FIT_OK 0
#define T2FIT_EINVAL (-1)    /* bad argument (sizes, NULL, n_echo out of range, len(bounds)) */
#define T2FIT_ENODEVICE (-2) /* no usable CUDA device */
#define T2FIT_ENOTINIT (-3)  /* t2fit_init() has not succeeded in this process */
#define T2FIT_ECUDA (-4)     /* CUDA runtime error (text in t2fit_last_error) */
#define T2FIT_ENOMEM (-5)

/* fit model = the reference's `fit` string (run_t2mapping.py:37,48) */
#define T2FIT_MODEL_GAUSSIAN 0        /* 'gaussian'        k exp(-te/T2)                   :129-131 */
#define T2FIT_MODEL_GAUSSIAN_RICIAN 1 /* 'gaussian_rician' sqrt(k^2 exp(-2te/T2)+sigma^2)  :133-138 */
#define T2FIT_MODEL_RICIAN 2          /* 'rician'  Rician negative log-likelihood (i0e)     :157-177;
                                         T2FIT_SOLVER_LBFGSB[_DENSE] only (not a least-squares problem) */

/* which optimiser runs per voxel */
#define T2FIT_SOLVER_FAST 0   /* float32 register-resident Newton / Levenberg-Marquardt: converges to the bounded
                                 minimiser of the objective (what the reference's optimiser approaches) */
#define T2FIT_SOLVER_LBFGSB 1 /* float64 restatement of the reference's own optimiser: scipy L-BFGS-B (m = 10) with
                                 2-point finite-difference gradients, started from the clipped preset x0, stopped
                                 by the preset's ftol / gtol / maxls (:260-286).  Reproduces the reference's result
                                 -- params, success, nit, fun and the callback trace -- also where the reference
                                 stops before convergence (ftol = gtol = 1e-2 presets). */
#define T2FIT_SOLVER_LBFGSB_DENSE 2 /* the same optimiser, same objectives / differences / line search / stopping tests
                                 and lbfgsb_* options, with the limited-memory matrix held as the n x n matrix it
                                 represents (n <= 3) instead of scipy's compact 2m x 2m form: equal in exact
                                 arithmetic, equal parity with the reference on the golden fixtures, ~20-30x the
                                 throughput (csrc/t2fit_lbfgsb_dense.cuh, DESIGN.md 3b). */

/* echo layout */
#define T2FIT_LAYOUT_AOS 0 /* reshaped_t2w: [n_vox, n_echo] row-major float32 (run_t2mapping.py:411) */
#define T2FIT_LAYOUT_SOA 1 /* packed: [n_echo, ld] float32, column i = i-th fitted voxel            */
#define T2FIT_LAYOUT_PLANES 2 /* per-TE volumes as they come off disk: [n_echo, ld] float32, ld >= n_vox, plane e =
                                 the flattened recon volume of echo e (the list `t2w` BEFORE np.stack, :377-385);
                                 voxel mask_idx[i] of every plane is read -- no interleaving pass is needed */

/* where the data pointers of a call live */
#define T2FIT_MEM_HOST 0   /* library stages through pinned buffers, copies results back */
#define T2FIT_MEM_DEVICE 1 /* pointers are device memory on the initialised GPU; fully asynchronous */

/* per-voxel status byte */
#define T2FIT_ST_OK 0           /* result.success == True                                            */
#define T2FIT_ST_NONFINITE 1    /* NaN/Inf echo: reference returns success False, x = clipped x0     */
#define T2FIT_ST_NOTCONVERGED 2 /* optimiser gave up on finite input: iteration cap, or (L-BFGS-B) line-search
                                   failure / maxiter / maxfun (reference: success False)             */
#define T2FIT_ST_BADBOUNDS 3    /* --no_prior and S(TE0) > k upper bound: scipy raises ValueError    */

/* initial guess of the iteration */
#define T2FIT_INIT_LOGLINEAR 0 /* weighted log-linear fit of the echoes (default) */
#define T2FIT_INIT_PRESET 1    /* the preset's initial_guess, clipped, as the reference starts */
#define T2FIT_INIT_BEST 2      /* 3-parameter FAST solver: multi-start -- log-linear, preset x0, T2 on its lower bound, T2
                                  mid-box -- and the lowest cost wins (the noise-floor objective has several local minima on
                                  voxels whose signal has decayed into the floor); the 2-parameter solver treats it as
                                  T2FIT_INIT_LOGLINEAR (its reduced problem is solved by a bracketing Newton iteration) */

/* element type of t2fit_problem.mask_idx */
#define T2FIT_IDX_I64 0
#define T2FIT_IDX_I32 1

/* The fit of one call.  Mirrors fit_voxel's arguments (run_t2mapping.py:120). */
typedef struct t2fit_problem {
    const float *echoes;     /* see layout */
    int32_t layout;          /* T2FIT_LAYOUT_* */
    int32_t memory;          /* T2FIT_MEM_* (applies to echoes, mask_idx and every output pointer) */
    int64_t ld;              /* SOA / PLANES: elements between consecutive echo planes (SOA >= n_fit, PLANES >= n_vox) */
    const int64_t *mask_idx; /* [n_fit] ascending flat voxel indices = mask_indices (:421); NULL = rows 0..n_fit-1.
                                AOS / PLANES: voxel to read (and dense output slot).  SOA: dense output slot only. */
    int64_t n_vox;           /* rows of the AOS array = length of dense maps */
    int64_t n_fit;           /* voxels to fit (M) */
    int32_t n_echo;          /* E, 2..T2FIT_MAX_ECHO */
    int32_t model;           /* T2FIT_MODEL_* */
    const double *te_ms;     /* HOST pointer, [n_echo] echo times in ms = TEeffs (:386) */
    double x0[3];            /* fit_params['initial_guess'] (k, T2, sigma)          :38,49,74,85 */
    double lb[3], ub[3];     /* fit_params['param_bounds']                          :39,50,75,86 */
    int32_t no_prior;        /* prior == False: bounds[0]=(S(TE0), no_prior_k_ub), bounds[1]=(no_prior_t2_lb,_ub) :243-245 */
    double no_prior_k_ub;    /* 10000 */
    double no_prior_t2_lb;   /* 10    */
    double no_prior_t2_ub;   /* 2000  */
    int32_t norm;            /* divide each row by its maximum (:237-240; utils/t2map_utils.py:74-79) */
    int32_t max_iter;        /* cap on passes over the echoes per voxel; 0 = default */
    float tol;               /* relative step tolerance; 0 = default */
    int32_t init;            /* T2FIT_INIT_* (FAST solver only; LBFGSB always starts from the clipped x0) */
    int32_t solver;          /* T2FIT_SOLVER_* */
    /* fit_params['options'] of the reference's minimize() call (:40-45,:51-57,...); LBFGSB solver only.
       0 selects scipy's default: ftol 2.220446049250313e-09, gtol 1e-5, maxls 20, maxiter = maxfun = 15000. */
    double lbfgsb_ftol, lbfgsb_gtol;
    int32_t lbfgsb_maxls, lbfgsb_maxiter, lbfgsb_maxfun;
    /* Element type of `echoes` for T2FIT_MEM_HOST calls: 0 = float32 (default), or T2FIT_DT_I16 / _U16 / _I32 / _F64 --
       the volume as it comes out of the NIfTI reader.  The `.astype(np.float32)` of the reference (:411) then happens
       while the masked rows are gathered into the staging buffers: only the n_fit fitted rows are cast, not all n_vox.
       Device-memory calls take float32 only. */
    int32_t echo_dtype;
    /* Element type of mask_idx: T2FIT_IDX_I64 (0, np.where's int64) or T2FIT_IDX_I32 (the same indices as int32, n_vox <
       2^31: half the index bytes over PCIe / from HBM).  mask_idx is then really a const int32_t*. */
    int32_t idx_dtype;
} t2fit_problem;

/* Results.  Any pointer may be NULL (that output is skipped).  Parameter maps follow the reference's
 * (k, T2, sigma) naming: t2 = x[1], k = x[0], sigma = x[2] (run_t2mapping.py:455-458). */
typedef struct t2fit_outputs {
    float *t2, *k, *sigma, *res; /* dense != 0: [n_vox] maps, only masked slots written (caller zero-fills,
                                    as :415-418); dense == 0: [n_fit] compact */
    uint8_t *status;             /* [n_fit] T2FIT_ST_* (== 0  <=>  convergence_flags[i], :450) */
    int32_t *nit;                /* [n_fit] num_iterations_array (:451): L-BFGS-B iterations (LBFGSB solver) or passes
                                    of the FAST solver (a different count) */
    float *fun;                  /* [n_fit] mean squared error at the solution (final_errors_array, :452) */
    int32_t dense;
    int64_t status_count[4];     /* OUT (host): voxels per status; filled when the call is synchronous
                                    (T2FIT_MEM_HOST) or by t2fit_status_counts() */
    /* iteration_info of the callback (:180-234), LBFGSB solver only, any may be NULL: per voxel up to trace_cap
       entries of f_val and step_size (NaN for the first iteration, as the reference) and the entry count
       (= min(nit, trace_cap)).  Row i of trace_f / trace_step starts at i * trace_cap. */
    float *trace_f, *trace_step;
    int32_t *trace_len;
    int32_t trace_cap;
    const uint8_t *zero_fill_mask; /* device calls with dense != 0 only: the [n_vox] uint8 mask (1 byte per voxel,
                                    nonzero = masked, consistent with mask_idx, 4-byte aligned).  When given, the
                                    call also zero-fills every unmasked slot of the four maps (np.zeros_like,
                                    :415-418) -- and all of sigma for the 2-parameter model -- so the caller
                                    need not pre-zero them.  2-parameter fast solver with all four maps given and
                                    16-byte aligned: inside the fit launch itself (every fit thread zeroes a few
                                    4-voxel words while it waits for its echoes).  Otherwise (3-parameter fits,
                                    L-BFGS-B solver, very sparse masks, unaligned maps, T2FIT_FILL=stream): a
                                    kernel on a side stream concurrent with the fit (forked from / joined into
                                    `stream`; one such call at a time per process, the events are shared).
                                    NULL = caller zero-fills. */
    /* Fused all-gather (T2FIT_MEM_DEVICE, dense == 0): every compact result of this call is ALSO stored to n_dup further
       destinations -- the same slab of the peer GPUs' buffers, mapped with t2fit_shared_open -- straight from the kernel
       epilogue over NVLink (peer stores; no collective, the transfer overlaps the fit).  dup_*[j] may be NULL (skipped);
       element i of this call goes to dup_*[j][i].  After the call a cross-rank barrier that is ordered after the kernels
       (e.g. a one-element NCCL all-reduce on the same stream) completes the gather on every rank. */
    int32_t n_dup;
    float *dup_t2[T2FIT_MAX_DUP], *dup_k[T2FIT_MAX_DUP], *dup_sigma[T2FIT_MAX_DUP], *dup_res[T2FIT_MAX_DUP];
    uint8_t *dup_status[T2FIT_MAX_DUP];
    uint64_t *counts_dev;        /* T2FIT_MEM_DEVICE calls, optional: [4] DEVICE counters this call ADDS its voxels to
                                    (slot 0: mask_idx entries outside [0, n_vox), which read / write voxel 0 instead --
                                    the reference raises IndexError there; slots 1..3: voxels per non-OK status).  The caller
                                    zeroes and reads them on its own stream: the histogram of exactly this call, whatever
                                    else runs on other streams.  NULL: the per-process counters behind
                                    t2fit_status_counts(). */
} t2fit_outputs;

/* Bind this process to one GPU (one process per GPU; device = LOCAL_RANK) and create its context
 * (streams, pinned staging, counters).  Idempotent for the same device. */
int t2fit_init(int device);
void t2fit_shutdown(void);
const char *t2fit_last_error(void);
int t2fit_abi_version(void);
/* name, SM count and clock of the bound device; any pointer may be NULL */
int t2fit_device_info(char *name, int name_len, int *sm_count, int *cc_major, int *cc_minor);

/* The fit: replaces pool.map(fit_voxel) (:430-443) and compute_residuals (:461) in one launch.
 * stream: a cudaStream_t (NULL = the legacy default stream, as everywhere in CUDA).  T2FIT_MEM_DEVICE
 * calls only enqueue work on it; T2FIT_MEM_HOST calls ignore it (internal staging streams) and return
 * when the results are in the caller's buffers. */
int t2fit_run(const t2fit_problem *p, t2fit_outputs *o, void *stream);

/* Status histogram of the device-memory t2fit_run calls WITHOUT counts_dev of their own since the previous query
 * (synchronises `stream`, then resets the counters): counts[1..3] = voxels per non-OK status, counts[0] = mask_idx entries
 * that were out of range.  One set of counters per process: a t2fit_run call that finds counts nobody has queried clears
 * them first, so a call's histogram is its own as long as calls and queries alternate on one stream; concurrent streams
 * should pass t2fit_outputs.counts_dev instead. */
int t2fit_status_counts(void *stream, int64_t counts[4]);

/* mask = np.sum(mask4, axis=3) > 0 (:383-384) and mask_indices = np.where(mask.flat) (:412,421):
 * masks is [n_vox, n_masks] uint8 (n_masks = 1 for a plain mask).  Writes ascending indices to
 * idx_out (capacity n_vox) and the count to *n_out (host).  Device pointers; synchronises stream. */
int t2fit_mask_indices(const uint8_t *masks, int64_t n_vox, int32_t n_masks, int64_t *idx_out, int64_t *n_out,
                       void *stream);

/* Mask union straight from the per-TE mask volumes (:383-384) with the optional --in_vitro_fast label masking
 * (mask[label == 0] = 0, :393-400): mask_out[v] = (sum_p planes[p][v] > 0) && (label == NULL || label[v] != 0).
 * planes: HOST array of n_planes DEVICE pointers to [n_vox] arrays of element type `dtype`; label: DEVICE pointer
 * of type `label_dtype` or NULL.  dtype codes: T2FIT_DT_*.  mask_out: device uint8 [n_vox] (0/1). */
#define T2FIT_DT_U8 0
#define T2FIT_DT_I16 1
#define T2FIT_DT_U16 2
#define T2FIT_DT_I32 3
#define T2FIT_DT_F32 4
#define T2FIT_DT_F64 5
int t2fit_mask_union(const void *const *planes, int32_t n_planes, int32_t dtype, const void *label, int32_t label_dtype,
                     int64_t n_vox, uint8_t *mask_out, void *stream);

/* Host-side variant for sparse masks (pure host code on the library's worker threads; no GPU, no t2fit_init needed): the
 * same union + label masking from HOST mask volumes, plus np.where(mask.flatten())[0] (:421) in one call:
 * mask_out[v] as above (host uint8 [n_vox]), idx_out[0 .. *n_out) = ascending flat indices of the union (host int64,
 * room for n_vox entries). */
int t2fit_host_mask_union_indices(const void *const *masks, int32_t n_masks, int32_t mask_dtype, const void *label,
                                  int32_t label_dtype, int64_t n_vox, uint8_t *mask_out, int64_t *idx_out, int64_t *n_out);

/* ... and the gather of the masked voxels of every per-TE HOST volume with the float32 cast of :411-412, packed
 * echo-major: soa_out[p * ld + i] = (float)planes[p][idx[i]] (T2FIT_LAYOUT_SOA with this ld; ld >= n_fit).  planes: n_planes
 * host pointers to [n_vox] arrays of element type `dtype` (T2FIT_DT_*).  EINVAL if an index lies outside [0, n_vox). */
int t2fit_host_gather_planes(const void *const *planes, int32_t n_planes, int32_t dtype, const int64_t *idx, int64_t n_fit,
                             int64_t n_vox, float *soa_out, int64_t ld);

/* Phantom ROI statistics (save_phantom_csv, utils/t2map_utils.py:30-59): for every label value 1..n_roi the
 * NaN-skipping mean and population standard deviation (np.nanmean / np.nanstd) of each of n_maps float32 maps
 * over the voxels with label == value.  maps: HOST array of n_maps DEVICE pointers to [n_vox] float32; label:
 * DEVICE int32 [n_vox].  Outputs are HOST arrays [n_maps, n_roi] (mean, std: float64; count: int64 non-NaN voxels);
 * an empty ROI gives NaN as numpy does.  Synchronises `stream`. */
int t2fit_roi_stats(const float *const *maps, int32_t n_maps, const int32_t *label, int64_t n_vox, int32_t n_roi,
                    double *mean_out, double *std_out, int64_t *count_out, void *stream);

/* Fused final gather (SURVEY.md 8(e)): instead of fitting into local vectors and then running a collective, every rank's
 * fit kernel stores its slab of results STRAIGHT INTO THE ROOT GPU'S BUFFER over NVLink (peer stores from the kernel
 * epilogue; no collective launch, the transfer overlaps the fit).  The root allocates the full-length buffer with
 * t2fit_shared_alloc and publishes the 64-byte handle (any transport: torch.distributed, MPI, a file); the other
 * processes map it with t2fit_shared_open and pass `mapped + slab offset` as the t2fit_outputs pointers of an ordinary
 * T2FIT_MEM_DEVICE t2fit_run; a barrier after the ranks have synchronised their streams completes the gather. */
#define T2FIT_IPC_HANDLE_BYTES 64
int t2fit_shared_alloc(int64_t bytes, void **dev_ptr, unsigned char handle[T2FIT_IPC_HANDLE_BYTES]);
int t2fit_shared_free(void *dev_ptr);
int t2fit_shared_open(const unsigned char handle[T2FIT_IPC_HANDLE_BYTES], void **dev_ptr); /* in ANOTHER process */
int t2fit_shared_close(void *dev_ptr);

/* pack_masked_soa: gather rows mask_idx[i] of the AOS array into the echo-contiguous SOA buffer
 * soa[e*ld + i] (device pointers).  The host-memory path of t2fit_run does this on the CPU side
 * while staging; this is the device-resident variant. */
int t2fit_pack_soa(const float *aos, int64_t n_vox, int32_t n_echo, const int64_t *mask_idx, int64_t n_fit, float *soa,
                   int64_t ld, void *stream);

/* scatter_maps: dense[mask_idx[i]] = compact[i] for n_maps float maps (run_t2mapping.py:455-458).
 * Device pointers. */
int t2fit_scatter(const float *const *compact, float *const *dense, int32_t n_maps, const int64_t *mask_idx,
                  int64_t n_fit, void *stream);

/* compute_residuals (utils/t2map_utils.py:62-89) as a stand-alone pass for callers that keep the
 * reference's two-step structure: res_map[row] = sum_e (y_e - model_e(k_map, t2_map, sigma_map)) / E on
 * the masked rows.  Uses echoes/mask_idx/n_fit/n_echo/te_ms/model/norm of *p (device pointers, AOS);
 * maps are dense [n_vox] device arrays.  t2fit_run already returns the same residuals. */
int t2fit_residuals(const t2fit_problem *p, const float *k_map, const float *t2_map, const float *sigma_map,
                    float *res_map, void *stream);

/* Per-voxel standard errors of the fitted parameters (DESIGN.md section 11), at the parameters given: the unconstrained local
 * linearisation of the fit's objective, bounds ignored, FP64 per voxel (csrc/t2fit_stderr.cuh).
 *   gaussian, gaussian_rician: Cov = s^2 (J'J)^-1, J[e][j] = d model_e / d theta_j, s^2 = sum_e r_e^2 / (E - P)
 *                              (scipy.optimize.curve_fit's pcov with absolute_sigma=False)
 *   rician:                    Cov = H^-1, H the analytic Hessian of the summed negative log-likelihood (rician_obj :157-177)
 * theta = (k, T2[, sigma]) in the units of the maps; se_j = sqrt(Cov_jj) from a Cholesky factorisation of D A D,
 * D = diag(A_jj^-1/2).  The echoes are those of the fit: float32, scaled by y / max(y) in float32 when p->norm.
 * NaN rule: all standard errors of a voxel are NaN when an echo is not finite (rician: or <= 0), a parameter is not finite
 * or T2 <= 0, n_echo <= P, a diagonal entry of A is <= 0, or a Cholesky pivot is <= 0 or not finite; otherwise they are
 * finite (huge for a near-singular voxel: reported, not clipped).
 * Reads echoes / layout / memory / mask_idx / idx_dtype / n_vox / n_fit / n_echo / te_ms / model / norm of *p, as
 * t2fit_residuals; T2FIT_LAYOUT_AOS and T2FIT_MEM_DEVICE only.  k, t2 (and sigma for the 3-parameter models) are device
 * float32 parameters: dense == 0 compact [n_fit] (element i = voxel mask_idx[i]), dense != 0 [n_vox] maps indexed by row.
 * se_k / se_t2 / se_sigma are written the same way; any may be NULL (skipped); se_sigma is not written for gaussian.  A
 * mask_idx entry outside [0, n_vox) reads nothing and gives NaN in a compact output (a dense one is left untouched).
 * Asynchronous on `stream`.  EINVAL: bad layout / memory kind, NULL pointers, n_echo outside 2..T2FIT_MAX_ECHO;
 * ENOTINIT before t2fit_init.  n_fit == 0 is a no-op. */
int t2fit_stderr(const t2fit_problem *p, const float *k, const float *t2, const float *sigma, int32_t dense, float *se_k,
                 float *se_t2, float *se_sigma, void *stream);

/* Per-voxel profile-likelihood confidence interval for T2 (DESIGN.md section 12), FP64 per voxel (csrc/t2fit_interval.cuh).
 * For one voxel, with the fit's objective f (gaussian, gaussian_rician: the mean squared error; rician: the summed negative
 * log-likelihood of rician_obj :157-177) on the fit's echoes (float32, scaled by y / max(y) in float32 when p->norm) and
 * the fit's box (lb / ub, or under p->no_prior k in [y(TE_0), no_prior_k_ub] and T2 in [no_prior_t2_lb, no_prior_t2_ub],
 * sigma keeping lb[2] / ub[2]):
 *   p(T2) = min over (k[, sigma]) in the box of f;  p* = min over T2 in the box of p, reached at t2_best;
 *   the set {T2 : p(T2) <= thr}, thr = p* (1 + q / (E - P)) for the least-squares fits (q = t^2_{E-P}(1 - alpha/2), the
 *   profile-t interval), thr = p* + q / 2 for rician (q = chi^2_1(1 - alpha), the likelihood ratio);
 *   t2_lo / t2_hi = the smallest / largest member of the set (its hull when it is not connected).
 * flags: bit 0 t2_lo is the lower T2 bound; bit 1 t2_hi is the upper T2 bound (upper end not determined); bit 2 a grid
 * point strictly between t2_lo and t2_hi lies outside the set; bit 3 invalid: t2_lo / t2_hi / t2_best NaN, when an echo is
 * not finite (rician: or <= 0), n_echo <= P, the box is empty (--no_prior with y(TE_0) > no_prior_k_ub: the fit's status
 * 3) or p* is not finite.  A least-squares voxel with p* == 0 is valid; its set is where p == 0.
 * Procedure: p on n_grid (16..256) points T2_g = lb (ub/lb)^(g/(n_grid-1)); golden-section refinement of p* / t2_best
 * (relative T2 tolerance 1e-7 or better); bisection of the crossings that bound the hull (1e-6 or better).
 * Reads echoes / layout / memory / mask_idx / idx_dtype / n_vox / n_fit / n_echo / te_ms / model / norm / lb / ub / no_prior*
 * of *p; T2FIT_LAYOUT_AOS and T2FIT_MEM_DEVICE only.  dense == 0: t2_lo / t2_hi / t2_best / flags compact [n_fit] (element
 * i = voxel mask_idx[i]); dense != 0: [n_vox] indexed by row.  profile (optional): [n_fit, n_grid] float64 p(T2_g), compact
 * in either case (NaN for an invalid voxel).  Any output may be NULL (skipped).  A mask_idx entry outside [0, n_vox) reads
 * nothing: NaN and flag 8 in a compact output (a dense one is left untouched).  Asynchronous on `stream`.
 * EINVAL: bad layout / memory kind, NULL echoes / te_ms, n_echo outside 2..T2FIT_MAX_ECHO, n_grid outside 16..256, q not
 * finite or < 0, T2 bounds not finite with 0 < lb < ub, a sigma lower bound <= 0 (3-parameter models); ENOTINIT before
 * t2fit_init.  n_fit == 0 is a no-op. */
int t2fit_t2_interval(const t2fit_problem *p, double q, int32_t n_grid, int32_t dense, float *t2_lo, float *t2_hi,
                      float *t2_best, uint8_t *flags, double *profile, void *stream);

/* Per-voxel parametric bootstrap (DESIGN.md section 13, csrc/t2fit_bootstrap.cuh): simulate n_rep noisy replicates of every
 * voxel from its fitted curve, refit them with t2fit_run (same problem: solver, init, x0 / bounds / options, no_prior, norm),
 * and summarise the refitted parameters.  The two passes below bracket that refit.
 *
 * t2fit_bootstrap_replicates: for voxel i with the float32 parameters k[i], t2[i] (, sigma[i]) and the fit's echoes y (float32,
 * scaled by y / max(y) in float32 when p->norm), rows[(i n_rep + r) n_echo + e] = replicate r, echo e, u_e = exp(-te_e / T2):
 *   gaussian         k u_e + s z_e                          s = noise_sd[i] if given, else sqrt(sum_e r_e^2 / (E - P)) at
 *   gaussian_rician  sqrt((k u_e)^2 + sigma^2) + s z_e        the parameters (FP64, as t2fit_stderr's s)
 *   rician           sqrt((k u_e + sn z_2e)^2 + (sn z_2e+1)^2)   sn = noise_sd[i] if given, else sigma[i]
 * FP64, stored as float32.  A given noise_sd is in the units of the stored echoes (divided by max(y) under norm).  z: standard
 * normals from Philox4x32-10, key (seed lo32, seed hi32), counter (j, r, v lo32, v hi32), v = voxel_id[i] if given, else the
 * row read (mask_idx[i], or i without an index); each word w gives u = (w + 0.5) 2^-32 and block j gives z_4j..z_4j+3 by
 * Box-Muller on (w0, w1), (w2, w3): sqrt(-2 ln u_a) (cos 2 pi u_b, sin 2 pi u_b).  The rows of a voxel are all NaN (every
 * refit gets status 1) when its index is outside [0, n_vox), an echo is not finite (rician: or <= 0), a parameter is not
 * finite or T2 <= 0, the noise level is not finite or < 0, or E <= P with s to estimate.
 * Reads echoes / layout / memory / mask_idx / idx_dtype / n_vox / n_fit / n_echo / te_ms / model / norm of *p; T2FIT_LAYOUT_AOS
 * and T2FIT_MEM_DEVICE only.  k, t2, sigma (3-parameter models), noise_sd, voxel_id: device [n_fit] compact (element i =
 * voxel mask_idx[i]), noise_sd / voxel_id may be NULL.  rows: device [n_fit * n_rep, n_echo].  Asynchronous on `stream`.
 *
 * t2fit_bootstrap_stats: for voxel i, replicate r at element i n_rep + r of rep_k / rep_t2 / rep_sigma / rep_status (the
 * compact outputs of the refit; rep_sigma unused for gaussian): a replicate is used when its status is 0 or 2 and its
 * parameters are finite.  n_used[i] = used replicates, n_ok[i] = replicates with status 0; mean[j n_fit + i] / sd[j n_fit + i]
 * = FP64 mean / standard deviation (ddof 1) of parameter j = (k, T2, sigma) over the used replicates; t2_lo / t2_hi = the T2
 * quantiles at (1 - level) / 2 and (1 + level) / 2 (numpy.quantile's default linear method).  NaN when n_used < 2, and for
 * sigma of gaussian.  Sums run in a fixed order: deterministic.  Any output may be NULL (skipped).  Device pointers,
 * asynchronous on `stream`.
 *
 * EINVAL: n_rep outside 16..4096, level outside (0, 1), NULL inputs, and the checks of t2fit_stderr; ENOTINIT before
 * t2fit_init.  n_fit == 0 is a no-op. */
int t2fit_bootstrap_replicates(const t2fit_problem *p, const float *k, const float *t2, const float *sigma,
                               const float *noise_sd, const int64_t *voxel_id, uint64_t seed, int32_t n_rep, float *rows,
                               void *stream);
int t2fit_bootstrap_stats(int32_t model, int64_t n_fit, int32_t n_rep, const float *rep_k, const float *rep_t2,
                          const float *rep_sigma, const uint8_t *rep_status, double level, float *mean, float *sd,
                          float *t2_lo, float *t2_hi, int32_t *n_used, int32_t *n_ok, void *stream);

/* Algorithmic work of the shipped kernels, for roofline accounting (DESIGN.md): FLOPs and MUFU ops
 * of one pass over the echoes, and the fixed per-voxel part. */
int t2fit_work_model(int32_t model, int32_t n_echo, double *flop_per_pass, double *mufu_per_pass,
                     double *flop_fixed, double *mufu_fixed, double *bytes_per_voxel);

#ifdef __cplusplus
}
#endif
#endif /* T2FIT_H */
