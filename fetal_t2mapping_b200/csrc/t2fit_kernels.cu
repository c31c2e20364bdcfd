// libt2fit: sm_100a kernels + the C ABI of include/t2fit.h.
//
// Kernels (DESIGN.md has the data layout and the roofline of each):
//   fit_kernel<MODEL,E,LAYOUT,FILL>  one thread per masked voxel: gather echoes (AoS rows through
//                                mask_idx, or SoA planes), solve in registers (t2fit_core.cuh),
//                                residual epilogue, write compact or scatter into dense maps.
//                                Replaces pool.map(fit_voxel) + compute_residuals + the scatter
//                                (run_t2mapping.py:430-461).  FILL: the same threads also zero-fill the dense maps.
//   floor_queue_kernel<E,LAYOUT> the 3-parameter fast solver: persistent grid, lanes pull voxels from a queue
//                                (pass counts vary 3..64 between neighbouring voxels).
//   lbfgsb_kernel<OBJ>           the reference's own optimiser (L-BFGS-B + finite differences, FP64, t2fit_lbfgsb.cuh) for
//                                all three objectives; persistent grid, lanes pull voxels from a queue.
//   zero_fill_kernel             np.zeros_like x4 of the dense maps (:415-418) beside the fit, on a side stream (where FILL does not apply)
//   mask_count / mask_scan / mask_write   mask union + ordered compaction (:383-384,:412,:421)
//   mask_union_kernel            union straight from per-TE mask volumes + --in_vitro_fast label masking (:381-400)
//   roi_stats_kernel             per-label nanmean / nanstd of the maps (save_phantom_csv, utils/t2map_utils.py:30-59)
//   pack_soa_kernel              AoS rows -> echo-contiguous SoA (pack_masked_soa)
//   scatter_kernel               compact -> dense maps (:455-458)
//   residual_kernel              compute_residuals as a stand-alone pass (utils/t2map_utils.py:62-89)
// Host side: per-process context (one GPU per process); host-memory calls either stage chunks through pinned buffers with
// worker threads (gather the next chunk while the previous ones are in flight) or, when the caller's arrays are
// page-locked, let the kernels read / write them in place; CUDA-IPC buffers for the fused multi-GPU gather.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <chrono>
#include <atomic>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <string>
#include <thread>
#include <type_traits>
#include <vector>

#include "t2fit_consts.h"
#include "t2fit_lbfgsb_coop.cuh"
#include "t2fit_lbfgsb_dense.cuh"
#include "t2fit_stderr.cuh"
#include "t2fit_interval.cuh"
#include "t2fit_bootstrap.cuh"
#include "t2fit_workers.h"

using namespace t2fit;

namespace {

constexpr int kBlock = 256;

struct KernelIO {
    const float* echoes;
    const int64_t* idx;   // may be null
    const int32_t* idx32; // the same vector as int32 (t2fit_problem::idx_dtype = T2FIT_IDX_I32); at most one of the two is set
    int64_t ld;
    int64_t n_fit;
    float* t2;
    float* k;
    float* sigma;
    float* res;
    float* fun;
    int32_t* nit;
    uint8_t* status;
    unsigned long long* counts;  // [4] per-status voxel counts of this launch (OK slot unused)
    int dense;                   // outputs indexed by idx[i] instead of i (status/nit/fun stay compact)
    int vec_ok;                  // AoS base pointer is 16-byte aligned
    int layout;                  // T2FIT_LAYOUT_* (run-time for the L-BFGS-B kernel)
    float* trace_f;              // L-BFGS-B solver only: callback trace, row i at i * trace_cap
    float* trace_step;
    int32_t* trace_len;
    int trace_cap;
    // fused zero-fill (fit_kernel<..., FILL = true>): every fit thread also zeroes a few 4-voxel words of the dense maps
    const uint8_t* fill_mask;    // dense [n_vox] mask, 4-byte aligned
    int64_t fill_words;          // n_vox / 4 full words; the ragged tail is left to thread 0
    int64_t fill_nvox;
    int fill_wpb;                // mask words per block (host: ceil(fill_words / blocks), rounded up to whole 128-byte lines of the maps)
    // fused all-gather: compact results are also stored to these peer-GPU destinations (t2fit_outputs::dup_*)
    struct Dup { int n; float* t2[T2FIT_MAX_DUP]; float* k[T2FIT_MAX_DUP]; float* sigma[T2FIT_MAX_DUP]; float* res[T2FIT_MAX_DUP]; uint8_t* status[T2FIT_MAX_DUP]; } dup;
    // > 0: idx comes unchecked from the caller's host memory -- entries outside [0, n_rows) are counted in counts[0] and
    // read row 0 instead (the host raises IndexError afterwards, as the reference's fancy indexing would)
    int64_t n_rows;
    // fit_kernel, device-resident inputs: > 0 = this block also pulls the index entries, echo rows and fill-mask words of the
    // block `ahead` blocks further on into L2, so that block's two dependent DRAM round trips (index -> row) become L2 hits
    int ahead;
};

__device__ __forceinline__ int64_t guarded_row(const KernelIO& io, int64_t row) {
    if (io.n_rows > 0 && (unsigned long long)row >= (unsigned long long)io.n_rows) {
        atomicAdd(io.counts, 1ull);
        row = 0;
    }
    return row;
}
// the fused all-gather: element i of this launch to the same slot of every peer buffer (NVLink peer stores)
__device__ __forceinline__ void store_dups(const KernelIO& io, int64_t i, float t2, float k, float sigma, float res, int status) {
    for (int j = 0; j < io.dup.n; ++j) {
        if (io.dup.t2[j]) io.dup.t2[j][i] = t2;
        if (io.dup.k[j]) io.dup.k[j][i] = k;
        if (io.dup.sigma[j]) io.dup.sigma[j][i] = sigma;
        if (io.dup.res[j]) io.dup.res[j][i] = res;
        if (io.dup.status[j]) io.dup.status[j][i] = (uint8_t)status;
    }
}
__device__ __forceinline__ bool has_idx(const KernelIO& io) { return io.idx != nullptr || io.idx32 != nullptr; }
// mask_indices[i] (int64 or int32 vector), unchecked
__device__ __forceinline__ int64_t raw_row(const KernelIO& io, int64_t i) {
    return io.idx ? __ldg(io.idx + i) : (int64_t)__ldg(io.idx32 + i);
}

// ------------------------------------------------------------------------------------------------
// echo loads
// ------------------------------------------------------------------------------------------------
template <int E>
__device__ __forceinline__ void load_aos(const float* __restrict__ base, int64_t row, bool vec_ok, float (&y)[E]) {
    const float* p = base + row * E;
    if constexpr (E % 4 == 0) {
        if (vec_ok) {
            const float4* p4 = reinterpret_cast<const float4*>(p);
#pragma unroll
            for (int q = 0; q < E / 4; ++q) {
                const float4 v = __ldg(p4 + q);
                y[4 * q] = v.x; y[4 * q + 1] = v.y; y[4 * q + 2] = v.z; y[4 * q + 3] = v.w;
            }
            return;
        }
    } else if constexpr (E % 2 == 0) {
        if (vec_ok) {
            const float2* p2 = reinterpret_cast<const float2*>(p);
#pragma unroll
            for (int q = 0; q < E / 2; ++q) {
                const float2 v = __ldg(p2 + q);
                y[2 * q] = v.x; y[2 * q + 1] = v.y;
            }
            return;
        }
    }
#pragma unroll
    for (int e = 0; e < E; ++e) y[e] = __ldg(p + e);
}

template <int E>
__device__ __forceinline__ void load_soa(const float* __restrict__ base, int64_t ld, int64_t i, float (&y)[E]) {
#pragma unroll
    for (int e = 0; e < E; ++e) y[e] = __ldg(base + (int64_t)e * ld + i);
}

// ------------------------------------------------------------------------------------------------
// the fit kernel
// ------------------------------------------------------------------------------------------------
constexpr int kQueueRefill = 8;      // floor_queue_kernel: waiting lanes per warp that trigger epilogue + refill
constexpr int kFusedFillMaxWpt = 16; // fused fill only while a fit thread gets at most this many mask words
constexpr int kFillChunk = 512;    // dense voxels zero-filled by one warp per round (32 lanes x 4 words x 4 voxels)

// ------------------------------------------------------------------------------------------------
// zero_fill_kernel: np.zeros_like x4 (run_t2mapping.py:415-418) restricted to the slots the fit will
// NOT write.  Runs on a side stream concurrently with fit_kernel (no ordering needed: the two kernels
// write disjoint slots), so the HBM-bound fill hides under the compute-bound fit.
// Persistent grid (a couple of blocks per SM); per round a warp covers 512 consecutive voxels: lane l
// loads mask word (j*32+l), j = 0..3 (4 voxels each) and, where none of the 4 is masked, issues one
// coalesced 16-byte store per map (512 B per warp instruction).  Words with both masked and unmasked
// voxels (mask boundary), unaligned maps and the ragged tail take a per-voxel path.
// SIGMA_ALL: the 2-parameter model never writes sigma, so that map is zeroed everywhere.
// ------------------------------------------------------------------------------------------------
struct FillArgs {
    float* t2; float* k; float* res; float* sigma;   // any may be null
    const uint8_t* mask;                            // [n_vox], nonzero = masked
    int64_t n_vox;
    int vec;                                        // every non-null map is 16-byte aligned
};

template <bool SIGMA_ALL>
__device__ __forceinline__ void fill_voxel(const FillArgs& a, int64_t v, bool unmasked) {
    if (unmasked) {
        if (a.t2) a.t2[v] = 0.f;
        if (a.k) a.k[v] = 0.f;
        if (a.res) a.res[v] = 0.f;
    }
    if (a.sigma && (unmasked || SIGMA_ALL)) a.sigma[v] = 0.f;
}

template <bool SIGMA_ALL>
__global__ void __launch_bounds__(256) zero_fill_kernel(const __grid_constant__ FillArgs a) {
    const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
    const int lane = threadIdx.x & 31;
    const int64_t gw = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int64_t full_chunks = a.n_vox / kFillChunk;
    const bool fast = a.vec && a.t2 && a.k && a.res && a.sigma;
    if (fast) {
#pragma unroll 1
        for (int64_t c = gw; c < full_chunks; c += nw) {
            const int64_t off = c * kFillChunk + lane * 4;
            const uint32_t* pm = reinterpret_cast<const uint32_t*>(a.mask + c * kFillChunk) + lane;
            uint32_t w[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) w[j] = __ldg(pm + j * 32);
            float* q0 = a.t2 + off;
            float* q1 = a.k + off;
            float* q2 = a.res + off;
            float* q3 = a.sigma + off;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const uint32_t wj = w[j];
                if (SIGMA_ALL || wj == 0u) *reinterpret_cast<float4*>(q3 + j * 128) = z4;
                if (wj == 0u) {
                    *reinterpret_cast<float4*>(q0 + j * 128) = z4;
                    *reinterpret_cast<float4*>(q1 + j * 128) = z4;
                    *reinterpret_cast<float4*>(q2 + j * 128) = z4;
                } else if (wj != 0x01010101u) {             // mask boundary inside the word: predicated scalar stores
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        if (((wj >> (8 * q)) & 0xffu) == 0u) {
                            q0[j * 128 + q] = 0.f; q1[j * 128 + q] = 0.f; q2[j * 128 + q] = 0.f;
                            if (!SIGMA_ALL) q3[j * 128 + q] = 0.f;
                        }
                    }
                }
            }
        }
    }
    // per-voxel path: everything if not `fast`, else only the ragged tail after the last full chunk
    const int64_t v0 = fast ? full_chunks * kFillChunk : 0;
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, nt = (int64_t)gridDim.x * blockDim.x;
#pragma unroll 1
    for (int64_t v = v0 + t; v < a.n_vox; v += nt) fill_voxel<SIGMA_ALL>(a, v, a.mask[v] == 0);
}

// resident blocks per SM the register allocator is asked to allow (256 threads each)
// (mono2, E <= 6: 6 blocks = 40 registers with 8 bytes spilled and 8 blocks = 32 registers with 56 bytes spilled were measured on the
// c2 step: 69.8 / 79.4 us against 69.8 us -- the step does not respond to occupancy)
constexpr int min_blocks(int model, int e) {
    return model == kMono2 ? (e <= 6 ? 5 : e <= 12 ? 4 : e <= 16 ? 3 : 2) : (e <= 8 ? 4 : e <= 16 ? 3 : 2);
}

// Fused zero-fill (FILL): the np.zeros_like x4 of the dense maps (run_t2mapping.py:415-418) is spread over the fit
// blocks themselves.  Block b owns ONE contiguous window of fill_wpb 4-voxel mask words, each of its warps a 128-word
// chunk of it: the mask words are loaded beside the thread's own index load; a chunk without a masked voxel goes out as one
// bulk shared -> global copy per map (fill_chunk_bulk), a chunk that meets the mask as 16-byte / 4-byte stores to the unmasked
// slots only (fill_word; the fit writes the masked ones, so no slot is written twice).  Every resident block carries both
// kinds of work, so the HBM-bound fill rides in the memory stalls of the fit without a second kernel holding SM slots (the
// side-stream zero_fill_kernel remains for callers this path does not cover).
template <int MODEL, bool SIGMA = true>
__device__ __forceinline__ void fill_word(const KernelIO& io, int64_t w, uint32_t m) {
    const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
    const int64_t v = w * 4;
    if (SIGMA && (MODEL == kMono2 || m == 0u)) *reinterpret_cast<float4*>(io.sigma + v) = z4;   // the 2-parameter fit never writes sigma
    if (m == 0u) {
        *reinterpret_cast<float4*>(io.t2 + v) = z4;
        *reinterpret_cast<float4*>(io.k + v) = z4;
        *reinterpret_cast<float4*>(io.res + v) = z4;
    } else if (m != 0x01010101u) {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            if (((m >> (8 * q)) & 0xffu) == 0u) {
                io.t2[v + q] = 0.f; io.k[v + q] = 0.f; io.res[v + q] = 0.f;
                if (SIGMA && MODEL != kMono2) io.sigma[v + q] = 0.f;
            }
        }
    }
}

// Zero runs of the dense maps leave the SM as bulk asynchronous shared -> global copies (cp.async.bulk, the TMA unit) of a zeroed
// shared line buffer: one instruction per map and 2 KB chunk, issued by one lane, instead of 16-byte stores queued in the
// load/store unit in front of the fit's own dependent loads (profiles/r02_notes.md section 8: c2 step 66.5 -> 65.7 us).
constexpr int kBulkWords = 128;                            // mask words (x 16 bytes per map) per warp chunk
__device__ __forceinline__ void bulk_zero(float* dst, const float* zeros_smem, int bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                 :: "l"(dst), "r"((uint32_t)__cvta_generic_to_shared(zeros_smem)), "r"(bytes) : "memory");
}
// One warp, one chunk of up to 128 consecutive mask words starting at window word cw0 (n of them inside the window).
template <int MODEL>
__device__ __forceinline__ void fill_chunk_bulk(const KernelIO& io, const float* zeros, int64_t w0, int cw0, int n, const uint32_t (&mw)[4]) {
    const int lane = (int)threadIdx.x & 31;
    uint32_t any = 0u;
#pragma unroll
    for (int g = 0; g < 4; ++g) any |= (g * 32 + lane < n) ? mw[g] : 0u;
    const bool all_zero = __all_sync(0xffffffffu, any == 0u);
    const int64_t v = (w0 + cw0) * 4;
    if (n > 0) {
        if (MODEL == kMono2 && lane == 3) bulk_zero(io.sigma + v, zeros, n * 16);     // the 2-parameter fit never writes sigma
        if (all_zero) {
            if (lane == 0) bulk_zero(io.t2 + v, zeros, n * 16);
            if (lane == 1) bulk_zero(io.k + v, zeros, n * 16);
            if (lane == 2) bulk_zero(io.res + v, zeros, n * 16);
            if (MODEL != kMono2 && lane == 3) bulk_zero(io.sigma + v, zeros, n * 16);
        } else {
#pragma unroll
            for (int g = 0; g < 4; ++g)
                if (g * 32 + lane < n) {
                    if (MODEL == kMono2) fill_word<MODEL, false>(io, w0 + cw0 + g * 32 + lane, mw[g]);
                    else fill_word<MODEL, true>(io, w0 + cw0 + g * 32 + lane, mw[g]);
                }
        }
    }
}

template <int MODEL, int E, int LAYOUT, bool FILL>
__global__ void __launch_bounds__(kBlock, min_blocks(MODEL, E)) fit_kernel(const __grid_constant__ FitConsts c,
                                                     const __grid_constant__ KernelIO io) {
    constexpr int kGroup = 4;                              // mask words in flight per thread
    __shared__ __align__(128) float zeros[FILL ? kBulkWords * 4 : 4];   // FILL: the line of zeros the bulk copies read
    if (FILL) {
        reinterpret_cast<float2*>(zeros)[threadIdx.x] = make_float2(0.f, 0.f);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncthreads();
    }
    // Programmatic dependent launch (launch_fit sets the attribute): the next fit launch of the stream may become resident while
    // this one drains; it touches no global memory before the wait, which returns once the previous grid has completed and
    // its stores are visible.  Both are no-ops for a launch without the attribute.
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");
    const int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x;
    const bool valid = i < io.n_fit;
    const int64_t ii = valid ? i : io.n_fit - 1;           // whole warps stay in the solver (warp votes)
    const int64_t row = has_idx(io) ? guarded_row(io, raw_row(io, ii)) : ii;
    int64_t row_ahead = -1;                                // the index entry of the thread `ahead` blocks on (an ordinary load)
    if (io.ahead > 0 && LAYOUT == T2FIT_LAYOUT_AOS && has_idx(io)) {
        const int64_t ia = i + (int64_t)io.ahead * kBlock;
        if (ia < io.n_fit) row_ahead = raw_row(io, ia);
    }
    // FILL: block b owns the contiguous window of fill_wpb mask words starting at b * fill_wpb (one window per map and block:
    // few concurrent write streams); warp w of the block owns window words [w * 128, w * 128 + 128) (+ 1024 per further
    // round), 2 KB of every map
    const int64_t w0 = (int64_t)blockIdx.x * io.fill_wpb;
    uint32_t mw[kGroup];
    const int wlim = FILL ? (int)min((int64_t)io.fill_wpb, io.fill_words - w0) : 0;   // words of this block's window (<= 0: none)
    const int cbase = ((int)threadIdx.x >> 5) * kBulkWords;
    if (FILL) {                                            // this warp's mask words: loads in flight beside the index load
        const uint32_t* pm = reinterpret_cast<const uint32_t*>(io.fill_mask);
#pragma unroll
        for (int g = 0; g < kGroup; ++g) {
            const int lw = cbase + g * 32 + ((int)threadIdx.x & 31);
            mw[g] = lw < wlim ? __ldg(pm + w0 + lw) : 0u;
        }
    }
    float y[E];
    if (LAYOUT == T2FIT_LAYOUT_AOS) load_aos<E>(io.echoes, row, io.vec_ok != 0, y);
    else if (LAYOUT == T2FIT_LAYOUT_SOA) load_soa<E>(io.echoes, io.ld, ii, y);
    else load_soa<E>(io.echoes, io.ld, row, y);            // PLANES: per-TE volumes, voxel `row` of every plane
    if (FILL) {                                            // zero stores go out while the echoes are on their way
        fill_chunk_bulk<MODEL>(io, zeros, w0, cbase, max(0, min(kBulkWords, wlim - cbase)), mw);
#pragma unroll 1
        for (int r0 = (kBlock / 32) * kBulkWords; r0 < wlim; r0 += (kBlock / 32) * kBulkWords) {   // sparse masks: further rounds
            const uint32_t* pm = reinterpret_cast<const uint32_t*>(io.fill_mask);
#pragma unroll
            for (int g = 0; g < kGroup; ++g) {
                const int lw = r0 + cbase + g * 32 + ((int)threadIdx.x & 31);
                mw[g] = lw < wlim ? __ldg(pm + w0 + lw) : 0u;
            }
            fill_chunk_bulk<MODEL>(io, zeros, w0, r0 + cbase, max(0, min(kBulkWords, wlim - r0 - cbase)), mw);
        }
        if (io.ahead > 0 && threadIdx.x < 32) {            // mask words of the window `ahead` blocks on: one 128-byte line per lane
            const int64_t wa = w0 + (int64_t)io.ahead * io.fill_wpb + (int64_t)threadIdx.x * 32;
            if (threadIdx.x * 32 < io.fill_wpb && wa < io.fill_words)
                asm volatile("prefetch.global.L2 [%0];" :: "l"(reinterpret_cast<const uint32_t*>(io.fill_mask) + wa));
        }
        if (i == 0) {                                               // ragged tail of the volume (n_vox % 4 voxels)
            for (int64_t v = io.fill_words * 4; v < io.fill_nvox; ++v) {
                const bool unmasked = io.fill_mask[v] == 0;
                if (unmasked) { io.t2[v] = 0.f; io.k[v] = 0.f; io.res[v] = 0.f; }
                if (unmasked || MODEL == kMono2) io.sigma[v] = 0.f;
            }
        }
    }

    if (row_ahead >= 0 && (io.n_rows <= 0 || row_ahead < io.n_rows))       // its echo row (20 bytes for E = 5: lanes share lines)
        asm volatile("prefetch.global.L2 [%0];" :: "l"(io.echoes + row_ahead * E));

    const VoxelFit f = fit_voxel<float, MODEL, E>(y, c, valid);

    if (valid) {
        const int64_t o = io.dense ? row : i;
        if (io.t2) io.t2[o] = f.t2;
        if (io.k) io.k[o] = f.k;
        if (MODEL != kMono2 && io.sigma) io.sigma[o] = f.sigma;
        if (io.res) io.res[o] = f.res;
        if (io.fun) io.fun[i] = f.fun;
        if (io.nit) io.nit[i] = f.nit;
        if (io.status) io.status[i] = (uint8_t)f.status;
        if (io.dup.n) store_dups(io, i, f.t2, f.k, f.sigma, f.res, f.status);
    }
    // warp-aggregated status histogram: one atomic per warp per non-OK status (normally none)
    const int st = valid ? f.status : 0;
    const unsigned any_bad = __ballot_sync(0xffffffffu, st != 0);
    if (any_bad && io.counts) {
#pragma unroll
        for (int s = 1; s < 4; ++s) {
            const unsigned m = __ballot_sync(0xffffffffu, st == s);
            if (m && (threadIdx.x & 31) == 0) atomicAdd(io.counts + s, (unsigned long long)__popc(m));
        }
    }
    if (FILL) {                                            // the zero line buffer must outlive the bulk copies that read it
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    }
}

// ------------------------------------------------------------------------------------------------
// floor_queue_kernel: the 3-parameter fast solver as a persistent grid with a lane-level voxel queue.
// The projected LM iteration needs 3..64 passes over the echoes depending on the voxel (noise-floor voxels run to the
// cap), so a warp of the one-shot kernel spends most of its time waiting for its slowest lane (c5: 6.4 passes per voxel
// on average, ~25 per warp).  Here a lane whose run has stopped gets the next voxel from a queue counter
// (warp-aggregated atomicAdd) while its neighbours keep iterating.  Epilogue (residuals, stores) and prologue (echo
// loads, log-linear start point) of the replaced lanes are batched: they run only once `refill` lanes of the warp
// are waiting, so their instructions are shared by that many lanes.  Same per-voxel arithmetic as fit_kernel<kFloor3>
// (voxel_prepare / FloorRun::step / voxel_finish), hence the same results.
// ------------------------------------------------------------------------------------------------
constexpr int kQBlock = 128;
constexpr int queue_min_blocks(int e) { return e <= 8 ? 6 : e <= 16 ? 4 : 2; }

template <int E, int LAYOUT>
__global__ void __launch_bounds__(kQBlock, queue_min_blocks(E)) floor_queue_kernel(const __grid_constant__ FitConsts c,
                                                                                   const __grid_constant__ KernelIO io,
                                                                                   unsigned long long* __restrict__ queue,
                                                                                   const int refill) {
    constexpr unsigned kFull = 0xffffffffu;
    const unsigned lane = threadIdx.x & 31;
    FloorRun<float> run;
    run.active = false;
    VoxelPre<float> pre{};
    float y[E];
    int64_t i = 0, row = 0;
    bool have = false;                       // this lane holds a voxel whose result has not been stored yet
    bool more = true;                        // the queue still has voxels (warp-uniform)
    unsigned cnt1 = 0, cnt2 = 0, cnt3 = 0;   // non-OK voxels of this lane, by status
    for (;;) {
        const unsigned m_done = __ballot_sync(kFull, have && !run.active);
        const unsigned m_empty = __ballot_sync(kFull, !have);
        const bool any_active = __any_sync(kFull, run.active);
        const int waiting = __popc(m_done) + __popc(m_empty);
        const bool turn = !any_active || ((waiting >= refill || !more) && (m_done != 0u || (more && m_empty != 0u)));
        if (turn) {
            if (have && !run.active) {       // epilogue of the lanes that have stopped
                const VoxelFit f = voxel_finish<float, kFloor3, E>(y, c, pre, run.x[0], run.x[1], run.sigma(c), run.nit, run.status);
                const int64_t o = io.dense ? row : i;
                if (io.t2) io.t2[o] = f.t2;
                if (io.k) io.k[o] = f.k;
                if (io.sigma) io.sigma[o] = f.sigma;
                if (io.res) io.res[o] = f.res;
                if (io.fun) io.fun[i] = f.fun;
                if (io.nit) io.nit[i] = f.nit;
                if (io.status) io.status[i] = (uint8_t)f.status;
                if (io.dup.n) store_dups(io, i, f.t2, f.k, f.sigma, f.res, f.status);
                cnt1 += f.status == 1; cnt2 += f.status == 2; cnt3 += f.status == 3;
                have = false;
            }
            if (more) {                      // next voxels for every lane without one
                const unsigned m_need = __ballot_sync(kFull, !have);
                const int n_need = __popc(m_need);
                unsigned long long base = 0;
                if (lane == 0) base = atomicAdd(queue, (unsigned long long)n_need);
                base = __shfl_sync(kFull, base, 0);
                more = (int64_t)(base + (unsigned long long)n_need) < io.n_fit;
                const int64_t cand = (int64_t)base + __popc(m_need & ((1u << lane) - 1u));
                if (!have && cand < io.n_fit) {
                    i = cand;
                    row = has_idx(io) ? guarded_row(io, raw_row(io, i)) : i;
                    if (LAYOUT == T2FIT_LAYOUT_AOS) load_aos<E>(io.echoes, row, io.vec_ok != 0, y);
                    else if (LAYOUT == T2FIT_LAYOUT_SOA) load_soa<E>(io.echoes, io.ld, i, y);
                    else load_soa<E>(io.echoes, io.ld, row, y);
                    pre = voxel_prepare<float, kFloor3, E>(y, c);
                    run.start(c, pre.kl, pre.ku, pre.k0, pre.r0, pre.s0, pre.status == kOk);
                    have = true;
                }
            }
            if (!__any_sync(kFull, have)) break;
        }
        if (__any_sync(kFull, run.active)) run.template step<E>(y, c);
    }
    // per-status voxel counts of the launch: one atomic per warp and status
    if (io.counts) {
        const unsigned t1 = __reduce_add_sync(kFull, cnt1), t2 = __reduce_add_sync(kFull, cnt2), t3 = __reduce_add_sync(kFull, cnt3);
        if (lane == 0) {
            if (t1) atomicAdd(io.counts + 1, (unsigned long long)t1);
            if (t2) atomicAdd(io.counts + 2, (unsigned long long)t2);
            if (t3) atomicAdd(io.counts + 3, (unsigned long long)t3);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// lbfgsb_kernel: the reference-faithful solver (t2fit_lbfgsb.cuh), one voxel per thread, FP64.
// The optimiser state (compact L-BFGS matrices, ~10 KB) lives in per-thread local memory; the kernel
// is bound by FP64 issue and L1/L2 traffic of that state, not by HBM (DESIGN.md).  Epilogue as
// fit_kernel: maps store float32(x) as the reference's scatter does (:455-458), res is evaluated from
// those stored values as compute_residuals does (utils/t2map_utils.py:62-89).
// ------------------------------------------------------------------------------------------------
constexpr int kLbBlock = 128;

template <int OBJ, int YS = 1>           // YS: stride of the signal row y (1 = contiguous; kLbBlock = a column of shared memory)
__device__ __noinline__ void lb_store(const lb::LbConsts& c, const KernelIO& io, const lb::LbVoxel& v, const float* y, int64_t i, int64_t row) {
    const int E = c.n_echo;
    const float kf = (float)v.x[0], t2f = (float)v.x[1], sf = (OBJ == 0) ? 0.f : (float)v.x[2];
    // residual epilogue on the stored float32 values; run.y is the signal as the fit saw it (normalised if norm)
    double acc = 0.0;
    for (int e = 0; e < E; ++e) {
        double pred = (double)kf * exp(-c.te[e] / (double)t2f);
        if (OBJ != 0) pred = sqrt(pred * pred + (double)sf * (double)sf);
        acc += (double)y[e * YS] - (double)(float)pred;
    }
    const int64_t o = io.dense ? row : i;
    if (io.t2) io.t2[o] = t2f;
    if (io.k) io.k[o] = kf;
    if (OBJ != 0 && io.sigma) io.sigma[o] = sf;
    if (io.res) io.res[o] = (float)(acc / (double)E);
    if (io.fun) io.fun[i] = (float)v.fun;
    if (io.nit) io.nit[i] = v.nit;
    if (io.status) io.status[i] = (uint8_t)v.status;
    if (io.trace_len) io.trace_len[i] = v.trace_len;
    if (io.dup.n) store_dups(io, i, t2f, kf, sf, (float)(acc / (double)E), v.status);
    if (v.status != 0 && io.counts) atomicAdd(io.counts + v.status, 1ull);
}

// Persistent grid; every LANE pulls its next voxel from a global queue as soon as its current one has
// terminated (warp-aggregated atomicAdd), so lanes whose optimiser stopped early do not idle until the
// slowest voxel of the warp is done (iteration counts vary 3..40 between neighbouring voxels).
// 8 blocks x 128 threads per SM = at most 64 registers: the kernel waits on its own local-memory state, so resident warps pay
// more than registers do (profiles/r02_notes.md section 7: 5 / 7 / 8 / 10 / 12 blocks per SM measured).
#ifndef T2_LB_MIN_BLOCKS
#define T2_LB_MIN_BLOCKS 8
#endif
template <int OBJ, class Run>
__device__ __forceinline__ void lb_queue_loop(const lb::LbConsts& c, const KernelIO& io, unsigned long long* __restrict__ queue) {
    const unsigned full = 0xffffffffu, lane = threadIdx.x & 31;
    const int E = c.n_echo;
    Run run;
    run.active = false;
    int64_t cur = -1, row = 0;
    bool exhausted = false;
    for (;;) {
        const bool need = !run.active && !exhausted;
        const unsigned m = __ballot_sync(full, need);
        if (m) {
            const int leader = __ffs(m) - 1;
            unsigned long long base = 0;
            if ((int)lane == leader) base = atomicAdd(queue, (unsigned long long)__popc(m));
            base = __shfl_sync(full, base, leader);
            if (need) {
                const int64_t i = (int64_t)base + __popc(m & ((1u << lane) - 1u));
                if (i < io.n_fit) {
                    cur = i;
                    row = has_idx(io) ? guarded_row(io, raw_row(io, i)) : i;
                    float yraw[kMaxEcho];
                    if (io.layout == T2FIT_LAYOUT_AOS) { for (int e = 0; e < E; ++e) yraw[e] = __ldg(io.echoes + row * E + e); }
                    else {
                        const int64_t col = io.layout == T2FIT_LAYOUT_SOA ? i : row;
                        for (int e = 0; e < E; ++e) yraw[e] = __ldg(io.echoes + (int64_t)e * io.ld + col);
                    }
                    const bool tr = io.trace_cap > 0;
                    run.start(yraw, c, (tr && io.trace_f) ? io.trace_f + i * io.trace_cap : nullptr,
                              (tr && io.trace_step) ? io.trace_step + i * io.trace_cap : nullptr, tr ? io.trace_cap : 0);
                    if (!run.active) lb_store<OBJ>(c, io, run.finish(), run.y, cur, row);      // non-finite input / bad bounds: no optimiser run
                } else {
                    exhausted = true;
                }
            }
        }
        if (!__any_sync(full, run.active)) {
            if (__all_sync(full, exhausted)) break;
            continue;
        }
        if (run.active) {
            run.pass(c);
            if (!run.active) lb_store<OBJ>(c, io, run.finish(), run.y, cur, row);
        }
    }
}


template <int OBJ>
__global__ void __launch_bounds__(kLbBlock, T2_LB_MIN_BLOCKS) lbfgsb_kernel(const __grid_constant__ lb::LbConsts c,
                                                          const __grid_constant__ KernelIO io,
                                                          unsigned long long* __restrict__ queue) {
    lb_queue_loop<OBJ, lb::VoxelRun<OBJ>>(c, io, queue);
}

// ------------------------------------------------------------------------------------------------
// lbfgsb_dense_kernel: the same optimiser with the limited-memory matrix as a dense n x n matrix (t2fit_lbfgsb_dense.cuh),
// one voxel per thread, FP64, same lane queue.  The state of a voxel is the <= 10 correction pairs (480 B of local memory)
// plus ~50 doubles in registers; the optimiser core is a few hundred flops per iteration, so the run time is the objective
// evaluations: N + 1 values per gradient, walked in ONE loop over the echoes whose N + 1 dependent chains overlap
// (DenseRun::fun_and_grad).  What that loop reads and writes -- the signal row and the 8 running sums of numpy's pairwise
// np.sum per point -- lives in SHARED memory as [slot][thread] columns (4 E + 64 (N + 1) bytes per thread), not in local
// memory: the loop issues no LDL / STL.
// ------------------------------------------------------------------------------------------------
#ifndef T2_LBD_MIN_BLOCKS
#define T2_LBD_MIN_BLOCKS 4
#endif
// T2_LBD_THREADS: threads per block.  T2_LBD_SYNC = 1: the warps of a block meet at a barrier before every pass, so that they
// run the echo loop -- and then the optimiser core -- at the same time and fetch the same instructions (the kernel stalls on
// instruction fetch: 83 KB of code, 32 KB L1.5 instruction cache); A/B in profiles/r02_notes.md section 10.
#ifndef T2_LBD_THREADS
#define T2_LBD_THREADS 128
#endif
#ifndef T2_LBD_SYNC
#define T2_LBD_SYNC 1
#endif
constexpr int kLbdBlock = T2_LBD_THREADS;
constexpr size_t dense_smem_bytes(int n_par, int n_echo) { return (size_t)kLbdBlock * (((size_t)(n_par + 1) * 8 + lb::kLsSlots) * sizeof(double) + (size_t)n_echo * sizeof(float)); }

// Epilogue of the voxels that ended in this pass of the warp (`fin` lanes, usually 2-3 of 32): what lb_store does, with the
// residual (compute_residuals, utils/t2map_utils.py:62-89: E double-precision exp / sqrt per voxel) evaluated BY THE WHOLE
// WARP, one echo per lane, instead of by the 2-3 finished lanes while the others wait: the same operations on the same
// operands, summed in echo order, so `res` is bit for bit lb_store's.  ys = the block's signal rows in shared memory.
template <int OBJ>
__device__ __noinline__ void dense_finish(const lb::LbConsts& c, const KernelIO& io, const lb::LbVoxel& v, bool fin, unsigned fm,
                                          const float* ys, int64_t i, int64_t row) {
    const unsigned full = 0xffffffffu, lane = threadIdx.x & 31;
    const int E = c.n_echo, warp0 = threadIdx.x & ~31;
    const float kf = (float)v.x[0], t2f = (float)v.x[1], sf = (OBJ == 0) ? 0.f : (float)v.x[2];
    const double te = c.te[lane < (unsigned)E ? lane : 0];
    double res = 0.0;
    for (unsigned mm = fm; mm; mm &= mm - 1) {
        const int src = __ffs(mm) - 1;
        const float kk = __shfl_sync(full, kf, src), tt = __shfl_sync(full, t2f, src), ss = __shfl_sync(full, sf, src);
        double term = 0.0;
        if (lane < (unsigned)E) {
            double pred = (double)kk * exp(-te / (double)tt);
            if (OBJ != 0) pred = sqrt(pred * pred + (double)ss * (double)ss);
            term = (double)ys[lane * kLbdBlock + warp0 + src] - (double)(float)pred;
        }
        double acc = 0.0;
        for (int e = 0; e < E; ++e) acc += __shfl_sync(full, term, e);
        if ((int)lane == src) res = acc;
    }
    if (!fin) return;
    const float resf = (float)(res / (double)E);
    const int64_t o = io.dense ? row : i;
    if (io.t2) io.t2[o] = t2f;
    if (io.k) io.k[o] = kf;
    if (OBJ != 0 && io.sigma) io.sigma[o] = sf;
    if (io.res) io.res[o] = resf;
    if (io.fun) io.fun[i] = (float)v.fun;
    if (io.nit) io.nit[i] = v.nit;
    if (io.status) io.status[i] = (uint8_t)v.status;
    if (io.trace_len) io.trace_len[i] = v.trace_len;
    if (io.dup.n) store_dups(io, i, t2f, kf, sf, resf, v.status);
    if (v.status != 0 && io.counts) atomicAdd(io.counts + v.status, 1ull);
}

// blocks per SM: 4 x 128 threads (128 registers) for the 3-parameter objectives; the 2-parameter fit measured + 15 % at 3 (168
// registers, no spills: its echo loop is short, the spilled state weighs more) -- profiles/r02_notes.md section 10
constexpr int dense_min_blocks(int obj) { return (obj == 0 && T2_LBD_MIN_BLOCKS == 4 && T2_LBD_THREADS == 128) ? 3 : T2_LBD_MIN_BLOCKS; }

template <int OBJ>
__global__ void __launch_bounds__(kLbdBlock, dense_min_blocks(OBJ)) lbfgsb_dense_kernel(const __grid_constant__ lb::LbConsts c,
                                                                const __grid_constant__ KernelIO io,
                                                                unsigned long long* __restrict__ queue) {
    extern __shared__ __align__(16) unsigned char dense_smem[];
    constexpr int N = OBJ == 0 ? 2 : 3;
    using Run = lb::DenseRun<OBJ, lb::DenseStridedMem<kLbdBlock>>;
    const unsigned full = 0xffffffffu, lane = threadIdx.x & 31;
    const int E = c.n_echo;
    double* const lsb = reinterpret_cast<double*>(dense_smem) + (size_t)(N + 1) * 8 * kLbdBlock;                  // [kLsSlots][kLbdBlock]
    float* const ys = reinterpret_cast<float*>(lsb + (size_t)lb::kLsSlots * kLbdBlock);                          // [E][kLbdBlock]
    double pairs[lb::DenseSolver<N>::kPairDoubles];           // the correction pairs: the one dynamically indexed array, an object of its own
    Run run;
    run.m.acc_ = reinterpret_cast<double*>(dense_smem) + threadIdx.x;                                   // [(N + 1) * 8][kLbdBlock]
    run.m.y_ = ys + threadIdx.x;
    run.m.pairs_ = pairs;
    run.m.ls_ = lsb + threadIdx.x;
    run.active = false;
    int64_t cur = -1, row = 0;
    bool exhausted = false, warp_done = false;
    for (;;) {
        bool fin = false;                                     // this lane's voxel ended in this round of the loop
        const bool need = !run.active && !exhausted;
        const unsigned m = __ballot_sync(full, need);
        if (m) {
            const int leader = __ffs(m) - 1;
            unsigned long long base = 0;
            if ((int)lane == leader) base = atomicAdd(queue, (unsigned long long)__popc(m));
            base = __shfl_sync(full, base, leader);
            if (need) {
                const int64_t i = (int64_t)base + __popc(m & ((1u << lane) - 1u));
                if (i < io.n_fit) {
                    cur = i;
                    row = has_idx(io) ? guarded_row(io, raw_row(io, i)) : i;
                    if (io.layout == T2FIT_LAYOUT_AOS) { for (int e = 0; e < E; ++e) run.m.y(e) = __ldg(io.echoes + row * E + e); }
                    else {
                        const int64_t col = io.layout == T2FIT_LAYOUT_SOA ? i : row;
                        for (int e = 0; e < E; ++e) run.m.y(e) = __ldg(io.echoes + (int64_t)e * io.ld + col);
                    }
                    const bool tr = io.trace_cap > 0;
                    run.start(c, (tr && io.trace_f) ? io.trace_f + i * io.trace_cap : nullptr,
                              (tr && io.trace_step) ? io.trace_step + i * io.trace_cap : nullptr, tr ? io.trace_cap : 0);
                    fin = !run.active;                        // non-finite input / bad bounds: no optimiser run
                } else {
                    exhausted = true;
                }
            }
        }
        const bool any_active = __any_sync(full, run.active);
#if T2_LBD_SYNC
        if (!__syncthreads_or(!warp_done)) break;             // every warp of the block has run dry
#endif
        if (run.active) {
            run.pass(c);
            fin = !run.active;
        }
        __syncwarp(full);
        const unsigned fm = __ballot_sync(full, fin);
        if (fm) {
            lb::LbVoxel v;
            if (fin) v = run.finish();
            dense_finish<OBJ>(c, io, v, fin, fm, ys, cur, row);
        }
        if (!any_active && __all_sync(full, exhausted)) warp_done = true;
#if !T2_LBD_SYNC
        if (warp_done) break;
#endif
    }
}

// ------------------------------------------------------------------------------------------------
// lbfgsb_coop_kernel: the same reference-faithful solver with ONE VOXEL PER GROUP OF G LANES and the optimiser state in
// SHARED MEMORY (t2fit_lbfgsb_coop.cuh).  Persistent blocks, one per SM, as many groups as fit into the 227 KB of shared
// memory (~7.6 KB per voxel); every group pulls its next voxel from the global queue as soon as its current one has
// terminated.  The groups of a warp run the same code: where they are in the same phase they share its instructions,
// where they are not (different iteration counts, different numbers of correction pairs) the warp pays the longest of
// them, not the sum.  No block-level barrier anywhere: groups only ever synchronise among their own lanes.
// ------------------------------------------------------------------------------------------------
template <int OBJ, int G>
__global__ void __launch_bounds__(G == 8 ? 256 : G == 16 ? 512 : 1024, 1) lbfgsb_coop_kernel(const __grid_constant__ lb::LbConsts c,
                                                            const __grid_constant__ KernelIO io,
                                                            unsigned long long* __restrict__ queue, const int stride_bytes) {
    extern __shared__ __align__(16) unsigned char coop_smem[];
    using Run = lb::CoopRun<OBJ, G>;
    const int gi = threadIdx.x / G;
    Run* run = reinterpret_cast<Run*>(coop_smem + (size_t)gi * stride_bytes);
    lb::Group<G> grp;
    grp.lane = threadIdx.x % G;
    grp.mask = G == 32 ? 0xffffffffu : (((1u << (G & 31)) - 1u) << (((threadIdx.x & 31) / G) * G));
    const int E = c.n_echo;
    bool have = false, exhausted = false;
    long long cur = -1, row = 0;
    for (;;) {
        if (!have && !exhausted) {
            long long i = 0;
            if (grp.master()) i = (long long)atomicAdd(queue, 1ull);
            i = grp.shfl(i, 0);
            if (i < io.n_fit) {
                cur = i;
                row = has_idx(io) ? raw_row(io, i) : i;
                if (io.n_rows > 0 && (unsigned long long)row >= (unsigned long long)io.n_rows) {      // unchecked host index vector
                    if (grp.master()) atomicAdd(io.counts, 1ull);
                    row = 0;
                }
                for (int e = grp.lane; e < E; e += G) {
                    float v;
                    if (io.layout == T2FIT_LAYOUT_AOS) v = __ldg(io.echoes + row * E + e);
                    else v = __ldg(io.echoes + (int64_t)e * io.ld + (io.layout == T2FIT_LAYOUT_SOA ? i : row));
                    run->yraw[e] = v;
                }
                grp.sync();
                const bool tr = io.trace_cap > 0;
                run->start(grp, c, (tr && io.trace_f) ? io.trace_f + i * io.trace_cap : nullptr,
                           (tr && io.trace_step) ? io.trace_step + i * io.trace_cap : nullptr, tr ? io.trace_cap : 0);
                have = true;
            } else {
                exhausted = true;
            }
        }
        if (!have) break;                                   // queue empty and nothing in flight: this group is done
        if (run->active) run->pass(grp, c);
        if (!run->active) {
            // epilogue as lb_store: float32(x) into the maps, residual from those stored values; the echo terms across the
            // lanes, their sum on the master lane in the serial order
            const float kf = (float)run->s.x[0], t2f = (float)run->s.x[1], sf = (OBJ == 0) ? 0.f : (float)run->s.x[OBJ == 0 ? 0 : 2];
            double* term = run->s.scr.fterm;
            for (int e = grp.lane; e < E; e += G) {
                double pred = (double)kf * exp(-c.te[e] / (double)t2f);
                if (OBJ != 0) pred = sqrt(pred * pred + (double)sf * (double)sf);
                term[e] = (double)run->y[e] - (double)(float)pred;
            }
            grp.sync();
            if (grp.master()) {
                const lb::LbVoxel v = run->finish();
                double acc = 0.0;
                for (int e = 0; e < E; ++e) acc += term[e];
                const int64_t o = io.dense ? row : cur;
                if (io.t2) io.t2[o] = t2f;
                if (io.k) io.k[o] = kf;
                if (OBJ != 0 && io.sigma) io.sigma[o] = sf;
                if (io.res) io.res[o] = (float)(acc / (double)E);
                if (io.fun) io.fun[cur] = (float)v.fun;
                if (io.nit) io.nit[cur] = v.nit;
                if (io.status) io.status[cur] = (uint8_t)v.status;
                if (io.trace_len) io.trace_len[cur] = v.trace_len;
                if (io.dup.n) store_dups(io, cur, t2f, kf, sf, (float)(acc / (double)E), v.status);
                if (v.status != 0 && io.counts) atomicAdd(io.counts + v.status, 1ull);
            }
            grp.sync();
            have = false;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// mask union + ordered compaction: three small passes over the mask bytes
// ------------------------------------------------------------------------------------------------
constexpr int kMaskTile = 2048;  // voxels per block (256 threads x 8)

__device__ __forceinline__ bool mask_any(const uint8_t* __restrict__ masks, int64_t v, int n_masks) {
    const uint8_t* p = masks + v * n_masks;
    int acc = 0;
    for (int m = 0; m < n_masks; ++m) acc |= p[m];      // np.sum(mask4, axis=3) > 0
    return acc != 0;
}

__global__ void __launch_bounds__(256) mask_count_kernel(const uint8_t* __restrict__ masks, int64_t n_vox, int n_masks,
                                                         int* __restrict__ tile_counts) {
    const int64_t base = (int64_t)blockIdx.x * kMaskTile;
    int cnt = 0;
#pragma unroll
    for (int j = 0; j < kMaskTile / 256; ++j) {
        const int64_t v = base + j * 256 + threadIdx.x;
        if (v < n_vox && mask_any(masks, v, n_masks)) ++cnt;
    }
    __shared__ int wsum[8];
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_down_sync(0xffffffffu, cnt, o);
    if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = cnt;
    __syncthreads();
    if (threadIdx.x == 0) {
        int t = 0;
        for (int w = 0; w < 8; ++w) t += wsum[w];
        tile_counts[blockIdx.x] = t;
    }
}

// exclusive scan of the tile counts (one block; tiles <= a few 100k)
__global__ void __launch_bounds__(1024) mask_scan_kernel(const int* __restrict__ tile_counts, int64_t* __restrict__ tile_offsets,
                                                         int n_tiles, int64_t* __restrict__ total) {
    __shared__ int64_t wsum[32];
    __shared__ int64_t carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (int base = 0; base < n_tiles; base += 1024) {
        const int t = base + threadIdx.x;
        const int64_t v = t < n_tiles ? tile_counts[t] : 0;
        int64_t incl = v;
        for (int o = 1; o < 32; o <<= 1) {
            const int64_t n = __shfl_up_sync(0xffffffffu, incl, o);
            if ((threadIdx.x & 31) >= o) incl += n;
        }
        if ((threadIdx.x & 31) == 31) wsum[threadIdx.x >> 5] = incl;
        __syncthreads();
        if (threadIdx.x < 32) {
            int64_t w = wsum[threadIdx.x];
            int64_t wi = w;
            for (int o = 1; o < 32; o <<= 1) {
                const int64_t n = __shfl_up_sync(0xffffffffu, wi, o);
                if (threadIdx.x >= o) wi += n;
            }
            wsum[threadIdx.x] = wi - w;  // exclusive warp offsets
        }
        __syncthreads();
        const int64_t excl = carry + wsum[threadIdx.x >> 5] + incl - v;
        if (t < n_tiles) tile_offsets[t] = excl;
        __syncthreads();
        if (threadIdx.x == 1023) carry = excl + v;
        __syncthreads();
    }
    if (threadIdx.x == 0) *total = carry;
}

__global__ void __launch_bounds__(256) mask_write_kernel(const uint8_t* __restrict__ masks, int64_t n_vox, int n_masks,
                                                         const int64_t* __restrict__ tile_offsets, int64_t* __restrict__ idx_out) {
    const int64_t base = (int64_t)blockIdx.x * kMaskTile;
    __shared__ int wcnt[8];
    __shared__ int running;
    if (threadIdx.x == 0) running = 0;
    __syncthreads();
    const int64_t out0 = tile_offsets[blockIdx.x];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int j = 0; j < kMaskTile / 256; ++j) {          // keeps ascending order: j-major, thread-minor
        const int64_t v = base + j * 256 + threadIdx.x;
        const bool f = v < n_vox && mask_any(masks, v, n_masks);
        const unsigned b = __ballot_sync(0xffffffffu, f);
        if (lane == 0) wcnt[warp] = __popc(b);
        __syncthreads();
        int woff = 0, tot = 0;
        for (int w = 0; w < 8; ++w) { if (w < warp) woff += wcnt[w]; tot += wcnt[w]; }
        const int before = running;
        if (f) idx_out[out0 + before + woff + __popc(b & ((1u << lane) - 1u))] = v;
        __syncthreads();
        if (threadIdx.x == 0) running = before + tot;
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------------
// mask union from per-TE mask volumes + --in_vitro_fast label masking (run_t2mapping.py:383-384,393-400)
// ------------------------------------------------------------------------------------------------
struct UnionArgs {
    const void* planes[kMaxEcho];
    const void* label;
    int n_planes, dtype, label_dtype;
    int64_t n_vox;
};

__device__ __forceinline__ double load_as_double(const void* p, int dtype, int64_t v) {
    switch (dtype) {
        case T2FIT_DT_U8: return (double)static_cast<const uint8_t*>(p)[v];
        case T2FIT_DT_I16: return (double)static_cast<const int16_t*>(p)[v];
        case T2FIT_DT_U16: return (double)static_cast<const uint16_t*>(p)[v];
        case T2FIT_DT_I32: return (double)static_cast<const int32_t*>(p)[v];
        case T2FIT_DT_F32: return (double)static_cast<const float*>(p)[v];
        default: return static_cast<const double*>(p)[v];
    }
}

__global__ void __launch_bounds__(256) mask_union_kernel(const __grid_constant__ UnionArgs a, uint8_t* __restrict__ out) {
    const int64_t nt = (int64_t)gridDim.x * 256;
    for (int64_t v = (int64_t)blockIdx.x * 256 + threadIdx.x; v < a.n_vox; v += nt) {
        double sum = 0.0;
        for (int p = 0; p < a.n_planes; ++p) sum += load_as_double(a.planes[p], a.dtype, v);   // np.sum(mask, axis=3)
        bool m = sum > 0.0;
        if (a.label && load_as_double(a.label, a.label_dtype, v) == 0.0) m = false;            // mask[label == 0] = 0
        out[v] = m ? 1 : 0;
    }
}

// ------------------------------------------------------------------------------------------------
// phantom ROI statistics (save_phantom_csv): NaN-skipping mean / population std per label, two passes
// (mean first, then squared deviations, as np.nanstd does).  Per-block shared accumulators (float64),
// one atomicAdd per (map, roi) per block into the global accumulators.
// ------------------------------------------------------------------------------------------------
constexpr int kMaxRoi = 64;
constexpr int kMaxStatMaps = 4;

struct RoiArgs {
    const float* maps[kMaxStatMaps];
    const int32_t* label;
    int64_t n_vox;
    int n_maps, n_roi, pass;       // pass 0: count + sum, pass 1: sum of squared deviations from mean[]
};

__global__ void __launch_bounds__(256) roi_stats_kernel(const __grid_constant__ RoiArgs a, double* __restrict__ sum,
                                                        unsigned long long* __restrict__ cnt, const double* __restrict__ mean) {
    __shared__ double s_sum[kMaxStatMaps * kMaxRoi];
    __shared__ unsigned long long s_cnt[kMaxStatMaps * kMaxRoi];
    const int slots = a.n_maps * a.n_roi;
    for (int i = threadIdx.x; i < slots; i += 256) { s_sum[i] = 0.0; s_cnt[i] = 0ull; }
    __syncthreads();
    const int64_t nt = (int64_t)gridDim.x * 256;
    for (int64_t v = (int64_t)blockIdx.x * 256 + threadIdx.x; v < a.n_vox; v += nt) {
        const int lab = __ldg(a.label + v);
        if (lab < 1 || lab > a.n_roi) continue;
        for (int m = 0; m < a.n_maps; ++m) {
            const float x = __ldg(a.maps[m] + v);
            if (x != x) continue;                                   // nanmean / nanstd skip NaN
            const int slot = m * a.n_roi + lab - 1;
            if (a.pass == 0) { atomicAdd(&s_sum[slot], (double)x); atomicAdd(&s_cnt[slot], 1ull); }
            else { const double d = (double)x - mean[slot]; atomicAdd(&s_sum[slot], d * d); }
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < slots; i += 256) {
        if (s_sum[i] != 0.0 || s_cnt[i]) { atomicAdd(sum + i, s_sum[i]); if (a.pass == 0) atomicAdd(cnt + i, s_cnt[i]); }
    }
}

// ------------------------------------------------------------------------------------------------
// pack / scatter
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) pack_soa_kernel(const float* __restrict__ aos, int n_echo, const int64_t* __restrict__ idx,
                                                       int64_t n_fit, float* __restrict__ soa, int64_t ld) {
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= n_fit) return;
    const int64_t row = idx ? __ldg(idx + i) : i;
    const float* p = aos + row * n_echo;
    for (int e = 0; e < n_echo; ++e) soa[(int64_t)e * ld + i] = __ldg(p + e);
}

struct ScatterArgs {
    const float* src[4];
    float* dst[4];
    int n_maps;
};

__global__ void __launch_bounds__(256) scatter_kernel(const __grid_constant__ ScatterArgs a, const int64_t* __restrict__ idx,
                                                      int64_t n_fit) {
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= n_fit) return;
    const int64_t o = __ldg(idx + i);
#pragma unroll
    for (int m = 0; m < 4; ++m)
        if (m < a.n_maps) a.dst[m][o] = __ldg(a.src[m] + i);
}

// compute_residuals as a stand-alone pass (utils/t2map_utils.py:62-89): res[row] = sum_e (y_e - pred_e)/E from given maps
__global__ void __launch_bounds__(256) residual_kernel(const __grid_constant__ FitConsts c, const float* __restrict__ aos,
                                                       const int64_t* __restrict__ idx, int64_t n_fit, int model,
                                                       const float* __restrict__ k_map, const float* __restrict__ t2_map,
                                                       const float* __restrict__ sigma_map, float* __restrict__ res_map) {
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= n_fit) return;
    const int64_t row = idx ? __ldg(idx + i) : i;
    const float* p = aos + row * c.n_echo;
    const float k = k_map[row], rr = 1.0f / t2_map[row];
    const float s = (model != T2FIT_MODEL_GAUSSIAN && sigma_map) ? sigma_map[row] : 0.f;
    float scale = 1.f;
    if (c.norm) {
        float mx = __ldg(p);
        for (int e = 1; e < c.n_echo; ++e) mx = fmaxf(mx, __ldg(p + e));
        scale = 1.0f / mx;
    }
    float acc = 0.f;
    for (int e = 0; e < c.n_echo; ++e) {
        float pred = k * fast_ex2(c.nte2[e] * rr);
        if (model != T2FIT_MODEL_GAUSSIAN) pred = sqrtf(pred * pred + s * s);
        acc += __ldg(p + e) * scale - pred;
    }
    res_map[row] = acc / (float)c.n_echo;
}

// ------------------------------------------------------------------------------------------------
// Per-voxel analysis passes (t2fit_stderr, t2fit_t2_interval): one FP64 thread per voxel on AoS device rows, read as the fit
// kernels read them (vector loads where E and the base allow).  PassInput is what both take from the problem.
// ------------------------------------------------------------------------------------------------
struct PassInput {
    double te[kMaxEcho];
    const float* echoes;
    const int64_t* idx;        // at most one of idx / idx32 is set; neither = rows 0..n_fit-1
    const int32_t* idx32;
    int64_t n_fit, n_vox;
    int dense;                 // outputs indexed by row instead of i
    int norm;
    int vec_ok;
};

struct PassSlot {
    int64_t row;               // echo row of voxel i
    int64_t o;                 // its output slot: row (dense) or i (compact)
    bool in_range;             // row < n_vox
};

__device__ __forceinline__ PassSlot pass_slot(const PassInput& in, int64_t i) {
    const int64_t row = in.idx ? __ldg(in.idx + i) : in.idx32 ? (int64_t)__ldg(in.idx32 + i) : i;
    const bool in_range = (unsigned long long)row < (unsigned long long)in.n_vox;
    return {row, in.dense ? row : i, in_range};
}

// stderr_kernel: standard errors of (k, T2[, sigma]) at given parameters (csrc/t2fit_stderr.cuh)
struct StderrArgs {
    PassInput in;
    const float *k, *t2, *sigma;
    float *se_k, *se_t2, *se_sigma;
};

template <int MODEL, int E>
__global__ void __launch_bounds__(256) stderr_kernel(const __grid_constant__ StderrArgs a) {
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= a.in.n_fit) return;
    const auto [row, o, in_range] = pass_slot(a.in, i);
    if (!in_range) {                        // an index outside the volume: nothing to read; a compact slot gets NaN
        if (!a.in.dense) {
            if (a.se_k) a.se_k[o] = NAN;
            if (a.se_t2) a.se_t2[o] = NAN;
            if (MODEL != T2FIT_MODEL_GAUSSIAN && a.se_sigma) a.se_sigma[o] = NAN;
        }
        return;
    }
    float y[E];
    load_aos<E>(a.in.echoes, row, a.in.vec_ok, y);
    double s[3];
    se::voxel_stderr<MODEL, E>(y, a.in.te, a.in.norm != 0, __ldg(a.k + o), __ldg(a.t2 + o),
                               MODEL == T2FIT_MODEL_GAUSSIAN ? 0.0f : __ldg(a.sigma + o), s);
    if (a.se_k) a.se_k[o] = (float)s[0];
    if (a.se_t2) a.se_t2[o] = (float)s[1];
    if (MODEL != T2FIT_MODEL_GAUSSIAN && a.se_sigma) a.se_sigma[o] = (float)s[2];
}

using StderrFn = void (*)(const StderrArgs);

StderrFn pick_stderr(int model, int n_echo) {
    return with_echo_count(n_echo, [model](auto e) -> StderrFn {
        constexpr int E = decltype(e)::value;
        if (model == T2FIT_MODEL_GAUSSIAN) return stderr_kernel<T2FIT_MODEL_GAUSSIAN, E>;
        if (model == T2FIT_MODEL_GAUSSIAN_RICIAN) return stderr_kernel<T2FIT_MODEL_GAUSSIAN_RICIAN, E>;
        if (model == T2FIT_MODEL_RICIAN) return stderr_kernel<T2FIT_MODEL_RICIAN, E>;
        return nullptr;
    });
}

// interval_kernel: profile-likelihood interval for T2 (csrc/t2fit_interval.cuh).  The kernel is instantiated per echo count
// for the row load only; the model is a run-time argument and the profile work is one out-of-line routine with E at run
// time, so its code is compiled 31 times rather than 93 (ptxas gives every kernel its own copy of the routine).  The grid
// work space (iv::Grid, 6 KB) is thread-local memory.
struct IntervalArgs {
    PassInput in;
    iv::Box box;               // k / T2 / sigma bounds in force; k_lo replaced by y(TE_0) per voxel when no_prior
    double q;
    float *lo, *hi, *best;
    uint8_t* flags;
    double* profile;           // [n_fit, n_grid] or NULL
    int model;
    int n_grid;
    int no_prior;
};

template <int E>
__global__ void __launch_bounds__(128) interval_kernel(const __grid_constant__ IntervalArgs a) {
    const int64_t i = (int64_t)blockIdx.x * 128 + threadIdx.x;
    if (i >= a.in.n_fit) return;
    const auto [row, o, in_range] = pass_slot(a.in, i);
    double* prof = a.profile ? a.profile + i * a.n_grid : nullptr;
    if (!in_range) {                        // an index outside the volume: nothing to read; a compact slot gets NaN / invalid
        if (!a.in.dense) {
            if (a.lo) a.lo[o] = NAN;
            if (a.hi) a.hi[o] = NAN;
            if (a.best) a.best[o] = NAN;
            if (a.flags) a.flags[o] = iv::kInvalid;
        }
        if (prof) for (int g = 0; g < a.n_grid; ++g) prof[g] = NAN;
        return;
    }
    float y[E];
    load_aos<E>(a.in.echoes, row, a.in.vec_ok, y);
    iv::Voxel v;
    iv::Grid w;
    const bool ok = iv::load_voxel<E>(y, a.in.te, a.model, a.in.norm != 0, a.box, a.no_prior != 0, v);
    double lo, hi, best;
    int fl;
    iv::voxel_interval(v, ok, a.q, a.n_grid, w, lo, hi, best, fl, prof);
    if (a.lo) a.lo[o] = (float)lo;
    if (a.hi) a.hi[o] = (float)hi;
    if (a.best) a.best[o] = (float)best;
    if (a.flags) a.flags[o] = (uint8_t)fl;
}

using IntervalFn = void (*)(const IntervalArgs);

IntervalFn pick_interval(int n_echo) {
    return with_echo_count(n_echo, [](auto e) -> IntervalFn { return interval_kernel<decltype(e)::value>; });
}

// replicate_kernel: the parametric-bootstrap rows of every voxel (csrc/t2fit_bootstrap.cuh).  One thread per (voxel,
// replicate): thread g writes row g = i n_rep + r, so consecutive threads store consecutive rows.  The threads of a voxel
// read the same observed row (served by L1) and recompute its source; the model is a run-time argument.
struct ReplicateArgs {
    PassInput in;
    const float *k, *t2, *sigma;
    const float* noise_sd;     // [n_fit] or NULL
    const int64_t* voxel_id;   // [n_fit] or NULL = the row read
    uint64_t seed;
    float* rows;               // [n_fit * n_rep, E]
    int n_rep;
    int model;
};

template <int E>
__global__ void __launch_bounds__(128) replicate_kernel(const __grid_constant__ ReplicateArgs a) {
    const int64_t g = (int64_t)blockIdx.x * 128 + threadIdx.x;
    if (g >= a.in.n_fit * a.n_rep) return;
    const int64_t i = g / a.n_rep;
    const int r = (int)(g - i * a.n_rep);
    const auto [row, o, in_range] = pass_slot(a.in, i);
    bs::Source<E> src;
    src.ok = false;
    if (in_range) {
        float y[E];
        load_aos<E>(a.in.echoes, row, a.in.vec_ok, y);
        bs::load_source<E>(y, a.in.te, a.model, a.in.norm != 0, __ldg(a.k + i), __ldg(a.t2 + i),
                           a.model == T2FIT_MODEL_GAUSSIAN ? 0.0f : __ldg(a.sigma + i), a.noise_sd != nullptr,
                           a.noise_sd ? __ldg(a.noise_sd + i) : 0.0f, src);
    }
    const uint64_t v = a.voxel_id ? (uint64_t)__ldg(a.voxel_id + i) : (uint64_t)row;
    float out[E];
    bs::replicate_row<E>(src, a.model, a.seed, r, v, out);
    float* dst = a.rows + g * E;
#pragma unroll
    for (int e = 0; e < E; ++e) dst[e] = out[e];
}

using ReplicateFn = void (*)(const ReplicateArgs);

ReplicateFn pick_replicate(int n_echo) {
    return with_echo_count(n_echo, [](auto e) -> ReplicateFn { return replicate_kernel<decltype(e)::value>; });
}

// bootstrap_stats_kernel: one block of kStatThreads per voxel.  Thread t sums the used replicates t, t + kStatThreads, ...
// in ascending order, a halving tree adds the partial sums (the fixed order of csrc/t2fit_bootstrap.cuh), and a bitonic
// sort of the used T2 values (unused slots +inf, padded to a power of two) in shared memory gives the quantiles.
struct BootstrapStatsArgs {
    const float *k, *t2, *sigma;
    const uint8_t* status;
    float *mean, *sd;          // [3][n_fit]
    float *lo, *hi;
    int32_t *n_used, *n_ok;
    int64_t n_fit;
    double q_lo, q_hi;
    int n_rep, n_pad;          // n_pad: the power of two >= n_rep the sort runs over
    int model;
};

__global__ void __launch_bounds__(bs::kStatThreads) bootstrap_stats_kernel(const __grid_constant__ BootstrapStatsArgs a) {
    constexpr int T = bs::kStatThreads;
    extern __shared__ float key[];                 // [n_pad]
    __shared__ double part[3][T];
    __shared__ int cnt[2][T];
    const int t = threadIdx.x;
    const int64_t i = blockIdx.x;
    const int P = a.model == T2FIT_MODEL_GAUSSIAN ? 2 : 3;
    const float* rk = a.k + i * a.n_rep;
    const float* rt = a.t2 + i * a.n_rep;
    const float* rs = P == 3 ? a.sigma + i * a.n_rep : nullptr;
    const uint8_t* st = a.status + i * a.n_rep;
    double s[3] = {0.0, 0.0, 0.0};
    int nu = 0, no = 0;
    for (int r = t; r < a.n_pad; r += T) {
        float kt = INFINITY;
        if (r < a.n_rep) {
            const float vk = rk[r], vt = rt[r], vs = rs ? rs[r] : 0.0f;
            const uint8_t sr = st[r];
            no += sr == T2FIT_ST_OK;
            if (bs::rep_used(sr, vk, vt, vs, P)) {
                ++nu;
                kt = vt;
                s[0] = lb::add(s[0], (double)vk);
                s[1] = lb::add(s[1], (double)vt);
                if (P == 3) s[2] = lb::add(s[2], (double)vs);
            }
        }
        key[r] = kt;
    }
    for (int j = 0; j < 3; ++j) part[j][t] = s[j];
    cnt[0][t] = nu;
    cnt[1][t] = no;
    __syncthreads();
    for (int h = T / 2; h >= 1; h /= 2) {
        if (t < h) {
            for (int j = 0; j < 3; ++j) part[j][t] = lb::add(part[j][t], part[j][t + h]);
            cnt[0][t] += cnt[0][t + h];
            cnt[1][t] += cnt[1][t + h];
        }
        __syncthreads();
    }
    const int n_used = cnt[0][0], n_ok = cnt[1][0];
    double m[3];
    for (int j = 0; j < 3; ++j) m[j] = part[j][0] / (double)n_used;
    __syncthreads();                               // everyone has read the sums before part[] is reused
    s[0] = s[1] = s[2] = 0.0;
    for (int r = t; r < a.n_rep; r += T) {
        const float vk = rk[r], vt = rt[r], vs = rs ? rs[r] : 0.0f;
        if (!bs::rep_used(st[r], vk, vt, vs, P)) continue;
        const double dk = lb::sub((double)vk, m[0]), dt = lb::sub((double)vt, m[1]);
        s[0] = lb::add(s[0], lb::mul(dk, dk));
        s[1] = lb::add(s[1], lb::mul(dt, dt));
        if (P == 3) {
            const double ds = lb::sub((double)vs, m[2]);
            s[2] = lb::add(s[2], lb::mul(ds, ds));
        }
    }
    for (int j = 0; j < 3; ++j) part[j][t] = s[j];
    __syncthreads();
    for (int h = T / 2; h >= 1; h /= 2) {
        if (t < h)
            for (int j = 0; j < 3; ++j) part[j][t] = lb::add(part[j][t], part[j][t + h]);
        __syncthreads();
    }
    for (int size = 2; size <= a.n_pad; size *= 2) {          // bitonic sort, ascending
        for (int stride = size / 2; stride > 0; stride /= 2) {
            for (int x = t; x < a.n_pad / 2; x += T) {
                const int lo = 2 * x - (x & (stride - 1)), hi = lo + stride;
                const bool up = (lo & size) == 0;
                const float u = key[lo], w = key[hi];
                if ((u > w) == up) { key[lo] = w; key[hi] = u; }
            }
            __syncthreads();
        }
    }
    if (t != 0) return;
    const bool enough = n_used >= 2;
    for (int j = 0; j < 3; ++j) {
        const bool has = enough && j < P;
        if (a.mean) a.mean[j * a.n_fit + i] = has ? (float)m[j] : NAN;
        if (a.sd) a.sd[j * a.n_fit + i] = has ? (float)sqrt(part[j][0] / (double)(n_used - 1)) : NAN;
    }
    if (a.lo) a.lo[i] = enough ? (float)bs::quantile_sorted(key, n_used, a.q_lo) : NAN;
    if (a.hi) a.hi[i] = enough ? (float)bs::quantile_sorted(key, n_used, a.q_hi) : NAN;
    if (a.n_used) a.n_used[i] = n_used;
    if (a.n_ok) a.n_ok[i] = n_ok;
}

// ------------------------------------------------------------------------------------------------
// launch table
// ------------------------------------------------------------------------------------------------
using FitFn = void (*)(const FitConsts, const KernelIO);

template <int MODEL, int LAYOUT, bool FILL>
FitFn pick_e(int n_echo) {
    return with_echo_count(n_echo, [](auto e) -> FitFn { return fit_kernel<MODEL, decltype(e)::value, LAYOUT, FILL>; });
}

template <bool FILL>
FitFn pick_layout(int model, int n_echo, int layout) {
    if (model == T2FIT_MODEL_GAUSSIAN)
        return layout == T2FIT_LAYOUT_AOS ? pick_e<kMono2, T2FIT_LAYOUT_AOS, FILL>(n_echo)
               : layout == T2FIT_LAYOUT_PLANES ? pick_e<kMono2, T2FIT_LAYOUT_PLANES, FILL>(n_echo)
               : FILL ? nullptr : pick_e<kMono2, T2FIT_LAYOUT_SOA, false>(n_echo);
    if (FILL) return nullptr;            // the 3-parameter fit runs in floor_queue_kernel; its dense maps are zeroed by zero_fill_kernel
    return layout == T2FIT_LAYOUT_AOS ? pick_e<kFloor3, T2FIT_LAYOUT_AOS, false>(n_echo)
           : layout == T2FIT_LAYOUT_PLANES ? pick_e<kFloor3, T2FIT_LAYOUT_PLANES, false>(n_echo)
           : pick_e<kFloor3, T2FIT_LAYOUT_SOA, false>(n_echo);
}

// fill: the launch also zero-fills the dense maps (AoS / PLANES input only; SoA input is compact by construction)
FitFn pick_kernel(int model, int n_echo, int layout, bool fill) {
    return fill ? pick_layout<true>(model, n_echo, layout) : pick_layout<false>(model, n_echo, layout);
}

using QueueFn = void (*)(const FitConsts, const KernelIO, unsigned long long*, const int);

template <int LAYOUT>
QueueFn pick_queue_e(int n_echo) {
    return with_echo_count(n_echo, [](auto e) -> QueueFn { return floor_queue_kernel<decltype(e)::value, LAYOUT>; });
}

QueueFn pick_queue_kernel(int n_echo, int layout) {
    return layout == T2FIT_LAYOUT_AOS ? pick_queue_e<T2FIT_LAYOUT_AOS>(n_echo)
           : layout == T2FIT_LAYOUT_SOA ? pick_queue_e<T2FIT_LAYOUT_SOA>(n_echo) : pick_queue_e<T2FIT_LAYOUT_PLANES>(n_echo);
}

using LbFn = void (*)(const lb::LbConsts, const KernelIO, unsigned long long*);

LbFn pick_lb_kernel(int model, int n_echo, bool dense) {
    if (n_echo < 2 || n_echo > kMaxEcho) return nullptr;
    if (dense) {
        if (model == T2FIT_MODEL_GAUSSIAN) return lbfgsb_dense_kernel<0>;
        if (model == T2FIT_MODEL_GAUSSIAN_RICIAN) return lbfgsb_dense_kernel<1>;
        return lbfgsb_dense_kernel<2>;
    }
    if (model == T2FIT_MODEL_GAUSSIAN) return lbfgsb_kernel<0>;
    if (model == T2FIT_MODEL_GAUSSIAN_RICIAN) return lbfgsb_kernel<1>;
    return lbfgsb_kernel<2>;
}

// ------------------------------------------------------------------------------------------------
// host context
// ------------------------------------------------------------------------------------------------
thread_local std::string tl_err;

int fail(int code, const std::string& msg) { tl_err = msg; return code; }

#define CU_TRY(expr)                                                                         \
    do {                                                                                     \
        cudaError_t _e = (expr);                                                             \
        if (_e != cudaSuccess)                                                               \
            return fail(T2FIT_ECUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));    \
    } while (0)

// minimal fork-join pool for the host-memory path (pack / unpack of staging chunks)
constexpr int kSlots = 3;
// voxels per staging chunk (T2FIT_HOST_CHUNK overrides, for tuning)
// Sized by BYTES, not voxels: measured on the B200 boxes (profiles/r01_notes.md), per-chunk transfers of ~2.6 MB pipeline
// cleanly (c2: 1.2-1.4 ms per volume) while >= 3.9 MB per chunk stalls the PCIe side 3x; ~2.6 MB of input per chunk.
constexpr int64_t kChunkInBytes = 2621440;
constexpr int64_t kChunkMax = 1 << 18;
static const int64_t kChunkEnv = [] { const char* e = getenv("T2FIT_HOST_CHUNK"); const long long v = e ? atoll(e) : 0; return v >= 1024 ? (int64_t)v : (int64_t)0; }();
inline int64_t chunk_for(int n_echo) {
    if (kChunkEnv) return kChunkEnv;
    const int64_t n = (kChunkInBytes / (4 * (int64_t)n_echo)) & ~(int64_t)4095;
    return std::min(kChunkMax, std::max<int64_t>(4096, n));
}
constexpr size_t kOutPerVoxel = 5 * sizeof(float) + sizeof(int32_t) + 1;

struct Slot {
    float* h_in = nullptr;     // pinned, E_cap * kChunk floats: gathered rows [n, E] (AoS) or planes [E, n] (SoA)
    float* d_in = nullptr;
    // results of one chunk, the same layout on both sides so that one copy moves everything:
    //   [t2 | k | sigma | res | fun] 5 x kChunk float, [nit] kChunk int32, [status] kChunk uint8
    uint8_t* h_out = nullptr;  // pinned
    uint8_t* d_out = nullptr;
    cudaStream_t stream = nullptr;
    cudaEvent_t done = nullptr;
    int64_t first = -1, count = 0;  // chunk in flight
    bool direct = false;            // results were copied straight into the caller's (pinned) arrays
};

constexpr int kQueues = 16;

struct Context {
    int device = -1;
    cudaDeviceProp prop{};
    cudaStream_t stream = nullptr;           // default stream of the library
    unsigned long long* d_counts = nullptr;  // [4]
    unsigned long long* h_counts = nullptr;  // pinned [4]
    Slot slots[kSlots];
    int e_cap = 0;                           // slots hold chunk_for(E) voxels of E echoes for every E <= e_cap seen so far
    size_t in_cap = 0, out_cap = 0;
    Workers* workers = nullptr;
    // scratch of t2fit_mask_indices
    int* d_tile_counts = nullptr;
    int64_t* d_tile_offsets = nullptr;
    int64_t* d_total = nullptr;
    int64_t* d_idx = nullptr;                // mapped-input host calls: device copy of a pageable mask_idx
    int64_t d_idx_cap = 0;
    int64_t* h_total = nullptr;
    int64_t tiles_cap = 0;
    unsigned long long* d_queue = nullptr;   // [kQueues] voxel queue counters of the L-BFGS-B launches (round robin)
    unsigned queue_next = 0;
    bool counts_dirty = false;               // device-memory launches may have bumped d_counts
    cudaStream_t fill_stream = nullptr;      // side stream of the zero-fill kernel
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
};

Context* g_ctx = nullptr;
std::mutex g_mu;

void free_slots(Context* c) {
    for (auto& s : c->slots) {
        if (s.h_in) cudaFreeHost(s.h_in);
        if (s.d_in) cudaFree(s.d_in);
        if (s.h_out) cudaFreeHost(s.h_out);
        if (s.d_out) cudaFree(s.d_out);
        s.h_in = s.d_in = nullptr;
        s.h_out = s.d_out = nullptr;
    }
    c->e_cap = 0; c->in_cap = 0; c->out_cap = 0;
}

int ensure_slots(Context* c, int n_echo) {
    const size_t need_in = sizeof(float) * (size_t)n_echo * (size_t)chunk_for(n_echo);
    const size_t need_out = kOutPerVoxel * (size_t)chunk_for(n_echo);
    if (c->in_cap >= need_in && c->out_cap >= need_out) return T2FIT_OK;
    const size_t in_b = std::max(need_in, c->in_cap), out_b = std::max(need_out, c->out_cap);
    free_slots(c);
    for (auto& s : c->slots) {
        CU_TRY(cudaMallocHost(&s.h_in, in_b));
        CU_TRY(cudaMalloc(&s.d_in, in_b));
        CU_TRY(cudaMallocHost(&s.h_out, out_b));
        CU_TRY(cudaMalloc(&s.d_out, out_b));
        if (!s.stream) CU_TRY(cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking));
        if (!s.done) CU_TRY(cudaEventCreateWithFlags(&s.done, cudaEventDisableTiming));
    }
    c->in_cap = in_b; c->out_cap = out_b;
    c->e_cap = n_echo;
    return T2FIT_OK;
}

// Mask words per block if the fit launch can take the zero-fill of the dense maps on, else 0: all four maps present and
// 16-byte aligned, AoS / PLANES input, and no more than a handful of words per thread (a sparse mask -- few fit threads for a
// large volume -- leaves the fill to the side-stream kernel).  Rounded up to 8 words = whole 128-byte lines of every map.
int fused_fill_wpb(const FillArgs& fa, int64_t n_fit, int layout) {
    if (!(fa.vec && fa.t2 && fa.k && fa.res && fa.sigma) || layout == T2FIT_LAYOUT_SOA || n_fit <= 0) return 0;
    const int64_t blocks = (n_fit + kBlock - 1) / kBlock;
    const int64_t words = fa.n_vox / 4;
    const int64_t wpb = std::max<int64_t>(8, (((words + blocks - 1) / blocks) + 7) & ~(int64_t)7);
    return wpb <= (int64_t)kFusedFillMaxWpt * kBlock ? (int)wpb : 0;
}

int launch_floor_queue(Context* c, const FitConsts& fc, const KernelIO& io, int n_echo, int layout, cudaStream_t st) {
    QueueFn fn = pick_queue_kernel(n_echo, layout);
    if (!fn) return fail(T2FIT_EINVAL, "no kernel for this n_echo");
    static std::mutex mu;
    static std::vector<std::pair<QueueFn, int>> occ;         // resident blocks per SM, per kernel
    int per_sm = 0;
    {
        std::lock_guard<std::mutex> lk(mu);
        for (auto& e : occ) if (e.first == fn) per_sm = e.second;
        if (per_sm == 0) {
            CU_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, kQBlock, 0));
            if (per_sm <= 0) per_sm = 1;
            occ.emplace_back(fn, per_sm);
        }
    }
    const char* er = getenv("T2FIT_QUEUE_REFILL");           // lanes of a warp that must be waiting before they are replaced
    const int refill = er ? std::min(32, std::max(1, atoi(er))) : kQueueRefill;
    const int64_t want = (io.n_fit + kQBlock - 1) / kQBlock;
    const unsigned grid = (unsigned)std::min<int64_t>(want, (int64_t)per_sm * c->prop.multiProcessorCount);
    unsigned long long* q = c->d_queue + (c->queue_next++ % kQueues);
    CU_TRY(cudaMemsetAsync(q, 0, sizeof(unsigned long long), st));
    fn<<<grid, kQBlock, 0, st>>>(fc, io, q, refill);
    CU_TRY(cudaGetLastError());
    return T2FIT_OK;
}

// fa (may be null): dense maps to zero-fill in the same launch; the caller has checked fused_fill_wpb() > 0.
int launch_fit(Context* c, const FitConsts& fc, KernelIO io, int model, int n_echo, int layout, cudaStream_t st,
               const FillArgs* fa = nullptr) {
    if (io.n_fit <= 0) return T2FIT_OK;
    if (model != T2FIT_MODEL_GAUSSIAN && !fa) {
        // 3-parameter fit: persistent grid + voxel queue (T2FIT_FLOOR_KERNEL=oneshot keeps the one-thread-per-voxel launch)
        const char* ek = getenv("T2FIT_FLOOR_KERNEL");
        if (!(ek && !strcmp(ek, "oneshot"))) return launch_floor_queue(c, fc, io, n_echo, layout, st);
    }
    const int64_t blocks = (io.n_fit + kBlock - 1) / kBlock;
    if (blocks > 0x7fffffffLL) return fail(T2FIT_EINVAL, "n_fit too large for one launch");
    if (fa) {
        io.fill_mask = fa->mask; io.fill_words = fa->n_vox / 4; io.fill_nvox = fa->n_vox;
        io.fill_wpb = fused_fill_wpb(*fa, io.n_fit, layout);
        io.sigma = fa->sigma;
        if (io.fill_wpb <= 0) return fail(T2FIT_EINVAL, "internal: fused fill not applicable");
    }
    FitFn fn = pick_kernel(model, n_echo, layout, fa != nullptr);
    if (!fn) return fail(T2FIT_EINVAL, "no kernel for this n_echo");
    // T2FIT_PDL=0: plain stream order (the default lets back-to-back fit launches overlap launch latency and ramp-up with the
    // previous launch's tail; the kernel waits for the previous grid before its first global access)
    static const bool pdl = [] { const char* e = getenv("T2FIT_PDL"); return !(e && !strcmp(e, "0")); }();
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)blocks); cfg.blockDim = dim3(kBlock); cfg.dynamicSmemBytes = 0; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = pdl ? 1 : 0;
    CU_TRY(cudaLaunchKernelEx(&cfg, fn, fc, io));
    CU_TRY(cudaGetLastError());
    return T2FIT_OK;
}

int launch_lbfgsb_coop(Context* c, const lb::LbConsts& lc, const KernelIO& io, int model, int lanes, cudaStream_t st);

int launch_lbfgsb(Context* c, const lb::LbConsts& lc, KernelIO io, int model, int n_echo, cudaStream_t st) {
    if (io.n_fit <= 0) return T2FIT_OK;
    if (n_echo < 2 || n_echo > kMaxEcho) return fail(T2FIT_EINVAL, "no kernel for this n_echo");
    // T2FIT_LB_KERNEL = thread (default) | coop8 | coop16 | coop32: the one-thread-per-voxel kernel with the state in local
    // memory, or a lane group per voxel with the state in shared memory (bit-identical results; measured 2.6-3x slower,
    // profiles/r02_notes.md -- kept as the cross-check of the thread kernel).  Read per call: tests and A/B runs switch it.
    const char* ek = getenv("T2FIT_LB_KERNEL");
    const int lanes = !ek ? 0 : !strcmp(ek, "coop8") ? 8 : !strcmp(ek, "coop16") ? 16 : !strcmp(ek, "coop32") ? 32 : 0;
    if (lanes && !lc.dense) return launch_lbfgsb_coop(c, lc, io, model, lanes, st);
    LbFn fn = pick_lb_kernel(model, n_echo, lc.dense != 0);
    if (!fn) return fail(T2FIT_EINVAL, "no kernel for this n_echo");
    // persistent grid sized to what is resident at once; voxels are handed out through a queue counter
    static const int env_per_sm = [] { const char* e = getenv("T2FIT_LB_BLOCKS_PER_SM"); return e ? atoi(e) : 0; }();
    static const int env_per_sm_dense = [] { const char* e = getenv("T2FIT_LBD_BLOCKS_PER_SM"); return e ? atoi(e) : 0; }();
    int per_sm = lc.dense ? env_per_sm_dense : env_per_sm;
    // the dense kernel keeps the signal row and the running sums of its objective loop in shared memory
    const size_t smem = lc.dense ? dense_smem_bytes(model == T2FIT_MODEL_GAUSSIAN ? 2 : 3, n_echo) : 0;
    if (smem > 48 * 1024) {
        static std::mutex mu;
        static std::vector<LbFn> prepared;
        std::lock_guard<std::mutex> lk(mu);
        if (std::find(prepared.begin(), prepared.end(), fn) == prepared.end()) {
            CU_TRY(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dense_smem_bytes(3, kMaxEcho)));
            prepared.push_back(fn);
        }
    }
    const int threads = lc.dense ? kLbdBlock : kLbBlock;
    if (per_sm <= 0) {
        CU_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, threads, smem));
        if (per_sm <= 0) per_sm = 1;
    }
    const int64_t want = (io.n_fit + threads - 1) / threads;
    const unsigned grid = (unsigned)std::min<int64_t>(want, (int64_t)per_sm * c->prop.multiProcessorCount);
    unsigned long long* q = c->d_queue + (c->queue_next++ % kQueues);
    CU_TRY(cudaMemsetAsync(q, 0, sizeof(unsigned long long), st));
    fn<<<grid, threads, smem, st>>>(lc, io, q);
    CU_TRY(cudaGetLastError());
    return T2FIT_OK;
}

// cooperative form: one block per SM, as many lane groups as the shared memory holds
using LbCoopFn = void (*)(const lb::LbConsts, const KernelIO, unsigned long long*, const int);

template <int G>
LbCoopFn pick_lb_coop(int model, size_t* run_bytes) {
    if (model == T2FIT_MODEL_GAUSSIAN) { *run_bytes = sizeof(lb::CoopRun<0, G>); return lbfgsb_coop_kernel<0, G>; }
    if (model == T2FIT_MODEL_GAUSSIAN_RICIAN) { *run_bytes = sizeof(lb::CoopRun<1, G>); return lbfgsb_coop_kernel<1, G>; }
    *run_bytes = sizeof(lb::CoopRun<2, G>);
    return lbfgsb_coop_kernel<2, G>;
}

int launch_lbfgsb_coop(Context* c, const lb::LbConsts& lc, const KernelIO& io, int model, int lanes, cudaStream_t st) {
    size_t run_bytes = 0;
    LbCoopFn fn = lanes == 8 ? pick_lb_coop<8>(model, &run_bytes) : lanes == 16 ? pick_lb_coop<16>(model, &run_bytes)
                                                                                 : pick_lb_coop<32>(model, &run_bytes);
    // per-voxel stride: a multiple of 16 bytes and = 8 (mod 16) in 8-byte words, so that the two groups of a half-warp
    // (G = 8) hit different banks when they read the same element of their own state
    size_t words = (run_bytes + 7) / 8;
    words += (8 + 16 - (words % 16)) % 16;
    const int stride = (int)(words * 8);
    const int smem_max = (int)c->prop.sharedMemPerBlockOptin;
    const int per_warp = 32 / lanes;
    int groups = (smem_max / stride) / per_warp * per_warp;
    groups = std::min(groups, 1024 / lanes);
    static const int env_groups = [] { const char* e = getenv("T2FIT_LB_GROUPS"); return e ? atoi(e) : 0; }();
    if (env_groups > 0) groups = std::min(groups, env_groups / per_warp * per_warp);
    if (groups < per_warp) return fail(T2FIT_EINVAL, "shared memory too small for the cooperative L-BFGS-B kernel");
    const int smem = groups * stride;
    static std::mutex mu;
    static std::vector<LbCoopFn> prepared;
    {
        std::lock_guard<std::mutex> lk(mu);
        if (std::find(prepared.begin(), prepared.end(), fn) == prepared.end()) {
            CU_TRY(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max));
            prepared.push_back(fn);
        }
    }
    const int64_t want = (io.n_fit + groups - 1) / groups;
    const unsigned grid = (unsigned)std::min<int64_t>(want, (int64_t)c->prop.multiProcessorCount);
    unsigned long long* q = c->d_queue + (c->queue_next++ % kQueues);
    CU_TRY(cudaMemsetAsync(q, 0, sizeof(unsigned long long), st));
    fn<<<grid, groups * lanes, smem, st>>>(lc, io, q, stride);
    CU_TRY(cudaGetLastError());
    return T2FIT_OK;
}

// zero-fill of the dense maps on the side stream, forked from and joined back into `st`
int launch_zero_fill(Context* c, const FillArgs& fa, bool sigma_all, cudaStream_t st, bool* forked) {
    *forked = false;
    if (fa.n_vox <= 0) return T2FIT_OK;
    CU_TRY(cudaEventRecord(c->ev_fork, st));
    CU_TRY(cudaStreamWaitEvent(c->fill_stream, c->ev_fork, 0));
    const int64_t chunks = (fa.n_vox + kFillChunk - 1) / kFillChunk;
    static const int threads = [] { const char* e = getenv("T2FIT_FILL_THREADS"); const int v = e ? atoi(e) : 256; return (v >= 32 && v <= 256 && v % 32 == 0) ? v : 256; }();
    const int64_t want = (chunks + threads / 32 - 1) / (threads / 32);      // one chunk per warp per round
    static const int per_sm = [] { const char* e = getenv("T2FIT_FILL_BLOCKS_PER_SM"); return e ? std::max(1, atoi(e)) : 1; }();
    const unsigned grid = (unsigned)std::max<int64_t>(1, std::min<int64_t>(want, (int64_t)per_sm * c->prop.multiProcessorCount));
    if (sigma_all) zero_fill_kernel<true><<<grid, threads, 0, c->fill_stream>>>(fa);
    else zero_fill_kernel<false><<<grid, threads, 0, c->fill_stream>>>(fa);
    CU_TRY(cudaGetLastError());
    CU_TRY(cudaEventRecord(c->ev_join, c->fill_stream));
    *forked = true;
    return T2FIT_OK;
}

// host-memory path: stage chunks through pinned buffers.  Worker threads gather the masked rows of the
// next chunk (run-aware memcpy: consecutive mask indices are contiguous rows) while the GPU works on
// the previous ones; per chunk ONE H2D copy, one kernel, and either direct D2H copies into the caller's
// arrays (when those are page-locked) or one D2H into pinned staging + a threaded unpack / scatter.
// Host echo arrays may hold int16 / uint16 / int32 / float64 elements (t2fit_problem::echo_dtype): the reference's
// `.astype(np.float32)` (:411) is applied while the fitted rows are gathered into the float32 staging buffers.
template <typename T>
inline void cast_copy(float* dst, const T* src, int64_t n) {
    for (int64_t i = 0; i < n; ++i) dst[i] = (float)src[i];
}
inline size_t echo_elem_size(int dt) {
    return dt == T2FIT_DT_F64 ? 8 : (dt == T2FIT_DT_I16 || dt == T2FIT_DT_U16) ? 2 : 4;
}
inline void echo_copy(float* dst, const void* base, int dt, int64_t off, int64_t n) {
    switch (dt) {
        case T2FIT_DT_I16: cast_copy(dst, static_cast<const int16_t*>(base) + off, n); break;
        case T2FIT_DT_U16: cast_copy(dst, static_cast<const uint16_t*>(base) + off, n); break;
        case T2FIT_DT_I32: cast_copy(dst, static_cast<const int32_t*>(base) + off, n); break;
        case T2FIT_DT_F64: cast_copy(dst, static_cast<const double*>(base) + off, n); break;
        default: memcpy(dst, static_cast<const float*>(base) + off, sizeof(float) * n); break;
    }
}
inline float echo_at(const void* base, int dt, int64_t off) {
    float v;
    echo_copy(&v, base, dt, off, 1);
    return v;
}

// mask_indices[i] of a HOST index vector (int64, or int32 when t2fit_problem::idx_dtype says so)
inline int64_t host_idx(const t2fit_problem& p, int64_t i) {
    return p.idx_dtype == T2FIT_IDX_I32 ? (int64_t)reinterpret_cast<const int32_t*>(p.mask_idx)[i] : p.mask_idx[i];
}

bool is_pinned(const void* p) {
    if (!p) return true;
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return at.type == cudaMemoryTypeHost;
}

double now_ms() {
    using namespace std::chrono;
    return duration<double, std::milli>(steady_clock::now().time_since_epoch()).count();
}

// Host-memory call whose INPUT is page-locked too (cudaHostAlloc / torch pin_memory / cudaHostRegister) and whose compact
// result arrays are page-locked: no staging at all.  ONE launch over all voxels; the kernel gathers the masked rows
// straight from host memory over PCIe (only the masked rows cross the bus, consecutive voxels coalesce into 128-byte
// reads, ~190 k threads in flight hide the latency) and stores the results straight back.  No host thread touches the
// data, so N ranks on one node do not compete for host cores.  Returns 1 if this path does not apply.
int run_host_mapped(Context* c, const t2fit_problem& p, t2fit_outputs& o, const FitConsts& fc, const lb::LbConsts* lc) {
    // T2FIT_HOST_IN = mapped | staged | auto (default = mapped whenever the arrays are page-locked).  Measured on c2
    // (profiles/r01_notes.md): 1.16-1.17 ms per volume, call after call, with no host thread touching the data (the kernel
    // runs at 47 GB/s PCIe reads + 41 GB/s writes); the staged pipeline with all 16 host cores to itself needs 1.35-1.55 ms
    // with 4 ms outliers, and 1.4x (2 ranks) to 4x (8 ranks) more when ranks share the cores.
    const char* env_in = getenv("T2FIT_HOST_IN");       // read per call (tests switch it)
    const int mode = !env_in ? 0 : !strcmp(env_in, "mapped") ? 1 : !strcmp(env_in, "staged") ? 2 : 0;
    const bool want = mode != 2;
    const bool mono = p.model == T2FIT_MODEL_GAUSSIAN;
    const double t_begin = now_ms();
    if (!want || o.dense || !p.echoes || !is_pinned(p.echoes)) return 1;
    if (p.echo_dtype != 0 && p.echo_dtype != T2FIT_DT_F32) return 1;      // the kernels read float32: other element types are staged (cast)
    if (o.trace_cap > 0 && (o.trace_f || o.trace_step || o.trace_len)) return 1;
    if (!(is_pinned(o.t2) && is_pinned(o.k) && is_pinned(o.res) && is_pinned(o.fun) && is_pinned(o.nit) && is_pinned(o.status) &&
          (mono || is_pinned(o.sigma)))) return 1;
    KernelIO io{};
    auto map = [&](const void* h, void** d) { *d = nullptr; return !h || cudaHostGetDevicePointer(d, const_cast<void*>(h), 0) == cudaSuccess; };
    void* d_echo = nullptr;
    if (!(map(p.echoes, &d_echo) && map(o.t2, (void**)&io.t2) && map(o.k, (void**)&io.k) && map(mono ? nullptr : o.sigma, (void**)&io.sigma) &&
          map(o.res, (void**)&io.res) && map(o.fun, (void**)&io.fun) && map(o.nit, (void**)&io.nit) && map(o.status, (void**)&io.status))) {
        cudaGetLastError();
        return 1;
    }
    cudaStream_t st = c->slots[0].stream;
    if (!st) { int rc0 = ensure_slots(c, p.n_echo); if (rc0) return rc0; st = c->slots[0].stream; }
    const int64_t M = p.n_fit;
    if (p.mask_idx) {
        // no host pass over the index vector: the kernel checks the range itself (KernelIO::n_rows)
        io.n_rows = p.n_vox;
        const bool i32 = p.idx_dtype == T2FIT_IDX_I32;
        const size_t isz = i32 ? sizeof(int32_t) : sizeof(int64_t);
        void* d_idx = nullptr;
        if (is_pinned(p.mask_idx) && map(p.mask_idx, &d_idx)) {
            // read in place too (measured: 1.6 ms vs 2.35 ms with a DMA copy first)
        } else {                                      // pageable index vector: one copy to the device (4 or 8 B per voxel)
            cudaGetLastError();
            if (c->d_idx_cap < M) {
                if (c->d_idx) cudaFree(c->d_idx);
                c->d_idx = nullptr; c->d_idx_cap = 0;
                CU_TRY(cudaMalloc(&c->d_idx, sizeof(int64_t) * M));
                c->d_idx_cap = M;
            }
            CU_TRY(cudaMemcpyAsync(c->d_idx, p.mask_idx, isz * M, cudaMemcpyHostToDevice, st));
            d_idx = c->d_idx;
        }
        if (i32) io.idx32 = static_cast<const int32_t*>(d_idx);
        else io.idx = static_cast<const int64_t*>(d_idx);
    }
    if (c->counts_dirty) {
        CU_TRY(cudaMemsetAsync(c->d_counts, 0, 4 * sizeof(unsigned long long), st));
        c->counts_dirty = false;
    }
    io.echoes = static_cast<const float*>(d_echo); io.ld = p.ld; io.n_fit = M;
    io.counts = c->d_counts; io.dense = 0; io.layout = p.layout;
    io.vec_ok = (reinterpret_cast<uintptr_t>(d_echo) % 16) == 0;
    int rc = lc ? launch_lbfgsb(c, *lc, io, p.model, p.n_echo, st) : launch_fit(c, fc, io, p.model, p.n_echo, p.layout, st);
    if (rc) return rc;
    const double t_launched = now_ms();
    CU_TRY(cudaMemcpyAsync(c->h_counts, c->d_counts, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaMemsetAsync(c->d_counts, 0, 4 * sizeof(unsigned long long), st));
    CU_TRY(cudaStreamSynchronize(st));
    if (c->h_counts[0] != 0) return fail(T2FIT_EINVAL, "mask_idx out of range");      // IndexError upstream
    int64_t bad_n = 0;
    for (int s = 1; s < 4; ++s) { o.status_count[s] = (int64_t)c->h_counts[s]; bad_n += o.status_count[s]; }
    o.status_count[0] = M - bad_n;
    static const bool profile = getenv("T2FIT_HOST_PROFILE") != nullptr;
    if (profile) fprintf(stderr, "[t2fit host] M=%lld mapped input (no staging): %.3f ms to launch, %.3f ms in all\n", (long long)M, t_launched - t_begin, now_ms() - t_begin);
    return T2FIT_OK;
}

int run_host(Context* c, const t2fit_problem& p, t2fit_outputs& o, const FitConsts& fc, const lb::LbConsts* lc) {
    int rc = ensure_slots(c, p.n_echo);
    if (rc) return rc;
    rc = run_host_mapped(c, p, o, fc, lc);
    if (rc != 1) return rc;
    // callback traces (L-BFGS-B solver, sampled voxels): per-slot device scratch for this call only
    const bool tracing = lc && p.n_fit > 0 && o.trace_cap > 0 && (o.trace_f || o.trace_step || o.trace_len);
    struct TraceScratch { float* f = nullptr; float* s = nullptr; int32_t* n = nullptr; } tsc[kSlots];
    auto free_trace = [&]() {
        for (auto& t : tsc) { if (t.f) cudaFree(t.f); if (t.s) cudaFree(t.s); if (t.n) cudaFree(t.n); t = TraceScratch{}; }
    };
    if (tracing) {
        const int64_t nmax = std::min<int64_t>(chunk_for(p.n_echo), p.n_fit);
        for (auto& t : tsc) {
            if (cudaMalloc(&t.f, sizeof(float) * nmax * o.trace_cap) != cudaSuccess ||
                cudaMalloc(&t.s, sizeof(float) * nmax * o.trace_cap) != cudaSuccess ||
                cudaMalloc(&t.n, sizeof(int32_t) * nmax) != cudaSuccess) {
                cudaGetLastError();
                free_trace();
                return fail(T2FIT_ENOMEM, "trace scratch: ask for traces of a sampled subset of voxels");
            }
        }
    }
    const int E = p.n_echo;
    const int64_t M = p.n_fit;
    static const bool profile = getenv("T2FIT_HOST_PROFILE") != nullptr;
    double t_pack = 0, t_wait = 0, t_unpack = 0, t0 = now_ms();
    if (c->counts_dirty) {                        // device-memory calls since the last query left counts behind
        CU_TRY(cudaMemsetAsync(c->d_counts, 0, 4 * sizeof(unsigned long long), c->slots[0].stream));
        CU_TRY(cudaStreamSynchronize(c->slots[0].stream));
        c->counts_dirty = false;
    }
    const int64_t kChunk = chunk_for(E);
    const int64_t n_chunks = (M + kChunk - 1) / kChunk;
    const bool mono = p.model == T2FIT_MODEL_GAUSSIAN;
    std::atomic<bool> bad_index{false};
    const int edt = p.echo_dtype == T2FIT_DT_F32 ? 0 : p.echo_dtype;     // 0 = float32
    // compact results can go straight into the caller's arrays if every one of them is page-locked
    // How compact results reach the caller's arrays (T2FIT_HOST_OUT overrides, for measurements):
    //   zerocopy  every result array is page-locked: the kernel stores straight into host memory through its device
    //             mapping (coalesced 128-byte writes over PCIe while it runs; no D2H copy, no unpack)      [default if pinned]
    //   direct    page-locked arrays, per-chunk cudaMemcpyAsync per field (measured erratic: 2-4.5 ms per c2 volume)
    //   staged    one D2H per chunk into pinned staging + threaded unpack / scatter                      [default otherwise]
    static const int out_mode_env = [] {
        const char* e = getenv("T2FIT_HOST_OUT");
        return !e ? 0 : !strcmp(e, "zerocopy") ? 0 : !strcmp(e, "direct") ? 1 : 2;
    }();
    const bool all_pinned = !o.dense && is_pinned(o.t2) && is_pinned(o.k) && is_pinned(o.res) && is_pinned(o.fun) &&
                            is_pinned(o.nit) && is_pinned(o.status) && (mono || is_pinned(o.sigma));
    bool zerocopy = all_pinned && out_mode_env == 0;
    struct DevView { float *t2 = nullptr, *k = nullptr, *sigma = nullptr, *res = nullptr, *fun = nullptr; int32_t* nit = nullptr; uint8_t* status = nullptr; } dv;
    if (zerocopy) {
        auto map = [&](void* h, void** d) { *d = nullptr; return !h || cudaHostGetDevicePointer(d, h, 0) == cudaSuccess; };
        zerocopy = map(o.t2, (void**)&dv.t2) && map(o.k, (void**)&dv.k) && map(mono ? nullptr : o.sigma, (void**)&dv.sigma) &&
                   map(o.res, (void**)&dv.res) && map(o.fun, (void**)&dv.fun) && map(o.nit, (void**)&dv.nit) &&
                   map(o.status, (void**)&dv.status);
        if (!zerocopy) cudaGetLastError();
    }
    const bool direct = zerocopy || (all_pinned && out_mode_env == 1);

    auto unpack = [&](Slot& s) {
        if (s.first < 0) return;
        const int64_t first = s.first, n = s.count;
        s.first = -1;
        if (s.direct) return;
        const double tu = now_ms();
        float* outs[5] = {o.t2, o.k, o.sigma, o.res, o.fun};
        const float* hf = reinterpret_cast<const float*>(s.h_out);
        const int32_t* hn = reinterpret_cast<const int32_t*>(s.h_out + (size_t)5 * n * sizeof(float));
        const uint8_t* hs = s.h_out + (size_t)5 * n * sizeof(float) + (size_t)n * sizeof(int32_t);
        c->workers->run([&](int part, int parts) {
            const int64_t lo = n * part / parts, hi = n * (part + 1) / parts;
            if (hi <= lo) return;
            for (int m = 0; m < 5; ++m) {
                float* dst = outs[m];
                if (!dst) continue;
                if (m == 2 && mono) continue;                     // sigma map stays as the caller zeroed it
                const float* src = hf + (int64_t)m * n;
                if (o.dense && m < 4 && p.mask_idx) {
                    for (int64_t i = lo; i < hi; ++i) dst[host_idx(p, first + i)] = src[i];   // scatter (:455-458)
                } else {
                    memcpy(dst + first + lo, src + lo, sizeof(float) * (hi - lo));
                }
            }
            if (o.nit) memcpy(o.nit + first + lo, hn + lo, sizeof(int32_t) * (hi - lo));
            if (o.status) memcpy(o.status + first + lo, hs + lo, hi - lo);
        });
        t_unpack += now_ms() - tu;
    };

    for (int64_t ch = 0; ch < n_chunks; ++ch) {
        Slot& s = c->slots[ch % kSlots];
        if (s.first >= 0) {                       // slot still holds an older chunk: drain it
            const double tw = now_ms();
            CU_TRY(cudaEventSynchronize(s.done));
            t_wait += now_ms() - tw;
            unpack(s);
        }
        const int64_t first = ch * kChunk, n = std::min(kChunk, M - first);
        const double tp = now_ms();
        c->workers->run([&](int part, int parts) {
            const int64_t lo = n * part / parts, hi = n * (part + 1) / parts;
            if (hi <= lo) return;
            if (p.layout == T2FIT_LAYOUT_AOS) {   // rows -> packed rows [n, E]; runs of consecutive indices in one copy (+ cast)
                if (!p.mask_idx) {
                    echo_copy(s.h_in + lo * E, p.echoes, edt, (first + lo) * E, (int64_t)E * (hi - lo));
                } else {
                    int64_t i = lo;
                    while (i < hi) {
                        int64_t j = i + 1;
                        while (j < hi && host_idx(p, first + j) == host_idx(p, first + j - 1) + 1) ++j;
                        const int64_t r0 = host_idx(p, first + i), r1 = host_idx(p, first + j - 1);
                        if (r0 < 0 || r1 >= p.n_vox) { bad_index.store(true); return; }   // IndexError upstream
                        echo_copy(s.h_in + i * E, p.echoes, edt, r0 * E, (int64_t)E * (j - i));
                        i = j;
                    }
                }
            } else if (p.layout == T2FIT_LAYOUT_SOA) {   // SoA planes [E, ld] -> planes [E, n]
                for (int e = 0; e < E; ++e)
                    echo_copy(s.h_in + (int64_t)e * n + lo, p.echoes, edt, (int64_t)e * p.ld + first + lo, hi - lo);
            } else {                              // per-TE volumes [E, ld >= n_vox] -> planes [E, n] of the masked voxels
                const bool idx = p.mask_idx != nullptr;
                for (int64_t i = lo; i < hi; ++i) {
                    const int64_t v = idx ? host_idx(p, first + i) : first + i;
                    if (v < 0 || v >= p.n_vox) { bad_index.store(true); return; }
                }
                for (int e = 0; e < E; ++e) {
                    const int64_t plane = (int64_t)e * p.ld;
                    float* dst = s.h_in + (int64_t)e * n;
                    if (!idx) echo_copy(dst + lo, p.echoes, edt, plane + first + lo, hi - lo);
                    else if (edt == 0) { const float* src = p.echoes + plane; for (int64_t i = lo; i < hi; ++i) dst[i] = src[host_idx(p, first + i)]; }
                    else for (int64_t i = lo; i < hi; ++i) dst[i] = echo_at(p.echoes, edt, plane + host_idx(p, first + i));
                }
            }
        });
        t_pack += now_ms() - tp;
        if (bad_index.load()) {
            for (auto& sl : c->slots) { cudaStreamSynchronize(sl.stream); sl.first = -1; }
            return fail(T2FIT_EINVAL, "mask_idx out of range");
        }
        CU_TRY(cudaMemcpyAsync(s.d_in, s.h_in, sizeof(float) * E * n, cudaMemcpyHostToDevice, s.stream));
        float* df = reinterpret_cast<float*>(s.d_out);
        KernelIO io{};
        io.echoes = s.d_in; io.idx = nullptr; io.ld = n; io.n_fit = n;
        io.t2 = df; io.k = df + n; io.sigma = df + 2 * n; io.res = df + 3 * n; io.fun = df + 4 * n;
        io.nit = reinterpret_cast<int32_t*>(s.d_out + (size_t)5 * n * sizeof(float));
        io.status = s.d_out + (size_t)5 * n * sizeof(float) + (size_t)n * sizeof(int32_t);
        if (zerocopy) {                               // results go straight to the caller's page-locked arrays
            io.t2 = dv.t2 ? dv.t2 + first : nullptr; io.k = dv.k ? dv.k + first : nullptr;
            io.sigma = dv.sigma ? dv.sigma + first : nullptr; io.res = dv.res ? dv.res + first : nullptr;
            io.fun = dv.fun ? dv.fun + first : nullptr; io.nit = dv.nit ? dv.nit + first : nullptr;
            io.status = dv.status ? dv.status + first : nullptr;
        }
        io.counts = c->d_counts; io.dense = 0; io.vec_ok = 1;
        io.layout = p.layout == T2FIT_LAYOUT_AOS ? T2FIT_LAYOUT_AOS : T2FIT_LAYOUT_SOA;     // staged chunks are packed
        if (tracing) {
            TraceScratch& t = tsc[ch % kSlots];
            io.trace_f = t.f; io.trace_step = t.s; io.trace_len = t.n; io.trace_cap = o.trace_cap;
        }
        rc = lc ? launch_lbfgsb(c, *lc, io, p.model, E, s.stream) : launch_fit(c, fc, io, p.model, E, io.layout, s.stream);
        if (rc) { free_trace(); return rc; }
        if (tracing) {
            const size_t tb = sizeof(float) * (size_t)n * o.trace_cap;
            if (o.trace_f) CU_TRY(cudaMemcpyAsync(o.trace_f + first * o.trace_cap, io.trace_f, tb, cudaMemcpyDeviceToHost, s.stream));
            if (o.trace_step) CU_TRY(cudaMemcpyAsync(o.trace_step + first * o.trace_cap, io.trace_step, tb, cudaMemcpyDeviceToHost, s.stream));
            if (o.trace_len) CU_TRY(cudaMemcpyAsync(o.trace_len + first, io.trace_len, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, s.stream));
        }
        s.direct = direct;
        if (zerocopy) {
            // nothing to copy
        } else if (direct) {
            auto d2h = [&](void* dst, const void* src, size_t bytes) {
                return dst ? cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, s.stream) : cudaSuccess;
            };
            CU_TRY(d2h(o.t2 ? o.t2 + first : nullptr, io.t2, sizeof(float) * n));
            CU_TRY(d2h(o.k ? o.k + first : nullptr, io.k, sizeof(float) * n));
            if (!mono) CU_TRY(d2h(o.sigma ? o.sigma + first : nullptr, io.sigma, sizeof(float) * n));
            CU_TRY(d2h(o.res ? o.res + first : nullptr, io.res, sizeof(float) * n));
            CU_TRY(d2h(o.fun ? o.fun + first : nullptr, io.fun, sizeof(float) * n));
            CU_TRY(d2h(o.nit ? o.nit + first : nullptr, io.nit, sizeof(int32_t) * n));
            CU_TRY(d2h(o.status ? o.status + first : nullptr, io.status, n));
        } else {
            CU_TRY(cudaMemcpyAsync(s.h_out, s.d_out, (size_t)n * kOutPerVoxel,
                                   cudaMemcpyDeviceToHost, s.stream));
        }
        CU_TRY(cudaEventRecord(s.done, s.stream));
        s.first = first; s.count = n;
    }
    // drain in submission order
    for (int64_t ch = std::max<int64_t>(0, n_chunks - kSlots); ch < n_chunks; ++ch) {
        Slot& s = c->slots[ch % kSlots];
        if (s.first >= 0) {
            const double tw = now_ms();
            CU_TRY(cudaEventSynchronize(s.done));
            t_wait += now_ms() - tw;
            unpack(s);
        }
    }
    // all slot streams are idle now: read the status histogram and leave the counters zeroed for the next call
    CU_TRY(cudaMemcpyAsync(c->h_counts, c->d_counts, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->slots[0].stream));
    CU_TRY(cudaMemsetAsync(c->d_counts, 0, 4 * sizeof(unsigned long long), c->slots[0].stream));
    CU_TRY(cudaStreamSynchronize(c->slots[0].stream));
    free_trace();
    int64_t bad = 0;
    for (int s = 1; s < 4; ++s) { o.status_count[s] = (int64_t)c->h_counts[s]; bad += o.status_count[s]; }
    o.status_count[0] = M - bad;
    if (profile)
        fprintf(stderr, "[t2fit host] M=%lld chunks=%lld direct=%d total %.3f ms: pack %.3f wait %.3f unpack %.3f\n", (long long)M,
                (long long)n_chunks, zerocopy ? 2 : (int)direct, now_ms() - t0, t_pack, t_wait, t_unpack);
    return T2FIT_OK;
}

// The checks t2fit_stderr and t2fit_t2_interval (`name`) make first, in this order, before their own.
int check_pass_problem(const t2fit_problem* p, const char* name) {
    if (!p) return fail(T2FIT_EINVAL, "NULL problem");
    if (p->layout != T2FIT_LAYOUT_AOS) return fail(T2FIT_EINVAL, std::string(name) + " reads T2FIT_LAYOUT_AOS echoes only");
    if (p->memory != T2FIT_MEM_DEVICE) return fail(T2FIT_EINVAL, std::string(name) + " takes T2FIT_MEM_DEVICE pointers only");
    if (p->n_echo < 2 || p->n_echo > T2FIT_MAX_ECHO) return fail(T2FIT_EINVAL, "n_echo out of range (2..T2FIT_MAX_ECHO)");
    if (p->model != T2FIT_MODEL_GAUSSIAN && p->model != T2FIT_MODEL_GAUSSIAN_RICIAN && p->model != T2FIT_MODEL_RICIAN)
        return fail(T2FIT_EINVAL, "unknown model");
    if (p->n_fit < 0 || p->n_vox < 0) return fail(T2FIT_EINVAL, "negative size");
    if (p->idx_dtype != T2FIT_IDX_I64 && p->idx_dtype != T2FIT_IDX_I32) return fail(T2FIT_EINVAL, "bad idx_dtype");
    if (!p->te_ms) return fail(T2FIT_EINVAL, "NULL te_ms");
    return T2FIT_OK;
}

// The kernel input of a checked problem with n_fit > 0 and echoes set; n_fit > n_vox is each entry's last argument check.
int pass_input(const t2fit_problem* p, int32_t dense, PassInput& in) {
    if (!p->mask_idx && p->n_fit > p->n_vox) return fail(T2FIT_EINVAL, "n_fit > n_vox");
    for (int e = 0; e < p->n_echo; ++e) in.te[e] = p->te_ms[e];
    in.echoes = p->echoes;
    if (p->mask_idx) {
        if (p->idx_dtype == T2FIT_IDX_I32) in.idx32 = reinterpret_cast<const int32_t*>(p->mask_idx);
        else in.idx = p->mask_idx;
    }
    in.n_fit = p->n_fit; in.n_vox = p->n_vox;
    in.dense = dense != 0; in.norm = p->norm != 0;
    in.vec_ok = (reinterpret_cast<uintptr_t>(p->echoes) % 16) == 0;
    return T2FIT_OK;
}

}  // namespace

// ================================================================================================
// C ABI
// ================================================================================================
// ------------------------------------------------------------------------------------------------
// Host-side front of the loader for sparse masks: the union / label masking / np.where of run_t2mapping.py:383-384,393-400,421
// and the gather + float32 cast of the masked voxels (:411-412 restricted to the rows the fit reads), on the library's own
// worker threads.  No GPU involved: with a brain mask covering ~10 % of the volume the loader then ships [E, M] floats and
// one mask plane over PCIe instead of E volumes and E masks.
// ------------------------------------------------------------------------------------------------
namespace {

std::mutex g_host_mu;                       // one host-side call at a time (Workers::run has one caller)
Workers* g_host_workers = nullptr;

Workers& host_workers() {                   // g_host_mu held
    if (!g_host_workers) {
        unsigned hw = std::thread::hardware_concurrency();
        const char* env = getenv("T2FIT_HOST_THREADS");
        g_host_workers = new Workers(env ? atoi(env) : (int)std::min(16u, hw ? hw : 4u));
    }
    return *g_host_workers;
}

constexpr int kHostTile = 512;              // voxels per inner tile (accumulators stay in L1)

template <typename T>
void union_range(const void* const* planes, int n_planes, int64_t a, int64_t b, uint8_t* __restrict__ out) {
    // np.sum(mask, axis=3) > 0 per voxel.  Unsigned masks: the sum is positive iff any plane is non-zero (bitwise OR, no
    // widening); signed integers sum exactly in int64; floating-point masks sum in float64 in plane order as numpy does.
    using Acc = std::conditional_t<std::is_unsigned<T>::value, T, std::conditional_t<std::is_integral<T>::value, int64_t, double>>;
    Acc acc[kHostTile];
    for (int64_t v0 = a; v0 < b; v0 += kHostTile) {
        const int n = (int)std::min<int64_t>(kHostTile, b - v0);
        for (int j = 0; j < n; ++j) acc[j] = Acc(0);
        for (int p = 0; p < n_planes; ++p) {
            const T* __restrict__ src = static_cast<const T*>(planes[p]) + v0;
            if constexpr (std::is_unsigned<T>::value) { for (int j = 0; j < n; ++j) acc[j] = (Acc)(acc[j] | src[j]); }
            else { for (int j = 0; j < n; ++j) acc[j] += (Acc)src[j]; }
        }
        for (int j = 0; j < n; ++j) out[v0 + j] = acc[j] > Acc(0) ? 1 : 0;
    }
}

template <typename T>
void label_range(const void* label, int64_t a, int64_t b, uint8_t* __restrict__ out) {      // mask[label == 0] = 0
    const T* __restrict__ l = static_cast<const T*>(label);
    for (int64_t v = a; v < b; ++v) out[v] = (l[v] == T(0)) ? 0 : out[v];
}

// the 0/1 mask of [a, b), eight voxels per step (a is a multiple of 64; whole-zero words -- most of a brain volume -- are skipped)
int64_t count_ones(const uint8_t* __restrict__ mask, int64_t a, int64_t b) {
    int64_t n = 0, v = a;
    for (; v + 8 <= b; v += 8) {
        uint64_t w;
        memcpy(&w, mask + v, 8);
        n += (int64_t)((w * 0x0101010101010101ull) >> 56);                     // bytes are 0 or 1: their sum lands in the top byte
    }
    for (; v < b; ++v) n += mask[v];
    return n;
}

void write_indices(const uint8_t* __restrict__ mask, int64_t a, int64_t b, int64_t* __restrict__ out) {
    int64_t v = a;
    for (; v + 8 <= b; v += 8) {
        uint64_t w;
        memcpy(&w, mask + v, 8);
        if (w == 0) continue;
        if (w == 0x0101010101010101ull) { for (int j = 0; j < 8; ++j) out[j] = v + j; out += 8; continue; }
        for (int j = 0; j < 8; ++j) if (mask[v + j]) *out++ = v + j;
    }
    for (; v < b; ++v) if (mask[v]) *out++ = v;
}

template <typename F>
bool by_dtype(int dtype, F&& f) {
    switch (dtype) {
        case T2FIT_DT_U8: f(uint8_t{}); return true;
        case T2FIT_DT_I16: f(int16_t{}); return true;
        case T2FIT_DT_U16: f(uint16_t{}); return true;
        case T2FIT_DT_I32: f(int32_t{}); return true;
        case T2FIT_DT_F32: f(float{}); return true;
        case T2FIT_DT_F64: f(double{}); return true;
        default: return false;
    }
}

}  // namespace

extern "C" {

int t2fit_abi_version(void) { return T2FIT_ABI_VERSION; }

const char* t2fit_last_error(void) { return tl_err.c_str(); }

int t2fit_init(int device) {
    std::lock_guard<std::mutex> g(g_mu);
    if (g_ctx) {
        if (g_ctx->device == device) return T2FIT_OK;
        return fail(T2FIT_EINVAL, "already initialised on another device (one process per GPU)");
    }
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0)
        return fail(T2FIT_ENODEVICE, std::string("no CUDA device: ") + cudaGetErrorString(e) +
                                         " (libt2fit has no CPU implementation of the fit)");
    if (device < 0 || device >= n) return fail(T2FIT_EINVAL, "device index out of range");
    CU_TRY(cudaSetDevice(device));
    Context* c = new Context();
    c->device = device;
    CU_TRY(cudaGetDeviceProperties(&c->prop, device));
    if (c->prop.major < 10)
        return fail(T2FIT_ENODEVICE, "libt2fit is built for sm_100a only; device is sm_" + std::to_string(c->prop.major) +
                                         std::to_string(c->prop.minor));
    CU_TRY(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    CU_TRY(cudaStreamCreateWithFlags(&c->fill_stream, cudaStreamNonBlocking));
    CU_TRY(cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming));
    CU_TRY(cudaEventCreateWithFlags(&c->ev_join, cudaEventDisableTiming));
    CU_TRY(cudaMalloc(&c->d_counts, 4 * sizeof(unsigned long long)));
    CU_TRY(cudaMemset(c->d_counts, 0, 4 * sizeof(unsigned long long)));
    CU_TRY(cudaMallocHost(&c->h_counts, 4 * sizeof(unsigned long long)));
    CU_TRY(cudaMalloc(&c->d_queue, kQueues * sizeof(unsigned long long)));
    CU_TRY(cudaMalloc(&c->d_total, sizeof(int64_t)));
    CU_TRY(cudaMallocHost(&c->h_total, sizeof(int64_t)));
    unsigned hw = std::thread::hardware_concurrency();
    const char* env = getenv("T2FIT_HOST_THREADS");
    int nt = env ? atoi(env) : (int)std::min(16u, hw ? hw : 4u);
    c->workers = new Workers(nt);
    g_ctx = c;
    return T2FIT_OK;
}

void t2fit_shutdown(void) {
    std::lock_guard<std::mutex> g(g_mu);
    Context* c = g_ctx;
    if (!c) return;
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();
    free_slots(c);
    for (auto& s : c->slots) {
        if (s.stream) cudaStreamDestroy(s.stream);
        if (s.done) cudaEventDestroy(s.done);
    }
    if (c->d_counts) cudaFree(c->d_counts);
    if (c->h_counts) cudaFreeHost(c->h_counts);
    if (c->d_tile_counts) cudaFree(c->d_tile_counts);
    if (c->d_tile_offsets) cudaFree(c->d_tile_offsets);
    if (c->d_queue) cudaFree(c->d_queue);
    if (c->d_total) cudaFree(c->d_total);
    if (c->d_idx) cudaFree(c->d_idx);
    if (c->h_total) cudaFreeHost(c->h_total);
    if (c->stream) cudaStreamDestroy(c->stream);
    if (c->fill_stream) cudaStreamDestroy(c->fill_stream);
    if (c->ev_fork) cudaEventDestroy(c->ev_fork);
    if (c->ev_join) cudaEventDestroy(c->ev_join);
    delete c->workers;
    delete c;
    g_ctx = nullptr;
}

int t2fit_device_info(char* name, int name_len, int* sm_count, int* cc_major, int* cc_minor) {
    if (!g_ctx) return fail(T2FIT_ENOTINIT, "t2fit_init() has not succeeded");
    if (name && name_len > 0) { strncpy(name, g_ctx->prop.name, name_len - 1); name[name_len - 1] = 0; }
    if (sm_count) *sm_count = g_ctx->prop.multiProcessorCount;
    if (cc_major) *cc_major = g_ctx->prop.major;
    if (cc_minor) *cc_minor = g_ctx->prop.minor;
    return T2FIT_OK;
}

int t2fit_run(const t2fit_problem* p, t2fit_outputs* o, void* stream) {
    Context* c = g_ctx;
    if (!c) return fail(T2FIT_ENOTINIT, "t2fit_init() has not succeeded (no CUDA device bound; there is no CPU fit)");
    if (!p || !o) return fail(T2FIT_EINVAL, "NULL problem/outputs");
    FitConsts fc;
    lb::LbConsts lc;
    memset(&fc, 0, sizeof(fc));
    memset(&lc, 0, sizeof(lc));
    std::string err;
    if (p->solver != T2FIT_SOLVER_FAST && p->solver != T2FIT_SOLVER_LBFGSB && p->solver != T2FIT_SOLVER_LBFGSB_DENSE)
        return fail(T2FIT_EINVAL, "unknown solver");
    const bool lbs = p->solver != T2FIT_SOLVER_FAST;
    if (!lbs && p->model == T2FIT_MODEL_RICIAN)
        return fail(T2FIT_EINVAL, "fit 'rician' (negative log-likelihood) needs solver T2FIT_SOLVER_LBFGSB");
    int rc = lbs ? make_lb_consts(*p, lc, err) : make_consts(*p, fc, err);
    if (rc) return fail(rc, err);
    const bool fill_only = p->n_fit == 0 && p->memory == T2FIT_MEM_DEVICE && o->dense && o->zero_fill_mask;
    if (p->n_fit == 0 && !fill_only) { memset(o->status_count, 0, sizeof(o->status_count)); return T2FIT_OK; }
    if (!p->echoes && !fill_only) return fail(T2FIT_EINVAL, "echoes is NULL");
    if (p->layout != T2FIT_LAYOUT_AOS && p->layout != T2FIT_LAYOUT_SOA && p->layout != T2FIT_LAYOUT_PLANES)
        return fail(T2FIT_EINVAL, "bad layout");
    if (p->layout == T2FIT_LAYOUT_SOA && p->ld < p->n_fit) return fail(T2FIT_EINVAL, "ld < n_fit");
    if (p->layout == T2FIT_LAYOUT_PLANES && p->ld < p->n_vox) return fail(T2FIT_EINVAL, "ld < n_vox");
    if (p->layout != T2FIT_LAYOUT_SOA && !p->mask_idx && p->n_fit > p->n_vox) return fail(T2FIT_EINVAL, "n_fit > n_vox");
    if (o->dense && !p->mask_idx && p->n_fit > p->n_vox) return fail(T2FIT_EINVAL, "dense output needs n_vox >= n_fit");
    const bool f32 = p->echo_dtype == 0 || p->echo_dtype == T2FIT_DT_F32;
    if (!f32 && p->echo_dtype != T2FIT_DT_I16 && p->echo_dtype != T2FIT_DT_U16 && p->echo_dtype != T2FIT_DT_I32 && p->echo_dtype != T2FIT_DT_F64)
        return fail(T2FIT_EINVAL, "bad echo_dtype");
    if (!f32 && p->memory != T2FIT_MEM_HOST) return fail(T2FIT_EINVAL, "device-memory echoes must be float32");
    CU_TRY(cudaSetDevice(c->device));
    if (p->memory == T2FIT_MEM_HOST && o->n_dup != 0) return fail(T2FIT_EINVAL, "the fused all-gather (dup_*) is for T2FIT_MEM_DEVICE calls");
    if (p->memory == T2FIT_MEM_HOST) return run_host(c, *p, *o, fc, lbs ? &lc : nullptr);
    if (p->memory != T2FIT_MEM_DEVICE) return fail(T2FIT_EINVAL, "bad memory kind");

    cudaStream_t st = (cudaStream_t)stream;   // NULL = the legacy default stream, as in CUDA
    KernelIO io{};
    io.echoes = p->echoes; io.ld = p->ld; io.n_fit = p->n_fit;
    if (p->idx_dtype == T2FIT_IDX_I32) io.idx32 = reinterpret_cast<const int32_t*>(p->mask_idx);
    else io.idx = p->mask_idx;
    // a caller-supplied index vector is range-checked by the kernels (entries outside [0, n_vox) are counted in slot 0 of
    // the counters and read / write voxel 0 instead): the reference's fancy indexing raises IndexError there
    if (p->mask_idx && p->layout != T2FIT_LAYOUT_SOA) io.n_rows = p->n_vox;
    io.t2 = o->t2; io.k = o->k; io.sigma = o->sigma; io.res = o->res; io.fun = o->fun; io.nit = o->nit;
    io.status = o->status; io.dense = o->dense;
    // status histogram of THIS call: the caller's own device counters, or the per-process ones (cleared first if an earlier
    // call left counts nobody asked for, so that they cannot leak into this call's t2fit_status_counts)
    if (o->counts_dev) io.counts = reinterpret_cast<unsigned long long*>(o->counts_dev);
    else {
        io.counts = c->d_counts;
        if (c->counts_dirty) CU_TRY(cudaMemsetAsync(c->d_counts, 0, 4 * sizeof(unsigned long long), st));
    }
    io.vec_ok = (reinterpret_cast<uintptr_t>(p->echoes) % 16) == 0;
    io.layout = p->layout;
    {   // T2FIT_PREFETCH_AHEAD: distance of the L2 prefetch in blocks (0 = off).  Default: 3/4 of the resident blocks -- c2 on
        // 148 SMs x 5 blocks: 63.4 us per pass without, 62.9 / 62.2 / 61.9 / 61.9 / 62.0 / 62.4 / 63.2 / 63.9 at 148 / 296 / 444 /
        // 592 / 740 / 888 / 1036 / 1184 blocks (profiles/r02_notes.md section 8)
        static const int env_ahead = [] { const char* e = getenv("T2FIT_PREFETCH_AHEAD"); return e ? atoi(e) : -1; }();
        const int resident = c->prop.multiProcessorCount * min_blocks(p->model == T2FIT_MODEL_GAUSSIAN ? kMono2 : kFloor3, p->n_echo);
        io.ahead = env_ahead >= 0 ? env_ahead : (3 * resident) / 4;
    }
    if (o->n_dup < 0 || o->n_dup > T2FIT_MAX_DUP) return fail(T2FIT_EINVAL, "n_dup out of range");
    if (o->n_dup > 0 && o->dense) return fail(T2FIT_EINVAL, "the fused all-gather (dup_*) takes compact outputs (dense = 0)");
    io.dup.n = o->n_dup;
    for (int j = 0; j < o->n_dup; ++j) {
        io.dup.t2[j] = o->dup_t2[j]; io.dup.k[j] = o->dup_k[j]; io.dup.res[j] = o->dup_res[j]; io.dup.status[j] = o->dup_status[j];
        io.dup.sigma[j] = p->model == T2FIT_MODEL_GAUSSIAN ? nullptr : o->dup_sigma[j];
    }
    if (lbs && o->trace_cap > 0) {
        io.trace_f = o->trace_f; io.trace_step = o->trace_step; io.trace_len = o->trace_len; io.trace_cap = o->trace_cap;
    }
    bool forked = false;
    if (!o->counts_dev) c->counts_dirty = true;
    if (o->dense && o->zero_fill_mask) {
        // np.zeros_like x4 (:415-418): inside the fit launch (every fit thread zeroes a few words of the maps while it
        // waits for its echoes) or, where that does not apply, by zero_fill_kernel on the side stream (disjoint slots)
        if ((reinterpret_cast<uintptr_t>(o->zero_fill_mask) % 4) != 0)
            return fail(T2FIT_EINVAL, "zero_fill_mask must be 4-byte aligned");
        FillArgs fa{};
        fa.t2 = o->t2; fa.k = o->k; fa.res = o->res; fa.sigma = o->sigma;
        fa.mask = o->zero_fill_mask; fa.n_vox = p->n_vox; fa.vec = 1;
        float* mp[4] = {o->t2, o->k, o->sigma, o->res};
        for (float* q : mp) if (q && (reinterpret_cast<uintptr_t>(q) % 16) != 0) fa.vec = 0;
        const char* env_fill = getenv("T2FIT_FILL");      // fused (default) | stream; read per call (tests switch it)
        const bool want_fused = !lbs && p->model == T2FIT_MODEL_GAUSSIAN && p->n_fit > 0 && !(env_fill && !strcmp(env_fill, "stream"));
        if (want_fused && fused_fill_wpb(fa, p->n_fit, p->layout) > 0)
            return launch_fit(c, fc, io, p->model, p->n_echo, p->layout, st, &fa);
        rc = launch_zero_fill(c, fa, p->model == T2FIT_MODEL_GAUSSIAN, st, &forked);
        if (rc) return rc;
    }
    rc = lbs ? launch_lbfgsb(c, lc, io, p->model, p->n_echo, st) : launch_fit(c, fc, io, p->model, p->n_echo, p->layout, st);
    if (forked) CU_TRY(cudaStreamWaitEvent(st, c->ev_join, 0));           // join: results complete on `st`
    return rc;
}

int t2fit_status_counts(void* stream, int64_t counts[4]) {
    Context* c = g_ctx;
    if (!c) return fail(T2FIT_ENOTINIT, "t2fit_init() has not succeeded");
    if (!counts) return fail(T2FIT_EINVAL, "NULL counts");
    cudaStream_t st = (cudaStream_t)stream;   // NULL = the legacy default stream, as in CUDA
    CU_TRY(cudaMemcpyAsync(c->h_counts, c->d_counts, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaStreamSynchronize(st));
    for (int s = 0; s < 4; ++s) counts[s] = (int64_t)c->h_counts[s];   // slot 0: mask_idx entries out of range (IndexError upstream)
    CU_TRY(cudaMemsetAsync(c->d_counts, 0, 4 * sizeof(unsigned long long), st));   // counts are "since the last query"
    CU_TRY(cudaStreamSynchronize(st));
    c->counts_dirty = false;
    return T2FIT_OK;
}

int t2fit_mask_indices(const uint8_t* masks, int64_t n_vox, int32_t n_masks, int64_t* idx_out, int64_t* n_out, void* stream) {
    Context* c = g_ctx;
    if (!c) return fail(T2FIT_ENOTINIT, "t2fit_init() has not succeeded");
    if (!masks || !idx_out || !n_out || n_vox < 0 || n_masks < 1) return fail(T2FIT_EINVAL, "bad mask arguments");
    if (n_vox == 0) { *n_out = 0; return T2FIT_OK; }
    CU_TRY(cudaSetDevice(c->device));
    cudaStream_t st = (cudaStream_t)stream;   // NULL = the legacy default stream, as in CUDA
    const int64_t tiles = (n_vox + kMaskTile - 1) / kMaskTile;
    if (tiles > 0x7fffffffLL) return fail(T2FIT_EINVAL, "volume too large");
    if (tiles > c->tiles_cap) {
        CU_TRY(cudaStreamSynchronize(st));
        if (c->d_tile_counts) cudaFree(c->d_tile_counts);
        if (c->d_tile_offsets) cudaFree(c->d_tile_offsets);
        c->d_tile_counts = nullptr; c->d_tile_offsets = nullptr; c->tiles_cap = 0;
        CU_TRY(cudaMalloc(&c->d_tile_counts, sizeof(int) * tiles));
        CU_TRY(cudaMalloc(&c->d_tile_offsets, sizeof(int64_t) * tiles));
        c->tiles_cap = tiles;
    }
    mask_count_kernel<<<(unsigned)tiles, 256, 0, st>>>(masks, n_vox, n_masks, c->d_tile_counts);
    mask_scan_kernel<<<1, 1024, 0, st>>>(c->d_tile_counts, c->d_tile_offsets, (int)tiles, c->d_total);
    mask_write_kernel<<<(unsigned)tiles, 256, 0, st>>>(masks, n_vox, n_masks, c->d_tile_offsets, idx_out);
    CU_TRY(cudaGetLastError());
    CU_TRY(cudaMemcpyAsync(c->h_total, c->d_total, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaStreamSynchronize(st));
    *n_out = *c->h_total;
    return T2FIT_OK;
}

int t2fit_mask_union(const void* const* planes, int32_t n_planes, int32_t dtype, const void* label, int32_t label_dtype,
                     int64_t n_vox, uint8_t* mask_out, void* stream) {
    Context* c = g_ctx;
    if (!c) return fail(T2FIT_ENOTINIT, "t2fit_init() has not succeeded");
    if (!planes || n_planes < 1 || n_planes > kMaxEcho || !mask_out || n_vox < 0) return fail(T2FIT_EINVAL, "bad mask_union arguments");
    if (dtype < T2FIT_DT_U8 || dtype > T2FIT_DT_F64 || (label && (label_dtype < T2FIT_DT_U8 || label_dtype > T2FIT_DT_F64)))
        return fail(T2FIT_EINVAL, "bad dtype code");
    if (n_vox == 0) return T2FIT_OK;
    CU_TRY(cudaSetDevice(c->device));
    UnionArgs a{};
    for (int p = 0; p < n_planes; ++p) { if (!planes[p]) return fail(T2FIT_EINVAL, "NULL mask plane"); a.planes[p] = planes[p]; }
    a.label = label; a.n_planes = n_planes; a.dtype = dtype; a.label_dtype = label_dtype; a.n_vox = n_vox;
    const int64_t want = (n_vox + 255) / 256;
    const unsigned grid = (unsigned)std::min<int64_t>(want, (int64_t)c->prop.multiProcessorCount * 16);
    mask_union_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(a, mask_out);
    CU_TRY(cudaGetLastError());
    return T2FIT_OK;
}

int t2fit_host_mask_union_indices(const void* const* masks, int32_t n_masks, int32_t mask_dtype, const void* label,
                                  int32_t label_dtype, int64_t n_vox, uint8_t* mask_out, int64_t* idx_out, int64_t* n_out) {
    if (!masks || n_masks < 1 || n_masks > kMaxEcho || !mask_out || !idx_out || !n_out || n_vox < 0)
        return fail(T2FIT_EINVAL, "bad host_mask_union_indices arguments");
    if (mask_dtype < T2FIT_DT_U8 || mask_dtype > T2FIT_DT_F64 || (label && (label_dtype < T2FIT_DT_U8 || label_dtype > T2FIT_DT_F64)))
        return fail(T2FIT_EINVAL, "bad dtype code");
    for (int p = 0; p < n_masks; ++p) if (!masks[p]) return fail(T2FIT_EINVAL, "NULL mask plane");
    *n_out = 0;
    if (n_vox == 0) return T2FIT_OK;
    std::lock_guard<std::mutex> g(g_host_mu);
    Workers& w = host_workers();
    const int parts = w.size();
    std::vector<int64_t> count(parts + 1, 0);
    const int64_t per = ((n_vox + parts - 1) / parts + 63) & ~(int64_t)63;
    const bool prof = getenv("T2FIT_HOST_PROFILE") != nullptr;
    const double t0 = prof ? now_ms() : 0.0;
    w.run([&](int part, int) {                                                 // union (+ label) and the count of every range
        const int64_t a = std::min<int64_t>(n_vox, part * per), b = std::min<int64_t>(n_vox, a + per);
        if (a >= b) return;
        by_dtype(mask_dtype, [&](auto t) { union_range<decltype(t)>(masks, n_masks, a, b, mask_out); });
        if (label) by_dtype(label_dtype, [&](auto t) { label_range<decltype(t)>(label, a, b, mask_out); });
        count[part + 1] = count_ones(mask_out, a, b);
    });
    for (int q = 0; q < parts; ++q) count[q + 1] += count[q];
    const double t1 = prof ? now_ms() : 0.0;
    w.run([&](int part, int) {                                                 // np.where(mask.flatten())[0], ascending
        const int64_t a = std::min<int64_t>(n_vox, part * per), b = std::min<int64_t>(n_vox, a + per);
        if (a < b) write_indices(mask_out, a, b, idx_out + count[part]);
    });
    *n_out = count[parts];
    if (prof) fprintf(stderr, "[t2fit] host_mask_union_indices: %d threads, union + count %.3f ms, indices %.3f ms\n", parts, t1 - t0, now_ms() - t1);
    return T2FIT_OK;
}

int t2fit_host_gather_planes(const void* const* planes, int32_t n_planes, int32_t dtype, const int64_t* idx, int64_t n_fit,
                             int64_t n_vox, float* soa_out, int64_t ld) {
    if (!planes || n_planes < 1 || n_planes > kMaxEcho || n_fit < 0 || n_vox < 0 || (n_fit > 0 && (!idx || !soa_out)) || ld < n_fit)
        return fail(T2FIT_EINVAL, "bad host_gather_planes arguments");
    if (dtype < T2FIT_DT_U8 || dtype > T2FIT_DT_F64) return fail(T2FIT_EINVAL, "bad dtype code");
    for (int p = 0; p < n_planes; ++p) if (!planes[p]) return fail(T2FIT_EINVAL, "NULL plane");
    if (n_fit == 0) return T2FIT_OK;
    std::lock_guard<std::mutex> g(g_host_mu);
    Workers& w = host_workers();
    const int parts = w.size();
    const int64_t per = ((n_fit + parts - 1) / parts + 63) & ~(int64_t)63;
    std::atomic<int> bad{0};
    w.run([&](int part, int) {
        const int64_t a = std::min<int64_t>(n_fit, part * per), b = std::min<int64_t>(n_fit, a + per);
        for (int64_t j = a; j < b; ++j) if (idx[j] < 0 || idx[j] >= n_vox) { bad.store(1); return; }
        by_dtype(dtype, [&](auto t) {
            using T = decltype(t);
            const int64_t* __restrict__ ix = idx;
            for (int p = 0; p < n_planes; ++p) {                               // .astype(np.float32) of the rows the fit reads
                const T* __restrict__ src = static_cast<const T*>(planes[p]);
                float* __restrict__ dst = soa_out + (int64_t)p * ld;
                int64_t j = a;
                for (; j + 8 <= b; j += 8) {                                   // masked voxels come in runs along x: 8 in a row
                    const int64_t v = ix[j];
                    __builtin_prefetch(src + ix[std::min<int64_t>(j + 256, b - 1)]);       // the next runs' first lines
                    if (ix[j + 7] - v == 7) { for (int q = 0; q < 8; ++q) dst[j + q] = (float)src[v + q]; }
                    else { for (int q = 0; q < 8; ++q) dst[j + q] = (float)src[ix[j + q]]; }
                }
                for (; j < b; ++j) dst[j] = (float)src[ix[j]];
            }
        });
    });
    if (bad.load()) return fail(T2FIT_EINVAL, "host_gather_planes: index outside [0, n_vox)");
    return T2FIT_OK;
}

int t2fit_roi_stats(const float* const* maps, int32_t n_maps, const int32_t* label, int64_t n_vox, int32_t n_roi, double* mean_out,
                    double* std_out, int64_t* count_out, void* stream) {
    Context* c = g_ctx;
    if (!c) return fail(T2FIT_ENOTINIT, "t2fit_init() has not succeeded");
    if (!maps || !label || n_maps < 1 || n_maps > kMaxStatMaps || n_roi < 1 || n_roi > kMaxRoi || n_vox < 0 || !mean_out || !std_out)
        return fail(T2FIT_EINVAL, "bad roi_stats arguments (n_maps <= 4, n_roi <= 64)");
    CU_TRY(cudaSetDevice(c->device));
    cudaStream_t st = (cudaStream_t)stream;
    const int slots = n_maps * n_roi;
    double *d_sum = nullptr, *d_mean = nullptr;
    unsigned long long* d_cnt = nullptr;
    CU_TRY(cudaMalloc(&d_sum, sizeof(double) * slots * 2));
    d_mean = d_sum + slots;
    if (cudaMalloc(&d_cnt, sizeof(unsigned long long) * slots) != cudaSuccess) { cudaFree(d_sum); return fail(T2FIT_ENOMEM, "roi_stats scratch"); }
    std::vector<double> h_sum(slots), h_mean(slots), h_sq(slots);
    std::vector<unsigned long long> h_cnt(slots);
    RoiArgs a{};
    for (int m = 0; m < n_maps; ++m) a.maps[m] = maps[m];
    a.label = label; a.n_vox = n_vox; a.n_maps = n_maps; a.n_roi = n_roi;
    const int64_t want = (n_vox + 255) / 256;
    const unsigned grid = (unsigned)std::max<int64_t>(1, std::min<int64_t>(want, (int64_t)c->prop.multiProcessorCount * 8));
    auto cleanup = [&]() { cudaFree(d_sum); cudaFree(d_cnt); };
    cudaError_t e = cudaMemsetAsync(d_sum, 0, sizeof(double) * slots * 2, st);
    if (e == cudaSuccess) e = cudaMemsetAsync(d_cnt, 0, sizeof(unsigned long long) * slots, st);
    a.pass = 0;
    if (e == cudaSuccess) { roi_stats_kernel<<<grid, 256, 0, st>>>(a, d_sum, d_cnt, d_mean); e = cudaGetLastError(); }
    if (e == cudaSuccess) e = cudaMemcpyAsync(h_sum.data(), d_sum, sizeof(double) * slots, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(h_cnt.data(), d_cnt, sizeof(unsigned long long) * slots, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) { cleanup(); return fail(T2FIT_ECUDA, std::string("roi_stats pass 0: ") + cudaGetErrorString(e)); }
    for (int i = 0; i < slots; ++i) h_mean[i] = h_cnt[i] ? h_sum[i] / (double)h_cnt[i] : NAN;
    e = cudaMemcpyAsync(d_mean, h_mean.data(), sizeof(double) * slots, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaMemsetAsync(d_sum, 0, sizeof(double) * slots, st);
    a.pass = 1;
    if (e == cudaSuccess) { roi_stats_kernel<<<grid, 256, 0, st>>>(a, d_sum, d_cnt, d_mean); e = cudaGetLastError(); }
    if (e == cudaSuccess) e = cudaMemcpyAsync(h_sq.data(), d_sum, sizeof(double) * slots, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    cleanup();
    if (e != cudaSuccess) return fail(T2FIT_ECUDA, std::string("roi_stats pass 1: ") + cudaGetErrorString(e));
    for (int i = 0; i < slots; ++i) {
        mean_out[i] = h_mean[i];
        std_out[i] = h_cnt[i] ? sqrt(h_sq[i] / (double)h_cnt[i]) : NAN;
        if (count_out) count_out[i] = (int64_t)h_cnt[i];
    }
    return T2FIT_OK;
}

int t2fit_shared_alloc(int64_t bytes, void** dev_ptr, unsigned char handle[T2FIT_IPC_HANDLE_BYTES]) {
    Context* c = g_ctx;
    if (!c) return fail(T2FIT_ENOTINIT, "t2fit_init() has not succeeded");
    if (bytes <= 0 || !dev_ptr || !handle) return fail(T2FIT_EINVAL, "bad shared_alloc arguments");
    static_assert(sizeof(cudaIpcMemHandle_t) == T2FIT_IPC_HANDLE_BYTES, "IPC handle size");
    CU_TRY(cudaSetDevice(c->device));
    void* p = nullptr;
    CU_TRY(cudaMalloc(&p, (size_t)bytes));
    cudaIpcMemHandle_t h;
    cudaError_t e = cudaIpcGetMemHandle(&h, p);
    if (e != cudaSuccess) { cudaFree(p); return fail(T2FIT_ECUDA, std::string("cudaIpcGetMemHandle: ") + cudaGetErrorString(e)); }
    memcpy(handle, &h, sizeof(h));
    *dev_ptr = p;
    return T2FIT_OK;
}

int t2fit_shared_free(void* dev_ptr) {
    if (!g_ctx) return fail(T2FIT_ENOTINIT, "t2fit_init() has not succeeded");
    if (dev_ptr) CU_TRY(cudaFree(dev_ptr));
    return T2FIT_OK;
}

int t2fit_shared_open(const unsigned char handle[T2FIT_IPC_HANDLE_BYTES], void** dev_ptr) {
    Context* c = g_ctx;
    if (!c) return fail(T2FIT_ENOTINIT, "t2fit_init() has not succeeded");
    if (!handle || !dev_ptr) return fail(T2FIT_EINVAL, "bad shared_open arguments");
    CU_TRY(cudaSetDevice(c->device));
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, sizeof(h));
    CU_TRY(cudaIpcOpenMemHandle(dev_ptr, h, cudaIpcMemLazyEnablePeerAccess));     // maps the peer GPU's memory (NVLink)
    return T2FIT_OK;
}

int t2fit_shared_close(void* dev_ptr) {
    if (!g_ctx) return fail(T2FIT_ENOTINIT, "t2fit_init() has not succeeded");
    if (dev_ptr) CU_TRY(cudaIpcCloseMemHandle(dev_ptr));
    return T2FIT_OK;
}

int t2fit_pack_soa(const float* aos, int64_t n_vox, int32_t n_echo, const int64_t* mask_idx, int64_t n_fit, float* soa,
                   int64_t ld, void* stream) {
    Context* c = g_ctx;
    if (!c) return fail(T2FIT_ENOTINIT, "t2fit_init() has not succeeded");
    if (!aos || !soa || n_echo < 1 || ld < n_fit || n_fit < 0 || n_vox < 0) return fail(T2FIT_EINVAL, "bad pack arguments");
    if (n_fit == 0) return T2FIT_OK;
    CU_TRY(cudaSetDevice(c->device));
    cudaStream_t st = (cudaStream_t)stream;   // NULL = the legacy default stream, as in CUDA
    pack_soa_kernel<<<(unsigned)((n_fit + 255) / 256), 256, 0, st>>>(aos, n_echo, mask_idx, n_fit, soa, ld);
    CU_TRY(cudaGetLastError());
    return T2FIT_OK;
}

int t2fit_scatter(const float* const* compact, float* const* dense, int32_t n_maps, const int64_t* mask_idx, int64_t n_fit,
                  void* stream) {
    Context* c = g_ctx;
    if (!c) return fail(T2FIT_ENOTINIT, "t2fit_init() has not succeeded");
    if (!compact || !dense || !mask_idx || n_maps < 1 || n_maps > 4 || n_fit < 0) return fail(T2FIT_EINVAL, "bad scatter arguments");
    if (n_fit == 0) return T2FIT_OK;
    CU_TRY(cudaSetDevice(c->device));
    cudaStream_t st = (cudaStream_t)stream;   // NULL = the legacy default stream, as in CUDA
    ScatterArgs a{};
    a.n_maps = n_maps;
    for (int m = 0; m < n_maps; ++m) { a.src[m] = compact[m]; a.dst[m] = dense[m]; }
    scatter_kernel<<<(unsigned)((n_fit + 255) / 256), 256, 0, st>>>(a, mask_idx, n_fit);
    CU_TRY(cudaGetLastError());
    return T2FIT_OK;
}

int t2fit_residuals(const t2fit_problem* p, const float* k_map, const float* t2_map, const float* sigma_map, float* res_map,
                    void* stream) {
    Context* c = g_ctx;
    if (!c) return fail(T2FIT_ENOTINIT, "t2fit_init() has not succeeded");
    if (!p || !k_map || !t2_map || !res_map || !p->echoes) return fail(T2FIT_EINVAL, "NULL argument");
    if (p->memory != T2FIT_MEM_DEVICE || p->layout != T2FIT_LAYOUT_AOS) return fail(T2FIT_EINVAL, "device AOS input only");
    FitConsts fc;
    memset(&fc, 0, sizeof(fc));
    std::string err;
    t2fit_problem q = *p;                     // 'rician' maps are evaluated with the noise-floor model, as the reference
    if (q.model == T2FIT_MODEL_RICIAN) q.model = T2FIT_MODEL_GAUSSIAN_RICIAN;   // does (utils/t2map_utils.py:68-71)
    int rc = make_consts(q, fc, err);
    if (rc) return fail(rc, err);
    if (p->n_fit == 0) return T2FIT_OK;
    CU_TRY(cudaSetDevice(c->device));
    cudaStream_t st = (cudaStream_t)stream;   // NULL = the legacy default stream, as in CUDA
    residual_kernel<<<(unsigned)((p->n_fit + 255) / 256), 256, 0, st>>>(fc, p->echoes, p->mask_idx, p->n_fit, q.model, k_map,
                                                                       t2_map, sigma_map, res_map);
    CU_TRY(cudaGetLastError());
    return T2FIT_OK;
}

int t2fit_stderr(const t2fit_problem* p, const float* k, const float* t2, const float* sigma, int32_t dense, float* se_k,
                 float* se_t2, float* se_sigma, void* stream) {
    Context* c = g_ctx;
    if (!c) return fail(T2FIT_ENOTINIT, "t2fit_init() has not succeeded");
    if (int rc = check_pass_problem(p, "t2fit_stderr")) return rc;
    if (p->n_fit == 0) return T2FIT_OK;
    if (!p->echoes || !k || !t2 || (p->model != T2FIT_MODEL_GAUSSIAN && !sigma)) return fail(T2FIT_EINVAL, "NULL echoes / parameters");
    StderrArgs a{};
    if (int rc = pass_input(p, dense, a.in)) return rc;
    a.k = k; a.t2 = t2; a.sigma = sigma;
    a.se_k = se_k; a.se_t2 = se_t2; a.se_sigma = se_sigma;
    const StderrFn fn = pick_stderr(p->model, p->n_echo);
    CU_TRY(cudaSetDevice(c->device));
    fn<<<(unsigned)((p->n_fit + 255) / 256), 256, 0, (cudaStream_t)stream>>>(a);
    CU_TRY(cudaGetLastError());
    return T2FIT_OK;
}

int t2fit_t2_interval(const t2fit_problem* p, double q, int32_t n_grid, int32_t dense, float* t2_lo, float* t2_hi,
                      float* t2_best, uint8_t* flags, double* profile, void* stream) {
    Context* c = g_ctx;
    if (!c) return fail(T2FIT_ENOTINIT, "t2fit_init() has not succeeded");
    if (int rc = check_pass_problem(p, "t2fit_t2_interval")) return rc;
    if (n_grid < iv::kMinGrid || n_grid > iv::kMaxGrid) return fail(T2FIT_EINVAL, "n_grid out of range (16..256)");
    if (!(q >= 0.0) || !(q - q == 0.0)) return fail(T2FIT_EINVAL, "q must be finite and >= 0");
    iv::Box b{p->lb[0], p->ub[0], p->lb[1], p->ub[1], p->lb[2], p->ub[2]};
    if (p->no_prior) { b.k_hi = p->no_prior_k_ub; b.t_lo = p->no_prior_t2_lb; b.t_hi = p->no_prior_t2_ub; }
    if (!(b.t_lo > 0.0) || !(b.t_lo < b.t_hi) || !(b.t_hi - b.t_hi == 0.0))
        return fail(T2FIT_EINVAL, "the T2 bounds must be finite with 0 < lb < ub");
    if (p->model == T2FIT_MODEL_GAUSSIAN) b.s_lo = b.s_hi = 1.0;
    else if (!(b.s_lo > 0.0)) return fail(T2FIT_EINVAL, "the sigma lower bound must be > 0");
    if (p->n_fit == 0) return T2FIT_OK;
    if (!p->echoes) return fail(T2FIT_EINVAL, "NULL echoes");
    IntervalArgs a{};
    if (int rc = pass_input(p, dense, a.in)) return rc;
    a.box = b;
    a.q = q;
    a.lo = t2_lo; a.hi = t2_hi; a.best = t2_best; a.flags = flags; a.profile = profile;
    a.model = p->model; a.n_grid = n_grid; a.no_prior = p->no_prior != 0;
    const IntervalFn fn = pick_interval(p->n_echo);
    CU_TRY(cudaSetDevice(c->device));
    fn<<<(unsigned)((p->n_fit + 127) / 128), 128, 0, (cudaStream_t)stream>>>(a);
    CU_TRY(cudaGetLastError());
    return T2FIT_OK;
}

int t2fit_bootstrap_replicates(const t2fit_problem* p, const float* k, const float* t2, const float* sigma,
                               const float* noise_sd, const int64_t* voxel_id, uint64_t seed, int32_t n_rep, float* rows,
                               void* stream) {
    Context* c = g_ctx;
    if (!c) return fail(T2FIT_ENOTINIT, "t2fit_init() has not succeeded");
    if (int rc = check_pass_problem(p, "t2fit_bootstrap_replicates")) return rc;
    if (n_rep < bs::kMinRep || n_rep > bs::kMaxRep) return fail(T2FIT_EINVAL, "n_rep out of range (16..4096)");
    if (p->n_fit == 0) return T2FIT_OK;
    if (!p->echoes || !k || !t2 || (p->model != T2FIT_MODEL_GAUSSIAN && !sigma) || !rows)
        return fail(T2FIT_EINVAL, "NULL echoes / parameters / rows");
    if (p->n_fit > INT64_MAX / n_rep) return fail(T2FIT_EINVAL, "n_fit * n_rep overflows");
    ReplicateArgs a{};
    if (int rc = pass_input(p, 0, a.in)) return rc;
    a.k = k; a.t2 = t2; a.sigma = sigma; a.noise_sd = noise_sd; a.voxel_id = voxel_id;
    a.seed = seed; a.rows = rows; a.n_rep = n_rep; a.model = p->model;
    const ReplicateFn fn = pick_replicate(p->n_echo);
    const int64_t n = p->n_fit * n_rep;
    if ((n + 127) / 128 > INT32_MAX) return fail(T2FIT_EINVAL, "n_fit * n_rep too large for one launch");
    CU_TRY(cudaSetDevice(c->device));
    fn<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(a);
    CU_TRY(cudaGetLastError());
    return T2FIT_OK;
}

int t2fit_bootstrap_stats(int32_t model, int64_t n_fit, int32_t n_rep, const float* rep_k, const float* rep_t2,
                          const float* rep_sigma, const uint8_t* rep_status, double level, float* mean, float* sd,
                          float* t2_lo, float* t2_hi, int32_t* n_used, int32_t* n_ok, void* stream) {
    Context* c = g_ctx;
    if (!c) return fail(T2FIT_ENOTINIT, "t2fit_init() has not succeeded");
    if (model != T2FIT_MODEL_GAUSSIAN && model != T2FIT_MODEL_GAUSSIAN_RICIAN && model != T2FIT_MODEL_RICIAN)
        return fail(T2FIT_EINVAL, "unknown model");
    if (n_fit < 0) return fail(T2FIT_EINVAL, "negative size");
    if (n_rep < bs::kMinRep || n_rep > bs::kMaxRep) return fail(T2FIT_EINVAL, "n_rep out of range (16..4096)");
    if (!(level > 0.0 && level < 1.0)) return fail(T2FIT_EINVAL, "level must lie in (0, 1)");
    if (n_fit == 0) return T2FIT_OK;
    if (!rep_k || !rep_t2 || !rep_status || (model != T2FIT_MODEL_GAUSSIAN && !rep_sigma))
        return fail(T2FIT_EINVAL, "NULL replicate results");
    if (n_fit > INT32_MAX) return fail(T2FIT_EINVAL, "n_fit too large for one launch");
    BootstrapStatsArgs a{};
    a.k = rep_k; a.t2 = rep_t2; a.sigma = rep_sigma; a.status = rep_status;
    a.mean = mean; a.sd = sd; a.lo = t2_lo; a.hi = t2_hi; a.n_used = n_used; a.n_ok = n_ok;
    a.n_fit = n_fit;
    a.q_lo = 0.5 * (1.0 - level);
    a.q_hi = 0.5 * (1.0 + level);
    a.n_rep = n_rep;
    a.n_pad = 1;
    while (a.n_pad < n_rep) a.n_pad *= 2;
    a.model = model;
    CU_TRY(cudaSetDevice(c->device));
    bootstrap_stats_kernel<<<(unsigned)n_fit, bs::kStatThreads, a.n_pad * sizeof(float), (cudaStream_t)stream>>>(a);
    CU_TRY(cudaGetLastError());
    return T2FIT_OK;
}

int t2fit_work_model(int32_t model, int32_t n_echo, double* flop_per_pass, double* mufu_per_pass, double* flop_fixed,
                     double* mufu_fixed, double* bytes_per_voxel) {
    if (n_echo < 1) return fail(T2FIT_EINVAL, "bad n_echo");
    const double E = n_echo;
    // counts of the shipped device code (t2fit_core.cuh), FMA = 2 FLOP; see DESIGN.md "work model"
    if (model == T2FIT_MODEL_GAUSSIAN) {
        if (flop_per_pass) *flop_per_pass = 12.0 * E + 48.0;   // echo loop: 2 FMUL + 5 FFMA; solve/bracket ~48
        if (mufu_per_pass) *mufu_per_pass = E + 4.0;           // EX2 per echo; RCP + divides in the solve
        if (flop_fixed) *flop_fixed = (10.0 * E + 16.0) + (7.0 * E + 8.0);  // log-linear init + residual epilogue
        if (mufu_fixed) *mufu_fixed = 2.0 * E + 4.0;           // LG2 per echo (init) + EX2 per echo (epilogue)
        if (bytes_per_voxel) *bytes_per_voxel = 4.0 * E + 4.0 * 3 + 1;      // echoes in; t2,k,res + status out
    } else if (model == T2FIT_MODEL_GAUSSIAN_RICIAN) {
        if (flop_per_pass) *flop_per_pass = 33.0 * E + 110.0;  // echo loop: 13 mul/add + 10 FFMA; 3x3 solve ~110
        if (mufu_per_pass) *mufu_per_pass = 2.0 * E + 5.0;     // EX2 + RSQ per echo; 3 RSQ + RCP in the solve
        if (flop_fixed) *flop_fixed = (10.0 * E + 16.0) + (12.0 * E + 5.0) + (11.0 * E + 8.0);
        if (mufu_fixed) *mufu_fixed = 4.0 * E + 4.0;
        if (bytes_per_voxel) *bytes_per_voxel = 4.0 * E + 4.0 * 4 + 1;
    } else {
        return fail(T2FIT_EINVAL, "unknown model");
    }
    return T2FIT_OK;
}

}  // extern "C"
