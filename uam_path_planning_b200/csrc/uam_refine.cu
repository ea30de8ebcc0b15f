// Batched refinement of candidate paths by descent on the raster cost (uam_refine_paths_raster; the rule is in the
// header comment of its declaration in include/uam_b200.h).  SURVEY 8f item 1: the local step after scoring, here a
// monotone per-path step-controlled descent, not the reference's OpEn / PANOC solver.
//
// One trip = one gradient launch of the raster scorer on the whole trial batch (uam_raster_grad_enqueue: same B, so
// the same kernels and bits as uam_grad_paths_raster) + one uam_k_refine_step, which takes or drops the trial just
// evaluated and writes the next one.  The loop is stream-ordered: no host synchronisation or read-back per trip, and
// every path is evaluated on every trip (a path's bits do not depend on the rest of the batch, and the kernel choice
// stays the one of the call's B).
//
// uam_refine_paths_raster_swept adds one uam_k_sweep_paths launch of the trial batch per trip (uam_sweep_enqueue) and
// the swept terms of the accept test (UAM_REFINE_SWEPT); everything else is the same loop.
// uam_refine_paths_raster_keepout adds one launch of the analytic sweep, or with a margin of the analytic clearance, of
// the trial batch per trip (uam_sweep_analytic_enqueue / uam_clearance_analytic_enqueue) and its terms of the accept
// test (UAM_REFINE_KEEPOUT).
#include <algorithm>
#include <cmath>

#include "uam_internal.cuh"

namespace {

// what a launch of uam_k_refine_step does
enum : int {
    UAM_REFINE_START = 1,      // tau = step_cells, accepted = 0 (first launch, after the gradient of Z)
    UAM_REFINE_ACCEPT = 2,     // take or drop the trial in zt, evaluated into (ct, kt, gt)
    UAM_REFINE_PROPOSE = 4,    // write the next trial into zt and whether it moved the path into active
    UAM_REFINE_SWEPT = 8,      // the accept test also needs the trial's swept flags (ft) and clearance (d2t)
    UAM_REFINE_KEEPOUT = 16,   // ... the trial's analytic sweep flags (ft) and clearance (clt)
};

struct UamRefineState {
    double2* z;               // (B, Wp) the caller's paths, refined in place
    double2* g;               // (B, Wp) gradient at z (free waypoints only are kept up to date)
    double2* zt;              // (B, Wp) trial
    const double2* gt;        // (B, Wp) gradient at zt
    float* c;                 // cost / collide at z: the caller's outputs
    uint8_t* k;
    const float* ct;          // cost / collide at zt
    const uint8_t* kt;
    double* tau;              // step, in cells
    uint8_t* active;          // the trial in zt is a proposed move (not a copy of z)
    int32_t* accepted;
    long long B;
    int Wp;
    double h;                 // cell size: min(|dx|, |dy|)
    double step, max_step, min_step;
    // UAM_REFINE_SWEPT: swept flags and clearance at z (the caller's outputs or scratch) and at zt; d2 / d2t are NULL
    // when no clearance is computed, min_d2 > 0 only with them
    uint8_t* f;
    const uint8_t* ft;
    int32_t* d2;
    const int32_t* d2t;
    int min_d2;
    // UAM_REFINE_KEEPOUT: f / ft hold the analytic sweep's flags; the analytic clearance capped at the margin at z (the
    // caller's output or scratch) and at zt, both NULL with margin 0
    double* cl;
    const double* clt;
};

__device__ __forceinline__ double uam_warp_max(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// Warp per path, lanes stride the waypoints (16 B each).  Waypoints 0 and Wp-1 (start and goal) are never written
// into z.  The proposal is fp64 with explicit rounded operations: nvcc would otherwise contract z - r g into an FMA.
template <int MODE>
__global__ void __launch_bounds__(UAM_CTA_THREADS) uam_k_refine_step(const UamRefineState s) {
    const int lane = threadIdx.x & 31;
    const long long nwarps = (long long)gridDim.x * UAM_WARPS_PER_CTA;
    for (long long b = (long long)blockIdx.x * UAM_WARPS_PER_CTA + (threadIdx.x >> 5); b < s.B; b += nwarps) {
        const size_t row = (size_t)b * s.Wp;
        double tau = (MODE & UAM_REFINE_START) ? s.step : s.tau[b];
        float c = s.c[b];
        bool take = false, was_active = false;
        float ct = 0.0f;
        uint8_t kt = 0;
        if (MODE & UAM_REFINE_ACCEPT) {
            was_active = s.active[b] != 0;
            ct = s.ct[b];
            kt = s.kt[b];
            take = was_active && kt <= s.k[b] && ct < c;
        }
        uint8_t ft = 0;
        int d2t = 0;
        if (MODE & UAM_REFINE_SWEPT) {
            ft = s.ft[b];
            take = take && (ft & ~s.f[b]) == 0;
            if (s.d2) {
                d2t = s.d2t[b];
                take = take && (s.min_d2 == 0 || min(d2t, s.min_d2) >= min(s.d2[b], s.min_d2));
            }
        }
        double clt = 0.0;
        if (MODE & UAM_REFINE_KEEPOUT) {
            ft = s.ft[b];
            take = take && (ft & ~s.f[b]) == 0;
            if (s.cl) {
                clt = s.clt[b];
                take = take && clt >= s.cl[b];     // a NaN rejects
            }
        }
        __syncwarp();                  // every lane has read the per-path scalars before lane 0 overwrites them
        if (MODE & UAM_REFINE_ACCEPT) {
            if (take) {
                c = ct;
                tau = fmin(2.0 * tau, s.max_step);
                if (lane == 0) { s.c[b] = ct; s.k[b] = kt; s.accepted[b] += 1; }
                if ((MODE & UAM_REFINE_SWEPT) && lane == 0) {
                    s.f[b] = ft;
                    if (s.d2) s.d2[b] = d2t;
                }
                if ((MODE & UAM_REFINE_KEEPOUT) && lane == 0) {
                    s.f[b] = ft;
                    if (s.cl) s.cl[b] = clt;
                }
            } else if (was_active) {
                tau = 0.5 * tau;
            }
        }
        if ((MODE & UAM_REFINE_START) && lane == 0) s.accepted[b] = 0;
        if (MODE & UAM_REFINE_PROPOSE) {
            // the state's gradient: the trial's when it was taken (kept in g for the trips that follow)
            const double2* gs = take ? s.gt + row : s.g + row;
            double m = 0.0;
            bool finite = true;
            for (int w = 1 + lane; w < s.Wp - 1; w += 32) {
                const double2 v = gs[w];
                if (take) s.g[row + w] = v;
                finite = finite && isfinite(v.x) && isfinite(v.y);
                m = fmax(m, fmax(fabs(v.x), fabs(v.y)));
            }
            m = uam_warp_max(m);
            finite = __all_sync(0xffffffffu, finite);
            const bool act = tau >= s.min_step && finite && m > 0.0 && isfinite(c);
            const double r = act ? __ddiv_rn(__dmul_rn(tau, s.h), m) : 0.0;      // no waypoint moves more than tau cells
            const double2* zs = take ? s.zt + row : s.z + row;
            for (int w = lane; w < s.Wp; w += 32) {
                double2 v = zs[w];
                const bool free_wp = w >= 1 && w < s.Wp - 1;
                if (take && free_wp) s.z[row + w] = v;
                if (act && free_wp) {
                    const double2 d = gs[w];
                    v.x = __dsub_rn(v.x, __dmul_rn(r, d.x));
                    v.y = __dsub_rn(v.y, __dmul_rn(r, d.y));
                }
                s.zt[row + w] = v;
            }
            if (lane == 0) s.active[b] = act ? 1 : 0;
        } else if (take) {
            for (int w = 1 + lane; w < s.Wp - 1; w += 32) s.z[row + w] = s.zt[row + w];
        }
        if (lane == 0) s.tau[b] = tau;
    }
}

template <int MODE>
int uam_refine_step_launch(uam_ctx* ctx, const UamRefineState& s, cudaStream_t st) {
    const long long ctas = std::min<long long>((s.B + UAM_WARPS_PER_CTA - 1) / UAM_WARPS_PER_CTA, (long long)ctx->sm_count * 16);
    uam_k_refine_step<MODE><<<(unsigned)ctas, UAM_CTA_THREADS, 0, st>>>(s);
    UAM_CHECK_LAUNCH(ctx, "uam_k_refine_step");
    return UAM_OK;
}

}  // namespace

// the analytic check of the keep-out refinement on a batch: the sweep's flags, or with margin > 0 the clearance's flags
// and clearance capped at the margin
static int uam_keepout_enqueue(uam_ctx* ctx, const double* d_z, int64_t B, int N, double margin, uint8_t* d_flags,
                               double* d_clearance, cudaStream_t st) {
    if (margin > 0.0) return uam_clearance_analytic_enqueue(ctx, d_z, B, N, margin, d_flags, d_clearance, nullptr, nullptr, st);
    return uam_sweep_analytic_enqueue(ctx, d_z, B, N, d_flags, nullptr, nullptr, st);
}

// All entry points: swept = uam_refine_paths_raster_swept (min_d2, d_sweep_flags and d_d2min are only read then),
// keepout = uam_refine_paths_raster_keepout (margin, d_sweep_flags and d_clearance are only read then).
static int uam_refine_run(uam_ctx* ctx, double* d_z, int64_t B, int N, const double* h_p, int n_p, int flags,
                          double samples_per_cell, int iterations, double step_cells, double max_step_cells,
                          double min_step_cells, float* d_cost, uint8_t* d_collide, int32_t* d_accepted, bool swept,
                          int min_d2, uint8_t* d_sweep_flags, int32_t* d_d2min, bool keepout, double margin,
                          double* d_clearance, void* stream) {
    if (!ctx) return UAM_ERR_INVALID;
    if (iterations < 0) return uam_fail(ctx, UAM_ERR_INVALID, "iterations must be >= 0 (got %d)", iterations);
    if (!(std::isfinite(step_cells) && std::isfinite(max_step_cells) && std::isfinite(min_step_cells) && min_step_cells > 0.0 &&
          min_step_cells <= step_cells && step_cells <= max_step_cells))
        return uam_fail(ctx, UAM_ERR_INVALID, "step sizes must be finite with 0 < min <= step <= max (got %g, %g, %g)",
                        min_step_cells, step_cells, max_step_cells);
    if (swept && (min_d2 < 0 || min_d2 > 65535)) return uam_fail(ctx, UAM_ERR_INVALID, "min_d2 must be in 0 .. 65535 (got %d)", min_d2);
    if (keepout && !(margin >= 0.0 && margin <= 1e100))
        return uam_fail(ctx, UAM_ERR_INVALID, "margin must be in [0, 1e100] (got %g)", margin);
    if (keepout && N > (1 << 28)) return uam_fail(ctx, UAM_ERR_INVALID, "need N <= 2^28 for the analytic check (got %d)", N);
    UamRasterParams rp;
    UAM_TRY(uam_raster_prepare(ctx, B, N, h_p, n_p, flags, samples_per_cell, &rp));
    if (B == 0) return UAM_OK;
    if (!d_z || !d_cost || !d_collide) return uam_fail(ctx, UAM_ERR_INVALID, "paths, cost or collide pointer is NULL");
    if ((swept || keepout) && !d_sweep_flags) return uam_fail(ctx, UAM_ERR_INVALID, "sweep flags pointer is NULL");
    if (keepout && d_clearance && margin == 0.0)
        return uam_fail(ctx, UAM_ERR_INVALID, "a clearance pointer needs margin > 0 (the clearance is capped at the margin)");
    UAM_TRY(uam_raster_grad_supported(ctx, rp));
    const bool clearance = swept && (min_d2 > 0 || d_d2min);
    if (swept) UAM_TRY(uam_sweep_supported(ctx, N, clearance));
    const bool keepout_cl = keepout && margin > 0.0;
    if (keepout && !ctx->has_shapes) return uam_fail(ctx, UAM_ERR_STATE, "no shapes: call uam_map_set_shapes first");
    UAM_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = uam_pick_stream(ctx, stream);
    UAM_NVTX(swept ? "uam.raster.refine_swept" : keepout ? "uam.raster.refine_keepout" : "uam.raster.refine");
    if (keepout) {
        UAM_TRY(uam_ensure_obs_tables(ctx, st));
        UAM_TRY(uam_obs_supported(ctx, keepout_cl));
        if (keepout_cl) UAM_TRY(uam_ensure_clr_lists(ctx, margin, st));
    }
    if (swept) UAM_TRY(uam_ensure_occ_bits(ctx, st));
    if (clearance) UAM_TRY(uam_sweep_ensure_d2(ctx, st));
    UAM_TRY(uam_raster_precompute(ctx, &rp, B, N, st));

    // scratch: zt | g | gt (B x Wp double2 each) | tau (f64) | [clt (f64) | cl (f64, when the caller passes none):
    // keep-out with a margin] | ct (f32) | accepted (i32, when the caller passes none) | [d2t (i32) | d2 (i32, when the
    // caller passes none): clearance] | kt (u8) | active (u8) | [ft (u8): swept or keep-out]
    const int Wp = N + 2;
    const size_t n = (size_t)B * Wp;
    const size_t swept_bytes = swept ? (size_t)B * (1 + (clearance ? 4 : 0) + (clearance && !d_d2min ? 4 : 0)) : 0;
    const size_t keepout_bytes = keepout ? (size_t)B * (1 + (keepout_cl ? 8 : 0) + (keepout_cl && !d_clearance ? 8 : 0)) : 0;
    UAM_TRY(uam_reserve(ctx, &ctx->d_refine_scratch, &ctx->refine_scratch_bytes,
                        3 * n * sizeof(double2) + (size_t)B * 18 + swept_bytes + keepout_bytes));
    UamRefineState s;
    s.zt = (double2*)ctx->d_refine_scratch;
    s.g = s.zt + n;
    double2* gt = s.g + n;
    s.gt = gt;
    s.tau = (double*)(gt + n);
    double* f64_end = s.tau + B;
    double* clt = nullptr;
    s.cl = nullptr;
    if (keepout_cl) {
        clt = f64_end;
        f64_end += B;
        s.cl = d_clearance ? d_clearance : f64_end;
        if (!d_clearance) f64_end += B;
    }
    s.clt = clt;
    float* ct = (float*)f64_end;
    s.ct = ct;
    int32_t* acc_scratch = (int32_t*)(ct + B);
    int32_t* i32_end = acc_scratch + B;
    int32_t* d2t = nullptr;
    s.d2 = nullptr;
    if (clearance) {
        d2t = i32_end;
        i32_end += B;
        s.d2 = d_d2min ? d_d2min : i32_end;
        if (!d_d2min) i32_end += B;
    }
    s.d2t = d2t;
    uint8_t* kt = (uint8_t*)i32_end;
    s.kt = kt;
    s.active = kt + B;
    uint8_t* ft = swept || keepout ? kt + 2 * B : nullptr;
    s.ft = ft;
    s.f = d_sweep_flags;
    s.min_d2 = min_d2;
    s.z = (double2*)d_z;
    s.c = d_cost;
    s.k = d_collide;
    s.accepted = d_accepted ? d_accepted : acc_scratch;
    s.B = B;
    s.Wp = Wp;
    s.h = std::min(std::fabs(rp.dx), std::fabs(rp.dy));
    s.step = step_cells;
    s.max_step = max_step_cells;
    s.min_step = min_step_cells;

    UAM_TRY(uam_raster_grad_enqueue(ctx, rp, d_z, B, N, d_cost, d_collide, (double*)s.g, st));
    if (swept) UAM_TRY(uam_sweep_enqueue(ctx, d_z, B, N, d_sweep_flags, nullptr, s.d2, st));
    if (keepout) UAM_TRY(uam_keepout_enqueue(ctx, d_z, B, N, margin, d_sweep_flags, s.cl, st));
    if (iterations == 0) {
        if (d_accepted) UAM_CUDA(ctx, cudaMemsetAsync(d_accepted, 0, (size_t)B * sizeof(int32_t), st));
        return UAM_OK;
    }
    UAM_TRY(uam_refine_step_launch<UAM_REFINE_START | UAM_REFINE_PROPOSE>(ctx, s, st));
    for (int it = 0; it < iterations; ++it) {
        const bool last = it + 1 == iterations;
        UAM_TRY(uam_raster_grad_enqueue(ctx, rp, (const double*)s.zt, B, N, ct, kt, (double*)gt, st));
        if (swept) {
            UAM_TRY(uam_sweep_enqueue(ctx, (const double*)s.zt, B, N, ft, nullptr, d2t, st));
            if (!last) UAM_TRY(uam_refine_step_launch<UAM_REFINE_ACCEPT | UAM_REFINE_PROPOSE | UAM_REFINE_SWEPT>(ctx, s, st));
            else UAM_TRY(uam_refine_step_launch<UAM_REFINE_ACCEPT | UAM_REFINE_SWEPT>(ctx, s, st));
        } else if (keepout) {
            UAM_TRY(uam_keepout_enqueue(ctx, (const double*)s.zt, B, N, margin, ft, clt, st));
            if (!last) UAM_TRY(uam_refine_step_launch<UAM_REFINE_ACCEPT | UAM_REFINE_PROPOSE | UAM_REFINE_KEEPOUT>(ctx, s, st));
            else UAM_TRY(uam_refine_step_launch<UAM_REFINE_ACCEPT | UAM_REFINE_KEEPOUT>(ctx, s, st));
        } else {
            if (!last) UAM_TRY(uam_refine_step_launch<UAM_REFINE_ACCEPT | UAM_REFINE_PROPOSE>(ctx, s, st));
            else UAM_TRY(uam_refine_step_launch<UAM_REFINE_ACCEPT>(ctx, s, st));
        }
    }
    return UAM_OK;
}

extern "C" int uam_refine_paths_raster(uam_ctx* ctx, double* d_z, int64_t B, int N, const double* h_p, int n_p, int flags,
                                       double samples_per_cell, int iterations, double step_cells, double max_step_cells,
                                       double min_step_cells, float* d_cost, uint8_t* d_collide, int32_t* d_accepted,
                                       void* stream) {
    return uam_refine_run(ctx, d_z, B, N, h_p, n_p, flags, samples_per_cell, iterations, step_cells, max_step_cells,
                          min_step_cells, d_cost, d_collide, d_accepted, false, 0, nullptr, nullptr, false, 0.0, nullptr,
                          stream);
}

extern "C" int uam_refine_paths_raster_swept(uam_ctx* ctx, double* d_z, int64_t B, int N, const double* h_p, int n_p,
                                             int flags, double samples_per_cell, int iterations, double step_cells,
                                             double max_step_cells, double min_step_cells, int min_d2, float* d_cost,
                                             uint8_t* d_collide, int32_t* d_accepted, uint8_t* d_sweep_flags,
                                             int32_t* d_d2min, void* stream) {
    return uam_refine_run(ctx, d_z, B, N, h_p, n_p, flags, samples_per_cell, iterations, step_cells, max_step_cells,
                          min_step_cells, d_cost, d_collide, d_accepted, true, min_d2, d_sweep_flags, d_d2min, false, 0.0,
                          nullptr, stream);
}

extern "C" int uam_refine_paths_raster_keepout(uam_ctx* ctx, double* d_z, int64_t B, int N, const double* h_p, int n_p,
                                               int flags, double samples_per_cell, int iterations, double step_cells,
                                               double max_step_cells, double min_step_cells, double margin, float* d_cost,
                                               uint8_t* d_collide, int32_t* d_accepted, uint8_t* d_sweep_flags,
                                               double* d_clearance, void* stream) {
    return uam_refine_run(ctx, d_z, B, N, h_p, n_p, flags, samples_per_cell, iterations, step_cells, max_step_cells,
                          min_step_cells, d_cost, d_collide, d_accepted, false, 0, d_sweep_flags, nullptr, true, margin,
                          d_clearance, stream);
}
