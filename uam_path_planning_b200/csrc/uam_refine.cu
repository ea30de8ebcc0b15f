// Batched refinement of candidate paths by descent on the raster cost (uam_refine_paths_raster; the rule is in the
// header comment of its declaration in include/uam_b200.h).  SURVEY 8f item 1: the local step after scoring, here a
// monotone per-path step-controlled descent, not the reference's OpEn / PANOC solver.
//
// One trip = one gradient launch of the raster scorer on the whole trial batch (uam_raster_grad_enqueue: same B, so
// the same kernels and bits as uam_grad_paths_raster) + one launch of the call's check (UamRefineCheck) of the trial
// batch, if it has one + one uam_k_refine_step, which takes or drops the trial just evaluated and writes the next one.
// The loop is stream-ordered: no host synchronisation or read-back per trip, and every path is evaluated on every trip
// (a path's bits do not depend on the rest of the batch, and the kernel choice stays the one of the call's B).
#include <algorithm>
#include <cmath>
#include <type_traits>

#include "uam_internal.cuh"

namespace {

// what a launch of uam_k_refine_step does
enum : int {
    UAM_REFINE_START = 1,      // tau = step_cells, accepted = 0 (first launch, after the gradient of Z)
    UAM_REFINE_ACCEPT = 2,     // take or drop the trial in zt, evaluated into (ct, kt, gt)
    UAM_REFINE_PROPOSE = 4,    // write the next trial into zt and whether it moved the path into active
    UAM_REFINE_CHECK = 8,      // the accept test also needs the trial's check flags (ft) and guard (d2t or clt)
};

struct UamRefineState {
    double2* z;               // (B, Wp) the caller's paths, refined in place
    double2* g;               // (B, Wp) gradient at z (free waypoints only are kept up to date)
    double2* zt;              // (B, Wp) trial
    double2* gt;              // (B, Wp) gradient at zt
    float* c;                 // cost / collide at z: the caller's outputs
    uint8_t* k;
    float* ct;                // cost / collide at zt
    uint8_t* kt;
    double* tau;              // step, in cells
    uint8_t* active;          // the trial in zt is a proposed move (not a copy of z)
    int32_t* accepted;
    long long B;
    int Wp;
    double h;                 // cell size: min(|dx|, |dy|)
    double step, max_step, min_step;
    // UAM_REFINE_CHECK: flags at z (the caller's output) and zt; at most one guard pair at z (output or scratch) and zt
    uint8_t* f;
    uint8_t* ft;
    int32_t* d2;              // raster sweep: d2min; may be set with min_d2 == 0 (the caller asked for d2min) and is
    int32_t* d2t;             // then not compared
    int min_d2;
    double* cl;               // analytic: the clearance capped at the margin
    double* clt;
};

__device__ __forceinline__ double uam_warp_max(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// Warp per path, lanes stride the waypoints (16 B each).  Waypoints 0 and Wp-1 (start and goal) are never written
// into z.  The proposal is fp64 with explicit rounded operations: nvcc would otherwise contract z - r g into an FMA.
// G is the type of the check's guard: int32_t (d2) or double (cl).  One body for both guards cost 2-3 % of this
// kernel's time on the C3 shard (ptxas took 45 registers for it).
template <int MODE, class G = void>
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
        double clt = 0.0;
        if (MODE & UAM_REFINE_CHECK) {
            ft = s.ft[b];
            take = take && (ft & ~s.f[b]) == 0;
            if (std::is_same<G, int32_t>::value && s.d2) {
                d2t = s.d2t[b];
                take = take && (s.min_d2 == 0 || min(d2t, s.min_d2) >= min(s.d2[b], s.min_d2));
            }
            if (std::is_same<G, double>::value && s.cl) {
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
                if ((MODE & UAM_REFINE_CHECK) && lane == 0) {
                    s.f[b] = ft;
                    if (std::is_same<G, int32_t>::value && s.d2) s.d2[b] = d2t;
                    if (std::is_same<G, double>::value && s.cl) s.cl[b] = clt;
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

// a launch in one of the modes the loop uses: START | PROPOSE first, then ACCEPT [| PROPOSE] [| CHECK], the check's
// guard being fp64 (the analytic clearance) or int32 (the raster sweep's d2)
int uam_refine_step_launch(uam_ctx* ctx, int mode, bool fp64_guard, const UamRefineState& s, cudaStream_t st) {
    constexpr int A = UAM_REFINE_ACCEPT, P = UAM_REFINE_PROPOSE, K = UAM_REFINE_CHECK;
    void (*kernel)(UamRefineState) = mode == (UAM_REFINE_START | P) ? uam_k_refine_step<UAM_REFINE_START | P>
                                     : mode == A                    ? uam_k_refine_step<A>
                                     : mode == (A | P)              ? uam_k_refine_step<A | P>
                                     : mode == (A | K) ? (fp64_guard ? uam_k_refine_step<A | K, double> : uam_k_refine_step<A | K, int32_t>)
                                     : fp64_guard      ? uam_k_refine_step<A | P | K, double>
                                                       : uam_k_refine_step<A | P | K, int32_t>;
    const long long ctas = std::min<long long>((s.B + UAM_WARPS_PER_CTA - 1) / UAM_WARPS_PER_CTA, (long long)ctx->sm_count * 16);
    kernel<<<(unsigned)ctas, UAM_CTA_THREADS, 0, st>>>(s);
    UAM_CHECK_LAUNCH(ctx, "uam_k_refine_step");
    return UAM_OK;
}

// the check of the trial batch in the accept test, filled by each entry point, with all that depends on its kind
struct UamRefineCheck {
    enum Kind { NONE, RASTER, ANALYTIC } kind = NONE;
    int min_d2 = 0;                   // RASTER: squared cells, 0 .. 65535
    double margin = 0.0;              // ANALYTIC: km, 0 = the sweep only
    uint8_t* d_flags = nullptr;       // the caller's flags (required with a check)
    int32_t* d_d2min = nullptr;       // RASTER: the caller's d2min (nullable)
    double* d_clearance = nullptr;    // ANALYTIC: the caller's clearance (nullable, only with margin > 0)
    // the guard: the raster d2min when min_d2 > 0 or the caller asks for it, the analytic clearance with a margin
    bool guard() const { return kind == RASTER ? min_d2 > 0 || d_d2min : kind == ANALYTIC && margin > 0.0; }

    int check_ranges(uam_ctx* ctx, int N) const {     // with the step sizes
        if (kind == RASTER && (min_d2 < 0 || min_d2 > 65535))
            return uam_fail(ctx, UAM_ERR_INVALID, "min_d2 must be in 0 .. 65535 (got %d)", min_d2);
        if (kind == ANALYTIC && !(margin >= 0.0 && margin <= 1e100))
            return uam_fail(ctx, UAM_ERR_INVALID, "margin must be in [0, 1e100] (got %g)", margin);
        if (kind == ANALYTIC && N > (1 << 28))
            return uam_fail(ctx, UAM_ERR_INVALID, "need N <= 2^28 for the analytic check (got %d)", N);
        return UAM_OK;
    }
    int check_pointers(uam_ctx* ctx) const {          // with the paths' pointers
        if (kind != NONE && !d_flags) return uam_fail(ctx, UAM_ERR_INVALID, "sweep flags pointer is NULL");
        if (kind == ANALYTIC && d_clearance && margin == 0.0)
            return uam_fail(ctx, UAM_ERR_INVALID, "a clearance pointer needs margin > 0 (the clearance is capped at the margin)");
        return UAM_OK;
    }
    int check_supported(uam_ctx* ctx, int N) const {  // before anything is built
        if (kind == RASTER) return uam_sweep_supported(ctx, N, guard());
        if (kind == ANALYTIC && !ctx->has_shapes) return uam_fail(ctx, UAM_ERR_STATE, "no shapes: call uam_map_set_shapes first");
        return UAM_OK;
    }
    // builds what the check reads when missing (each build may synchronise); the analytic record and form checks come
    // with its tables
    int build(uam_ctx* ctx, cudaStream_t st) const {
        if (kind == RASTER) {
            UAM_TRY(uam_ensure_occ_bits(ctx, st));
            if (guard()) UAM_TRY(uam_sweep_ensure_d2(ctx, st));
        } else if (kind == ANALYTIC) {
            UAM_TRY(uam_ensure_obs_tables(ctx, st));
            UAM_TRY(uam_obs_supported(ctx, guard()));
            if (guard()) UAM_TRY(uam_ensure_clr_lists(ctx, margin, st));
        }
        return UAM_OK;
    }
    // one launch of the check on the batch d_z, none without a check: its flags, and its guard into d2 or cl
    int enqueue(uam_ctx* ctx, const double* d_z, int64_t B, int N, uint8_t* flags, int32_t* d2, double* cl,
                cudaStream_t st) const {
        if (kind == RASTER) return uam_sweep_enqueue(ctx, d_z, B, N, flags, nullptr, d2, st);
        if (kind == ANALYTIC && margin > 0.0)
            return uam_clearance_analytic_enqueue(ctx, d_z, B, N, margin, flags, cl, nullptr, nullptr, st);
        if (kind == ANALYTIC) return uam_sweep_analytic_enqueue(ctx, d_z, B, N, flags, nullptr, nullptr, st);
        return UAM_OK;
    }
};

}  // namespace

static int uam_refine_run(uam_ctx* ctx, double* d_z, int64_t B, int N, const double* h_p, int n_p, int flags,
                          double samples_per_cell, int iterations, double step_cells, double max_step_cells,
                          double min_step_cells, float* d_cost, uint8_t* d_collide, int32_t* d_accepted,
                          const UamRefineCheck& chk, void* stream) {
    if (!ctx) return UAM_ERR_INVALID;
    if (iterations < 0) return uam_fail(ctx, UAM_ERR_INVALID, "iterations must be >= 0 (got %d)", iterations);
    if (!(std::isfinite(step_cells) && std::isfinite(max_step_cells) && std::isfinite(min_step_cells) && min_step_cells > 0.0 &&
          min_step_cells <= step_cells && step_cells <= max_step_cells))
        return uam_fail(ctx, UAM_ERR_INVALID, "step sizes must be finite with 0 < min <= step <= max (got %g, %g, %g)",
                        min_step_cells, step_cells, max_step_cells);
    UAM_TRY(chk.check_ranges(ctx, N));
    UamRasterParams rp;
    UAM_TRY(uam_raster_prepare(ctx, B, N, h_p, n_p, flags, samples_per_cell, &rp));
    if (B == 0) return UAM_OK;
    if (!d_z || !d_cost || !d_collide) return uam_fail(ctx, UAM_ERR_INVALID, "paths, cost or collide pointer is NULL");
    UAM_TRY(chk.check_pointers(ctx));
    UAM_TRY(uam_raster_grad_supported(ctx, rp));
    UAM_TRY(chk.check_supported(ctx, N));
    UAM_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = uam_pick_stream(ctx, stream);
    UAM_NVTX(chk.kind == UamRefineCheck::RASTER ? "uam.raster.refine_swept"
             : chk.kind == UamRefineCheck::ANALYTIC ? "uam.raster.refine_keepout" : "uam.raster.refine");
    UAM_TRY(chk.build(ctx, st));
    UAM_TRY(uam_raster_precompute(ctx, &rp, B, N, st));

    // scratch, widest type first so that no slice needs padding; cl / d2 only when the caller passes none
    const bool check = chk.kind != UamRefineCheck::NONE;
    const size_t n = (size_t)B * (N + 2);
    UamRefineState s{};
    auto carve = [&](uintptr_t at) {         // lays the scratch out from address `at` on; returns its size
        const uintptr_t base = at;
        auto take = [&at](size_t bytes) { const uintptr_t r = at; at += bytes; return r; };
        s.zt = (double2*)take(n * sizeof(double2));
        s.g = (double2*)take(n * sizeof(double2));
        s.gt = (double2*)take(n * sizeof(double2));
        s.tau = (double*)take(B * sizeof(double));
        if (chk.kind == UamRefineCheck::ANALYTIC && chk.guard()) {
            s.clt = (double*)take(B * sizeof(double));
            s.cl = chk.d_clearance ? chk.d_clearance : (double*)take(B * sizeof(double));
        }
        s.ct = (float*)take(B * sizeof(float));
        s.accepted = (int32_t*)take(B * sizeof(int32_t));
        if (chk.kind == UamRefineCheck::RASTER && chk.guard()) {
            s.d2t = (int32_t*)take(B * sizeof(int32_t));
            s.d2 = chk.d_d2min ? chk.d_d2min : (int32_t*)take(B * sizeof(int32_t));
        }
        s.kt = (uint8_t*)take(B);
        s.active = (uint8_t*)take(B);
        if (check) s.ft = (uint8_t*)take(B);
        return (size_t)(at - base);
    };
    UAM_TRY(uam_reserve(ctx, &ctx->d_refine_scratch, &ctx->refine_scratch_bytes, carve(0)));
    carve((uintptr_t)ctx->d_refine_scratch);
    if (d_accepted) s.accepted = d_accepted;
    s.f = chk.d_flags;
    s.min_d2 = chk.min_d2;
    s.z = (double2*)d_z;
    s.c = d_cost;
    s.k = d_collide;
    s.B = B;
    s.Wp = N + 2;
    s.h = std::min(std::fabs(rp.dx), std::fabs(rp.dy));
    s.step = step_cells;
    s.max_step = max_step_cells;
    s.min_step = min_step_cells;

    UAM_TRY(uam_raster_grad_enqueue(ctx, rp, d_z, B, N, d_cost, d_collide, (double*)s.g, st));
    UAM_TRY(chk.enqueue(ctx, d_z, B, N, s.f, s.d2, s.cl, st));
    if (iterations == 0) {
        if (d_accepted) UAM_CUDA(ctx, cudaMemsetAsync(d_accepted, 0, (size_t)B * sizeof(int32_t), st));
        return UAM_OK;
    }
    const bool fp64_guard = chk.kind == UamRefineCheck::ANALYTIC;
    UAM_TRY(uam_refine_step_launch(ctx, UAM_REFINE_START | UAM_REFINE_PROPOSE, fp64_guard, s, st));
    for (int it = 0; it < iterations; ++it) {
        UAM_TRY(uam_raster_grad_enqueue(ctx, rp, (const double*)s.zt, B, N, s.ct, s.kt, (double*)s.gt, st));
        UAM_TRY(chk.enqueue(ctx, (const double*)s.zt, B, N, s.ft, s.d2t, s.clt, st));
        const int mode = UAM_REFINE_ACCEPT | (it + 1 < iterations ? UAM_REFINE_PROPOSE : 0) | (check ? UAM_REFINE_CHECK : 0);
        UAM_TRY(uam_refine_step_launch(ctx, mode, fp64_guard, s, st));
    }
    return UAM_OK;
}

extern "C" int uam_refine_paths_raster(uam_ctx* ctx, double* d_z, int64_t B, int N, const double* h_p, int n_p, int flags,
                                       double samples_per_cell, int iterations, double step_cells, double max_step_cells,
                                       double min_step_cells, float* d_cost, uint8_t* d_collide, int32_t* d_accepted,
                                       void* stream) {
    return uam_refine_run(ctx, d_z, B, N, h_p, n_p, flags, samples_per_cell, iterations, step_cells, max_step_cells,
                          min_step_cells, d_cost, d_collide, d_accepted, UamRefineCheck{}, stream);
}

extern "C" int uam_refine_paths_raster_swept(uam_ctx* ctx, double* d_z, int64_t B, int N, const double* h_p, int n_p,
                                             int flags, double samples_per_cell, int iterations, double step_cells,
                                             double max_step_cells, double min_step_cells, int min_d2, float* d_cost,
                                             uint8_t* d_collide, int32_t* d_accepted, uint8_t* d_sweep_flags,
                                             int32_t* d_d2min, void* stream) {
    return uam_refine_run(ctx, d_z, B, N, h_p, n_p, flags, samples_per_cell, iterations, step_cells, max_step_cells,
                          min_step_cells, d_cost, d_collide, d_accepted,
                          UamRefineCheck{UamRefineCheck::RASTER, min_d2, 0.0, d_sweep_flags, d_d2min, nullptr}, stream);
}

extern "C" int uam_refine_paths_raster_keepout(uam_ctx* ctx, double* d_z, int64_t B, int N, const double* h_p, int n_p,
                                               int flags, double samples_per_cell, int iterations, double step_cells,
                                               double max_step_cells, double min_step_cells, double margin, float* d_cost,
                                               uint8_t* d_collide, int32_t* d_accepted, uint8_t* d_sweep_flags,
                                               double* d_clearance, void* stream) {
    return uam_refine_run(ctx, d_z, B, N, h_p, n_p, flags, samples_per_cell, iterations, step_cells, max_step_cells,
                          min_step_cells, d_cost, d_collide, d_accepted,
                          UamRefineCheck{UamRefineCheck::ANALYTIC, 0, margin, d_sweep_flags, nullptr, d_clearance}, stream);
}
