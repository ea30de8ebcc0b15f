// Shape grid of the analytic scorer: per-cell candidate lists over the map's convex shapes.
//
// Problem.get_cost evaluates every shape of every region at every waypoint (problem.py:49-82), but
// psi_s(x; e) = prod_i min(h_i(x) - e, 0)^2 is non-zero only where ALL h_i(x) < e, i.e. inside the (enlarged) shape,
// and Map.collides / the obstacle block of get_nonlincon likewise need all h_i(x) <= 1e-14.  A shape that has one
// inequality > max(e, 1e-14) on a whole grid cell therefore contributes exact zeros ("not contained") to every point of
// that cell, and x + 0.0 == x: leaving it out does not change a bit of the sums.  The lists are in ascending device
// order (obstacles, then regions in insertion order), so the surviving terms are added in the reference's order.
//
// Not culled, ever: shapes whose centre normaliser psi_s(c_s) is 0 or NaN (the reference's 0/0 = NaN must propagate).
// The grid is used only for smooth region penalties (the reference's default; the non-smooth form is non-zero OUTSIDE
// the shapes), finite inequality records and finite weights (uam_pick_shape_grid), and only for points inside the
// grid's box; everything else takes the full loops.  With obstacle_smooth off (the reference's default) the obstacles'
// psi values are non-zero outside them: the lists then serve only their `contains` test (obs_values = 0) and the
// constraint block / obstacle penalty loop over every obstacle.
//
// Build: count (one thread per cell tests every shape) -> exclusive scan -> fill (same test, ordered writes); one 4-byte
// read-back sizes the item array.  Redone when the shapes or the enlargement change (like the psi(centre) table).
#include <algorithm>
#include <cmath>

#include "uam_internal.cuh"

namespace {

__device__ __forceinline__ bool uam_shape_may_matter(const UamEdge* __restrict__ edges, const UamShape* __restrict__ shapes,
                                                     const double* __restrict__ psic, int s, double xa, double xb, double ya,
                                                     double yb, double thr, int obs_values) {
    const int4 meta = __ldg(reinterpret_cast<const int4*>(&shapes[s].e0));     // e0, e1, region, has_center
    if (meta.w && (meta.z >= 0 || obs_values)) {
        const double pc = __ldg(psic + s);
        if (pc == 0.0 || pc != pc) return true;        // 0/0, x/NaN: the reference's NaN reaches every point
    }
    for (int i = meta.x; i < meta.y; ++i)
        if (uam_edge_excludes_tile(uam_load_edge(edges + i), xa, xb, ya, yb, thr)) return false;
    return true;
}

// FILL = 0: counts[cell] = candidates; FILL = 1: items[start[cell] ..] = the candidates in ascending order.
// A cell's box is widened by 1/1000 of a cell on every side: the cell index of a point is computed in floating point.
template <int FILL>
__global__ void __launch_bounds__(128)
uam_k_shape_grid(const UamEdge* __restrict__ edges, const UamShape* __restrict__ shapes, const double* __restrict__ psic,
                 int n_shapes, int G, double gx0, double gy0, double cw, double ch, double thr, int obs_values, int* __restrict__ counts,
                 const int* __restrict__ start, int* __restrict__ items) {
    const int cell = blockIdx.x * blockDim.x + threadIdx.x;
    if (cell >= G * G) return;
    const int cy = cell / G, cx = cell - cy * G;
    const double xa = gx0 + ((double)cx - 1e-3) * cw, xb = gx0 + ((double)cx + 1.001) * cw;
    const double ya = gy0 + ((double)cy - 1e-3) * ch, yb = gy0 + ((double)cy + 1.001) * ch;
    int n = 0;
    int* dst = FILL ? items + start[cell] : nullptr;
    for (int s = 0; s < n_shapes; ++s) {
        if (uam_shape_may_matter(edges, shapes, psic, s, xa, xb, ya, yb, thr, obs_values)) {
            if (FILL) dst[n] = s;
            ++n;
        }
    }
    if (!FILL) counts[cell] = n;
}

// exclusive prefix sum of counts[0..n) into start[0..n], start[n] = total (single CTA)
__global__ void __launch_bounds__(1024)
uam_k_shape_grid_scan(const int* __restrict__ counts, int n, int* __restrict__ start) {
    __shared__ int warp_tot[32];
    const int per = (n + 1023) / 1024;
    const int lo = min((int)threadIdx.x * per, n), hi = min(lo + per, n);
    int local = 0;
    for (int i = lo; i < hi; ++i) local += counts[i];
    int incl = local;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) warp_tot[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        const int w = warp_tot[lane];
        int wi = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, wi, o);
            if (lane >= o) wi += t;
        }
        warp_tot[lane] = wi - w;
    }
    __syncthreads();
    int run = warp_tot[warp] + incl - local;
    for (int i = lo; i < hi; ++i) {
        const int c = counts[i];
        start[i] = run;
        run += c;
    }
    if (threadIdx.x == 1023) start[n] = run;
}

}  // namespace

// Called by uam_ensure_shape_norm after psi(centre) has been refreshed for (e, flags); the caller has synchronised the
// device, so no kernel still reads the old lists.
int uam_build_shape_grid(uam_ctx* ctx, double e, int flags, cudaStream_t st) {
    ctx->shape_grid = UamShapeGrid{};
    const int obs_values = (flags & UAM_OBSTACLE_SMOOTH) ? 1 : 0;
    if (!ctx->shape_grid_opt || !(flags & UAM_PENALTY_SMOOTH) || ctx->n_shapes < 4 || !ctx->edges_finite || !std::isfinite(e)) return UAM_OK;
    const double x0 = ctx->shape_bbox[0], x1 = ctx->shape_bbox[1], y0 = ctx->shape_bbox[2], y1 = ctx->shape_bbox[3];
    if (!(x1 > x0 && y1 > y0) || !std::isfinite(x1 - x0) || !std::isfinite(y1 - y0)) return UAM_OK;
    // about 8 cells per sqrt(shape), a power of two in [32, 256], and at most 2^26 shape tests for the build
    int G = 32;
    while (G < 256 && G < 8.0 * std::sqrt((double)ctx->n_shapes)) G *= 2;
    while (G > 8 && (double)G * G * ctx->n_shapes > 67108864.0) G /= 2;
    const double mx = 0.05 * (x1 - x0) + 0.5 * std::fabs(e), my = 0.05 * (y1 - y0) + 0.5 * std::fabs(e);
    const double gx0 = x0 - mx, gy0 = y0 - my;
    const double cw = (x1 - x0 + 2 * mx) / G, ch = (y1 - y0 + 2 * my) / G;
    if (!(cw > 0.0 && ch > 0.0) || !std::isfinite(1.0 / cw) || !std::isfinite(1.0 / ch)) return UAM_OK;
    const int cells = G * G;
    UAM_TRY(uam_reserve(ctx, (void**)&ctx->d_grid_start, &ctx->grid_start_bytes, (size_t)(2 * cells + 2) * sizeof(int)));
    int* start = ctx->d_grid_start;
    int* counts = start + cells + 1;
    const double thr = std::max(e, 1e-14);       // covers psi(x; e), psi(x; 0) of the constraint block and `contains`
    const int ctas = (cells + 127) / 128;
    uam_k_shape_grid<0><<<ctas, 128, 0, st>>>(ctx->d_edges, ctx->d_shapes, ctx->d_psic, ctx->n_shapes, G, gx0, gy0, cw, ch, thr,
                                              obs_values, counts, nullptr, nullptr);
    UAM_CHECK_LAUNCH(ctx, "uam_k_shape_grid");
    uam_k_shape_grid_scan<<<1, 1024, 0, st>>>(counts, cells, start);
    UAM_CHECK_LAUNCH(ctx, "uam_k_shape_grid_scan");
    int total = 0;
    UAM_CUDA(ctx, cudaMemcpyAsync(&total, start + cells, sizeof(int), cudaMemcpyDeviceToHost, st));
    UAM_CUDA(ctx, cudaStreamSynchronize(st));
    UAM_TRY(uam_reserve(ctx, (void**)&ctx->d_grid_items, &ctx->grid_items_bytes, (size_t)(total + 1) * sizeof(int)));
    uam_k_shape_grid<1><<<ctas, 128, 0, st>>>(ctx->d_edges, ctx->d_shapes, ctx->d_psic, ctx->n_shapes, G, gx0, gy0, cw, ch, thr,
                                              obs_values, nullptr, start, ctx->d_grid_items);
    UAM_CHECK_LAUNCH(ctx, "uam_k_shape_grid");
    UAM_CUDA(ctx, cudaStreamSynchronize(st));
    UamShapeGrid sg;
    sg.gx0 = gx0; sg.gy0 = gy0; sg.inv_cw = 1.0 / cw; sg.inv_ch = 1.0 / ch;
    sg.G = G;
    sg.obs_values = obs_values;
    sg.start = start;
    sg.items = ctx->d_grid_items;
    ctx->shape_grid = sg;
    ctx->grid_items_total = total;
    return UAM_OK;
}

int uam_shape_grid_scan(uam_ctx* ctx, const int* counts, int n, int* start, cudaStream_t st) {
    uam_k_shape_grid_scan<<<1, 1024, 0, st>>>(counts, n, start);
    UAM_CHECK_LAUNCH(ctx, "uam_k_shape_grid_scan");
    return UAM_OK;
}

UamShapeGrid uam_pick_shape_grid(const uam_ctx* ctx, const UamParams& prm) {
    UamShapeGrid none{};
    // (the grid was built for these flags: uam_ensure_shape_norm rebuilds it whenever e or the smooth flags change)
    if (!ctx->shape_grid_opt || ctx->shape_grid.G == 0 || !(prm.flags & UAM_PENALTY_SMOOTH)) return none;
    for (int r = 0; r < prm.n_regions; ++r)
        if (!std::isfinite(prm.w[r])) return none;      // w * 0 must be 0 for a skipped region
    return ctx->shape_grid;
}
