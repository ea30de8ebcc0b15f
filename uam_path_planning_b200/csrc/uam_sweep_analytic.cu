// Swept check of whole path segments against the analytic hard obstacles (uam_sweep_paths_analytic, include/uam_b200.h;
// DESIGN.md section 9g).
//
// HIT(k, o) is a pure function of the segment's two fp64 endpoints and obstacle o's records, computed with explicit
// round-to-nearest operations in a fixed order (tests/analytic_sweep_reference.py restates it in numpy bit for bit):
//   - the fp64 `contains` (all h_i <= 1e-14, uam_h_exact) at either endpoint;
//   - else, per affine record (line, box), the endpoint values lowered by their error bound, L = h - (2^-49 M + 2^-1000),
//     give the interval of t in [0, 1] where the affine interpolation of L is <= 1e-14; its crossing parameter is
//     rounded to nearest and widened outward by 2^-50; the intervals are intersected;
//   - a non-empty intersection [lo, hi] is a hit unless the obstacle has an ellipse record; that record is evaluated at
//     its scaled vertex t clamped to [lo, hi] and hits when its value minus the error bound s is <= 1e-14.
// The cell lists only choose which (segment, obstacle) pairs are evaluated: a pair the lists leave out cannot hit (the
// argument is in DESIGN.md 9g; uam_obs_grid_qmax checks its conditions for the uploaded records and grid).
#include <algorithm>
#include <climits>
#include <cmath>
#include <vector>

#include "uam_internal.cuh"

namespace {

constexpr double kThr = 1e-14;               // quadratic_obstacle.py:89-94
constexpr double kTiny = 0x1p-1000;          // absolute part of every error bound (underflow)
constexpr double kBig = 1e100;               // |coordinate| bound of a valid path, as in uam_psi
constexpr double kWalkMargin = 0x1p-20;      // cells: the walk visits every cell within this distance of the segment
constexpr double kListWiden = 1e-3;          // cells: a list covers its cell widened by this much (as the scorer's grid)

// M_i(x, y) of an affine record: the magnitude its fp64 evaluation error is bounded by (3.01 u M, u = 2^-53)
__device__ __forceinline__ double uam_affine_mag(const UamEdge& r, double x, double y) {
    if ((int)r.kind == UAM_EDGE_LINE) {
        const double mx = __dmul_rn(fabs(r.p3), __dadd_rn(fabs(x), fabs(r.p0)));
        const double my = __dmul_rn(fabs(r.p2), __dadd_rn(fabs(y), fabs(r.p1)));
        return __dmul_rn(fabs(r.p4), __dadd_rn(mx, my));
    }
    const double xd = ((int)r.p0 == 0) ? x : y;
    return __dadd_rn(__dadd_rn(fabs(xd), fabs(r.p2)), fabs(r.p3));
}

// a lower bound of the exact value of an affine record at (x, y) from its fp64 value h
__device__ __forceinline__ double uam_lowered(const UamEdge& r, double h, double x, double y) {
    return __dsub_rn(h, __dadd_rn(__dmul_rn(uam_affine_mag(r, x, y), 0x1p-49), kTiny));
}

// HIT(k, o) for the segment (ax, ay) -> (bx, by) and the records [e0, e1) of one obstacle (at most one ellipse record)
__device__ __forceinline__ bool uam_segment_hits(const UamEdge* __restrict__ edges, int e0, int e1, double ax, double ay, double bx,
                                 double by) {
    bool in_a = true, in_b = true;
    double lo = 0.0, hi = 1.0;
    int ell = -1;
    for (int i = e0; i < e1; ++i) {
        const UamEdge r = uam_load_edge(edges + i);
        const double ha = uam_h_exact(r, ax, ay), hb = uam_h_exact(r, bx, by);
        in_a = in_a && (ha <= kThr);
        in_b = in_b && (hb <= kThr);
        if ((int)r.kind == UAM_EDGE_ELLIPSE) {
            ell = i;
            continue;
        }
        const double la = uam_lowered(r, ha, ax, ay), lb = uam_lowered(r, hb, bx, by);
        if (la <= kThr) {
            if (lb > kThr) hi = fmin(hi, __dadd_rn(__ddiv_rn(__dsub_rn(kThr, la), __dsub_rn(lb, la)), 0x1p-50));
        } else if (lb <= kThr) {
            lo = fmax(lo, __dsub_rn(__ddiv_rn(__dsub_rn(la, kThr), __dsub_rn(la, lb)), 0x1p-50));
        } else {
            lo = 2.0;                               // both ends above: this record allows no t
        }
    }
    if (in_a || in_b) return true;
    if (!(lo <= hi)) return false;
    if (ell < 0) return true;
    // the ellipse in scaled coordinates p(t) = u + t w (u = (A - c) / r, w = (B - A) / r)
    const UamEdge r = uam_load_edge(edges + ell);
    const double ux = __ddiv_rn(__dsub_rn(ax, r.p0), r.p2), uy = __ddiv_rn(__dsub_rn(ay, r.p1), r.p3);
    const double wx = __ddiv_rn(__dsub_rn(bx, ax), r.p2), wy = __ddiv_rn(__dsub_rn(by, ay), r.p3);
    const double ww = __dadd_rn(__dmul_rn(wx, wx), __dmul_rn(wy, wy));
    const double uw = __dadd_rn(__dmul_rn(ux, wx), __dmul_rn(uy, wy));
    const double tv = ww > 0.0 ? __ddiv_rn(-uw, ww) : lo;
    const double t = fmin(fmax(tv, lo), hi);
    const double px = __dadd_rn(ux, __dmul_rn(t, wx)), py = __dadd_rn(uy, __dmul_rn(t, wy));
    const double v = __dsub_rn(__dadd_rn(__dmul_rn(px, px), __dmul_rn(py, py)), 1.0);
    const double S = __dadd_rn(__dadd_rn(__dadd_rn(fabs(ux), fabs(uy)), fabs(wx)), fabs(wy));
    const double X = __dadd_rn(fabs(px), fabs(py));
    const double s1 = __dmul_rn(__dadd_rn(__dadd_rn(1.0, __dmul_rn(X, X)), __dmul_rn(S, X)), 0x1p-46);
    const double s = __dadd_rn(s1, __dadd_rn(__dmul_rn(__dmul_rn(S, S), 0x1p-96), kTiny));
    return __dsub_rn(v, s) <= kThr;
}

__device__ __forceinline__ bool uam_obstacle_hits(const UamEdge* __restrict__ edges, const UamShape* __restrict__ shapes,
                                                  int o, double ax, double ay, double bx, double by) {
    const int2 er = __ldg(reinterpret_cast<const int2*>(&shapes[o].e0));
    return uam_segment_hits(edges, er.x, er.y, ax, ay, bx, by);
}

__device__ __forceinline__ int uam_clamp_cell(double f, int G) {
    return (int)fmin(fmax(floor(f), 0.0), (double)(G - 1));
}

// smallest obstacle index that segment (ax, ay) -> (bx, by) hits, INT_MAX if none
__device__ __forceinline__ int uam_segment_first_obstacle(const UamEdge* __restrict__ edges, const UamShape* __restrict__ shapes, int n_obs,
                                          const UamObsGrid& og, double ax, double ay, double bx, double by) {
    const double mag = fmax(fmax(fabs(ax), fabs(ay)), fmax(fabs(bx), fabs(by)));
    if (og.G == 0 || !(mag <= og.qmax)) {
        for (int o = 0; o < n_obs; ++o)
            if (uam_obstacle_hits(edges, shapes, o, ax, ay, bx, by)) return o;
        return INT_MAX;
    }
    // walk the cells along the major axis: strip j covers major coordinates [j - m, j + 1 + m] (the border strips reach
    // out to the segment's ends), its minor range comes from one slope |k| <= 1, widened by m
    const double fax = __dmul_rn(__dsub_rn(ax, og.gx0), og.inv_cw), fay = __dmul_rn(__dsub_rn(ay, og.gy0), og.inv_ch);
    const double fbx = __dmul_rn(__dsub_rn(bx, og.gx0), og.inv_cw), fby = __dmul_rn(__dsub_rn(by, og.gy0), og.inv_ch);
    const bool steep = fabs(fby - fay) > fabs(fbx - fax);
    double p0 = steep ? fay : fax, q0 = steep ? fax : fay, p1 = steep ? fby : fbx, q1 = steep ? fbx : fby;
    if (p1 < p0) {
        double tp = p0; p0 = p1; p1 = tp;
        tp = q0; q0 = q1; q1 = tp;
    }
    const double dp = p1 - p0;
    const double k = dp > 0.0 ? (q1 - q0) / dp : 0.0;
    const int G = og.G;
    const double m = kWalkMargin;
    const int j0 = uam_clamp_cell(p0 - m, G), j1 = uam_clamp_cell(p1 + m, G);
    int best = INT_MAX, last = -1;
    for (int j = j0; j <= j1; ++j) {
        const double s0 = (j == 0) ? p0 : fmin(fmax((double)j - m, p0), p1);
        const double s1 = (j == G - 1) ? p1 : fmin(fmax((double)j + 1.0 + m, p0), p1);
        const double qa = q0 + (s0 - p0) * k, qb = q0 + (s1 - p0) * k;
        const int i0 = uam_clamp_cell(fmin(qa, qb) - m, G), i1 = uam_clamp_cell(fmax(qa, qb) + m, G);
        for (int i = i0; i <= i1; ++i) {
            const int cell = steep ? j * G + i : i * G + j;
            const int l1 = __ldg(og.start + cell + 1);
            for (int li = __ldg(og.start + cell); li < l1; ++li) {
                const int o = __ldg(og.items + li);
                if (o >= best) break;                       // ascending lists: nothing smaller follows
                if (o == last) continue;                    // just tested in the previous cell
                last = o;
                if (uam_obstacle_hits(edges, shapes, o, ax, ay, bx, by)) best = o;
            }
        }
    }
    return best;
}

// one warp per path, segment k on lane k mod 32; the walk stops after the first window of 32 segments with a hit.  Two CTAs
// per SM leave 128 registers: it takes 94 and does not spill (the default heuristic picks 80 and spills 32 bytes)
__global__ void __launch_bounds__(UAM_CTA_THREADS, 2)
uam_k_sweep_analytic(const double2* __restrict__ z, int64_t B, int Wp, const UamEdge* __restrict__ edges,
                     const UamShape* __restrict__ shapes, int n_obs, UamObsGrid og, uint8_t* __restrict__ flags,
                     int32_t* __restrict__ first_hit, int32_t* __restrict__ first_obstacle) {
    const int lane = threadIdx.x & 31;
    const int64_t warps = (int64_t)gridDim.x * UAM_WARPS_PER_CTA;
    for (int64_t path = (int64_t)blockIdx.x * UAM_WARPS_PER_CTA + (threadIdx.x >> 5); path < B; path += warps) {
        const double2* zp = z + path * Wp;
        bool bad = false;
        for (int k = lane; k < Wp; k += 32) {
            const double2 p = zp[k];
            bad = bad || !(fabs(p.x) < kBig && fabs(p.y) < kBig);
        }
        bad = __any_sync(0xffffffffu, bad);
        int hitk = -1, hito = -1;
        if (!bad) {
            for (int k0 = 0; k0 < Wp - 1; k0 += 32) {
                const int k = k0 + lane;
                int o = INT_MAX;
                if (k < Wp - 1) {
                    const double2 a = zp[k], b = zp[k + 1];
                    o = uam_segment_first_obstacle(edges, shapes, n_obs, og, a.x, a.y, b.x, b.y);
                }
                const unsigned hits = __ballot_sync(0xffffffffu, o != INT_MAX);
                if (hits) {
                    const int src = __ffs(hits) - 1;
                    hitk = k0 + src;
                    hito = __shfl_sync(0xffffffffu, o, src);
                    break;
                }
            }
        }
        if (lane == 0) {
            flags[path] = (uint8_t)(bad ? UAM_SWEEP_INVALID : (hitk >= 0 ? UAM_SWEEP_HIT : 0));
            if (first_hit) first_hit[path] = hitk;
            if (first_obstacle) first_obstacle[path] = hito;
        }
    }
}

// FILL = 0: counts[cell] = listed obstacles; FILL = 1: items[start[cell] ..] = them in ascending order
template <int FILL>
__global__ void __launch_bounds__(128)
uam_k_obs_grid(const UamEdge* __restrict__ edges, const UamShape* __restrict__ shapes, int n_obs, int G, double gx0,
               double gy0, double cw, double ch, double ext, int* __restrict__ counts, const int* __restrict__ start,
               int* __restrict__ items) {
    const int cell = blockIdx.x * blockDim.x + threadIdx.x;
    if (cell >= G * G) return;
    const int cy = cell / G, cx = cell - cy * G;
    const double xa = cx == 0 ? -ext : gx0 + ((double)cx - kListWiden) * cw;
    const double xb = cx == G - 1 ? ext : gx0 + ((double)cx + 1.0 + kListWiden) * cw;
    const double ya = cy == 0 ? -ext : gy0 + ((double)cy - kListWiden) * ch;
    const double yb = cy == G - 1 ? ext : gy0 + ((double)cy + 1.0 + kListWiden) * ch;
    int n = 0;
    int* dst = FILL ? items + start[cell] : nullptr;
    for (int o = 0; o < n_obs; ++o) {
        const int2 er = __ldg(reinterpret_cast<const int2*>(&shapes[o].e0));
        bool listed = true;
        for (int i = er.x; i < er.y && listed; ++i)
            listed = !uam_edge_excludes_tile(uam_load_edge(edges + i), xa, xb, ya, yb, kThr);
        if (listed) {
            if (FILL) dst[n] = o;
            ++n;
        }
    }
    if (!FILL) counts[cell] = n;
}

// Largest coordinate magnitude Q for which a segment may use the lists of this grid (0 .. Q: the lists are exact for
// it).  With cmin the smaller cell side and every endpoint coordinate within [-Q, Q], for every obstacle record:
//   - the exclusion margin 1e-9 scale of uam_edge_excludes_tile, less that test's own fp64 error at the cell corners
//     (at most 2^-50 M at a corner <= 2Q + 1 away from the origin), exceeds the sweep's eta_i (include/uam_b200.h):
//       line:    scale >= (|Bx-Ax| + |By-Ay|) cmin / 2, eta + error <= |sgn| (|Bx-Ax| + |By-Ay|) 2^-44 (Q + P + 1),
//                P = max(|Ax|, |Ay|)                                          -> Q <= 5e-10 cmin 2^44 / |sgn| - P - 1
//       box:     scale >= cmin / 2 + |c| + |r|, eta + error <= 2^-44 (Q + 1 + |c| + |r|)  -> Q <= 5e-10 cmin 2^44 - 1
//       ellipse: scale >= 2, error <= 2^-50 scale, eta <= 2^-44 (2 + S) + 2^-94 S^2 with
//                S <= (6Q + |cx| + |cy|) / min(|r1|, |r2|); S <= 3e4 keeps eta below 1.71e-9 < (1e-9 - 2^-50) 2
//                                                                             -> Q <= (3e4 min(|r1|, |r2|) - |cx| - |cy|) / 6
//     so an obstacle a cell's list leaves out has no point of K_o^eta in that (widened) cell, and HIT implies such a
//     point on the real segment (G3);
//   - cell coordinates are then exact to ~4 u (Q + |grid|) / cmin <= 2^-22 cells, well inside the walk's margin
//     (Q <= 2^28 cmin - |grid|).
double uam_obs_grid_qmax(const std::vector<UamEdge>& recs, double cmin, double gmag) {
    double q = 0x1p28 * cmin - gmag;
    for (const UamEdge& r : recs) {
        const int kind = (int)r.kind;
        if (kind == UAM_EDGE_LINE) {
            if (r.p4 == 0.0 || (r.p2 == 0.0 && r.p3 == 0.0)) continue;     // h is +-0 everywhere: never excludes
            q = std::min(q, 5e-10 * cmin * 0x1p44 / std::fabs(r.p4) - std::max(std::fabs(r.p0), std::fabs(r.p1)) - 1.0);
        } else if (kind == UAM_EDGE_BOX) {
            q = std::min(q, 5e-10 * cmin * 0x1p44 - 1.0);
        } else {
            q = std::min(q, (3e4 * std::min(std::fabs(r.p2), std::fabs(r.p3)) - std::fabs(r.p0) - std::fabs(r.p1)) / 6.0);
        }
    }
    return q;
}

// On the first call after each upload: copy the obstacles' records back, check them, and (shape_grid option on, at
// least 4 obstacles) build the lists.  Synchronises `st`.
int uam_ensure_obs_tables(uam_ctx* ctx, cudaStream_t st) {
    if (ctx->obs_gen == ctx->shapes_gen) return UAM_OK;
    UAM_NVTX("uam.analytic.sweep.build_lists");
    const int n_obs = ctx->n_obs;
    std::vector<UamShape> shapes(n_obs);
    std::vector<UamEdge> recs;
    if (n_obs > 0) {
        UAM_CUDA(ctx, cudaMemcpy(shapes.data(), ctx->d_shapes, sizeof(UamShape) * n_obs, cudaMemcpyDeviceToHost));
        recs.resize(shapes[n_obs - 1].e1);
        if (!recs.empty())
            UAM_CUDA(ctx, cudaMemcpy(recs.data(), ctx->d_edges, sizeof(UamEdge) * recs.size(), cudaMemcpyDeviceToHost));
    }
    ctx->obs_rc = UAM_OK;
    ctx->obs_err.clear();
    for (int o = 0; o < n_obs && ctx->obs_rc == UAM_OK; ++o) {
        int n_ell = 0;
        for (int i = shapes[o].e0; i < shapes[o].e1; ++i) {
            const UamEdge& r = recs[i];
            const double f[7] = {r.p0, r.p1, r.p2, r.p3, r.p4, r.p5, r.p6};
            bool ok = true;
            for (double v : f) ok = ok && std::fabs(v) <= kBig;     // false for NaN
            const bool ellipse = (int)r.kind == UAM_EDGE_ELLIPSE;
            if (ellipse) ++n_ell;
            char msg[160];
            msg[0] = 0;
            if (!ok)
                snprintf(msg, sizeof msg, "obstacle %d: a record field is not finite or beyond 1e100 in magnitude", o);
            else if (ellipse && !(std::fabs(r.p2) >= 1e-50 && std::fabs(r.p3) >= 1e-50))
                snprintf(msg, sizeof msg, "obstacle %d: an ellipse radius is below 1e-50 in magnitude", o);
            else if (n_ell > 1)
                snprintf(msg, sizeof msg, "obstacle %d has more than one ellipse record", o);
            if (msg[0]) {
                ctx->obs_rc = UAM_ERR_UNSUPPORTED;
                ctx->obs_err = msg;
                break;
            }
        }
    }
    ctx->obs_grid = UamObsGrid{};
    ctx->obs_gen = ctx->shapes_gen;
    if (ctx->obs_rc != UAM_OK || n_obs < 4) return UAM_OK;
    // the grid's box: the obstacles' bounding box as far as the records tell, as for the scorer's grid (every
    // obstacle is listed wherever it may be, so the box only sets the resolution)
    double bx0 = INFINITY, bx1 = -INFINITY, by0 = INFINITY, by1 = -INFINITY;
    for (const UamEdge& r : recs) {
        const int k = (int)r.kind;
        if (k == UAM_EDGE_LINE) {
            bx0 = std::min(bx0, std::min(r.p0, r.p0 + r.p2)); bx1 = std::max(bx1, std::max(r.p0, r.p0 + r.p2));
            by0 = std::min(by0, std::min(r.p1, r.p1 + r.p3)); by1 = std::max(by1, std::max(r.p1, r.p1 + r.p3));
        } else if (k == UAM_EDGE_ELLIPSE) {
            bx0 = std::min(bx0, r.p0 - std::fabs(r.p2)); bx1 = std::max(bx1, r.p0 + std::fabs(r.p2));
            by0 = std::min(by0, r.p1 - std::fabs(r.p3)); by1 = std::max(by1, r.p1 + std::fabs(r.p3));
        } else if ((int)r.p0 == 0) {
            bx0 = std::min(bx0, r.p2 - std::fabs(r.p3)); bx1 = std::max(bx1, r.p2 + std::fabs(r.p3));
        } else {
            by0 = std::min(by0, r.p2 - std::fabs(r.p3)); by1 = std::max(by1, r.p2 + std::fabs(r.p3));
        }
    }
    if (!(bx1 > bx0 && by1 > by0) || !std::isfinite(bx1 - bx0) || !std::isfinite(by1 - by0)) return UAM_OK;
    int G = 32;
    while (G < 256 && G < 8.0 * std::sqrt((double)n_obs)) G *= 2;
    while (G > 8 && (double)G * G * n_obs > 67108864.0) G /= 2;
    const double mx = 0.05 * (bx1 - bx0), my = 0.05 * (by1 - by0);
    const double gx0 = bx0 - mx, gy0 = by0 - my;
    const double cw = (bx1 - bx0 + 2 * mx) / G, ch = (by1 - by0 + 2 * my) / G;
    if (!(cw > 0.0 && ch > 0.0) || !std::isfinite(1.0 / cw) || !std::isfinite(1.0 / ch)) return UAM_OK;
    const double gmag = std::max(std::max(std::fabs(gx0), std::fabs(gx0 + G * cw)), std::max(std::fabs(gy0), std::fabs(gy0 + G * ch)));
    const double qmax = uam_obs_grid_qmax(recs, std::min(cw, ch), gmag);
    if (!(qmax >= gmag)) return UAM_OK;                   // the lists would not be exact for segments inside the grid
    const double ext = 2.0 * qmax + 1.0;
    const int cells = G * G;
    UAM_TRY(uam_reserve(ctx, (void**)&ctx->d_obs_grid, &ctx->obs_grid_bytes, (size_t)(2 * cells + 2) * sizeof(int)));
    int* start = ctx->d_obs_grid;
    int* counts = start + cells + 1;
    const int ctas = (cells + 127) / 128;
    uam_k_obs_grid<0><<<ctas, 128, 0, st>>>(ctx->d_edges, ctx->d_shapes, n_obs, G, gx0, gy0, cw, ch, ext, counts, nullptr,
                                            nullptr);
    UAM_CHECK_LAUNCH(ctx, "uam_k_obs_grid");
    UAM_TRY(uam_shape_grid_scan(ctx, counts, cells, start, st));
    int total = 0;
    UAM_CUDA(ctx, cudaMemcpyAsync(&total, start + cells, sizeof(int), cudaMemcpyDeviceToHost, st));
    UAM_CUDA(ctx, cudaStreamSynchronize(st));
    UAM_TRY(uam_reserve(ctx, (void**)&ctx->d_obs_items, &ctx->obs_items_bytes, (size_t)(total + 1) * sizeof(int)));
    uam_k_obs_grid<1><<<ctas, 128, 0, st>>>(ctx->d_edges, ctx->d_shapes, n_obs, G, gx0, gy0, cw, ch, ext, nullptr, start,
                                            ctx->d_obs_items);
    UAM_CHECK_LAUNCH(ctx, "uam_k_obs_grid");
    UAM_CUDA(ctx, cudaStreamSynchronize(st));
    UamObsGrid og;
    og.gx0 = gx0; og.gy0 = gy0; og.inv_cw = 1.0 / cw; og.inv_ch = 1.0 / ch;
    og.qmax = qmax;
    og.G = G;
    og.start = start;
    og.items = ctx->d_obs_items;
    ctx->obs_grid = og;
    return UAM_OK;
}

}  // namespace

extern "C" int uam_sweep_paths_analytic(uam_ctx* ctx, const double* d_z, int64_t B, int N, uint8_t* d_flags,
                                        int32_t* d_first_hit, int32_t* d_first_obstacle, void* stream) {
    if (!ctx) return UAM_ERR_INVALID;
    if (B < 0 || N < 0 || N > (1 << 28))
        return uam_fail(ctx, UAM_ERR_INVALID, "need B >= 0 and 0 <= N <= 2^28 (got B=%lld N=%d)", (long long)B, N);
    if (B == 0) return UAM_OK;
    if (!d_z || !d_flags) return uam_fail(ctx, UAM_ERR_INVALID, "paths or flags pointer is NULL");
    if (!ctx->has_shapes) return uam_fail(ctx, UAM_ERR_STATE, "no shapes: call uam_map_set_shapes first");
    UAM_NVTX("uam.analytic.sweep");
    UAM_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = uam_pick_stream(ctx, stream);
    if (ctx->obs_gen != ctx->shapes_gen) {
        UAM_CUDA(ctx, cudaDeviceSynchronize());      // a sweep on another stream may still read the old lists
        UAM_TRY(uam_ensure_obs_tables(ctx, st));
    }
    if (ctx->obs_rc != UAM_OK) return uam_fail(ctx, ctx->obs_rc, "%s", ctx->obs_err.c_str());
    const UamObsGrid og = ctx->shape_grid_opt ? ctx->obs_grid : UamObsGrid{};
    const long long ctas = std::min<long long>((B + UAM_WARPS_PER_CTA - 1) / UAM_WARPS_PER_CTA, (long long)ctx->sm_count * 16);
    uam_k_sweep_analytic<<<(unsigned)ctas, UAM_CTA_THREADS, 0, st>>>(reinterpret_cast<const double2*>(d_z), B, N + 2,
                                                                     ctx->d_edges, ctx->d_shapes, ctx->n_obs, og, d_flags,
                                                                     d_first_hit, d_first_obstacle);
    UAM_CHECK_LAUNCH(ctx, "uam_k_sweep_analytic");
    return UAM_OK;
}
