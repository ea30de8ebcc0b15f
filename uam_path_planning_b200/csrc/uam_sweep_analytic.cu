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
// The clearance (uam_clearance_paths_analytic, DESIGN.md 9h) shares HIT, the walk and the table check: D(k, o) = 0 iff
// HIT(k, o), else the fp64 distance from the segment to the obstacle's polygon, box or ellipse.
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

// Visit, in the order of the cells' lists, the obstacles listed in every cell within kWalkMargin cells of the segment
// (ax, ay) -> (bx, by): stop(o) ends the current cell's list (the lists ascend), visit(o) sees each listed obstacle, an
// obstacle listed in consecutive cells once
template <class Stop, class Visit>
__device__ __forceinline__ void uam_walk_obs_lists(const UamObsGrid& og, double ax, double ay, double bx, double by, Stop stop,
                                                   Visit visit) {
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
    int last = -1;
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
                if (stop(o)) break;
                if (o == last) continue;                    // just visited in the previous cell
                last = o;
                visit(o);
            }
        }
    }
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
    int best = INT_MAX;
    uam_walk_obs_lists(og, ax, ay, bx, by, [&](int o) { return o >= best; },       // ascending lists: nothing smaller follows
                       [&](int o) {
                           if (uam_obstacle_hits(edges, shapes, o, ax, ay, bx, by)) best = o;
                       });
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

// ---- clearance (uam_clearance_paths_analytic; DESIGN.md section 9h) -------------------------------------------------
// D(k, o) = 0 iff HIT(k, o); else the fp64 distance from the segment to P_o, at least 2^-1022.  Every candidate below
// is the distance between a computed point near the segment and one near P_o; tests/analytic_clearance_reference.py
// restates the operations in this order.

// squared distance from (px, py) to the segment (ax, ay) + t (dx, dy), t in [0, 1], dd = dx^2 + dy^2
__device__ __forceinline__ double uam_point_segment_d2(double px, double py, double ax, double ay, double dx, double dy,
                                                       double dd) {
    const double wx = __dsub_rn(px, ax), wy = __dsub_rn(py, ay);
    double t = 0.0;
    if (dd > 0.0) t = fmin(fmax(__ddiv_rn(__dadd_rn(__dmul_rn(wx, dx), __dmul_rn(wy, dy)), dd), 0.0), 1.0);
    const double ex = __dsub_rn(px, __dadd_rn(ax, __dmul_rn(t, dx)));
    const double ey = __dsub_rn(py, __dadd_rn(ay, __dmul_rn(t, dy)));
    return __dadd_rn(__dmul_rn(ex, ex), __dmul_rn(ey, ey));
}

// the three point-to-segment candidates of the polygon edge V -> W: V to the path segment, A and B to the edge
__device__ __forceinline__ double uam_edge_d2(double vx, double vy, double wx, double wy, double ax, double ay, double bx,
                                              double by, double dx, double dy, double dd) {
    const double ex = __dsub_rn(wx, vx), ey = __dsub_rn(wy, vy);
    const double ee = __dadd_rn(__dmul_rn(ex, ex), __dmul_rn(ey, ey));
    const double d1 = uam_point_segment_d2(vx, vy, ax, ay, dx, dy, dd);
    const double d2 = uam_point_segment_d2(ax, ay, vx, vy, ex, ey, ee);
    const double d3 = uam_point_segment_d2(bx, by, vx, vy, ex, ey, ee);
    return fmin(d1, fmin(d2, d3));
}

// distance from (y0, y1) >= 0 to the ellipse of semi-axes e0 >= e1 > 0 (Eberly, "Distance from a Point to an Ellipse,
// an Ellipsoid, or a Hyperellipsoid": the root of G(s) by bisection until the midpoint repeats an end)
__device__ __forceinline__ double uam_point_ellipse_dist(double e0, double e1, double y0, double y1) {
    if (y1 > 0.0) {
        if (y0 > 0.0) {
            const double z0 = __ddiv_rn(y0, e0), z1 = __ddiv_rn(y1, e1);
            const double g = __dsub_rn(__dadd_rn(__dmul_rn(z0, z0), __dmul_rn(z1, z1)), 1.0);
            if (g == 0.0) return 0.0;
            const double q = __ddiv_rn(e0, e1), r0 = __dmul_rn(q, q);
            const double n0 = __dmul_rn(r0, z0);
            double s0 = __dsub_rn(z1, 1.0);
            double s1 = g < 0.0 ? 0.0 : __dsub_rn(__dsqrt_rn(__dadd_rn(__dmul_rn(n0, n0), __dmul_rn(z1, z1))), 1.0);
            double s = 0.0;
            for (int it = 0; it < 2200; ++it) {
                s = __dmul_rn(__dadd_rn(s0, s1), 0.5);
                if (s == s0 || s == s1) break;
                const double ra = __ddiv_rn(n0, __dadd_rn(s, r0)), rb = __ddiv_rn(z1, __dadd_rn(s, 1.0));
                const double gs = __dsub_rn(__dadd_rn(__dmul_rn(ra, ra), __dmul_rn(rb, rb)), 1.0);
                if (gs > 0.0) s0 = s;
                else if (gs < 0.0) s1 = s;
                else break;
            }
            const double x0 = __ddiv_rn(__dmul_rn(r0, y0), __dadd_rn(s, r0)), x1 = __ddiv_rn(y1, __dadd_rn(s, 1.0));
            const double u0 = __dsub_rn(x0, y0), u1 = __dsub_rn(x1, y1);
            return __dsqrt_rn(__dadd_rn(__dmul_rn(u0, u0), __dmul_rn(u1, u1)));
        }
        return fabs(__dsub_rn(y1, e1));
    }
    const double numer0 = __dmul_rn(e0, y0), denom0 = __dsub_rn(__dmul_rn(e0, e0), __dmul_rn(e1, e1));
    if (numer0 < denom0) {
        const double xd = __ddiv_rn(numer0, denom0);
        const double x0 = __dmul_rn(e0, xd), x1 = __dmul_rn(e1, __dsqrt_rn(__dsub_rn(1.0, __dmul_rn(xd, xd))));
        const double u0 = __dsub_rn(x0, y0);
        return __dsqrt_rn(__dadd_rn(__dmul_rn(u0, u0), __dmul_rn(x1, x1)));
    }
    return fabs(__dsub_rn(y0, e0));
}

__device__ __forceinline__ double uam_point_ellipse(double px, double py, double cx, double cy, double a, double b) {
    const double y0 = fabs(__dsub_rn(px, cx)), y1 = fabs(__dsub_rn(py, cy));
    return a >= b ? uam_point_ellipse_dist(a, b, y0, y1) : uam_point_ellipse_dist(b, a, y1, y0);
}

// distance from the segment to the boundary point q = c + sg (ox, oy) whose normal is perpendicular to it, if the foot
// of q on the segment's line lies in [0, 1]; +inf otherwise
__device__ __forceinline__ double uam_tangent_dist(double qx, double qy, double ax, double ay, double dx, double dy, double dd) {
    const double wx = __dsub_rn(qx, ax), wy = __dsub_rn(qy, ay);
    const double t = __ddiv_rn(__dadd_rn(__dmul_rn(wx, dx), __dmul_rn(wy, dy)), dd);
    if (!(t >= 0.0 && t <= 1.0)) return INFINITY;
    const double ex = __dsub_rn(qx, __dadd_rn(ax, __dmul_rn(t, dx)));
    const double ey = __dsub_rn(qy, __dadd_rn(ay, __dmul_rn(t, dy)));
    return __dsqrt_rn(__dadd_rn(__dmul_rn(ex, ex), __dmul_rn(ey, ey)));
}

// the fp64 distance from the segment to P_o for a pair that is not HIT, before the clamp at 2^-1022
__device__ double uam_obstacle_distance(const UamEdge* __restrict__ edges, int e0, int e1, const UamObsGeom& g, double ax,
                                        double ay, double bx, double by) {
    const double dx = __dsub_rn(bx, ax), dy = __dsub_rn(by, ay);
    const double dd = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
    if (g.form == UAM_FORM_POLYGON) {
        // the vertices are the records' origins (Ax, Ay), doubles 1 and 2 of each 8-double record
        const double* rec = reinterpret_cast<const double*>(edges);
        const double fx = __ldg(rec + 8 * e0 + 1), fy = __ldg(rec + 8 * e0 + 2);
        double d2 = INFINITY, vx = fx, vy = fy;
        for (int i = e0; i < e1; ++i) {
            const bool closing = i + 1 == e1;
            const double wx = closing ? fx : __ldg(rec + 8 * (i + 1) + 1), wy = closing ? fy : __ldg(rec + 8 * (i + 1) + 2);
            d2 = fmin(d2, uam_edge_d2(vx, vy, wx, wy, ax, ay, bx, by, dx, dy, dd));
            vx = wx; vy = wy;
        }
        return __dsqrt_rn(d2);
    }
    if (g.form == UAM_FORM_BOX) {
        double d2 = uam_edge_d2(g.x0, g.y0, g.x1, g.y0, ax, ay, bx, by, dx, dy, dd);
        d2 = fmin(d2, uam_edge_d2(g.x1, g.y0, g.x1, g.y1, ax, ay, bx, by, dx, dy, dd));
        d2 = fmin(d2, uam_edge_d2(g.x1, g.y1, g.x0, g.y1, ax, ay, bx, by, dx, dy, dd));
        d2 = fmin(d2, uam_edge_d2(g.x0, g.y1, g.x0, g.y0, ax, ay, bx, by, dx, dy, dd));
        return __dsqrt_rn(d2);
    }
    const UamEdge r = uam_load_edge(edges + e0);
    const double a = fabs(r.p2), b = fabs(r.p3);
    if (g.form == UAM_FORM_DISC)
        return __dsub_rn(__dsqrt_rn(uam_point_segment_d2(r.p0, r.p1, ax, ay, dx, dy, dd)), a);
    double d = fmin(uam_point_ellipse(ax, ay, r.p0, r.p1, a, b), uam_point_ellipse(bx, by, r.p0, r.p1, a, b));
    // normal n = (-dy, dx) scaled to max |n_i| = 1; q = c +- (a^2 n_x, b^2 n_y) / sqrt(a^2 n_x^2 + b^2 n_y^2)
    const double nm = fmax(fabs(dx), fabs(dy));
    if (nm > 0.0) {
        const double nx = __ddiv_rn(-dy, nm), ny = __ddiv_rn(dx, nm);
        const double px = __dmul_rn(__dmul_rn(a, a), nx), py = __dmul_rn(__dmul_rn(b, b), ny);
        const double den = __dsqrt_rn(__dadd_rn(__dmul_rn(px, nx), __dmul_rn(py, ny)));
        const double ox = __ddiv_rn(px, den), oy = __ddiv_rn(py, den);
        d = fmin(d, uam_tangent_dist(__dadd_rn(r.p0, ox), __dadd_rn(r.p1, oy), ax, ay, dx, dy, dd));
        d = fmin(d, uam_tangent_dist(__dsub_rn(r.p0, ox), __dsub_rn(r.p1, oy), ax, ay, dx, dy, dd));
    }
    return d;
}

// lower bound of the segment's distance to a box that contains P_o: the larger axis gap, less a margin that covers the
// distance's rounding (DESIGN.md 9h), so skipping a pair with bound > best never changes the result
__device__ __forceinline__ bool uam_prune(const UamObsGeom& g, double ax, double ay, double bx, double by, double best) {
    if (g.form == UAM_FORM_ELLIPSE) return false;
    const double gx = fmax(fmax(__dsub_rn(g.bx0, fmax(ax, bx)), __dsub_rn(fmin(ax, bx), g.bx1)), 0.0);
    const double gy = fmax(fmax(__dsub_rn(g.by0, fmax(ay, by)), __dsub_rn(fmin(ay, by), g.by1)), 0.0);
    const double mag = __dadd_rn(__dadd_rn(fmax(fabs(ax), fabs(bx)), fmax(fabs(ay), fabs(by))),
                                 __dadd_rn(fmax(fabs(g.bx0), fabs(g.bx1)), fmax(fabs(g.by0), fabs(g.by1))));
    return fmax(gx, gy) > __dadd_rn(best, __dadd_rn(__dmul_rn(mag, 0x1p-40), kTiny));
}

// pair (k, o): D and the running minimum (best, besto) of the segment, ties to the smaller o; only D < cap counts
__device__ __forceinline__ void uam_clearance_visit(const UamEdge* __restrict__ edges, const UamShape* __restrict__ shapes,
                                                    const UamObsGeom* __restrict__ geom, int o, double ax, double ay,
                                                    double bx, double by, double& best, int& besto) {
    const int2 er = __ldg(reinterpret_cast<const int2*>(&shapes[o].e0));
    double D = 0.0;
    if (!uam_segment_hits(edges, er.x, er.y, ax, ay, bx, by)) {
        const UamObsGeom g = geom[o];
        if (uam_prune(g, ax, ay, bx, by, best)) return;
        D = fmax(uam_obstacle_distance(edges, er.x, er.y, g, ax, ay, bx, by), 0x1p-1022);
    }
    if (D < best || (D == best && besto >= 0 && o < besto)) {
        best = D;
        besto = o;
    }
}

__device__ __forceinline__ void uam_segment_clearance(const UamEdge* __restrict__ edges, const UamShape* __restrict__ shapes,
                                                      const UamObsGeom* __restrict__ geom, int n_obs, const UamObsGrid& og,
                                                      double ax, double ay, double bx, double by, double& best, int& besto) {
    const double mag = fmax(fmax(fabs(ax), fabs(ay)), fmax(fabs(bx), fabs(by)));
    if (og.G == 0 || !(mag <= og.qmax)) {
        for (int o = 0; o < n_obs && !(best == 0.0 && o > besto); ++o)
            uam_clearance_visit(edges, shapes, geom, o, ax, ay, bx, by, best, besto);
        return;
    }
    uam_walk_obs_lists(og, ax, ay, bx, by, [&](int o) { return best == 0.0 && o >= besto; },   // nothing beats (0, besto)
                       [&](int o) { uam_clearance_visit(edges, shapes, geom, o, ax, ay, bx, by, best, besto); });
}

// one warp per path, segment k on lane k mod 32, as the sweep; each window of 32 segments is reduced to its (D, k, o)
// minimum, and the walk stops after the first window with a HIT (D = 0)
__global__ void __launch_bounds__(UAM_CTA_THREADS, 2)
uam_k_clearance_analytic(const double2* __restrict__ z, int64_t B, int Wp, const UamEdge* __restrict__ edges,
                         const UamShape* __restrict__ shapes, const UamObsGeom* __restrict__ geom, int n_obs, UamObsGrid og,
                         double cap, uint8_t* __restrict__ flags, double* __restrict__ clearance,
                         int32_t* __restrict__ nearest_segment, int32_t* __restrict__ nearest_obstacle) {
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
        double best = cap;
        int bk = -1, bo = -1;
        if (!bad) {
            for (int k0 = 0; k0 < Wp - 1; k0 += 32) {
                const int k = k0 + lane;
                double d = cap;
                int o = -1;
                if (k < Wp - 1) {
                    const double2 a = zp[k], b = zp[k + 1];
                    uam_segment_clearance(edges, shapes, geom, n_obs, og, a.x, a.y, b.x, b.y, d, o);
                }
                double wd = d;
                int wl = lane;
                for (int off = 16; off > 0; off >>= 1) {
                    const double od = __shfl_xor_sync(0xffffffffu, wd, off);
                    const int ol = __shfl_xor_sync(0xffffffffu, wl, off);
                    if (od < wd || (od == wd && ol < wl)) {
                        wd = od;
                        wl = ol;
                    }
                }
                const int wo = __shfl_sync(0xffffffffu, o, wl);
                if (wo >= 0 && wd < best) {
                    best = wd;
                    bk = k0 + wl;
                    bo = wo;
                }
                if (best == 0.0) break;
            }
        }
        if (lane == 0) {
            flags[path] = (uint8_t)(bad ? UAM_SWEEP_INVALID : (best == 0.0 ? UAM_SWEEP_HIT : 0));
            if (clearance) clearance[path] = bad ? (double)NAN : best;
            if (nearest_segment) nearest_segment[path] = bk;
            if (nearest_obstacle) nearest_obstacle[path] = bo;
        }
    }
}

// clearance lists: FILL = 0: counts[cell]; FILL = 1: items[start[cell] ..] ascending.  An obstacle is listed where the
// sweep lists it (no record excludes the cell) or where its box dilated by dil[o] meets the cell's box
template <int FILL>
__global__ void __launch_bounds__(128)
uam_k_clr_grid(const UamEdge* __restrict__ edges, const UamShape* __restrict__ shapes, const UamObsGeom* __restrict__ geom,
               const double* __restrict__ dil, int n_obs, int G, double gx0, double gy0, double cw, double ch, double ext,
               int* __restrict__ counts, const int* __restrict__ start, int* __restrict__ items) {
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
        const UamObsGeom g = geom[o];
        const double r = dil[o];
        const double gx = fmax(fmax(g.bx0 - xb, xa - g.bx1), 0.0), gy = fmax(fmax(g.by0 - yb, ya - g.by1), 0.0);
        bool listed = gx <= r && gy <= r && gx * gx + gy * gy <= r * r;
        if (!listed) {
            const int2 er = __ldg(reinterpret_cast<const int2*>(&shapes[o].e0));
            listed = true;
            for (int i = er.x; i < er.y && listed; ++i)
                listed = !uam_edge_excludes_tile(uam_load_edge(edges + i), xa, xb, ya, yb, kThr);
        }
        if (listed) {
            if (FILL) dst[n] = o;
            ++n;
        }
    }
    if (!FILL) counts[cell] = n;
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

// The clearance's form of every obstacle and a box that contains it (DESIGN.md 9h):
//   polygon: >= 3 line records, each direction ending at the next origin (to 2^-50 of the two origins' magnitudes, per
//            component, cyclically), and every origin but the record's own two strictly inside it (fp64 h < 0): the origins are a
//            strictly convex polygon in hull order and every sign points inward; P_o is their hull;
//   box:     4 box records, one per (axis, sign), with c - r <= c + r on each axis; P_o is the rectangle;
//   ellipse: one ellipse record (a disc when |r1| == |r2|).
// Anything else is UAM_ERR_UNSUPPORTED, with a message naming the obstacle.
int uam_obs_forms(const std::vector<UamShape>& shapes, const std::vector<UamEdge>& recs, std::vector<UamObsGeom>& geom,
                  std::string& err) {
    const int n_obs = (int)shapes.size();
    geom.assign(n_obs, UamObsGeom{});
    char msg[200];
    for (int o = 0; o < n_obs; ++o) {
        const int e0 = shapes[o].e0, n = shapes[o].e1 - shapes[o].e0;
        int n_line = 0, n_box = 0, n_ell = 0;
        for (int i = e0; i < e0 + n; ++i) {
            const int k = (int)recs[i].kind;
            n_line += k == UAM_EDGE_LINE;
            n_box += k == UAM_EDGE_BOX;
            n_ell += k == UAM_EDGE_ELLIPSE;
        }
        UamObsGeom& g = geom[o];
        g.rho = 1.0;
        const char* why = nullptr;
        if (n_line == n && n >= 3) {
            g.form = UAM_FORM_POLYGON;
            g.bx0 = g.by0 = INFINITY;
            g.bx1 = g.by1 = -INFINITY;
            for (int i = 0; i < n && !why; ++i) {
                const UamEdge& a = recs[e0 + i];
                const UamEdge& b = recs[e0 + (i + 1) % n];
                if (!(std::fabs((a.p0 + a.p2) - b.p0) <= 0x1p-50 * (std::fabs(a.p0) + std::fabs(b.p0)) &&
                      std::fabs((a.p1 + a.p3) - b.p1) <= 0x1p-50 * (std::fabs(a.p1) + std::fabs(b.p1))))
                    why = "a line record's direction does not end at the next record's origin";
                for (int j = 0; j < n && !why; ++j) {
                    if (j == i || j == (i + 1) % n) continue;
                    const UamEdge& v = recs[e0 + j];
                    const double h = -a.p4 * (a.p3 * (v.p0 - a.p0) - a.p2 * (v.p1 - a.p1));
                    if (!(h < 0.0)) why = "its line records' origins are not a strictly convex polygon with inward signs";
                }
                g.bx0 = std::min(g.bx0, a.p0); g.bx1 = std::max(g.bx1, a.p0);
                g.by0 = std::min(g.by0, a.p1); g.by1 = std::max(g.by1, a.p1);
            }
        } else if (n_box == n && n == 4) {
            g.form = UAM_FORM_BOX;
            int seen = 0;
            for (int i = e0; i < e0 + 4; ++i) {
                const UamEdge& r = recs[i];
                const bool x = (int)r.p0 == 0, plus = r.p1 > 0;
                seen |= 1 << ((x ? 0 : 2) + (plus ? 0 : 1));
                double& v = x ? (plus ? g.x1 : g.x0) : (plus ? g.y1 : g.y0);
                v = plus ? r.p2 + r.p3 : r.p2 - r.p3;      // sign > 0: x_d <= c + r; else x_d >= c - r
            }
            if (seen != 15) why = "its box records are not one for each axis and sign";
            else if (!(g.x0 <= g.x1 && g.y0 <= g.y1)) why = "its box records bound an empty rectangle";
            g.bx0 = g.x0; g.bx1 = g.x1; g.by0 = g.y0; g.by1 = g.y1;
        } else if (n_ell == 1 && n == 1) {
            const UamEdge& r = recs[e0];
            const double a = std::fabs(r.p2), b = std::fabs(r.p3);
            g.form = a == b ? UAM_FORM_DISC : UAM_FORM_ELLIPSE;
            if (g.form == UAM_FORM_ELLIPSE) g.rho = std::max(a, b) / std::min(a, b);
            g.bx0 = r.p0 - a; g.bx1 = r.p0 + a; g.by0 = r.p1 - b; g.by1 = r.p1 + b;
        } else {
            why = "not a polygon, a box or an ellipse (the forms polygon(), square() and ball() make)";
        }
        if (why) {
            snprintf(msg, sizeof msg, "clearance: obstacle %d: %s", o, why);
            err = msg;
            return UAM_ERR_UNSUPPORTED;
        }
        // outward by more than the rounding of c -+ r
        const double m = 0x1p-44 * std::max(std::max(std::fabs(g.bx0), std::fabs(g.bx1)), std::max(std::fabs(g.by0), std::fabs(g.by1))) + kTiny;
        g.bx0 -= m; g.bx1 += m; g.by0 -= m; g.by1 += m;
    }
    return UAM_OK;
}

}  // namespace

// On the first call after each upload: copy the obstacles' records back, check them, and (shape_grid option on, at
// least 4 obstacles) build the lists.  Synchronises the device first (a call on another stream may still read the old
// lists), then `st`.
int uam_ensure_obs_tables(uam_ctx* ctx, cudaStream_t st) {
    if (ctx->obs_gen == ctx->shapes_gen) return UAM_OK;
    UAM_NVTX("uam.analytic.sweep.build_lists");
    UAM_CUDA(ctx, cudaDeviceSynchronize());
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
    ctx->clr_gen = 0;
    ctx->clr_rc = UAM_OK;
    ctx->clr_err.clear();
    if (ctx->obs_rc != UAM_OK) return UAM_OK;
    {
        std::vector<UamObsGeom> geom;
        ctx->clr_rc = uam_obs_forms(shapes, recs, geom, ctx->clr_err);
        if (ctx->clr_rc == UAM_OK && n_obs > 0) {
            UAM_TRY(uam_reserve(ctx, (void**)&ctx->d_obs_geom, &ctx->obs_geom_bytes, sizeof(UamObsGeom) * n_obs));
            UAM_CUDA(ctx, cudaMemcpy(ctx->d_obs_geom, geom.data(), sizeof(UamObsGeom) * n_obs, cudaMemcpyHostToDevice));
        }
        ctx->h_obs_geom = geom;
    }
    if (n_obs < 4) return UAM_OK;
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
    ctx->obs_cw = cw; ctx->obs_ch = ch; ctx->obs_ext = ext;
    return UAM_OK;
}

// Clearance lists for `cap` (the first call after each upload or change of cap; synchronises `st`): in the sweep grid's
// cells, every obstacle the sweep lists there and every obstacle whose box lies within dil_o = cap (1 + 2^-40) +
// 2^-36 rho_o (qmax + |box|) of the cell (the second term exceeds the distance's error bound delta, DESIGN.md 9h).  No
// lists (every segment tests every obstacle) where the sweep has none or where they would hold over 3/4 of all pairs.
// Nothing is built with the shape_grid option off.  Synchronises the device first (a clearance call on another stream
// may still read the old lists), then `st`.
int uam_ensure_clr_lists(uam_ctx* ctx, double cap, cudaStream_t st) {
    if (!ctx->shape_grid_opt || (ctx->clr_gen == ctx->shapes_gen && ctx->clr_cap == cap)) return UAM_OK;
    UAM_NVTX("uam.analytic.clearance.build_lists");
    UAM_CUDA(ctx, cudaDeviceSynchronize());
    ctx->clr_grid = UamObsGrid{};
    ctx->clr_gen = ctx->shapes_gen;
    ctx->clr_cap = cap;
    const UamObsGrid& og = ctx->obs_grid;
    const int n_obs = ctx->n_obs;
    if (og.G == 0) return UAM_OK;
    std::vector<double> dil(n_obs);
    for (int o = 0; o < n_obs; ++o) {
        const UamObsGeom& g = ctx->h_obs_geom[o];
        const double bm = std::max(std::max(std::fabs(g.bx0), std::fabs(g.bx1)), std::max(std::fabs(g.by0), std::fabs(g.by1)));
        dil[o] = cap * (1.0 + 0x1p-40) + 0x1p-36 * g.rho * (og.qmax + bm);
    }
    const int G = og.G, cells = G * G;
    const size_t ints = ((size_t)(2 * cells + 2) + 1) & ~(size_t)1;          // keep the doubles after them 8-byte aligned
    UAM_TRY(uam_reserve(ctx, (void**)&ctx->d_clr_grid, &ctx->clr_grid_bytes, ints * sizeof(int) + n_obs * sizeof(double)));
    int* start = ctx->d_clr_grid;
    int* counts = start + cells + 1;
    double* d_dil = reinterpret_cast<double*>(start + ints);
    UAM_CUDA(ctx, cudaMemcpyAsync(d_dil, dil.data(), n_obs * sizeof(double), cudaMemcpyHostToDevice, st));
    const int ctas = (cells + 127) / 128;
    uam_k_clr_grid<0><<<ctas, 128, 0, st>>>(ctx->d_edges, ctx->d_shapes, ctx->d_obs_geom, d_dil, n_obs, G, og.gx0, og.gy0,
                                            ctx->obs_cw, ctx->obs_ch, ctx->obs_ext, counts, nullptr, nullptr);
    UAM_CHECK_LAUNCH(ctx, "uam_k_clr_grid");
    UAM_TRY(uam_shape_grid_scan(ctx, counts, cells, start, st));
    int total = 0;
    UAM_CUDA(ctx, cudaMemcpyAsync(&total, start + cells, sizeof(int), cudaMemcpyDeviceToHost, st));
    UAM_CUDA(ctx, cudaStreamSynchronize(st));
    if ((double)total > 0.75 * cells * n_obs) return UAM_OK;
    UAM_TRY(uam_reserve(ctx, (void**)&ctx->d_clr_items, &ctx->clr_items_bytes, (size_t)(total + 1) * sizeof(int)));
    uam_k_clr_grid<1><<<ctas, 128, 0, st>>>(ctx->d_edges, ctx->d_shapes, ctx->d_obs_geom, d_dil, n_obs, G, og.gx0, og.gy0,
                                            ctx->obs_cw, ctx->obs_ch, ctx->obs_ext, nullptr, start, ctx->d_clr_items);
    UAM_CHECK_LAUNCH(ctx, "uam_k_clr_grid");
    UAM_CUDA(ctx, cudaStreamSynchronize(st));
    UamObsGrid cg = og;
    cg.start = start;
    cg.items = ctx->d_clr_items;
    ctx->clr_grid = cg;
    return UAM_OK;
}

int uam_obs_supported(uam_ctx* ctx, bool clearance) {
    if (ctx->obs_rc != UAM_OK) return uam_fail(ctx, ctx->obs_rc, "%s", ctx->obs_err.c_str());
    if (clearance && ctx->clr_rc != UAM_OK) return uam_fail(ctx, ctx->clr_rc, "%s", ctx->clr_err.c_str());
    return UAM_OK;
}

int uam_sweep_analytic_enqueue(uam_ctx* ctx, const double* d_z, int64_t B, int N, uint8_t* d_flags, int32_t* d_first_hit,
                               int32_t* d_first_obstacle, cudaStream_t st) {
    const UamObsGrid og = ctx->shape_grid_opt ? ctx->obs_grid : UamObsGrid{};
    const long long ctas = std::min<long long>((B + UAM_WARPS_PER_CTA - 1) / UAM_WARPS_PER_CTA, (long long)ctx->sm_count * 16);
    uam_k_sweep_analytic<<<(unsigned)ctas, UAM_CTA_THREADS, 0, st>>>(reinterpret_cast<const double2*>(d_z), B, N + 2,
                                                                     ctx->d_edges, ctx->d_shapes, ctx->n_obs, og, d_flags,
                                                                     d_first_hit, d_first_obstacle);
    UAM_CHECK_LAUNCH(ctx, "uam_k_sweep_analytic");
    return UAM_OK;
}

int uam_clearance_analytic_enqueue(uam_ctx* ctx, const double* d_z, int64_t B, int N, double cap, uint8_t* d_flags,
                                   double* d_clearance, int32_t* d_nearest_segment, int32_t* d_nearest_obstacle,
                                   cudaStream_t st) {
    const UamObsGrid og = ctx->shape_grid_opt ? ctx->clr_grid : UamObsGrid{};
    const long long ctas = std::min<long long>((B + UAM_WARPS_PER_CTA - 1) / UAM_WARPS_PER_CTA, (long long)ctx->sm_count * 16);
    uam_k_clearance_analytic<<<(unsigned)ctas, UAM_CTA_THREADS, 0, st>>>(
        reinterpret_cast<const double2*>(d_z), B, N + 2, ctx->d_edges, ctx->d_shapes, ctx->d_obs_geom, ctx->n_obs, og, cap,
        d_flags, d_clearance, d_nearest_segment, d_nearest_obstacle);
    UAM_CHECK_LAUNCH(ctx, "uam_k_clearance_analytic");
    return UAM_OK;
}

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
    UAM_TRY(uam_ensure_obs_tables(ctx, st));
    UAM_TRY(uam_obs_supported(ctx, false));
    return uam_sweep_analytic_enqueue(ctx, d_z, B, N, d_flags, d_first_hit, d_first_obstacle, st);
}

extern "C" int uam_clearance_paths_analytic(uam_ctx* ctx, const double* d_z, int64_t B, int N, double cap, uint8_t* d_flags,
                                            double* d_clearance, int32_t* d_nearest_segment, int32_t* d_nearest_obstacle,
                                            void* stream) {
    if (!ctx) return UAM_ERR_INVALID;
    if (B < 0 || N < 0 || N > (1 << 28) || !(cap > 0.0 && cap <= kBig))
        return uam_fail(ctx, UAM_ERR_INVALID, "need B >= 0, 0 <= N <= 2^28 and 0 < cap <= 1e100 (got B=%lld N=%d cap=%g)",
                        (long long)B, N, cap);
    if (B == 0) return UAM_OK;
    if (!d_z || !d_flags) return uam_fail(ctx, UAM_ERR_INVALID, "paths or flags pointer is NULL");
    if (!ctx->has_shapes) return uam_fail(ctx, UAM_ERR_STATE, "no shapes: call uam_map_set_shapes first");
    UAM_NVTX("uam.analytic.clearance");
    UAM_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = uam_pick_stream(ctx, stream);
    UAM_TRY(uam_ensure_obs_tables(ctx, st));
    UAM_TRY(uam_obs_supported(ctx, true));
    UAM_TRY(uam_ensure_clr_lists(ctx, cap, st));
    return uam_clearance_analytic_enqueue(ctx, d_z, B, N, cap, d_flags, d_clearance, d_nearest_segment, d_nearest_obstacle,
                                          st);
}
