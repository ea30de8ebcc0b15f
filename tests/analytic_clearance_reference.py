"""Restatements of uam_clearance_paths_analytic (include/uam_b200.h) for the tests.

``obstacle_form`` is the host's form check, ``pair_distance`` the device's D(k, o) in numpy, in the kernel's fp64
operation order (numpy float64 arithmetic is round-to-nearest without contraction), vectorised over segments, and
``clearance_reference`` reduces it to the per-path outputs: the D3 reference, bit for bit.  HIT comes from
analytic_sweep_reference.segment_hits.  ``exact_distance`` is the oracle of D2: fractions.Fraction squared distances for
polygons and boxes, mpmath at 50 digits for discs and ellipses.
"""
from fractions import Fraction

import mpmath
import numpy as np

from analytic_sweep_reference import BIG, BOX, ELLIPSE, HIT, INVALID, LINE, segment_hits

POLYGON_FORM, ELLIPSE_FORM, BOX_FORM, DISC_FORM = 0, 1, 2, 3
TINY = 2.0 ** -1022


class Unsupported(ValueError):
    pass


def obstacle_form(recs):
    """(form, data) of one obstacle's records (n, 8), as the host decides it; data: polygon (n, 2) vertices, box
    (x0, x1, y0, y1), disc / ellipse the record.  Raises Unsupported for anything else."""
    recs = np.asarray(recs, dtype=np.float64).reshape(-1, 8)
    kinds = recs[:, 0].astype(int)
    n = len(recs)
    if n >= 3 and np.all(kinds == LINE):
        for i in range(n):
            a, b = recs[i], recs[(i + 1) % n]
            for c in (1, 2):
                if not abs((a[c] + a[c + 2]) - b[c]) <= 2.0 ** -50 * (abs(a[c]) + abs(b[c])):
                    raise Unsupported('direction does not end at the next origin')
            for j in range(n):
                if j != i and j != (i + 1) % n:
                    v = recs[j]
                    h = -a[5] * (a[4] * (v[1] - a[1]) - a[3] * (v[2] - a[2]))
                    if not h < 0.0:
                        raise Unsupported('not a strictly convex polygon with inward signs')
        return POLYGON_FORM, recs[:, 1:3].copy()
    if n == 4 and np.all(kinds == BOX):
        lim, seen = {}, set()
        for r in recs:
            x, plus = int(r[1]) == 0, r[2] > 0
            seen.add((x, plus))
            lim[(x, plus)] = r[3] + r[4] if plus else r[3] - r[4]
        if len(seen) != 4:
            raise Unsupported('box records are not one per axis and sign')
        x0, x1, y0, y1 = lim[(True, False)], lim[(True, True)], lim[(False, False)], lim[(False, True)]
        if not (x0 <= x1 and y0 <= y1):
            raise Unsupported('empty box')
        return BOX_FORM, (x0, x1, y0, y1)
    if n == 1 and kinds[0] == ELLIPSE:
        return (DISC_FORM if abs(recs[0, 3]) == abs(recs[0, 4]) else ELLIPSE_FORM), recs[0]
    raise Unsupported('not a polygon, a box or an ellipse')


# ---- the device's arithmetic -----------------------------------------------------------------------------------------
def point_segment_d2(px, py, ax, ay, dx, dy, dd):
    wx, wy = px - ax, py - ay
    pos = dd > 0.0
    t = np.where(pos, np.minimum(np.maximum((wx * dx + wy * dy) / np.where(pos, dd, 1.0), 0.0), 1.0), 0.0)
    ex = px - (ax + t * dx)
    ey = py - (ay + t * dy)
    return ex * ex + ey * ey


def edge_d2(vx, vy, wx, wy, ax, ay, bx, by, dx, dy, dd):
    ex, ey = wx - vx, wy - vy
    ee = ex * ex + ey * ey
    d1 = point_segment_d2(vx, vy, ax, ay, dx, dy, dd)
    d2 = point_segment_d2(ax, ay, vx, vy, ex, ey, ee)
    d3 = point_segment_d2(bx, by, vx, vy, ex, ey, ee)
    return np.minimum(d1, np.minimum(d2, d3))


def point_ellipse_dist(e0, e1, y0, y1):
    """Eberly's distance from (y0, y1) >= 0 to the ellipse of semi-axes e0 >= e1 (arrays), the device's bisection."""
    e0, e1, y0, y1 = np.broadcast_arrays(*(np.asarray(v, dtype=np.float64) for v in (e0, e1, y0, y1)))
    out = np.empty(y0.shape)
    # y1 == 0
    m = ~(y1 > 0.0)
    numer0, denom0 = e0 * y0, e0 * e0 - e1 * e1
    inner = m & (numer0 < denom0)
    xd = numer0 / np.where(inner, denom0, 1.0)
    x0, x1 = e0 * xd, e1 * np.sqrt(np.where(inner, 1.0 - xd * xd, 0.0))
    u0 = x0 - y0
    out = np.where(inner, np.sqrt(u0 * u0 + x1 * x1), np.abs(y0 - e0))
    # y1 > 0, y0 == 0
    out = np.where((y1 > 0.0) & ~(y0 > 0.0), np.abs(y1 - e1), out)
    # y1 > 0, y0 > 0
    gen = (y1 > 0.0) & (y0 > 0.0)
    z0, z1 = y0 / e0, y1 / e1
    g = (z0 * z0 + z1 * z1) - 1.0
    q = e0 / e1
    r0 = q * q
    n0 = r0 * z0
    s0 = z1 - 1.0
    s1 = np.where(g < 0.0, 0.0, np.sqrt(n0 * n0 + z1 * z1) - 1.0)
    s = np.zeros(y0.shape)
    act = gen & (g != 0.0)
    for _ in range(2200):
        if not act.any():
            break
        sm = (s0 + s1) * 0.5
        s = np.where(act, sm, s)
        stop = act & ((sm == s0) | (sm == s1))
        act = act & ~stop
        ra, rb = n0 / (sm + r0), z1 / (sm + 1.0)
        gs = (ra * ra + rb * rb) - 1.0
        s0 = np.where(act & (gs > 0.0), sm, s0)
        s1 = np.where(act & (gs < 0.0), sm, s1)
        act = act & (gs != 0.0)
    x0, x1 = (r0 * y0) / (s + r0), y1 / (s + 1.0)
    u0, u1 = x0 - y0, x1 - y1
    d = np.where(g == 0.0, 0.0, np.sqrt(u0 * u0 + u1 * u1))
    return np.where(gen, d, out)


def point_ellipse(px, py, cx, cy, a, b):
    y0, y1 = np.abs(px - cx), np.abs(py - cy)
    if a >= b:
        return point_ellipse_dist(a, b, y0, y1)
    return point_ellipse_dist(b, a, y1, y0)


def tangent_dist(qx, qy, ax, ay, dx, dy, dd):
    wx, wy = qx - ax, qy - ay
    t = (wx * dx + wy * dy) / np.where(dd > 0.0, dd, 1.0)
    ex = qx - (ax + t * dx)
    ey = qy - (ay + t * dy)
    return np.where((t >= 0.0) & (t <= 1.0) & (dd > 0.0), np.sqrt(ex * ex + ey * ey), np.inf)


def obstacle_distance(form, data, ax, ay, bx, by):
    """The fp64 distance of a pair that is not HIT, before the clamp (arrays of segments)."""
    with np.errstate(all='ignore'):
        dx, dy = bx - ax, by - ay
        dd = dx * dx + dy * dy
        if form in (POLYGON_FORM, BOX_FORM):
            if form == BOX_FORM:
                x0, x1, y0, y1 = data
                V = np.array([[x0, y0], [x1, y0], [x1, y1], [x0, y1]])
            else:
                V = data
            d2 = np.full(ax.shape, np.inf)
            for i in range(len(V)):
                v, w = V[i], V[(i + 1) % len(V)]
                d2 = np.minimum(d2, edge_d2(v[0], v[1], w[0], w[1], ax, ay, bx, by, dx, dy, dd))
            return np.sqrt(d2)
        r = data
        a, b = abs(r[3]), abs(r[4])
        if form == DISC_FORM:
            return np.sqrt(point_segment_d2(r[1], r[2], ax, ay, dx, dy, dd)) - a
        d = np.minimum(point_ellipse(ax, ay, r[1], r[2], a, b), point_ellipse(bx, by, r[1], r[2], a, b))
        nm = np.maximum(np.abs(dx), np.abs(dy))
        pos = nm > 0.0
        nms = np.where(pos, nm, 1.0)
        nx, ny = -dy / nms, dx / nms
        px, py = (a * a) * nx, (b * b) * ny
        den = np.sqrt(px * nx + py * ny)
        den = np.where(pos, den, 1.0)
        ox, oy = px / den, py / den
        d = np.minimum(d, np.where(pos, tangent_dist(r[1] + ox, r[2] + oy, ax, ay, dx, dy, dd), np.inf))
        d = np.minimum(d, np.where(pos, tangent_dist(r[1] - ox, r[2] - oy, ax, ay, dx, dy, dd), np.inf))
        return d


def pair_distance(recs, ax, ay, bx, by, form=None):
    """D(k, o) for one obstacle and segments given as float64 arrays of equal shape."""
    ax, ay, bx, by = (np.asarray(v, dtype=np.float64) for v in (ax, ay, bx, by))
    form = obstacle_form(recs) if form is None else form
    hit = segment_hits(recs, ax, ay, bx, by)
    with np.errstate(all='ignore'):
        D = np.fmax(obstacle_distance(*form, ax, ay, bx, by), TINY)
    return np.where(hit, 0.0, D)


def clearance_reference(Z, obstacle_records, cap):
    """Per-path (flags u8, clearance f64, nearest_segment i32, nearest_obstacle i32) for paths Z (B, 2(N+2))."""
    Z = np.asarray(Z, dtype=np.float64)
    B = Z.shape[0]
    P = Z.reshape(B, -1, 2)
    bad = ~np.all(np.abs(Z) < BIG, axis=1)
    A, Bp = P[:, :-1], P[:, 1:]
    best = np.full(A.shape[:2], float(cap))
    besto = np.full(A.shape[:2], -1, dtype=np.int64)
    for o, recs in enumerate(obstacle_records):
        D = pair_distance(recs, A[..., 0], A[..., 1], Bp[..., 0], Bp[..., 1])
        upd = D < best                                   # ascending o: a tie keeps the smaller o
        best = np.where(upd, D, best)
        besto = np.where(upd, o, besto)
    has = besto >= 0
    segmin = np.where(has, best, np.inf)
    k = segmin.argmin(axis=1) if segmin.shape[1] else np.zeros(B, dtype=np.int64)
    dmin = segmin[np.arange(B), k] if segmin.shape[1] else np.full(B, np.inf)
    near = np.isfinite(dmin) & ~bad
    clearance = np.where(bad, np.nan, np.where(near, dmin, float(cap)))
    kk = np.where(near, k, -1)
    oo = np.where(near, besto[np.arange(B), np.maximum(k, 0)], -1)
    flags = np.where(bad, INVALID, np.where(near & (dmin == 0.0), HIT, 0)).astype(np.uint8)
    return flags, clearance, kk.astype(np.int32), oo.astype(np.int32)


# ---- the oracle ------------------------------------------------------------------------------------------------------
def _F(v):
    return Fraction(float(v))


def _pt_seg_d2_exact(P, A, B):
    d = (B[0] - A[0], B[1] - A[1])
    dd = d[0] * d[0] + d[1] * d[1]
    w = (P[0] - A[0], P[1] - A[1])
    t = Fraction(0) if dd == 0 else min(max((w[0] * d[0] + w[1] * d[1]) / dd, Fraction(0)), Fraction(1))
    e = (P[0] - A[0] - t * d[0], P[1] - A[1] - t * d[1])
    return e[0] * e[0] + e[1] * e[1]


def _mp_point_ellipse(px, py, cx, cy, a, b):
    """Distance from a point outside (or on) the ellipse to it, at mpmath's precision (bisection on Eberly's G)."""
    y0, y1 = abs(px - cx), abs(py - cy)
    if b > a:
        a, b, y0, y1 = b, a, y1, y0
    if y1 == 0:
        return abs(y0 - a) if a * y0 >= a * a - b * b else None
    if y0 == 0:
        return abs(y1 - b)
    z0, z1 = y0 / a, y1 / b
    r0 = (a / b) ** 2
    lo, hi = z1 - 1, mpmath.sqrt((r0 * z0) ** 2 + z1 ** 2) - 1
    for _ in range(400):
        s = (lo + hi) / 2
        g = (r0 * z0 / (s + r0)) ** 2 + (z1 / (s + 1)) ** 2 - 1
        if g > 0:
            lo = s
        else:
            hi = s
    s = (lo + hi) / 2
    x0, x1 = r0 * y0 / (s + r0), y1 / (s + 1)
    return mpmath.sqrt((x0 - y0) ** 2 + (x1 - y1) ** 2)


def exact_distance(recs, ax, ay, bx, by):
    """dist(segment, P_o) for a segment disjoint from P_o, as an mpmath number at 50 digits."""
    form, data = obstacle_form(recs)
    with mpmath.workdps(50):
        if form in (POLYGON_FORM, BOX_FORM):
            if form == BOX_FORM:
                x0, x1, y0, y1 = data
                V = [(_F(x0), _F(y0)), (_F(x1), _F(y0)), (_F(x1), _F(y1)), (_F(x0), _F(y1))]
            else:
                V = [(_F(v[0]), _F(v[1])) for v in data]
            A, B = (_F(ax), _F(ay)), (_F(bx), _F(by))
            d2 = min(min(_pt_seg_d2_exact(V[i], A, B), _pt_seg_d2_exact(A, V[i], V[(i + 1) % len(V)]),
                         _pt_seg_d2_exact(B, V[i], V[(i + 1) % len(V)])) for i in range(len(V)))
            return mpmath.sqrt(mpmath.mpf(d2.numerator) / d2.denominator)
        m = mpmath.mpf
        cx, cy, a, b = m(float(data[1])), m(float(data[2])), abs(m(float(data[3]))), abs(m(float(data[4])))
        A, B = (m(float(ax)), m(float(ay))), (m(float(bx)), m(float(by)))
        d = (B[0] - A[0], B[1] - A[1])
        dd = d[0] ** 2 + d[1] ** 2
        cands = [_mp_point_ellipse(A[0], A[1], cx, cy, a, b), _mp_point_ellipse(B[0], B[1], cx, cy, a, b)]
        if dd > 0:
            n = (-d[1], d[0])
            den = mpmath.sqrt(a * a * n[0] ** 2 + b * b * n[1] ** 2)
            for sg in (1, -1):
                q = (cx + sg * a * a * n[0] / den, cy + sg * b * b * n[1] / den)
                t = ((q[0] - A[0]) * d[0] + (q[1] - A[1]) * d[1]) / dd
                if 0 <= t <= 1:
                    cands.append(mpmath.sqrt((q[0] - A[0] - t * d[0]) ** 2 + (q[1] - A[1] - t * d[1]) ** 2))
        return min(c for c in cands if c is not None)


def delta(recs, ax, ay, bx, by, D):
    """D2's bound for a pair that is not HIT (D the exact distance, float)."""
    form, data = obstacle_form(recs)
    M = max(abs(ax), abs(ay), abs(bx), abs(by))
    rho = 1.0
    if form == POLYGON_FORM:
        M = max(M, float(np.abs(data).max()))
    elif form == BOX_FORM:
        M = max(M, *(abs(v) for v in data))
    else:
        e0, e1 = max(abs(data[3]), abs(data[4])), min(abs(data[3]), abs(data[4]))
        M = max(M, abs(data[1]) + e0, abs(data[2]) + e0)
        if form == ELLIPSE_FORM:
            rho = e0 / e1
            return 2.0 ** -40 * rho * M + 4 * 2.0 ** -53 * D + 2.0 ** -1000
    return 2.0 ** -48 * M + 4 * 2.0 ** -53 * D + 2.0 ** -1000
