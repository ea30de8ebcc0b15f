"""Restatements of uam_sweep_paths_analytic (include/uam_b200.h) for the tests.

``segment_hits`` is the device's HIT(k, o) in numpy, in the kernel's fp64 operation order (numpy float64 arithmetic is
round-to-nearest without contraction), vectorised over segments: the G4 reference, bit for bit.  ``sweep_reference``
reduces it to the per-path outputs.  ``exact_meets`` decides in exact rational arithmetic (fractions.Fraction) whether a
segment meets K_o, or K_o^eta with per-record slack: the oracle of G1 and G3.  Records are the 8-double rows of
``uam_map_set_shapes`` (``QuadraticObstacle.records()``).
"""
from fractions import Fraction

import numpy as np

HIT, OUTSIDE, INVALID = 1, 2, 4
THR = 1e-14
TINY = 2.0 ** -1000
BIG = 1e100
LINE, ELLIPSE, BOX = 0, 1, 2


def h_exact(r, x, y):
    """uam_h_exact (fp64, the reference's order)."""
    k = int(r[0])
    if k == LINE:
        return -r[5] * (r[4] * (x - r[1]) - r[3] * (y - r[2]))
    if k == ELLIPSE:
        a = (x - r[1]) / r[3]
        b = (y - r[2]) / r[4]
        return (a * a + b * b) - 1.0
    xd = x if int(r[1]) == 0 else y
    return (xd - r[3]) - r[4] if r[2] > 0 else (-xd + r[3]) - r[4]


def affine_mag(r, x, y):
    """M_i(x, y) of an affine record."""
    if int(r[0]) == LINE:
        mx = abs(r[4]) * (np.abs(x) + abs(r[1]))
        my = abs(r[3]) * (np.abs(y) + abs(r[2]))
        return abs(r[5]) * (mx + my)
    xd = x if int(r[1]) == 0 else y
    return (np.abs(xd) + abs(r[3])) + abs(r[4])


def segment_hits(recs, ax, ay, bx, by):
    """HIT(k, o) for one obstacle's records (n, 8) and segments given as float64 arrays of equal shape."""
    recs = np.asarray(recs, dtype=np.float64).reshape(-1, 8)
    ax, ay, bx, by = (np.asarray(v, dtype=np.float64) for v in (ax, ay, bx, by))
    with np.errstate(all='ignore'):
        in_a = np.ones(ax.shape, dtype=bool)
        in_b = np.ones(ax.shape, dtype=bool)
        lo = np.zeros(ax.shape)
        hi = np.ones(ax.shape)
        ell = None
        for r in recs:
            ha, hb = h_exact(r, ax, ay), h_exact(r, bx, by)
            in_a &= ha <= THR
            in_b &= hb <= THR
            if int(r[0]) == ELLIPSE:
                ell = r
                continue
            la = ha - (affine_mag(r, ax, ay) * 2.0 ** -49 + TINY)
            lb = hb - (affine_mag(r, bx, by) * 2.0 ** -49 + TINY)
            up = (la <= THR) & (lb > THR)
            down = (la > THR) & (lb <= THR)
            none = (la > THR) & (lb > THR)
            hi = np.where(up, np.minimum(hi, (THR - la) / np.where(up, lb - la, 1.0) + 2.0 ** -50), hi)
            lo = np.where(down, np.maximum(lo, (la - THR) / np.where(down, la - lb, 1.0) - 2.0 ** -50), lo)
            lo = np.where(none, 2.0, lo)
        ok = lo <= hi
        if ell is not None:
            r = ell
            ux, uy = (ax - r[1]) / r[3], (ay - r[2]) / r[4]
            wx, wy = (bx - ax) / r[3], (by - ay) / r[4]
            ww = wx * wx + wy * wy
            uw = ux * wx + uy * wy
            tv = np.where(ww > 0.0, -uw / np.where(ww > 0.0, ww, 1.0), lo)
            t = np.minimum(np.maximum(tv, lo), hi)
            px, py = ux + t * wx, uy + t * wy
            v = (px * px + py * py) - 1.0
            S = ((np.abs(ux) + np.abs(uy)) + np.abs(wx)) + np.abs(wy)
            X = np.abs(px) + np.abs(py)
            s = ((1.0 + X * X) + S * X) * 2.0 ** -46 + ((S * S) * 2.0 ** -96 + TINY)
            ok = ok & ((v - s) <= THR)
        return in_a | in_b | ok


def sweep_reference(Z, obstacle_records):
    """Per-path (flags u8, first_hit i32, first_obstacle i32) for paths Z (B, 2(N+2)) and a list of record arrays."""
    Z = np.asarray(Z, dtype=np.float64)
    B = Z.shape[0]
    P = Z.reshape(B, -1, 2)
    bad = ~np.all(np.abs(Z) < BIG, axis=1)
    A, Bp = P[:, :-1], P[:, 1:]
    seg_first = np.full(A.shape[:2], np.iinfo(np.int32).max, dtype=np.int64)
    for o, recs in enumerate(obstacle_records):
        hit = segment_hits(recs, A[..., 0], A[..., 1], Bp[..., 0], Bp[..., 1])
        seg_first = np.where(hit & (seg_first == np.iinfo(np.int32).max), o, seg_first)
    seg_hit = seg_first != np.iinfo(np.int32).max
    anyhit = seg_hit.any(axis=1) & ~bad
    k = np.where(anyhit, seg_hit.argmax(axis=1), -1)
    fo = np.where(anyhit, seg_first[np.arange(B), np.maximum(k, 0)], -1)
    flags = np.where(bad, INVALID, np.where(anyhit, HIT, 0)).astype(np.uint8)
    return flags, k.astype(np.int32), fo.astype(np.int32)


# ---- exact arithmetic ------------------------------------------------------------------------------------------------
def _F(v):
    return Fraction(float(v))


def h_real(r, x, y):
    """h_i^R: the record's formula in exact arithmetic on its doubles (x, y Fractions)."""
    k = int(r[0])
    if k == LINE:
        return -_F(r[5]) * (_F(r[4]) * (x - _F(r[1])) - _F(r[3]) * (y - _F(r[2])))
    if k == ELLIPSE:
        a = (x - _F(r[1])) / _F(r[3])
        b = (y - _F(r[2])) / _F(r[4])
        return a * a + b * b - 1
    xd = x if int(r[1]) == 0 else y
    return (xd - _F(r[3]) - _F(r[4])) if r[2] > 0 else (-xd + _F(r[3]) - _F(r[4]))


def eta(r, ax, ay, bx, by):
    """eta_i of include/uam_b200.h as a Fraction (inputs floats)."""
    A, B = (_F(ax), _F(ay)), (_F(bx), _F(by))
    tail = Fraction(1, 2 ** 990)
    k = int(r[0])
    if k == ELLIPSE:
        S = (abs(A[0] - _F(r[1])) + abs(B[0] - A[0])) / abs(_F(r[3])) + (abs(A[1] - _F(r[2])) + abs(B[1] - A[1])) / abs(_F(r[4]))
        return Fraction(1, 2 ** 44) * (2 + S) + Fraction(1, 2 ** 94) * S * S + tail

    def M(P):
        if k == LINE:
            return abs(_F(r[5])) * (abs(_F(r[4])) * (abs(P[0]) + abs(_F(r[1]))) + abs(_F(r[3])) * (abs(P[1]) + abs(_F(r[2]))))
        xd = P[0] if int(r[1]) == 0 else P[1]
        return abs(xd) + abs(_F(r[3])) + abs(_F(r[4]))
    return Fraction(1, 2 ** 46) * (M(A) + M(B)) + tail


def exact_meets(recs, ax, ay, bx, by, relax=False):
    """Does the real segment (ax, ay) -> (bx, by) meet K_o (relax=False) or K_o^eta (relax=True)?"""
    recs = np.asarray(recs, dtype=np.float64).reshape(-1, 8)
    A, B = (_F(ax), _F(ay)), (_F(bx), _F(by))
    lo, hi = Fraction(0), Fraction(1)
    quads = []
    for r in recs:
        thr = _F(THR) + (eta(r, ax, ay, bx, by) if relax else 0)
        if int(r[0]) == ELLIPSE:
            quads.append((r, thr))
            continue
        ha, hb = h_real(r, *A), h_real(r, *B)
        if ha <= thr and hb <= thr:
            continue
        if ha <= thr:
            hi = min(hi, (thr - ha) / (hb - ha))
        elif hb <= thr:
            lo = max(lo, (ha - thr) / (ha - hb))
        else:
            return False
    if lo > hi:
        return False
    if not quads:
        return True
    assert len(quads) == 1, 'one ellipse record per obstacle'
    r, thr = quads[0]
    ex, ey = (A[0] - _F(r[1])) / _F(r[3]), (A[1] - _F(r[2])) / _F(r[4])
    fx, fy = (B[0] - A[0]) / _F(r[3]), (B[1] - A[1]) / _F(r[4])
    a, b, c = fx * fx + fy * fy, 2 * (ex * fx + ey * fy), ex * ex + ey * ey - 1
    if a > 0:
        t = min(max(-b / (2 * a), lo), hi)
    else:
        t = lo if b >= 0 else hi
    return a * t * t + b * t + c <= thr
