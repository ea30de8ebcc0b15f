"""numpy restatement of uam_sweep_paths_raster (include/uam_b200.h has the definition).

A different algorithm from the kernel's strip walk: for every segment, every raster cell whose dilated box meets the
segment's bounding box is tested on its own with the separating-axis test of a closed segment against a closed box (the
two axes of the box, then the segment's normal: the four corners must not lie strictly on one side of the segment's
line), in exact integer arithmetic.  Products of fixed-point differences pass 2^63 for far-away points; those segments are
tested with Python integers.
"""
import numpy as np

Q = 1 << 16
HALF = (1 << 15) + 1          # half a cell + one quantum
HIT, OUTSIDE, INVALID = 1, 2, 4
D2_CLIP = 65535


def pixel_coords_unclamped(X, geo):
    x0, dx, y0, dy = geo
    return (X[..., 0] - x0) / dx - 0.5, (X[..., 1] - y0) / dy - 0.5


def touched_cells(u0, v0, u1, v1, H, W):
    """(rows, cols) of the raster cells the closed segment (u0, v0) -> (u1, v1) (fixed point, Python ints) touches."""
    jlo = max(-((HALF - min(u0, u1)) // Q), 0)       # first column whose dilated box reaches the bounding box
    jhi = min((max(u0, u1) + HALF) // Q, W - 1)
    ilo = max(-((HALF - min(v0, v1)) // Q), 0)
    ihi = min((max(v0, v1) + HALF) // Q, H - 1)
    if jlo > jhi or ilo > ihi:
        return np.zeros(0, dtype=np.int64), np.zeros(0, dtype=np.int64)
    big = max(abs(u0), abs(v0), abs(u1), abs(v1)) >= (1 << 29)
    dt = object if big else np.int64
    ii, jj = np.meshgrid(np.arange(ilo, ihi + 1), np.arange(jlo, jhi + 1), indexing='ij')
    ii, jj = ii.ravel(), jj.ravel()
    ulo = jj.astype(dt) * Q - HALF
    uhi = jj.astype(dt) * Q + HALF
    vlo = ii.astype(dt) * Q - HALF
    vhi = ii.astype(dt) * Q + HALF
    du, dv = u1 - u0, v1 - v0
    # orientation of each corner against the segment's line: du (cv - v0) - dv (cu - u0)
    side = [du * (cv - v0) - dv * (cu - u0) for cu, cv in ((ulo, vlo), (ulo, vhi), (uhi, vlo), (uhi, vhi))]
    pos = np.ones(ii.shape, dtype=bool)
    neg = np.ones(ii.shape, dtype=bool)
    for s in side:
        pos &= np.asarray(s > 0, dtype=bool)
        neg &= np.asarray(s < 0, dtype=bool)
    keep = ~(pos | neg)
    # the box axes: the bounding boxes overlap (true by the enumeration above, kept for the statement's sake)
    keep &= np.asarray((uhi >= min(u0, u1)) & (ulo <= max(u0, u1)) & (vhi >= min(v0, v1)) & (vlo <= max(v0, v1)),
                       dtype=bool)
    return ii[keep], jj[keep]


def sweep_reference(occ, geo, Z, d2=None):
    """occ (H, W), geo = (x0, dx, y0, dy), Z (B, 2(N+2)) float64; d2 (H, W) = the squared EDT (oracle.edt_sq) or None.
    -> (flags uint8 (B,), first_hit int32 (B,), d2min int32 (B,) or None)."""
    occ = np.asarray(occ) != 0
    H, W = occ.shape
    Z = np.asarray(Z, dtype=np.float64)
    B = Z.shape[0]
    P = Z.reshape(B, -1, 2)
    U, V = pixel_coords_unclamped(P, geo)
    d2c = None if d2 is None else np.minimum(np.asarray(d2, dtype=np.int64), D2_CLIP)
    flags = np.zeros(B, dtype=np.uint8)
    first = np.full(B, -1, dtype=np.int32)
    d2min = None if d2 is None else np.full(B, -1, dtype=np.int32)
    with np.errstate(invalid='ignore'):
        for b in range(B):
            if not (np.all(np.abs(U[b]) < 2.0 ** 31) and np.all(np.abs(V[b]) < 2.0 ** 31)):
                flags[b] = INVALID
                continue
            if not np.all((U[b] >= -0.5) & (U[b] <= W - 0.5) & (V[b] >= -0.5) & (V[b] <= H - 0.5)):
                flags[b] |= OUTSIDE
            uq = [int(x) for x in np.rint(U[b] * Q).astype(np.int64)]
            vq = [int(x) for x in np.rint(V[b] * Q).astype(np.int64)]
            best = None
            for k in range(len(uq) - 1):
                ii, jj = touched_cells(uq[k], vq[k], uq[k + 1], vq[k + 1], H, W)
                if ii.size == 0:
                    continue
                if first[b] < 0 and occ[ii, jj].any():
                    first[b] = k
                    flags[b] |= HIT
                if d2c is not None:
                    m = int(d2c[ii, jj].min())
                    best = m if best is None else min(best, m)
            if d2min is not None and best is not None:
                d2min[b] = best
    return flags, first, d2min
