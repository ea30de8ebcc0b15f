"""The refinement rule of uam_refine_paths_raster in numpy float64 -- TEST INFRASTRUCTURE ONLY.

Driven by any ``evaluate(Z) -> (cost f32, collide u8, grad f64)`` on the whole batch: the device gradient
(RasterMap.cost_gradient) for bit-equality tests, the float64 oracle (raster_gradient_oracle) on the CPU.  The
operations are elementwise and in the device's order (tau h, then / m, then r g, then Z - r g, each rounded once) plus
an order-independent max, so with the device's evaluate the result has the device's bits.
"""
from __future__ import annotations

import numpy as np

F64 = np.float64


def refine_reference(evaluate, Z, h: float, iterations: int, step_cells: float = 1.0, max_step_cells: float = 64.0,
                     min_step_cells: float = 1.0 / 256, trace=None):
    """-> (Z_out, cost, collide, accepted).  `trace` (a list, optional) receives per trip a dict with the trial, the
    active and accepted masks, and Z, cost, collide and tau after the trip."""
    Z = np.array(Z, dtype=F64, copy=True)
    c, k, g = evaluate(Z)
    c = np.asarray(c, dtype=np.float32).copy()
    k = np.asarray(k, dtype=np.uint8).copy()
    g = np.array(g, dtype=F64, copy=True)
    B, cols = Z.shape
    free = slice(2, cols - 2)
    tau = np.full(B, float(step_cells), dtype=F64)
    accepted = np.zeros(B, dtype=np.int32)
    for _ in range(int(iterations)):
        gf = g[:, free]
        finite = np.isfinite(gf).all(axis=1)
        m = np.where(finite, np.abs(np.where(np.isfinite(gf), gf, 0.0)).max(axis=1), 0.0)
        active = (tau >= min_step_cells) & finite & (m > 0) & np.isfinite(c)
        r = np.zeros(B, dtype=F64)
        r[active] = (tau[active] * h) / m[active]
        Zt = Z.copy()
        Zt[active, free] = Z[active, free] - r[active, None] * g[active, free]
        ct, kt, gt = evaluate(Zt)
        ct = np.asarray(ct, dtype=np.float32)
        kt = np.asarray(kt, dtype=np.uint8)
        with np.errstate(invalid='ignore'):
            ok = active & (kt <= k) & (ct < c)
        Z[ok] = Zt[ok]
        c[ok] = ct[ok]
        k[ok] = kt[ok]
        g[ok] = np.asarray(gt, dtype=F64)[ok]
        tau = np.where(ok, np.minimum(2.0 * tau, max_step_cells), np.where(active, 0.5 * tau, tau))
        accepted += ok
        if trace is not None:
            trace.append(dict(Zt=Zt, active=active, accepted=ok, Z=Z.copy(), cost=c.copy(), collide=k.copy(),
                              tau=tau.copy()))
    return Z, c, k, accepted
