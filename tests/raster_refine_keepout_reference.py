"""The refinement rule of uam_refine_paths_raster_keepout in numpy float64 -- TEST INFRASTRUCTURE ONLY.

raster_refine_reference's rule with the analytic check against the no-fly shapes in the accept test.  Driven by
``evaluate(Z) -> (cost f32, collide u8, grad f64)`` and ``check(Z) -> (flags u8, clearance f64 or None)`` on the whole
batch: the device gradient and the device analytic sweep / clearance (RasterMap.cost_gradient, Engine.sweep_analytic,
Engine.clearance_analytic at cap = margin) for bit-equality tests, the float64 oracle and analytic_sweep_reference /
analytic_clearance_reference on the CPU.  check may return None for the clearance only when margin == 0.
"""
from __future__ import annotations

import numpy as np

F64 = np.float64


def refine_keepout_reference(evaluate, check, Z, h: float, iterations: int, step_cells: float = 1.0,
                             max_step_cells: float = 64.0, min_step_cells: float = 1.0 / 256, margin: float = 0.0,
                             trace=None):
    """-> (Z_out, cost, collide, accepted, flags, clearance).  `trace` (a list, optional) receives per trip a dict with
    the trial, the active mask, the plain rule's accept mask, the accept mask, and Z, cost, collide, flags, clearance
    and tau after the trip."""
    Z = np.array(Z, dtype=F64, copy=True)
    c, k, g = evaluate(Z)
    c = np.asarray(c, dtype=np.float32).copy()
    k = np.asarray(k, dtype=np.uint8).copy()
    g = np.array(g, dtype=F64, copy=True)
    f, cl = check(Z)
    f = np.asarray(f, dtype=np.uint8).copy()
    cl = None if cl is None else np.array(cl, dtype=F64, copy=True)
    assert cl is not None or margin == 0
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
        ft, clt = check(Zt)
        ft = np.asarray(ft, dtype=np.uint8)
        with np.errstate(invalid='ignore'):
            plain = active & (kt <= k) & (ct < c)
            ok = plain & ((ft & ~f) == 0)
            if margin > 0:
                clt = np.asarray(clt, dtype=F64)
                ok &= clt >= cl                     # a NaN on either side rejects
        Z[ok] = Zt[ok]
        c[ok] = ct[ok]
        k[ok] = kt[ok]
        g[ok] = np.asarray(gt, dtype=F64)[ok]
        f[ok] = ft[ok]
        if cl is not None:
            cl[ok] = np.asarray(clt, dtype=F64)[ok]
        tau = np.where(ok, np.minimum(2.0 * tau, max_step_cells), np.where(active, 0.5 * tau, tau))
        accepted += ok
        if trace is not None:
            trace.append(dict(Zt=Zt, active=active, plain=plain, accepted=ok, Z=Z.copy(), cost=c.copy(),
                              collide=k.copy(), flags=f.copy(), clearance=None if cl is None else cl.copy(),
                              tau=tau.copy()))
    return Z, c, k, accepted, f, cl
