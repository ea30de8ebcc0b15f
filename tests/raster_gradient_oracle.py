"""Float64 restatement of the raster cost gradient (uam_grad_paths_raster) -- TEST INFRASTRUCTURE ONLY.

Built on oracle.score_paths_raster: the same samples, clamps, sample counts S_k and float32 fractions; its cost,
collision flags and sample counts ARE that function's.  Pinned by tests/test_raster_gradient.py (a closed form on
planar layers and central differences of oracle.score_paths_raster).
"""
from __future__ import annotations

from typing import Sequence, Tuple

import numpy as np

from oracle import uam_oracle as orc

F64 = np.float64


def sample_uv_grad(layers: np.ndarray, u: np.ndarray, v: np.ndarray):
    """Slopes (dP/du, dP/dv) per layer of the bilinear interpolant on the cell orc.sample_uv samples, at its float32
    fractions; u, v already clamped (the caller zeroes the slope of a coordinate whose clamp is active)."""
    L, H, W = layers.shape
    j0 = np.minimum(np.floor(u), W - 2).astype(np.int64)
    i0 = np.minimum(np.floor(v), H - 2).astype(np.int64)
    fx = (u - j0).astype(np.float32).astype(F64)
    fy = (v - i0).astype(np.float32).astype(F64)
    t00 = layers[:, i0, j0].astype(F64)
    t01 = layers[:, i0, j0 + 1].astype(F64)
    t10 = layers[:, i0 + 1, j0].astype(F64)
    t11 = layers[:, i0 + 1, j0 + 1].astype(F64)
    return (1 - fy) * (t01 - t00) + fy * (t11 - t10), (1 - fx) * (t10 - t00) + fx * (t11 - t01)


def score_paths_raster_gradient(layers: np.ndarray, occ: np.ndarray, geo: Tuple[float, float, float, float],
                                Z: np.ndarray, weights: Sequence[float], samples_per_cell: float = 0.0,
                                length_smooth: bool = True, x_start=None):
    """orc.score_paths_raster + d cost / d Z (B, 2W) with the sample counts S_k held fixed (the cost is piecewise smooth
    in Z: S_k is piecewise constant and the cost jumps where it changes).  The slope of a clamped coordinate is 0;
    sample s of segment k moves with weight 1 - s/S_k with z_k and s/S_k with z_{k+1}, the goal sample with z_{N+1};
    the length part is orc.get_cost_gradient's (pairs (x_start, z_0) when x_start is given, (z_0, z_1) ..
    (z_{N-1}, z_N)).  Returns (cost, collide, nsamples, grad)."""
    cost, col, nsmp = orc.score_paths_raster(layers, occ, geo, Z, weights, samples_per_cell, length_smooth, x_start)
    x0, dx, y0, dy = geo
    L_, H, W_ = layers.shape
    Z = np.asarray(Z, dtype=F64)
    B = Z.shape[0]
    Wp = Z.shape[1] // 2
    N = Wp - 2
    P = Z.reshape(B, Wp, 2)
    w = np.asarray(weights, dtype=F64)
    U = (P[..., 0] - x0) / dx - 0.5
    V = (P[..., 1] - y0) / dy - 0.5
    dU = U[:, 1:] - U[:, :-1]
    dV = V[:, 1:] - V[:, :-1]
    if samples_per_cell > 0:
        S = np.maximum(1.0, np.ceil(np.sqrt(dU * dU + dV * dV) * samples_per_cell)).astype(np.int64)
    else:
        S = np.ones((B, Wp - 1), dtype=np.int64)

    def slopes(u_raw, v_raw):
        u = np.minimum(np.maximum(u_raw, 0.0), float(W_ - 1))
        v = np.minimum(np.maximum(v_raw, 0.0), float(H - 1))
        gu, gv = sample_uv_grad(layers, u, v)
        gu = np.where((u_raw >= 0) & (u_raw <= W_ - 1), w @ gu, 0.0)
        gv = np.where((v_raw >= 0) & (v_raw <= H - 1), w @ gv, 0.0)
        return np.stack([gu, gv], axis=-1)

    G = np.zeros((B, Wp, 2), dtype=F64)          # penalty part, pixel units, before the 1/N
    for k in range(Wp - 1):
        Sk = S[:, k]
        su, sv = dU[:, k] / Sk, dV[:, k] / Sk
        for s in range(int(Sk.max())):
            act = (s < Sk)[:, None]
            g = slopes(U[:, k] + s * su, V[:, k] + s * sv)
            t = (s / Sk)[:, None]
            G[:, k] += np.where(act, (1 - t) * g / Sk[:, None], 0.0)
            G[:, k + 1] += np.where(act, t * g / Sk[:, None], 0.0)
    G[:, -1] += slopes(U[:, -1], V[:, -1])
    G[..., 0] /= dx
    G[..., 1] /= dy
    G /= N
    # length part (quirk Q1): pairs (x_start, z_0) if given, (z_{k-1}, z_k) for k = 1..N
    Y = P if x_start is None else np.concatenate([np.broadcast_to(np.asarray(x_start, dtype=F64), (B, 1, 2)), P], axis=1)
    off = 0 if x_start is None else 1             # Y_{k + off} = z_k
    for m in range(1 - off, N + 1):               # pair (Y_{m-1+off}, Y_{m+off}) ends at z_m
        d = Y[:, m + off] - Y[:, m - 1 + off]
        if length_smooth:
            gk = 2 * d
        else:
            n = np.sqrt(d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1])[:, None]
            gk = np.divide(d, n, out=np.zeros_like(d), where=n > 0)
        G[:, m] += (N + 1) * gk
        if m >= 1:
            G[:, m - 1] -= (N + 1) * gk
    return cost, col, nsmp, G.reshape(B, 2 * Wp)
