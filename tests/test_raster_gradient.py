"""Gradient of the raster path cost with respect to the waypoints (uam_grad_paths_raster / RasterMap.cost_gradient).

CPU: the float64 restatement (raster_gradient_oracle.score_paths_raster_gradient) against a closed form and against central differences of
oracle.score_paths_raster.  GPU: the device gradient against the oracle, its cost / collide bits against the scorer's,
its independence from the rest of the batch, and its tie to the analytic gradient of the reference's cost.
"""
import os
import sys

import numpy as np
import pytest

from conftest import build_product_map, build_product_problem, full_paths
from oracle import uam_oracle as orc
from raster_gradient_oracle import score_paths_raster_gradient

GRAD_RTOL = 2e-5          # device vs oracle, per path, relative to the path's gradient max-norm (observed <= 6.3e-6)


def _random_raster(rng, L, H, W):
    yy, xx = np.mgrid[0:H, 0:W]
    lay = np.stack([(rng.uniform(0.2, 2.0) * np.exp(-((xx - rng.uniform(0, W)) ** 2 + (yy - rng.uniform(0, H)) ** 2) /
                                                    (2 * rng.uniform(8, 40) ** 2)) + 0.05 * rng.uniform(size=(H, W)))
                    for _ in range(L)]).astype(np.float32)
    occ = np.zeros((H, W), dtype=np.uint8)
    for _ in range(6):
        ci, cj, r = rng.uniform(0, H), rng.uniform(0, W), rng.uniform(2, 9)
        occ |= (((yy - ci) ** 2 + (xx - cj) ** 2) < r * r).astype(np.uint8)
    return lay, occ


def _random_paths(rng, B, Wp, geo, H, W, spill=0.0, jitter=2.0):
    x0, dx, y0, dy = geo
    lo = np.array([x0, y0]) - spill * np.array([dx * W, dy * H])
    hi = np.array([x0 + dx * W, y0 + dy * H]) + spill * np.array([dx * W, dy * H])
    s = lo + rng.uniform(size=(B, 1, 2)) * (hi - lo)
    g = lo + rng.uniform(size=(B, 1, 2)) * (hi - lo)
    t = np.linspace(0, 1, Wp).reshape(1, Wp, 1)
    P = s + t * (g - s) + rng.normal(0, jitter * abs(dx), (B, Wp, 2))
    return np.ascontiguousarray(P.reshape(B, 2 * Wp))


# ------------------------------------------------------------------------------------------------------------------
# CPU: the oracle
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('spc', [0.0, 0.7, 2.0])
@pytest.mark.parametrize('length_smooth,x_start', [(True, None), (False, [3.5, 41.0])])
def test_oracle_gradient_closed_form_on_planes(spc, length_smooth, x_start):
    """Layers a + b i + c j with small integers (exact in float32) and every sample inside the raster: the bilinear
    interpolant is the plane itself, so dP/du = sum_l w_l c_l, dP/dv = sum_l w_l b_l everywhere.  Segment k's S samples
    then give z_k the weight (S+1)/(2S) and z_{k+1} the weight (S-1)/(2S) of that constant slope, the goal sample 1."""
    H, W, geo = 60, 80, (2.0, 0.5, 50.0, -0.25)
    x0, dx, y0, dy = geo
    a, b, c = np.array([3.0, -2.0, 7.0]), np.array([2.0, 1.0, -1.0]), np.array([-1.0, 3.0, 2.0])
    ii, jj = np.mgrid[0:H, 0:W]
    lay = np.stack([a[l] + b[l] * ii + c[l] * jj for l in range(3)]).astype(np.float32)
    occ = np.zeros((H, W), dtype=np.uint8)
    w = np.array([1.5, 0.25, 2.0])
    rng = np.random.default_rng(5)
    B, Wp = 12, 9
    N = Wp - 2
    # waypoints well inside: pixel coordinates in [5, W-6] x [5, H-6]
    U = rng.uniform(5, W - 6, size=(B, Wp))
    V = rng.uniform(5, H - 6, size=(B, Wp))
    P = np.stack([x0 + (U + 0.5) * dx, y0 + (V + 0.5) * dy], axis=-1)
    Z = P.reshape(B, 2 * Wp)
    cost, col, ns, G = score_paths_raster_gradient(lay, occ, geo, Z, w, spc, length_smooth, x_start)
    c_ref, col_ref, ns_ref = orc.score_paths_raster(lay, occ, geo, Z, w, spc, length_smooth, x_start)
    assert np.array_equal(cost, c_ref) and np.array_equal(col, col_ref) and np.array_equal(ns, ns_ref)
    g = np.array([w @ c / dx, w @ b / dy])
    dUk, dVk = np.diff(U, axis=1), np.diff(V, axis=1)
    S = np.maximum(1, np.ceil(np.hypot(dUk, dVk) * spc)) if spc > 0 else np.ones_like(dUk)
    Gp = np.zeros((B, Wp, 2))
    Gp[:, :-1] += ((S + 1) / (2 * S))[..., None] * g
    Gp[:, 1:] += ((S - 1) / (2 * S))[..., None] * g
    Gp[:, -1] += g
    Gp /= N
    # length part: (x_start, z_0) if given, (z_{k-1}, z_k) for k = 1..N
    Gl = np.zeros((B, Wp, 2))
    pairs = [(k - 1, k) for k in range(1, N + 1)]
    for i0, i1 in pairs + ([(None, 0)] if x_start is not None else []):
        d = P[:, i1] - (P[:, i0] if i0 is not None else np.asarray(x_start))
        gk = 2 * d if length_smooth else d / np.linalg.norm(d, axis=1, keepdims=True)
        Gl[:, i1] += gk
        if i0 is not None:
            Gl[:, i0] -= gk
    Gref = (Gp + (N + 1) * Gl).reshape(B, 2 * Wp)
    np.testing.assert_allclose(G, Gref, rtol=1e-12, atol=1e-12 * np.abs(Gref).max())


@pytest.mark.parametrize('spc', [0.0, 0.37, 1.0, 2.5])
@pytest.mark.parametrize('length_smooth', [True, False])
@pytest.mark.parametrize('x_start', [None, [4.0, 39.0]])
def test_oracle_gradient_matches_finite_differences(spc, length_smooth, x_start):
    """Central differences of oracle.score_paths_raster, step h = 1e-3 cell, on random rasters with paths that spill
    outside the raster; errors relative to the max-norm of the path's PENALTY gradient (the length part is smooth and
    would hide them).  The cost is piecewise bilinear in each sample: central differences are exact except where a sample
    crosses a cell edge (the slope jumps) inside [z - h, z + h], and the float32 fractions move in steps of up to 2^-24
    cell (2^-24 / 2h = 3e-5 of a slope per sample, random in sign: the 1e-5 median).  A sample crosses an edge with
    probability ~h per axis; when one does, its coordinate is off by up to the slope jump / (N S_k): up to 1e-2 of the
    penalty gradient in waypoint mode (S_k = 1, observed 1.0e-2), less with more samples per segment."""
    rng = np.random.default_rng(31)
    H, W, geo = 70, 90, (3.0, 0.25, 40.0, -0.2)
    lay, occ = _random_raster(rng, 3, H, W)
    w = [200.0, 1500.0, 2700.0]
    Z = _random_paths(rng, 8, 8, geo, H, W, spill=0.1)
    cost, col, ns, G = score_paths_raster_gradient(lay, occ, geo, Z, w, spc, length_smooth, x_start)
    h = 1e-3 * abs(geo[1])
    Gfd = np.zeros_like(G)
    same = np.ones(Z.shape[0], dtype=bool)        # paths that stay on one piece (every S_k unchanged) at every z +- h
    for c in range(Z.shape[1]):
        Zp, Zm = Z.copy(), Z.copy()
        Zp[:, c] += h
        Zm[:, c] -= h
        cp, _, nsp = orc.score_paths_raster(lay, occ, geo, Zp, w, spc, length_smooth, x_start)
        cm, _, nsm = orc.score_paths_raster(lay, occ, geo, Zm, w, spc, length_smooth, x_start)
        same &= (nsp == ns) & (nsm == ns)
        Gfd[:, c] = (cp - cm) / (2 * h)
    # a segment whose length in cells times spc lies within h of an integer changes S_k across z +- h: the cost jumps
    # there and the difference quotient is not a derivative.  Those paths (rare) are left out, most must remain.
    assert same.sum() >= Z.shape[0] - 2, same
    G_len = score_paths_raster_gradient(lay, occ, geo, Z, [0.0, 0.0, 0.0], spc, length_smooth, x_start)[3]
    err = (np.abs(G - Gfd).max(axis=1) / np.abs(G - G_len).max(axis=1))[same]
    assert np.all(err < 3e-2), err
    assert np.median(err) < 1e-4, err


# ------------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope='module')
def uam():
    import uam_path_planning_b200 as u
    return u


@pytest.fixture(scope='module')
def torch():
    import torch as t
    assert t.cuda.is_available()
    return t


def _grad_err(g, g_ref):
    """per path: max |g - g_ref| / max |g_ref|"""
    return np.abs(g - g_ref).max(axis=1) / np.maximum(np.abs(g_ref).max(axis=1), 1e-300)


@pytest.mark.gpu
@pytest.mark.parametrize('L', [1, 2, 3])
@pytest.mark.parametrize('spc', [0.0, 0.37, 1.0, 2.5])
@pytest.mark.parametrize('layout', [0, 1])
@pytest.mark.parametrize('variant', [-1, 0, 2])
@pytest.mark.parametrize('combine', [0, 1, 2])
def test_raster_gradient_vs_oracle(uam, torch, L, spc, layout, variant, combine):
    """Every kernel of the gradient (waypoint mode, warp per path, binned) on every texel form (float2 / float4 texels,
    quads + bit-plane, sign-packed quads; a negative weight forces the bit-plane) against the oracle; cost / collide
    are the scorer's bits; the numpy and tensor paths agree bit for bit."""
    if spc == 0.0 and variant != -1:
        pytest.skip('waypoint mode has a single kernel')
    if combine != 1 and variant != 2:
        pytest.skip('quad texels are sampled by the binned pipeline only (at these batch sizes)')
    rng = np.random.default_rng(200 + L + 10 * layout)
    H, W = (150, 230) if layout else (151, 229)
    geo = (3.0, 0.25, 40.0, -0.2)
    lay, occ = _random_raster(rng, L, H, W)
    rm = uam.RasterMap.from_arrays(lay, geo, occ, options={'raster_layout': layout, 'integral_variant': variant,
                                                           'combine_layers': combine})
    w = [200.0, -15000.0, 27000.0][:L] if combine == 2 else [200.0, 15000.0, 27000.0][:L]
    worst = 0.0
    for Wp, spill, x_start in [(64, 0.0, None), (7, 0.15, [4.0, 39.0]), (3, 0.0, None), (130, 0.05, [0.0, 0.0])]:
        Z = _random_paths(rng, 96, Wp, geo, H, W, spill)
        for ls in (True, False):
            Zt = torch.from_numpy(Z).cuda()
            c, k, g = rm.cost_gradient(Zt, w, spc, ls, x_start)
            cs, ks = rm.score_paths(Zt, w, spc, ls, x_start)
            assert np.array_equal(c.cpu().numpy(), cs.cpu().numpy()) and np.array_equal(k.cpu().numpy(), ks.cpu().numpy())
            ch, kh, gh = rm.cost_gradient(Z, w, spc, ls, x_start)
            assert np.array_equal(ch, c.cpu().numpy()) and np.array_equal(kh, k.cpu().numpy())
            assert np.array_equal(gh, g.cpu().numpy())
            _, _, _, g_ref = score_paths_raster_gradient(lay, occ, geo, Z, w, spc, ls, x_start)
            e = _grad_err(gh, g_ref)
            worst = max(worst, float(e.max()))
            assert np.all(e <= GRAD_RTOL), (Wp, ls, e.max())
    print(f'worst gradient error vs oracle: {worst:.2e}')


@pytest.mark.gpu
def test_raster_gradient_large_batch(uam, torch):
    """8192 paths x 64 waypoints (2^19 segments: quad texels, binned pipeline in integral mode) on a 2048^2 raster: every
    cost equals score_paths' bit for bit, a seeded sample of 256 paths matches the oracle gradient."""
    rng = np.random.default_rng(77)
    n = 2048
    geo = (0.0, 1.0 / 32, 0.0, 1.0 / 32)
    lay, occ = _random_raster(rng, 3, n, n)
    rm = uam.RasterMap.from_arrays(lay, geo, occ)
    w = [200.0, 15000.0, 27000.0]
    Z = _random_paths(rng, 8192, 64, geo, n, n)
    Zt = torch.from_numpy(Z).cuda()
    idx = np.sort(np.random.default_rng(78).choice(8192, 256, replace=False))
    for spc in (1.0, 0.0):          # binned pipeline / waypoint kernel, both on sign-packed quads
        c, k, g = rm.cost_gradient(Zt, w, spc, True, None)
        cs, ks = rm.score_paths(Zt, w, spc, True, None)
        assert np.array_equal(c.cpu().numpy(), cs.cpu().numpy()) and np.array_equal(k.cpu().numpy(), ks.cpu().numpy())
        _, _, _, g_ref = score_paths_raster_gradient(lay, occ, geo, Z[idx], w, spc, True, None)
        e = _grad_err(g.cpu().numpy()[idx], g_ref)
        print(f'large batch, spc = {spc}: worst gradient error vs oracle {e.max():.2e}')
        assert np.all(e <= GRAD_RTOL), e.max()


@pytest.mark.gpu
@pytest.mark.parametrize('spc,variant', [(0.0, -1), (1.0, 0), (1.0, 2)])
def test_raster_gradient_independent_of_the_batch(uam, torch, spc, variant):
    """A clean path's gradient has the same bits whatever else the batch holds and in whatever order: permuted batch,
    NaN / inf / far-outside / zero-length rows; two identical calls give identical bits."""
    rng = np.random.default_rng(19)
    H, W, geo = 120, 90, (0.0, 0.5, 0.0, 0.5)
    lay, occ = _random_raster(rng, 3, H, W)
    rm = uam.RasterMap.from_arrays(lay, geo, occ, options={'integral_variant': variant})
    w = [1.0, 2.0, 3.0]
    Z = _random_paths(rng, 40, 16, geo, H, W)
    _, _, g0 = rm.cost_gradient(torch.from_numpy(Z).cuda(), w, spc)
    g0 = g0.cpu().numpy()
    _, _, g1 = rm.cost_gradient(torch.from_numpy(Z).cuda(), w, spc)
    assert np.array_equal(g0, g1.cpu().numpy())
    perm = np.random.default_rng(20).permutation(40)
    _, _, gp = rm.cost_gradient(torch.from_numpy(np.ascontiguousarray(Z[perm])).cuda(), w, spc)
    assert np.array_equal(gp.cpu().numpy(), g0[perm])
    Zb = Z.copy()
    Zb[3, 5] = np.nan
    Zb[7, 0] = np.inf
    Zb[11, 8:12] = 400.0
    Zb[13, :] = Zb[13, 0]
    Zb[17, 2:] = np.tile(Zb[17, :2], 15)
    _, _, gb = rm.cost_gradient(torch.from_numpy(Zb).cuda(), w, spc)
    gb = gb.cpu().numpy()
    ok = np.ones(40, dtype=bool)
    ok[[3, 7, 11, 13, 17]] = False
    assert np.array_equal(gb[ok], g0[ok])
    # the far-outside and zero-length rows still match the oracle
    _, _, _, g_ref = score_paths_raster_gradient(lay, occ, geo, Zb[[11, 13, 17]], w, spc, True, None)
    assert np.all(_grad_err(gb[[11, 13, 17]], g_ref) <= GRAD_RTOL)


@pytest.mark.gpu
def test_raster_gradient_converges_to_analytic_gradient(uam, torch, fixture_spec, golden):
    """Tie to the reference: the main.py map rasterised at 4096^2, 8192^2 and 16384^2 over the 64 km window; the
    waypoint-mode raster gradient of the jittered golden paths against Problem.get_cost_gradient (analytic, pinned by
    finite differences to the reference's cost).  Same length form and x_start on both sides, so only the penalty parts
    differ.  Bilinear slopes are first order in the cell size.  Measured (NVIDIA B200), |g_raster - g_analytic|_2 /
    |penalty part of g_analytic|_2 over all paths and waypoints: 2.1e-2 / 9.4e-3 / 4.9e-3 (x 2.3, x 1.9 per halving);
    worst single waypoint per path, relative to the path's penalty max-norm: 6.2e-2 / 2.9e-2 / 2.1e-2 (x 2.1, x 1.4) --
    those waypoints sit where the penalty's second derivative jumps (region boundaries, psi = prod m_i^2).  The inputs are
    fixed, so the figures reproduce."""
    f = fixture_spec
    N = 62
    Z = full_paths(f, golden['jit_x'])
    prob = build_product_problem(f, N)
    _, g_an = prob.get_cost_gradient(Z)
    g_len = orc.get_cost_gradient(orc.OMap(f), Z, N, [0.0] * len(f['weights']), 0.0, dict(f['options']))
    pen = g_an - g_len
    m = build_product_map(f)
    err, err_max = {}, {}
    for R in (4096, 8192, 16384):
        geo = (8.0, 64.0 / R, -42.0, 64.0 / R)
        rm = uam.RasterMap.from_map(m, R, R, geo)
        _, _, g = rm.cost_gradient(Z, f['weights'], 0.0, True, f['x_start'])
        err[R] = float(np.linalg.norm(g - g_an) / np.linalg.norm(pen))
        err_max[R] = float(np.max(np.abs(g - g_an).max(axis=1) / np.abs(pen).max(axis=1)))
        del rm
        torch.cuda.empty_cache()
    print('raster vs analytic gradient, relative 2-norm:', err, 'max per path:', err_max)
    assert err[4096] / err[8192] >= 1.5 and err[8192] / err[16384] >= 1.5, err
    assert err[16384] < 6e-3, err
    assert err_max[4096] / err_max[8192] >= 1.8 and err_max[8192] / err_max[16384] >= 1.3, err_max


@pytest.mark.gpu
def test_raster_gradient_descent_step(uam, torch):
    """One small step along -grad on the free waypoints (integral mode, C3-like paths on an 8192^2 C3-like map) lowers
    the raster cost of the large majority of paths (the use a refinement loop makes of it)."""
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    sys.dont_write_bytecode = True
    import bench
    lay, occ, geo = bench.make_raster(torch, 'cuda', n=2048)
    rm = uam.RasterMap.from_arrays(lay, geo, occ)
    Z = bench.make_paths(torch, 'cuda', 4096, 11, n=2048)
    c, _, g = rm.cost_gradient(Z, bench.WEIGHTS, bench.SPC)
    d = g.clone()
    d[:, :2] = 0.0
    d[:, -2:] = 0.0
    step = 0.01 * geo[1] / d.abs().amax(dim=1, keepdim=True)         # at most 1/100 cell per coordinate
    c2, _ = rm.score_paths((Z - step * d).contiguous(), bench.WEIGHTS, bench.SPC)
    frac = float((c2 < c).float().mean())
    print(f'descent: {frac:.4f} of the paths lower their cost')
    assert frac > 0.9, frac


@pytest.mark.gpu
def test_raster_gradient_errors(uam, torch):
    import ctypes as C
    from uam_path_planning_b200 import _lib
    rng = np.random.default_rng(3)
    lay, occ = _random_raster(rng, 2, 40, 50)
    geo = (0.0, 1.0, 0.0, 1.0)
    Z = torch.from_numpy(_random_paths(rng, 4, 6, geo, 40, 50)).cuda()
    for variant in (1, 3):
        rm = uam.RasterMap.from_arrays(lay, geo, occ, options={'integral_variant': variant})
        with pytest.raises(uam.UamError) as ei:
            rm.cost_gradient(Z, [1.0, 2.0], 1.0)
        assert ei.value.code == -5
        rm.cost_gradient(Z, [1.0, 2.0], 0.0)           # waypoint mode has one kernel, whatever the variant
    rm = uam.RasterMap.from_arrays(lay, geo, occ)
    with pytest.raises(uam.UamError) as ei:
        rm.cost_gradient(Z, [1.0], 1.0)                # wrong weight count
    assert ei.value.code == -1
    c, k, g = rm.cost_gradient(Z[:0], [1.0, 2.0], 1.0)   # B = 0
    assert c.shape == (0,) and g.shape == (0, 12)
    lib = _lib.load()
    eng = rm.engine
    p = rm.parameter_vector([1.0, 2.0])
    pp = p.ctypes.data_as(C.c_void_p)
    zp = C.c_void_p(Z.data_ptr())
    assert lib.uam_grad_paths_raster(eng._h, zp, 4, 4, pp, p.size, 0, 1.0, None, None, None, None) == -1   # NULL grad
    assert lib.uam_grad_paths_raster(eng._h, zp, 0, 4, pp, p.size, 0, 1.0, None, None, None, None) == 0    # B = 0
    h = C.c_void_p()
    assert lib.uam_ctx_create(0, C.byref(h)) == 0
    assert lib.uam_grad_paths_raster(h, zp, 4, 4, pp, p.size, 0, 1.0, None, None, None, None) == -4        # no raster
    assert lib.uam_ctx_destroy(h) == 0
