"""Refinement of candidate paths by descent on the raster cost (uam_refine_paths_raster / RasterMap.refine_paths).

CPU: the numpy restatement of the rule (raster_refine_reference.refine_reference) driven by the float64 oracle: the
invariants of the rule.  GPU: the device loop against the restatement driven by the device gradient, bit for bit, over
every kernel and texel form; the library interface; a large batch; the tie to the reference's analytic cost.
"""
import numpy as np
import pytest

from conftest import build_product_map, build_product_problem, full_paths
from raster_gradient_oracle import score_paths_raster_gradient
from raster_refine_reference import refine_reference
from test_raster_gradient import _random_paths, _random_raster


def _oracle_evaluate(lay, occ, geo, w, spc, length_smooth=True, x_start=None):
    def evaluate(Z):
        c, k, _, g = score_paths_raster_gradient(lay, occ, geo, Z, w, spc, length_smooth, x_start)
        return np.asarray(c).astype(np.float32), np.asarray(k).astype(np.uint8), g
    return evaluate


def _bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint8)


def _cpu_case(seed=41, B=24, Wp=9, spc=1.0, x_start=None, bad_rows=True):
    rng = np.random.default_rng(seed)
    H, W, geo = 70, 90, (3.0, 0.25, 40.0, -0.2)
    lay, occ = _random_raster(rng, 3, H, W)
    w = [200.0, 1500.0, 2700.0]
    Z = _random_paths(rng, B, Wp, geo, H, W, spill=0.05)
    ev0 = _oracle_evaluate(lay, occ, geo, w, spc, True, x_start)

    def ev(Zq):
        c, k, g = ev0(Zq)
        if bad_rows:            # a NaN and an inf in the gradient of rows 3 and 5 (the oracle has no NaN paths)
            g[3, 4] = np.nan
            g[5, 2 * Wp - 3] = -np.inf
        return c, k, g
    return Z, ev, min(abs(geo[1]), abs(geo[3]))


# ------------------------------------------------------------------------------------------------------------------
# CPU: the rule on the float64 oracle
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('spc', [0.0, 1.0])
@pytest.mark.parametrize('x_start', [None, [4.0, 39.0]])
def test_reference_monotone_endpoints_and_bad_rows(spc, x_start):
    Z, ev, h = _cpu_case(spc=spc, x_start=x_start)
    c0, k0, _ = ev(Z)
    Zo, c, k, acc = refine_reference(ev, Z, h, 8)
    good = np.ones(Z.shape[0], dtype=bool)
    good[[3, 5]] = False
    # (collide, cost) never gets worse; a clean path stays clean
    assert np.all(k <= k0)
    assert np.all(c[good] <= c0[good])
    assert not np.any((k0 == 0) & (k != 0))
    # start and goal are never written
    assert np.array_equal(_bits(Zo[:, :2]), _bits(Z[:, :2])) and np.array_equal(_bits(Zo[:, -2:]), _bits(Z[:, -2:]))
    # rows with NaN / inf in the gradient are untouched
    assert np.array_equal(_bits(Zo[~good]), _bits(Z[~good])) and np.all(acc[~good] == 0)
    # the result is the evaluation of the returned paths
    ce, ke, _ = ev(Zo)
    assert np.array_equal(_bits(ce), _bits(c)) and np.array_equal(ke, k)
    assert np.sum(c[good] < c0[good]) >= 0.9 * good.sum()
    assert np.array_equal(acc > 0, c < c0)


def test_reference_zero_iterations_is_the_identity():
    Z, ev, h = _cpu_case()
    c0, k0, _ = ev(Z)
    Zo, c, k, acc = refine_reference(ev, Z, h, 0)
    assert np.array_equal(_bits(Zo), _bits(Z))
    assert np.array_equal(_bits(c), _bits(c0)) and np.array_equal(k, k0) and np.all(acc == 0)


@pytest.mark.parametrize('step,max_step,min_step', [(1.0, 16.0, 1.0 / 256), (4.0, 4.0, 0.5), (0.25, 8.0, 0.125)])
def test_reference_step_schedule_and_bound(step, max_step, min_step):
    """tau starts at step_cells; a kept trial doubles it (up to max_step_cells), a dropped one halves it; a path whose tau
    fell below min_step_cells (or whose gradient is not finite) no longer moves; no waypoint moves more than tau cells in
    a trip, so never more than max_step_cells."""
    Z, ev, h = _cpu_case(seed=43, B=16, spc=0.7)
    trace = []
    Zo, _, _, acc = refine_reference(ev, Z, h, 12, step, max_step, min_step, trace=trace)
    tau = np.full(Z.shape[0], step)
    Zp = Z.copy()
    n_acc = np.zeros(Z.shape[0], dtype=np.int64)
    saw = set()
    for t in trace:
        act = t['active']
        assert np.all(act <= (tau >= min_step))
        expect = np.where(t['accepted'], np.minimum(2 * tau, max_step), np.where(act, tau / 2, tau))
        assert np.array_equal(t['tau'], expect)
        assert np.all(t['tau'] <= max_step)
        # tau stays step * 2^j (clamped to max_step, itself step * 2^j here)
        j = np.log2(t['tau'] / step)
        assert np.array_equal(j, np.round(j))
        B = Z.shape[0]
        moved = np.any(_bits(t['Z']).reshape(B, -1) != _bits(Zp).reshape(B, -1), axis=1)
        proposed = np.any(_bits(t['Zt']).reshape(B, -1) != _bits(Zp).reshape(B, -1), axis=1)
        assert np.array_equal(moved, t['accepted'] & proposed)
        d = np.abs(t['Zt'] - Zp)[:, 2:-2]
        fin = np.isfinite(Zp).all(axis=1)
        bound = tau[:, None] * h * (1 + 1e-12) + 4 * np.spacing(np.abs(Zp[:, 2:-2]))
        assert np.all(d[fin] <= bound[fin])
        assert np.all(d[fin] <= max_step * h * (1 + 1e-12) + 4 * np.spacing(np.abs(Zp[fin, 2:-2])))
        assert not np.any(d[~act & fin])
        saw.update(np.unique(np.sign(t['tau'] - tau)).tolist())
        n_acc += t['accepted']
        tau, Zp = t['tau'], t['Z']
    assert np.array_equal(n_acc, acc) and np.array_equal(_bits(Zp), _bits(Zo))
    assert {-1.0, 1.0} <= saw or max_step == step        # the schedule went both ways


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


def _device_evaluate(rm, w, spc, length_smooth=True, x_start=None):
    def evaluate(Z):
        return rm.cost_gradient(np.ascontiguousarray(Z), w, spc, length_smooth, x_start)
    return evaluate


@pytest.mark.gpu
@pytest.mark.parametrize('L', [1, 2, 3])
@pytest.mark.parametrize('spc', [0.0, 1.0])
@pytest.mark.parametrize('layout', [0, 1])
@pytest.mark.parametrize('variant', [-1, 0, 2])
@pytest.mark.parametrize('combine', [0, 1, 2])
def test_refine_matches_reference_bit_for_bit(uam, torch, L, spc, layout, variant, combine):
    """The device loop against refine_reference driven by the device gradient: Z_out, cost, collide and the accepted
    counts are identical after 0, 1, 3 and 8 trips, on every gradient kernel (waypoint mode, warp per path, binned) and
    texel form (float2 / float4 texels, quads + bit-plane, sign-packed quads; a negative weight forces the bit-plane)."""
    if spc == 0.0 and variant != -1:
        pytest.skip('waypoint mode has a single kernel')
    if combine != 1 and variant != 2:
        pytest.skip('quad texels are sampled by the binned pipeline only (at these batch sizes)')
    rng = np.random.default_rng(300 + L + 10 * layout)
    H, W = (150, 230) if layout else (151, 229)
    geo = (3.0, 0.25, 40.0, -0.2)
    h = min(abs(geo[1]), abs(geo[3]))
    lay, occ = _random_raster(rng, L, H, W)
    rm = uam.RasterMap.from_arrays(lay, geo, occ, options={'raster_layout': layout, 'integral_variant': variant,
                                                           'combine_layers': combine})
    w = [200.0, -15000.0, 27000.0][:L] if combine == 2 else [200.0, 15000.0, 27000.0][:L]
    for Wp, spill, x_start in [(64, 0.0, None), (7, 0.15, [4.0, 39.0]), (3, 0.0, None), (130, 0.05, [0.0, 0.0])]:
        Z = _random_paths(rng, 96, Wp, geo, H, W, spill)
        Z[5, 2] = np.nan
        trace = []
        ev = _device_evaluate(rm, w, spc, True, x_start)
        c0, k0, _ = ev(Z)
        refine_reference(ev, Z, h, 8, trace=trace)
        acc_ref = np.cumsum([t['accepted'] for t in trace], axis=0)
        for K in (0, 1, 3, 8):
            Zo, c, k, acc = rm.refine_paths(Z, w, spc, K, True, x_start)
            if K == 0:
                Zr, cr, kr, ar = Z, c0, k0, np.zeros(96, dtype=np.int32)
            else:
                t = trace[K - 1]
                Zr, cr, kr, ar = t['Z'], t['cost'], t['collide'], acc_ref[K - 1]
            assert np.array_equal(_bits(Zo), _bits(Zr)), (Wp, K)
            assert np.array_equal(_bits(c), _bits(cr)) and np.array_equal(k, kr), (Wp, K)
            assert np.array_equal(acc, ar), (Wp, K)
        assert np.array_equal(_bits(Zo[5]), _bits(Z[5]))          # NaN row untouched
        assert np.sum(acc_ref[-1] > 0) > 48                        # and the descent does move the others


@pytest.mark.gpu
@pytest.mark.parametrize('spc', [0.0, 1.0])
def test_refine_interface(uam, torch, spc):
    """numpy and tensor inputs give the same bits and the input tensor is left as it was; the returned cost / collide
    are score_paths' bits for the returned paths; a permuted batch gives the permuted result (equal B: same kernels)."""
    rng = np.random.default_rng(23)
    H, W, geo = 120, 90, (0.0, 0.5, 0.0, 0.5)
    lay, occ = _random_raster(rng, 3, H, W)
    rm = uam.RasterMap.from_arrays(lay, geo, occ)
    w = [1.0, 2.0, 3.0]
    Z = _random_paths(rng, 40, 16, geo, H, W)
    Zt = torch.from_numpy(Z).cuda()
    Zt_before = Zt.clone()
    Zo, c, k, acc = rm.refine_paths(Zt, w, spc, 6)
    assert Zo.is_cuda and c.is_cuda and k.is_cuda and acc.is_cuda and Zo.data_ptr() != Zt.data_ptr()
    assert torch.equal(Zt, Zt_before)
    Zh, ch, kh, ah = rm.refine_paths(Z, w, spc, 6)
    assert isinstance(Zh, np.ndarray)
    assert np.array_equal(_bits(Zh), _bits(Zo.cpu().numpy())) and np.array_equal(_bits(ch), _bits(c.cpu().numpy()))
    assert np.array_equal(kh, k.cpu().numpy()) and np.array_equal(ah, acc.cpu().numpy())
    cs, ks = rm.score_paths(Zo, w, spc)
    assert torch.equal(cs, c) and torch.equal(ks, k)
    perm = np.random.default_rng(24).permutation(40)
    Zp, cp, kp, ap = rm.refine_paths(np.ascontiguousarray(Z[perm]), w, spc, 6)
    assert np.array_equal(_bits(Zp), _bits(Zh[perm])) and np.array_equal(_bits(cp), _bits(ch[perm]))
    assert np.array_equal(kp, kh[perm]) and np.array_equal(ap, ah[perm])
    assert np.all(ch <= rm.score_paths(Z, w, spc)[0])


@pytest.mark.gpu
def test_refine_large_batch(uam, torch):
    """8192 paths x 64 waypoints on a 2048^2 raster (binned pipeline on sign-packed quads), 20 trips: no path gets
    worse, no new collision, at least 90 % of the paths strictly improve."""
    rng = np.random.default_rng(77)
    n = 2048
    geo = (0.0, 1.0 / 32, 0.0, 1.0 / 32)
    lay, occ = _random_raster(rng, 3, n, n)
    rm = uam.RasterMap.from_arrays(lay, geo, occ)
    w = [200.0, 15000.0, 27000.0]
    Z = torch.from_numpy(_random_paths(rng, 8192, 64, geo, n, n)).cuda()
    c0, k0 = rm.score_paths(Z, w, 1.0)
    Zo, c, k, acc = rm.refine_paths(Z, w, 1.0, 20)
    cs, ks = rm.score_paths(Zo, w, 1.0)
    assert torch.equal(cs, c) and torch.equal(ks, k)
    c0, k0, c, k = c0.cpu().numpy(), k0.cpu().numpy(), c.cpu().numpy(), k.cpu().numpy()
    assert np.all(c <= c0) and np.all(k <= k0)
    frac = float(np.mean(c < c0))
    red = (c0 - c) / np.abs(c0)
    print(f'large batch: {frac:.4f} of the paths improved, median relative reduction {np.median(red):.4f}, '
          f'mean accepted trips {acc.float().mean().item():.2f}')
    assert frac >= 0.9, frac


@pytest.mark.gpu
def test_refine_lowers_the_reference_cost(uam, torch, fixture_spec, golden):
    """Tie to the reference: the main.py map rasterised at 8192^2 over the 64 km window (raster and analytic cost agree
    to 1.5e-5 at that cell size); refining the jittered golden paths in waypoint mode lowers Problem.score -- the
    analytic form of the reference's get_cost -- for at least 90 % of them."""
    f = fixture_spec
    N = 62
    Z = full_paths(f, golden['jit_x'])
    prob = build_product_problem(f, N)
    R = 8192
    rm = uam.RasterMap.from_map(build_product_map(f), R, R, (8.0, 64.0 / R, -42.0, 64.0 / R))
    Zo, c, k, acc = rm.refine_paths(Z, f['weights'], 0.0, 20, True, f['x_start'])
    a0 = prob.score(Z)[0]
    a1 = prob.score(Zo)[0]
    red = (a0 - a1) / np.abs(a0)
    print('analytic cost reduction per path:', np.round(red, 5).tolist(), 'accepted trips:', acc.tolist())
    assert np.mean(a1 < a0) >= 0.9, red
    del rm
    torch.cuda.empty_cache()


@pytest.mark.gpu
def test_refine_errors(uam, torch):
    import ctypes as C
    from uam_path_planning_b200 import _lib
    rng = np.random.default_rng(3)
    lay, occ = _random_raster(rng, 2, 40, 50)
    geo = (0.0, 1.0, 0.0, 1.0)
    Z = torch.from_numpy(_random_paths(rng, 4, 6, geo, 40, 50)).cuda()
    for variant in (1, 3):
        rm = uam.RasterMap.from_arrays(lay, geo, occ, options={'integral_variant': variant})
        with pytest.raises(uam.UamError) as ei:
            rm.refine_paths(Z, [1.0, 2.0], 1.0, 2)
        assert ei.value.code == -5
        rm.refine_paths(Z, [1.0, 2.0], 0.0, 2)          # waypoint mode has one kernel, whatever the variant
    rm = uam.RasterMap.from_arrays(lay, geo, occ)
    for kw in (dict(iterations=-1), dict(min_step_cells=0.0), dict(step_cells=0.5, min_step_cells=1.0),
               dict(step_cells=2.0, max_step_cells=1.0), dict(step_cells=float('nan')), dict(max_step_cells=float('inf'))):
        with pytest.raises(uam.UamError) as ei:
            rm.refine_paths(Z, [1.0, 2.0], 1.0, **dict(dict(iterations=2), **kw))
        assert ei.value.code == -1, kw
    Zo, c, k, acc = rm.refine_paths(Z[:0], [1.0, 2.0], 1.0, 3)       # B = 0
    assert Zo.shape == (0, 12) and c.shape == (0,) and acc.shape == (0,)
    lib = _lib.load()
    eng = rm.engine
    p = rm.parameter_vector([1.0, 2.0])
    pp = p.ctypes.data_as(C.c_void_p)
    Zc = Z.clone()
    zp = C.c_void_p(Zc.data_ptr())
    cost = torch.empty(4, dtype=torch.float32, device='cuda')
    col = torch.empty(4, dtype=torch.uint8, device='cuda')
    cp, kp = C.c_void_p(cost.data_ptr()), C.c_void_p(col.data_ptr())
    args = (4, 4, pp, p.size, _lib.UAM_LENGTH_SMOOTH | _lib.UAM_OWN_START, 1.0, 2, 1.0, 16.0, 1.0 / 256)
    assert lib.uam_refine_paths_raster(eng._h, None, *args, cp, kp, None, None) == -1      # NULL paths
    assert lib.uam_refine_paths_raster(eng._h, zp, *args, None, kp, None, None) == -1      # NULL cost
    assert lib.uam_refine_paths_raster(eng._h, zp, *args, cp, None, None, None) == -1      # NULL collide
    assert lib.uam_refine_paths_raster(eng._h, zp, 0, *args[1:], None, None, None, None) == 0   # B = 0
    assert lib.uam_refine_paths_raster(eng._h, zp, *args, cp, kp, None, None) == 0         # accepted is optional
    torch.cuda.synchronize()
    cs, ks = rm.score_paths(Zc, [1.0, 2.0], 1.0)
    assert torch.equal(cs, cost) and torch.equal(ks, col)
    h = C.c_void_p()
    assert lib.uam_ctx_create(0, C.byref(h)) == 0
    assert lib.uam_refine_paths_raster(h, zp, *args, cp, kp, None, None) == -4             # no raster
    assert lib.uam_ctx_destroy(h) == 0
