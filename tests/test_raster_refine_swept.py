"""Refinement under the swept occupancy check (uam_refine_paths_raster_swept / RasterMap.refine_paths_swept).

CPU: the numpy restatement of the rule (raster_refine_swept_reference) driven by the float64 oracle and
raster_sweep_reference: the rule's invariants, and a hand case where the plain rule cuts through an occupied cell.  GPU:
the device loop against the restatement driven by the device gradient and sweep, bit for bit; the library interface;
bit identity with refine_paths where the swept terms never reject; errors; a large batch.
"""
import ctypes as C

import numpy as np
import pytest

from oracle import uam_oracle as orc
from raster_gradient_oracle import score_paths_raster_gradient
from raster_refine_reference import refine_reference
from raster_refine_swept_reference import refine_swept_reference
from raster_sweep_reference import HIT, OUTSIDE, sweep_reference
from test_raster_gradient import _random_paths, _random_raster

GEO = (3.0, 0.25, 40.0, -0.2)
GEO_PIX = (-0.5, 1.0, -0.5, 1.0)            # world = pixel coordinates, exactly


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint8)


def _oracle_evaluate(lay, occ, geo, w, spc, x_start=None, bad_rows=()):
    def evaluate(Z):
        c, k, _, g = score_paths_raster_gradient(lay, occ, geo, Z, w, spc, True, x_start)
        for r, col, v in bad_rows:          # NaN / inf in the gradient (the oracle has no NaN paths)
            g[r, col] = v
        return np.asarray(c).astype(np.float32), np.asarray(k).astype(np.uint8), g
    return evaluate


def _oracle_sweep(occ, geo):
    d2 = orc.edt_sq(occ)

    def sweep(Z):
        f, _, d = sweep_reference(occ, geo, Z, d2)
        return f, d
    return sweep


def _cpu_case(seed, spc, x_start, B=24, Wp=9):
    rng = np.random.default_rng(seed)
    H, W = 70, 90
    lay, occ = _random_raster(rng, 3, H, W)
    Z = _random_paths(rng, B, Wp, GEO, H, W, spill=0.05)
    ev = _oracle_evaluate(lay, occ, GEO, [200.0, 1500.0, 2700.0], spc, x_start,
                          bad_rows=[(3, 4, np.nan), (5, 2 * Wp - 3, -np.inf)])
    return Z, ev, _oracle_sweep(occ, GEO), min(abs(GEO[1]), abs(GEO[3]))


# ------------------------------------------------------------------------------------------------------------------
# CPU: the rule on the float64 oracle
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('spc', [0.0, 1.0])
@pytest.mark.parametrize('x_start', [None, [4.0, 39.0]])
@pytest.mark.parametrize('min_d2', [0, 1, 5])
def test_reference_invariants(spc, x_start, min_d2):
    Z, ev, sw, h = _cpu_case(51, spc, x_start)
    c0, k0, _ = ev(Z)
    f0, d0 = sw(Z)
    trace = []
    Zo, c, k, acc, f, d2 = refine_swept_reference(ev, sw, Z, h, 8, min_d2=min_d2, trace=trace)
    good = np.ones(Z.shape[0], dtype=bool)
    good[[3, 5]] = False
    # no swept flag is gained; the capped clearance never drops
    assert not np.any(f & ~f0)
    if min_d2 > 0:
        assert np.all(np.minimum(d2, min_d2) >= np.minimum(d0, min_d2))
    # (collide, cost) is monotone, as for refine_paths
    assert np.all(k <= k0) and np.all(c[good] <= c0[good])
    # rows with NaN / inf in the gradient come back bit-identical
    assert np.array_equal(_bits(Zo[~good]), _bits(Z[~good])) and np.all(acc[~good] == 0)
    assert np.array_equal(_bits(Zo[:, :2]), _bits(Z[:, :2])) and np.array_equal(_bits(Zo[:, -2:]), _bits(Z[:, -2:]))
    # the outputs are the evaluation and the sweep of the returned paths
    ce, ke, _ = ev(Zo)
    fe, de = sw(Zo)
    assert np.array_equal(_bits(ce), _bits(c)) and np.array_equal(ke, k)
    assert np.array_equal(fe, f) and np.array_equal(de, d2)
    # every accepted trial the plain rule accepts too; here the swept terms do reject some
    assert all(np.all(t['accepted'] <= t['plain']) for t in trace)
    assert sum(int(np.sum(t['plain'] & ~t['accepted'])) for t in trace) > 0
    assert np.sum(acc > 0) >= Z.shape[0] // 2


def test_reference_zero_iterations_is_the_identity():
    Z, ev, sw, h = _cpu_case(52, 1.0, None)
    c0, k0, _ = ev(Z)
    f0, d0 = sw(Z)
    Zo, c, k, acc, f, d2 = refine_swept_reference(ev, sw, Z, h, 0, min_d2=5)
    assert np.array_equal(_bits(Zo), _bits(Z)) and np.array_equal(_bits(c), _bits(c0)) and np.array_equal(k, k0)
    assert np.all(acc == 0) and np.array_equal(f, f0) and np.array_equal(d2, d0)


def _hand_case():
    """Waypoint mode on zero penalty layers: the path (0, 2) -> (5, 8) -> (10, 2) in pixels, one occupied cell (2, 2).
    The length term pulls the free waypoint towards (0, 2), which puts the second segment through the cell."""
    H = W = 16
    lay = np.zeros((1, H, W), dtype=np.float32)
    occ = np.zeros((H, W), dtype=np.uint8)
    occ[2, 2] = 1
    Z = np.array([[0.0, 2.0, 5.0, 8.0, 10.0, 2.0]])
    return lay, occ, Z


def test_hand_case_the_plain_rule_cuts_through_the_cell():
    lay, occ, Z = _hand_case()
    ev = _oracle_evaluate(lay, occ, GEO_PIX, [1.0], 0.0)
    sw = _oracle_sweep(occ, GEO_PIX)
    assert sw(Z)[0][0] == 0
    Zp, cp, kp, _ = refine_reference(ev, Z, 1.0, 20)
    assert kp[0] == 0 and sw(Zp)[0][0] == HIT
    Zs, cs, ks, acc, fs, _ = refine_swept_reference(ev, sw, Z, 1.0, 20)
    assert ks[0] == 0 and fs[0] == 0 and acc[0] > 0
    assert cp[0] < cs[0] < ev(Z)[0][0]           # it still descends, and stops short of the plain result


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


def _device_evaluate(rm, w, spc, x_start=None):
    def evaluate(Z):
        return rm.cost_gradient(np.ascontiguousarray(Z), w, spc, True, x_start)
    return evaluate


def _device_sweep(rm, N, clearance):
    def sweep(Z):
        f, _, d = rm.engine.sweep_raster(np.ascontiguousarray(Z), N, False, clearance)
        return f, d
    return sweep


def _refine_swept(rm, Z, w, spc, K, x_start, min_d2, want_d2min):
    """Engine.refine_raster_swept, which can also return d2min with min_d2 = 0"""
    from uam_path_planning_b200 import _lib
    flags = _lib.UAM_LENGTH_SMOOTH | (_lib.UAM_OWN_START if x_start is None else 0)
    return rm.engine.refine_raster_swept(Z, Z.shape[1] // 2 - 2, rm.parameter_vector(w, x_start), flags, spc, K, 1.0,
                                         64.0, 1.0 / 256, min_d2, want_d2min)


@pytest.mark.gpu
@pytest.mark.parametrize('L', [1, 3])
@pytest.mark.parametrize('spc', [0.0, 1.0])
@pytest.mark.parametrize('layout', [0, 1])
@pytest.mark.parametrize('variant', [-1, 0, 2])
@pytest.mark.parametrize('combine', [0, 1, 2])
def test_refine_swept_matches_reference_bit_for_bit(uam, torch, L, spc, layout, variant, combine):
    """The device loop against refine_swept_reference driven by the device gradient and sweep: Z_out, cost, collide,
    accepted, sweep flags and d2min are identical after 0, 1, 3 and 8 trips, for min_d2 = 0 (with and without d2min
    returned), 1 and 5, on every gradient kernel and texel form (float2 / float4 texels, quads + bit-plane,
    sign-packed quads)."""
    if spc == 0.0 and variant != -1:
        pytest.skip('waypoint mode has a single kernel')
    if combine != 1 and variant != 2:
        pytest.skip('quad texels are sampled by the binned pipeline only (at these batch sizes)')
    rng = np.random.default_rng(400 + L + 10 * layout)
    H, W = (150, 230) if layout else (151, 229)
    h = min(abs(GEO[1]), abs(GEO[3]))
    lay, occ = _random_raster(rng, L, H, W)
    rm = uam.RasterMap.from_arrays(lay, GEO, occ, options={'raster_layout': layout, 'integral_variant': variant,
                                                           'combine_layers': combine})
    w = [200.0, -15000.0, 27000.0][:L] if combine == 2 else [200.0, 15000.0, 27000.0][:L]
    rejected = 0
    cases = [(64, 0.0, None, 5, True), (7, 0.15, [4.0, 39.0], 0, True), (3, 0.0, None, 1, True),
             (130, 0.05, [0.0, 0.0], 0, False)]
    for Wp, spill, x_start, min_d2, want_d2 in cases:
        Z = _random_paths(rng, 96, Wp, GEO, H, W, spill)
        Z[5, 2] = np.nan
        trace = []
        ev = _device_evaluate(rm, w, spc, x_start)
        sw = _device_sweep(rm, Wp - 2, want_d2)
        c0, k0, _ = ev(Z)
        f0, d0 = sw(Z)
        refine_swept_reference(ev, sw, Z, h, 8, min_d2=min_d2, trace=trace)
        acc_ref = np.cumsum([t['accepted'] for t in trace], axis=0)
        rejected += sum(int(np.sum(t['plain'] & ~t['accepted'])) for t in trace)
        for K in (0, 1, 3, 8):
            Zo, c, k, acc, f, d2 = _refine_swept(rm, Z, w, spc, K, x_start, min_d2, want_d2)
            if K == 0:
                Zr, cr, kr, ar, fr, dr = Z, c0, k0, np.zeros(96, dtype=np.int32), f0, d0
            else:
                t = trace[K - 1]
                Zr, cr, kr, ar, fr, dr = t['Z'], t['cost'], t['collide'], acc_ref[K - 1], t['flags'], t['d2min']
            key = (Wp, min_d2, K)
            assert np.array_equal(_bits(Zo), _bits(Zr)), key
            assert np.array_equal(_bits(c), _bits(cr)) and np.array_equal(k, kr), key
            assert np.array_equal(acc, ar) and np.array_equal(f, fr), key
            assert (d2 is None and dr is None) or np.array_equal(d2, dr), key
        assert np.array_equal(_bits(Zo[5]), _bits(Z[5]))          # NaN row untouched
        assert np.sum(acc_ref[-1] > 0) > 48                        # the descent does move the others
    assert rejected > 0                                            # and the swept terms did reject trials


@pytest.mark.gpu
@pytest.mark.parametrize('spc', [0.0, 1.0])
def test_refine_swept_interface(uam, torch, spc):
    """The outputs are score_paths' and sweep_paths' bits for the returned paths; numpy and tensor inputs give the same
    bits and the input tensor is left as it was; a permuted batch gives the permuted result."""
    rng = np.random.default_rng(29)
    H, W, geo = 120, 90, (0.0, 0.5, 0.0, 0.5)
    lay, occ = _random_raster(rng, 3, H, W)
    rm = uam.RasterMap.from_arrays(lay, geo, occ)
    w = [1.0, 2.0, 3.0]
    Z = _random_paths(rng, 40, 16, geo, H, W, spill=0.05)
    Zt = torch.from_numpy(Z).cuda()
    Zt_before = Zt.clone()
    out = rm.refine_paths_swept(Zt, w, spc, 6, min_d2=3)
    Zo, c, k, acc, f, d2 = out
    assert all(t.is_cuda for t in out) and Zo.data_ptr() != Zt.data_ptr()
    assert torch.equal(Zt, Zt_before)
    cs, ks = rm.score_paths(Zo, w, spc)
    assert torch.equal(cs, c) and torch.equal(ks, k)
    fs, _, ds = rm.sweep_paths(Zo)
    assert torch.equal(fs, f) and torch.equal(ds, d2)
    host = rm.refine_paths_swept(Z, w, spc, 6, min_d2=3)
    assert all(isinstance(a, np.ndarray) for a in host)
    for a, b in zip(host, out):
        assert np.array_equal(_bits(a), _bits(b.cpu().numpy()))
    perm = np.random.default_rng(30).permutation(40)
    for a, b in zip(rm.refine_paths_swept(np.ascontiguousarray(Z[perm]), w, spc, 6, min_d2=3), host):
        assert np.array_equal(_bits(a), _bits(b[perm]))
    no_d2 = rm.refine_paths_swept(Z, w, spc, 6)
    assert no_d2[5] is None


@pytest.mark.gpu
@pytest.mark.parametrize('spc', [0.0, 1.0])
def test_refine_swept_equals_refine_paths_without_obstacles(uam, torch, spc):
    """No occupied cell and every path at least 50 cells inside the raster, with steps of at most 2 cells for 20 trips:
    the swept terms cannot reject a trial, so the result is refine_paths' bit for bit."""
    rng = np.random.default_rng(31)
    H, W, geo = 200, 240, (0.0, 0.5, 0.0, 0.5)
    lay, _ = _random_raster(rng, 3, H, W)
    occ = np.zeros((H, W), dtype=np.uint8)
    rm = uam.RasterMap.from_arrays(lay, geo, occ)
    w = [100.0, 200.0, 300.0]
    Z = _random_paths(rng, 64, 12, (geo[0] + 25.0, geo[1], geo[2] + 25.0, geo[3]), H - 100, W - 100, jitter=1.0)
    kw = dict(step_cells=1.0, max_step_cells=2.0)
    Zp, cp, kp, ap = rm.refine_paths(Z, w, spc, 20, **kw)
    assert np.sum(ap > 0) >= 48
    for min_d2 in (0, 5):
        Zs, cs, ks, as_, fs, _ = rm.refine_paths_swept(Z, w, spc, 20, min_d2=min_d2, **kw)
        assert np.array_equal(_bits(Zs), _bits(Zp)) and np.array_equal(_bits(cs), _bits(cp))
        assert np.array_equal(ks, kp) and np.array_equal(as_, ap) and not np.any(fs)


@pytest.mark.gpu
def test_refine_swept_errors(uam, torch):
    from uam_path_planning_b200 import _lib
    rng = np.random.default_rng(3)
    lay, occ = _random_raster(rng, 2, 40, 50)
    geo = (0.0, 1.0, 0.0, 1.0)
    Z = torch.from_numpy(_random_paths(rng, 4, 6, geo, 40, 50)).cuda()
    for variant in (1, 3):
        rm = uam.RasterMap.from_arrays(lay, geo, occ, options={'integral_variant': variant})
        with pytest.raises(uam.UamError) as ei:
            rm.refine_paths_swept(Z, [1.0, 2.0], 1.0, 2)
        assert ei.value.code == -5
        rm.refine_paths_swept(Z, [1.0, 2.0], 0.0, 2)        # waypoint mode has one kernel, whatever the variant
    rm = uam.RasterMap.from_arrays(lay, geo, occ)
    for kw in (dict(iterations=-1), dict(min_step_cells=0.0), dict(step_cells=2.0, max_step_cells=1.0),
               dict(max_step_cells=float('inf')), dict(min_d2=-1), dict(min_d2=65536)):
        with pytest.raises(uam.UamError) as ei:
            rm.refine_paths_swept(Z, [1.0, 2.0], 1.0, **dict(dict(iterations=2), **kw))
        assert ei.value.code == -1, kw
    with pytest.raises(TypeError):
        rm.refine_paths_swept(Z, [1.0, 2.0], 1.0, 2, min_d2=2.0)       # an integer in squared cells, not a radius
    rm.refine_paths_swept(Z, [1.0, 2.0], 1.0, 2, min_d2=65535)
    out = rm.refine_paths_swept(Z[:0], [1.0, 2.0], 1.0, 3, min_d2=1)     # B = 0
    assert out[0].shape == (0, 12) and out[4].shape == (0,) and out[5].shape == (0,)
    lib = _lib.load()
    eng = rm.engine
    p = rm.parameter_vector([1.0, 2.0])
    pp = p.ctypes.data_as(C.c_void_p)
    Zc = Z.clone()
    zp = C.c_void_p(Zc.data_ptr())
    cost = torch.empty(4, dtype=torch.float32, device='cuda')
    col = torch.empty(4, dtype=torch.uint8, device='cuda')
    fl = torch.empty(4, dtype=torch.uint8, device='cuda')
    cp, kp, fp = C.c_void_p(cost.data_ptr()), C.c_void_p(col.data_ptr()), C.c_void_p(fl.data_ptr())
    args = (4, 4, pp, p.size, _lib.UAM_LENGTH_SMOOTH | _lib.UAM_OWN_START, 1.0, 2, 1.0, 16.0, 1.0 / 256, 2)
    f = lib.uam_refine_paths_raster_swept
    assert f(eng._h, None, *args, cp, kp, None, fp, None, None) == -1       # NULL paths
    assert f(eng._h, zp, *args, None, kp, None, fp, None, None) == -1       # NULL cost
    assert f(eng._h, zp, *args, cp, None, None, fp, None, None) == -1       # NULL collide
    assert f(eng._h, zp, *args, cp, kp, None, None, None, None) == -1       # NULL sweep flags
    assert f(eng._h, zp, 0, *args[1:], None, None, None, None, None, None) == 0     # B = 0
    assert f(eng._h, zp, *args, cp, kp, None, fp, None, None) == 0          # accepted and d2min are optional
    torch.cuda.synchronize()
    cs, ks = rm.score_paths(Zc, [1.0, 2.0], 1.0)
    fs, _, _ = rm.sweep_paths(Zc, clearance=False)
    assert torch.equal(cs, cost) and torch.equal(ks, col) and torch.equal(fs, fl)
    h = C.c_void_p()
    assert lib.uam_ctx_create(0, C.byref(h)) == 0
    assert f(h, zp, *args, cp, kp, None, fp, None, None) == -4             # no raster
    assert lib.uam_ctx_destroy(h) == 0
    # an N beyond the sweep's shared-memory table; refine_paths takes it
    Zl = torch.from_numpy(_random_paths(rng, 2, 3659, geo, 40, 50)).cuda()
    rm.refine_paths(Zl, [1.0, 2.0], 0.0, 1)
    with pytest.raises(uam.UamError) as ei:
        rm.refine_paths_swept(Zl, [1.0, 2.0], 0.0, 1)
    assert ei.value.code == -5
    rm.refine_paths_swept(Zl[:, :-2].contiguous(), [1.0, 2.0], 0.0, 1)      # N = 3656 fits
    # over 23170 cells per side: flags only; the clearance (min_d2 > 0 or d2min wanted) is refused
    H, W = 3, 23171
    occ_w = np.zeros((H, W), dtype=np.uint8)
    occ_w[1, 20000] = 1
    rw = uam.RasterMap.from_arrays(np.ones((1, H, W), dtype=np.float32), GEO_PIX, occ_w)
    Zw = np.array([[10.0, 1.0, 5000.0, 0.5, 23160.0, 1.0], [0.0, 0.0, 50.0, 0.2, 100.0, 0.0]])
    for min_d2, want in ((1, False), (0, True)):
        with pytest.raises(uam.UamError) as ei:
            rw.engine.refine_raster_swept(Zw, 1, rw.parameter_vector([1.0]), _lib.UAM_OWN_START, 0.0, 2, 1.0, 4.0,
                                          1.0 / 256, min_d2, want)
        assert ei.value.code == -5
    out = rw.refine_paths_swept(Zw, [1.0], 0.0, 2)
    assert list(out[4]) == [HIT, 0]


@pytest.mark.gpu
def test_refine_swept_large_batch(uam, torch):
    """8192 paths x 64 waypoints on a 2048^2 raster (binned pipeline), 20 trips, min_d2 = 4: no path gains a sweep flag,
    no capped clearance drops, and no path that starts with collide = 0 ends HIT.  A path that starts colliding and
    HIT may lose its sampled collide flag while still crossing an occupied cell (it gains no flag), so the count of
    paths with collide = 0 yet HIT may grow by those only; refine_paths on the same input adds clean paths to it
    (printed, not asserted)."""
    import bench
    n = 2048
    layers, occ, geo = bench.make_raster(torch, 'cuda:0', n)
    rm = uam.RasterMap.from_arrays(layers, geo, occ)
    Z = bench.make_paths(torch, 'cuda:0', 8192, seed=5, n=n)
    w, spc = bench.WEIGHTS, 1.0
    _, k0 = rm.score_paths(Z, w, spc)
    f0, _, d0 = rm.sweep_paths(Z)
    Zo, c, k, acc, f, d2 = rm.refine_paths_swept(Z, w, spc, 20, min_d2=4)
    cs, ks = rm.score_paths(Zo, w, spc)
    assert torch.equal(cs, c) and torch.equal(ks, k)
    assert int((f & ~f0).sum()) == 0
    assert bool(torch.all(torch.clamp(d2, max=4) >= torch.clamp(d0, max=4)))
    hit0, hit = (f0 & HIT) != 0, (f & HIT) != 0
    clean_hit0 = int(((k0 == 0) & hit0).sum())
    clean_hit = int(((k == 0) & hit).sum())
    assert int(((k0 == 0) & ~hit0 & hit).sum()) == 0
    Zp, _, kp, _ = rm.refine_paths(Z, w, spc, 20)
    fp, _, _ = rm.sweep_paths(Zp, clearance=False)
    clean_hit_plain = int(((kp == 0) & ((fp & HIT) != 0)).sum())
    inside = int(((f0 & OUTSIDE) == 0).sum())
    print(f'large batch: {inside} paths inside; collide = 0 but HIT: {clean_hit0} before, {clean_hit} after the swept '
          f'refine ({int(((k0 != 0) & (k == 0) & hit).sum())} of them collided before), {clean_hit_plain} after '
          f'refine_paths; mean accepted trips {acc.float().mean().item():.2f}')
    assert float((acc > 0).float().mean()) >= 0.8
