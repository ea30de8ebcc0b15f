"""Refinement under the analytic obstacle check (uam_refine_paths_raster_keepout / RasterMap.refine_paths_keepout).

CPU: the numpy restatement of the rule (raster_refine_keepout_reference) driven by the float64 oracle and the numpy
restatements of the analytic sweep and clearance: the rule's invariants (K1, K2, monotone (collide, cost), K3), and a
hand case where the raster rules cut a disc between the cell centres and the keep-out rule stops short.  GPU: the device
loop against the restatement driven by the device gradient, sweep and clearance, bit for bit; the library interface;
set_obstacles; bit identity with refine_paths where the analytic terms never reject; errors; a large batch on C2's map.
"""
import ctypes as C

import numpy as np
import pytest

from analytic_clearance_reference import clearance_reference
from analytic_sweep_reference import HIT, INVALID, sweep_reference
from oracle import uam_oracle as orc
from raster_gradient_oracle import score_paths_raster_gradient
from raster_refine_keepout_reference import refine_keepout_reference
from raster_refine_reference import refine_reference
from raster_refine_swept_reference import refine_swept_reference
from raster_sweep_reference import sweep_reference as raster_sweep_reference
from test_analytic_sweep import _disc, _poly, _square
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


def _reference_check(recs, margin):
    """check(Z) of the rule from the numpy restatements: the sweep's flags, or with a margin the clearance's flags and
    clearance at cap = margin (its flags are the sweep's, D1)"""
    def check(Z):
        if margin > 0:
            f, cl, _, _ = clearance_reference(Z, recs, margin)
            return f, cl
        return sweep_reference(Z, recs)[0], None
    return check


def _obstacle_records(rng, geo, H, W, n=12):
    """Discs, boxes and convex pentagons spread over the raster's rectangle"""
    x0, dx, y0, dy = geo
    lo = np.array([min(x0, x0 + dx * W), min(y0, y0 + dy * H)])
    hi = np.array([max(x0, x0 + dx * W), max(y0, y0 + dy * H)])
    s = float(np.min(hi - lo))
    recs = []
    for i in range(n):
        c = lo + rng.uniform(0.05, 0.95, 2) * (hi - lo)
        if i % 3 == 0:
            recs.append(_disc(c[0], c[1], float(rng.uniform(0.02, 0.07) * s)))
        elif i % 3 == 1:
            recs.append(_square(c[0], c[1], float(rng.uniform(0.02, 0.06) * s), float(rng.uniform(0.02, 0.06) * s)))
        else:
            ang = np.sort(rng.uniform(0, 2 * np.pi, 5))
            r = rng.uniform(0.03, 0.08) * s
            recs.append(_poly(c + r * np.stack([np.cos(ang), np.sin(ang)], 1)))
    return recs


def _cpu_case(seed, spc, x_start, B=24, Wp=9):
    rng = np.random.default_rng(seed)
    H, W = 70, 90
    lay, occ = _random_raster(rng, 3, H, W)
    Z = _random_paths(rng, B, Wp, GEO, H, W, spill=0.05)
    ev = _oracle_evaluate(lay, occ, GEO, [200.0, 1500.0, 2700.0], spc, x_start,
                          bad_rows=[(3, 4, np.nan), (5, 2 * Wp - 3, -np.inf)])
    return Z, ev, _obstacle_records(rng, GEO, H, W), min(abs(GEO[1]), abs(GEO[3]))


# ------------------------------------------------------------------------------------------------------------------
# CPU: the rule on the float64 oracle
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('spc', [0.0, 1.0])
@pytest.mark.parametrize('x_start', [None, [4.0, 39.0]])
@pytest.mark.parametrize('margin', [0.0, 1e-3, 0.5])
def test_reference_invariants(spc, x_start, margin):
    Z, ev, recs, h = _cpu_case(61, spc, x_start)
    check = _reference_check(recs, margin)
    c0, k0, _ = ev(Z)
    f0, cl0 = check(Z)
    trace = []
    Zo, c, k, acc, f, cl = refine_keepout_reference(ev, check, Z, h, 8, margin=margin, trace=trace)
    good = np.ones(Z.shape[0], dtype=bool)
    good[[3, 5]] = False
    # K1: no HIT or INVALID is gained; K2: the clearance capped at the margin never drops
    assert not np.any(f & ~f0)
    if margin > 0:
        assert np.all(cl >= cl0) and np.all(cl <= margin)
    else:
        assert cl is None
    # (collide, cost) is monotone, as for refine_paths
    assert np.all(k <= k0) and np.all(c[good] <= c0[good])
    # rows with NaN / inf in the gradient come back bit-identical
    assert np.array_equal(_bits(Zo[~good]), _bits(Z[~good])) and np.all(acc[~good] == 0)
    assert np.array_equal(_bits(Zo[:, :2]), _bits(Z[:, :2])) and np.array_equal(_bits(Zo[:, -2:]), _bits(Z[:, -2:]))
    # the outputs are the evaluation and the analytic check of the returned paths
    ce, ke, _ = ev(Zo)
    fe, cle = check(Zo)
    assert np.array_equal(_bits(ce), _bits(c)) and np.array_equal(ke, k) and np.array_equal(fe, f)
    assert (cl is None and cle is None) or np.array_equal(_bits(cle), _bits(cl))
    # K3: every accepted trial the plain rule accepts too; here the analytic terms do reject some
    assert all(np.all(t['accepted'] <= t['plain']) for t in trace)
    assert sum(int(np.sum(t['plain'] & ~t['accepted'])) for t in trace) > 0
    assert np.sum(acc > 0) >= Z.shape[0] // 2


def test_reference_zero_iterations_is_the_identity():
    Z, ev, recs, h = _cpu_case(62, 1.0, None)
    check = _reference_check(recs, 0.5)
    c0, k0, _ = ev(Z)
    f0, cl0 = check(Z)
    Zo, c, k, acc, f, cl = refine_keepout_reference(ev, check, Z, h, 0, margin=0.5)
    assert np.array_equal(_bits(Zo), _bits(Z)) and np.array_equal(_bits(c), _bits(c0)) and np.array_equal(k, k0)
    assert np.all(acc == 0) and np.array_equal(f, f0) and np.array_equal(_bits(cl), _bits(cl0))


def test_reference_nan_clearance_takes_no_trial():
    """With a margin, a path whose clearance is NaN (as an INVALID path's is) takes no trial, even where the plain rule
    would take one.  Here check() reports row 7 as INVALID with a NaN clearance for every trial."""
    Z, ev, recs, h = _cpu_case(63, 0.0, None)
    inner = _reference_check(recs, 0.5)

    def check(Zq):
        f, cl = inner(Zq)
        f, cl = f.copy(), cl.copy()
        f[7] |= INVALID
        cl[7] = np.nan
        return f, cl
    trace = []
    refine_keepout_reference(ev, check, Z, h, 6, margin=0.5, trace=trace)
    assert any(t['plain'][7] for t in trace)
    assert not any(t['accepted'][7] for t in trace)


def _hand_case():
    """Waypoint mode on zero penalty layers, in pixel coordinates: a disc of radius 0.6 around the cell centre (2, 2),
    so the occupancy taken at cell centres marks that one cell, and the disc reaches 0.1 beyond its square between the
    centres.  The path (0, 2.55) -> (2, 8) -> (4, 2.55): the length term pulls the free waypoint down to (2, 2.55),
    inside the disc's rim and above the occupied square."""
    H = W = 16
    lay = np.zeros((1, H, W), dtype=np.float32)
    yy, xx = np.mgrid[0:H, 0:W]
    occ = (((xx - 2.0) ** 2 + (yy - 2.0) ** 2) <= 0.36).astype(np.uint8)
    assert occ.sum() == 1 and occ[2, 2] == 1
    Z = np.array([[0.0, 2.55, 2.0, 8.0, 4.0, 2.55]])
    return lay, occ, [_disc(2.0, 2.0, 0.6)], Z


def test_hand_case_the_raster_rules_cut_the_disc_between_centres():
    lay, occ, recs, Z = _hand_case()
    ev = _oracle_evaluate(lay, occ, GEO_PIX, [1.0], 0.0)
    d2 = orc.edt_sq(occ)

    def raster_sweep(Zq):
        f, _, d = raster_sweep_reference(occ, GEO_PIX, Zq, d2)
        return f, d
    assert raster_sweep(Z)[0][0] == 0 and sweep_reference(Z, recs)[0][0] == 0
    # the plain rule and the raster-swept rule both end inside the disc, clean in the raster's picture
    Zp, cp, kp, _ = refine_reference(ev, Z, 1.0, 20)
    Zs, cs, ks, _, fs, _ = refine_swept_reference(ev, raster_sweep, Z, 1.0, 20)
    for Zr, kr in ((Zp, kp), (Zs, ks)):
        assert kr[0] == 0 and raster_sweep(Zr)[0][0] == 0 and sweep_reference(Zr, recs)[0][0] == HIT
    assert fs[0] == 0
    # the keep-out rule stops short of the disc and still descends
    c0 = ev(Z)[0][0]
    Zk, ck, kk, acc, fk, _ = refine_keepout_reference(ev, _reference_check(recs, 0.0), Z, 1.0, 20)
    assert kk[0] == 0 and fk[0] == 0 and acc[0] > 0 and sweep_reference(Zk, recs)[0][0] == 0
    assert cs[0] < ck[0] < c0
    # with a margin it also stays that far away
    margin = 0.25
    Zm, cm, km, accm, fm, clm = refine_keepout_reference(ev, _reference_check(recs, margin), Z, 1.0, 20, margin=margin)
    assert km[0] == 0 and fm[0] == 0 and accm[0] > 0 and clm[0] == margin
    assert clearance_reference(Zm, recs, margin)[1][0] == margin
    assert ck[0] < cm[0] < c0
    assert clearance_reference(Zk, recs, margin)[1][0] < margin


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


def _shape_map(uam, recs):
    m = uam.Map()
    for r in recs:
        m.add(uam.QuadraticObstacle(*[uam.shapes.Inequality(row) for row in r]))
    return m


def _device_evaluate(rm, w, spc, x_start=None):
    def evaluate(Z):
        return rm.cost_gradient(np.ascontiguousarray(Z), w, spc, True, x_start)
    return evaluate


def _device_check(rm, N, margin):
    def check(Z):
        Z = np.ascontiguousarray(Z)
        if margin > 0:
            f, cl, _, _ = rm.engine.clearance_analytic(Z, N, margin, False)
            return f, cl
        return rm.engine.sweep_analytic(Z, N, False, False)[0], None
    return check


def _refine_keepout(rm, Z, w, spc, K, x_start, margin, want_clearance):
    """Engine.refine_raster_keepout, which can also keep the clearance in scratch (margin > 0, none returned)"""
    from uam_path_planning_b200 import _lib
    flags = _lib.UAM_LENGTH_SMOOTH | (_lib.UAM_OWN_START if x_start is None else 0)
    return rm.engine.refine_raster_keepout(Z, Z.shape[1] // 2 - 2, rm.parameter_vector(w, x_start), flags, spc, K, 1.0,
                                           64.0, 1.0 / 256, margin, want_clearance)


@pytest.mark.gpu
@pytest.mark.parametrize('L', [1, 3])
@pytest.mark.parametrize('spc', [0.0, 1.0])
@pytest.mark.parametrize('layout', [0, 1])
@pytest.mark.parametrize('variant', [-1, 0, 2])
@pytest.mark.parametrize('combine', [0, 1, 2])
def test_refine_keepout_matches_reference_bit_for_bit(uam, torch, L, spc, layout, variant, combine):
    """The device loop against refine_keepout_reference driven by the device gradient, sweep and clearance: Z_out, cost,
    collide, accepted, sweep flags and clearance are identical after 0, 1, 3 and 8 trips, for margin = 0, 1e-3 and 0.5
    km (with the clearance returned and kept in scratch), on every gradient kernel and texel form (float2 / float4
    texels, quads + bit-plane, sign-packed quads), on a map of discs, boxes and polygons."""
    if spc == 0.0 and variant != -1:
        pytest.skip('waypoint mode has a single kernel')
    if combine != 1 and variant != 2:
        pytest.skip('quad texels are sampled by the binned pipeline only (at these batch sizes)')
    rng = np.random.default_rng(500 + L + 10 * layout)
    H, W = (150, 230) if layout else (151, 229)
    h = min(abs(GEO[1]), abs(GEO[3]))
    lay, occ = _random_raster(rng, L, H, W)
    rm = uam.RasterMap.from_arrays(lay, GEO, occ, options={'raster_layout': layout, 'integral_variant': variant,
                                                           'combine_layers': combine})
    rm.set_obstacles(_shape_map(uam, _obstacle_records(rng, GEO, H, W, n=18)))
    w = [200.0, -15000.0, 27000.0][:L] if combine == 2 else [200.0, 15000.0, 27000.0][:L]
    rejected = 0
    cases = [(64, 0.0, None, 0.5, True), (7, 0.15, [4.0, 39.0], 0.0, False), (3, 0.0, None, 1e-3, True),
             (130, 0.05, [0.0, 0.0], 0.5, False)]
    for Wp, spill, x_start, margin, want_cl in cases:
        Z = _random_paths(rng, 96, Wp, GEO, H, W, spill)
        Z[5, 2] = np.nan
        trace = []
        ev = _device_evaluate(rm, w, spc, x_start)
        check = _device_check(rm, Wp - 2, margin)
        c0, k0, _ = ev(Z)
        f0, cl0 = check(Z)
        refine_keepout_reference(ev, check, Z, h, 8, margin=margin, trace=trace)
        acc_ref = np.cumsum([t['accepted'] for t in trace], axis=0)
        rejected += sum(int(np.sum(t['plain'] & ~t['accepted'])) for t in trace)
        for K in (0, 1, 3, 8):
            Zo, c, k, acc, f, cl = _refine_keepout(rm, Z, w, spc, K, x_start, margin, want_cl)
            if K == 0:
                Zr, cr, kr, ar, fr, clr = Z, c0, k0, np.zeros(96, dtype=np.int32), f0, cl0
            else:
                t = trace[K - 1]
                Zr, cr, kr, ar, fr, clr = t['Z'], t['cost'], t['collide'], acc_ref[K - 1], t['flags'], t['clearance']
            key = (Wp, margin, K)
            assert np.array_equal(_bits(Zo), _bits(Zr)), key
            assert np.array_equal(_bits(c), _bits(cr)) and np.array_equal(k, kr), key
            assert np.array_equal(acc, ar) and np.array_equal(f, fr), key
            if want_cl:
                assert np.array_equal(_bits(cl), _bits(clr)), key
            else:
                assert cl is None, key
        assert np.array_equal(_bits(Zo[5]), _bits(Z[5]))          # NaN row untouched
        assert np.sum(acc_ref[-1] > 0) > 48                        # the descent does move the others
    assert rejected > 0                                            # and the analytic terms did reject trials


@pytest.mark.gpu
@pytest.mark.parametrize('margin', [0.0, 0.5])
def test_refine_keepout_same_bits_with_and_without_cell_lists(uam, torch, margin):
    rng = np.random.default_rng(41)
    H, W = 160, 200
    lay, occ = _random_raster(rng, 3, H, W)
    rm = uam.RasterMap.from_arrays(lay, GEO, occ)
    rm.set_obstacles(_shape_map(uam, _obstacle_records(rng, GEO, H, W, n=30)))
    Z = _random_paths(rng, 200, 33, GEO, H, W, spill=0.05)
    w = [200.0, 15000.0, 27000.0]
    rm.engine.set_option('shape_grid', 1)
    a = rm.refine_paths_keepout(Z, w, 1.0, 8, margin=margin)
    rm.engine.set_option('shape_grid', 0)
    b = rm.refine_paths_keepout(Z, w, 1.0, 8, margin=margin)
    rm.engine.set_option('shape_grid', 1)
    for x, y in zip(a, b):
        assert (x is None and y is None) or np.array_equal(_bits(x), _bits(y))
    assert np.sum(a[3] > 0) > 100


@pytest.mark.gpu
@pytest.mark.parametrize('spc', [0.0, 1.0])
def test_refine_keepout_interface(uam, torch, spc):
    """The outputs are score_paths', Map.sweep_paths' and Map.path_clearance's bits for the returned paths; numpy and
    tensor inputs give the same bits and the input tensor is left as it was; a permuted batch gives the permuted
    result."""
    rng = np.random.default_rng(39)
    H, W, geo = 120, 90, (0.0, 0.5, 0.0, 0.5)
    lay, occ = _random_raster(rng, 3, H, W)
    rm = uam.RasterMap.from_arrays(lay, geo, occ)
    m = _shape_map(uam, _obstacle_records(rng, geo, H, W, n=9))
    rm.set_obstacles(m)
    w = [1.0, 2.0, 3.0]
    Z = _random_paths(rng, 40, 16, geo, H, W, spill=0.05)
    Zt = torch.from_numpy(Z).cuda()
    Zt_before = Zt.clone()
    out = rm.refine_paths_keepout(Zt, w, spc, 6, margin=0.5)
    Zo, c, k, acc, f, cl = out
    assert all(t.is_cuda for t in out) and Zo.data_ptr() != Zt.data_ptr()
    assert torch.equal(Zt, Zt_before)
    cs, ks = rm.score_paths(Zo, w, spc)
    assert torch.equal(cs, c) and torch.equal(ks, k)
    fs, _, _ = m.sweep_paths(Zo)
    _, cls, _, _ = m.path_clearance(Zo, 0.5)
    assert torch.equal(fs, f) and torch.equal(cls, cl)
    host = rm.refine_paths_keepout(Z, w, spc, 6, margin=0.5)
    assert all(isinstance(a, np.ndarray) for a in host)
    for a, b in zip(host, out):
        assert np.array_equal(_bits(a), _bits(b.cpu().numpy()))
    perm = np.random.default_rng(40).permutation(40)
    for a, b in zip(rm.refine_paths_keepout(np.ascontiguousarray(Z[perm]), w, spc, 6, margin=0.5), host):
        assert np.array_equal(_bits(a), _bits(b[perm]))
    no_cl = rm.refine_paths_keepout(Z, w, spc, 6)
    assert no_cl[5] is None
    assert np.array_equal(no_cl[4], m.sweep_paths(no_cl[0])[0])


@pytest.mark.gpu
@pytest.mark.parametrize('spc', [0.0, 1.0])
def test_refine_keepout_equals_refine_paths_where_nothing_rejects(uam, torch, spc):
    """No obstacles, and obstacles 1000 km from every path: the analytic terms cannot reject a trial, so the result is
    refine_paths' bit for bit, for margin 0 and 0.5."""
    rng = np.random.default_rng(31)
    H, W, geo = 200, 240, (0.0, 0.5, 0.0, 0.5)
    lay, occ = _random_raster(rng, 3, H, W)
    rm = uam.RasterMap.from_arrays(lay, geo, occ)
    w = [100.0, 200.0, 300.0]
    Z = _random_paths(rng, 64, 12, geo, H, W, spill=0.05)
    Zp, cp, kp, ap = rm.refine_paths(Z, w, spc, 20)
    assert np.sum(ap > 0) >= 48
    far = [_disc(1000.0, 1000.0, 5.0), _square(-1000.0, 50.0, 3.0),
           _poly([[1000.0, -900.0], [1010.0, -900.0], [1005.0, -890.0]]), _disc(50.0, 1200.0, 1.0, 2.0),
           _square(1100.0, 1100.0, 1.0, 4.0)]
    for recs in ([], far):
        rm.set_obstacles(_shape_map(uam, recs))
        for margin in (0.0, 0.5):
            Zk, ck, kk, ak, fk, clk = rm.refine_paths_keepout(Z, w, spc, 20, margin=margin)
            assert np.array_equal(_bits(Zk), _bits(Zp)) and np.array_equal(_bits(ck), _bits(cp))
            assert np.array_equal(kk, kp) and np.array_equal(ak, ap) and not np.any(fk)
            assert clk is None if margin == 0 else np.all(clk == margin)


@pytest.mark.gpu
def test_set_obstacles_changes_no_raster_output(uam, torch):
    """A shapes upload (set_obstacles after from_arrays) leaves score_paths, cost_gradient, sweep_paths and refine_paths
    bit for bit as they were; it is a snapshot, so a change to the map needs a new call."""
    rng = np.random.default_rng(45)
    H, W = 140, 170
    lay, occ = _random_raster(rng, 3, H, W)
    rm = uam.RasterMap.from_arrays(lay, GEO, occ)
    w = [200.0, 15000.0, 27000.0]
    Z = _random_paths(rng, 300, 20, GEO, H, W, spill=0.05)

    def outputs():
        return (*rm.score_paths(Z, w, 1.0), *rm.score_paths(Z, w, 0.0), *rm.cost_gradient(Z, w, 1.0),
                *rm.sweep_paths(Z), *rm.refine_paths(Z, w, 1.0, 4))
    before = outputs()
    m = _shape_map(uam, _obstacle_records(rng, GEO, H, W, n=20))
    rm.set_obstacles(m)
    assert np.array_equal(rm.engine.sweep_analytic(Z, 18, False, False)[0], m.sweep_paths(Z)[0])
    after = outputs()
    for a, b in zip(before, after):
        assert np.array_equal(_bits(a), _bits(b))
    # the upload is a snapshot: the raster's engine keeps the old shapes until set_obstacles runs again
    f_old = m.sweep_paths(Z)[0]
    x0, dx, y0, dy = GEO
    m.add(uam.square([x0 + dx * W / 2, y0 + dy * H / 2], abs(dx) * W, abs(dy) * H))    # covers the whole raster
    assert np.array_equal(rm.engine.sweep_analytic(Z, 18, False, False)[0], f_old)
    rm.set_obstacles(m)
    f_new = rm.engine.sweep_analytic(Z, 18, False, False)[0]
    assert np.array_equal(f_new, m.sweep_paths(Z)[0]) and np.all(f_new == HIT)


@pytest.mark.gpu
def test_refine_keepout_errors_in_order(uam, torch):
    from uam_path_planning_b200 import _lib
    rng = np.random.default_rng(3)
    lay, occ = _random_raster(rng, 2, 40, 50)
    geo = (0.0, 1.0, 0.0, 1.0)
    Z = torch.from_numpy(_random_paths(rng, 4, 6, geo, 40, 50)).cuda()
    good = _shape_map(uam, [_disc(10.0, 10.0, 2.0), _square(30.0, 20.0, 3.0)])
    # a forced integral variant without a gradient form comes before the missing shapes
    for variant in (1, 3):
        rm = uam.RasterMap.from_arrays(lay, geo, occ, options={'integral_variant': variant})
        with pytest.raises(uam.UamError) as ei:
            rm.refine_paths_keepout(Z, [1.0, 2.0], 1.0, 2)
        assert ei.value.code == -5
        rm.set_obstacles(good)
        rm.refine_paths_keepout(Z, [1.0, 2.0], 0.0, 2)        # waypoint mode has one kernel, whatever the variant
    rm = uam.RasterMap.from_arrays(lay, geo, occ)
    # argument errors come before the missing shapes
    for kw in (dict(iterations=-1), dict(min_step_cells=0.0), dict(step_cells=2.0, max_step_cells=1.0),
               dict(max_step_cells=float('inf')), dict(margin=-1e-9), dict(margin=float('nan')), dict(margin=2e100),
               dict(margin=float('inf'))):
        with pytest.raises(uam.UamError) as ei:
            rm.refine_paths_keepout(Z, [1.0, 2.0], 1.0, **dict(dict(iterations=2), **kw))
        assert ei.value.code == -1, kw
    with pytest.raises(uam.UamError) as ei:
        rm.refine_paths_keepout(Z, [1.0, 2.0], 1.0, 2)
    assert ei.value.code == -4                                             # no shapes uploaded
    out = rm.refine_paths_keepout(Z[:0], [1.0, 2.0], 1.0, 3, margin=0.1)   # B = 0 is a no-op, before the state
    assert out[0].shape == (0, 12) and out[4].shape == (0,) and out[5].shape == (0,)
    rm.set_obstacles(good)
    rm.refine_paths_keepout(Z, [1.0, 2.0], 1.0, 2, margin=1e100)
    lib = _lib.load()
    eng = rm.engine
    p = rm.parameter_vector([1.0, 2.0])
    pp = p.ctypes.data_as(C.c_void_p)
    Zc = Z.clone()
    zp = C.c_void_p(Zc.data_ptr())
    cost = torch.empty(4, dtype=torch.float32, device='cuda')
    col = torch.empty(4, dtype=torch.uint8, device='cuda')
    fl = torch.empty(4, dtype=torch.uint8, device='cuda')
    cl = torch.empty(4, dtype=torch.float64, device='cuda')
    cp, kp, fp, clp = (C.c_void_p(t.data_ptr()) for t in (cost, col, fl, cl))
    args = (4, 4, pp, p.size, _lib.UAM_LENGTH_SMOOTH | _lib.UAM_OWN_START, 1.0, 2, 1.0, 16.0, 1.0 / 256)
    f = lib.uam_refine_paths_raster_keepout
    assert f(None, zp, *args, 0.5, cp, kp, None, fp, clp, None) == -1      # no ctx
    assert f(eng._h, None, *args, 0.5, cp, kp, None, fp, clp, None) == -1  # NULL paths
    assert f(eng._h, zp, *args, 0.5, None, kp, None, fp, clp, None) == -1  # NULL cost
    assert f(eng._h, zp, *args, 0.5, cp, None, None, fp, clp, None) == -1  # NULL collide
    assert f(eng._h, zp, *args, 0.5, cp, kp, None, None, clp, None) == -1  # NULL sweep flags
    assert f(eng._h, zp, *args, 0.0, cp, kp, None, fp, clp, None) == -1    # a clearance pointer needs margin > 0
    assert f(eng._h, zp, 4, 0, *args[2:], 0.5, cp, kp, None, fp, clp, None) == -1          # N < 1
    assert f(eng._h, zp, 0, *args[1:], 0.5, None, None, None, None, None, None) == 0       # B = 0
    assert f(eng._h, zp, *args, 0.5, cp, kp, None, fp, None, None) == 0    # accepted and clearance are optional
    torch.cuda.synchronize()
    cs, ks = rm.score_paths(Zc, [1.0, 2.0], 1.0)
    assert torch.equal(cs, cost) and torch.equal(ks, col) and torch.equal(fl, good.sweep_paths(Zc)[0])
    assert f(eng._h, zp, *args, 0.5, cp, kp, None, fp, clp, None) == 0
    torch.cuda.synchronize()
    assert torch.equal(cl, good.path_clearance(Zc, 0.5)[1])
    h = C.c_void_p()
    assert lib.uam_ctx_create(0, C.byref(h)) == 0
    assert f(h, zp, *args, 0.5, cp, kp, None, fp, clp, None) == -4        # no raster
    assert lib.uam_ctx_destroy(h) == 0
    # the sweep's record checks, then (margin > 0 only) the clearance's form checks: before anything is launched
    bad_record = [[1, np.nan, 0, 1, 1, 0, 0, 0]]                             # a NaN centre
    bad_form = np.concatenate([_poly([[0.0, 0.0], [4.0, 0.0], [1.0, 3.0]]), _disc(1.0, 1.0, 0.5)])   # lines + ellipse
    for recs, margins_refused, margins_taken in (([_disc(10.0, 10.0, 2.0), bad_record], (0.0, 0.5), ()),
                                                 ([_disc(10.0, 10.0, 2.0), bad_form], (0.5,), (0.0,))):
        rm.set_obstacles(_shape_map(uam, recs))
        for margin in margins_refused:
            n0 = eng.launch_count()
            with pytest.raises(uam.UamError) as ei:
                rm.refine_paths_keepout(Z, [1.0, 2.0], 1.0, 2, margin=margin)
            assert ei.value.code == -5 and eng.launch_count() == n0, margin
            with pytest.raises(uam.UamError) as ei:                        # argument errors still come first
                rm.refine_paths_keepout(Z, [1.0, 2.0], 1.0, 2, margin=margin, step_cells=0.0)
            assert ei.value.code == -1
        for margin in margins_taken:
            rm.refine_paths_keepout(Z, [1.0, 2.0], 1.0, 2, margin=margin)


@pytest.mark.gpu
def test_refine_keepout_large_batch_on_c2(uam, torch):
    """C2's map rasterised with from_map at 2048^2, 8192 corridor paths x 64 waypoints, 20 trips, margin 0.25 km: no
    path gains an analytic HIT, no clearance capped at the margin drops, and the outputs are score_paths',
    Map.sweep_paths' and Map.path_clearance's bits for the returned paths."""
    import bench_analytic_sweep
    rng = np.random.default_rng(20260101)
    m = bench_analytic_sweep.c2_map(uam, rng)
    n, km, Wp, B, margin = 2048, 64.0, 64, 8192, 0.25
    rm = uam.RasterMap.from_map(m, n, n, (0.0, km / n, 0.0, km / n))
    prob = uam.Problem(m, Wp - 2, {'length_smooth': True, 'obstacle_smooth': True})
    prob.params.update(maxratio=1.04, maxalpha=np.pi / 80, enlargement=0)
    prob.set_weight('Risk', 5000.0)
    Zh = uam.Solver(prob, {}).candidates(rng.uniform(-0.9, 0.9, B), jitter=0.25 * km / 4096, rng=rng)
    Z = torch.from_numpy(np.ascontiguousarray(Zh)).cuda()
    w, spc = [5000.0], 1.0
    f0, _, _ = m.sweep_paths(Z)
    _, cl0, _, _ = m.path_clearance(Z, margin)
    Zo, c, k, acc, f, cl = rm.refine_paths_keepout(Z, w, spc, 20, margin=margin)
    cs, ks = rm.score_paths(Zo, w, spc)
    assert torch.equal(cs, c) and torch.equal(ks, k)
    fs, _, _ = m.sweep_paths(Zo)
    _, cls, _, _ = m.path_clearance(Zo, margin)
    assert torch.equal(fs, f) and torch.equal(cls, cl)
    assert int((f & ~f0).sum()) == 0
    assert bool(torch.all(cl >= cl0))
    Zp, _, kp, _ = rm.refine_paths(Z, w, spc, 20)
    fp, _, _ = m.sweep_paths(Zp)
    _, clp, _, _ = m.path_clearance(Zp, margin)
    print(f'C2 corridor: HIT before {int((f0 & HIT).sum())}; gained HIT: keep-out 0, refine_paths '
          f'{int(((fp & ~f0) & HIT).sum())}; capped clearance dropped: refine_paths {int((clp < cl0).sum())}; '
          f'mean accepted trips {acc.float().mean().item():.2f}')
    assert float((acc > 0).float().mean()) >= 0.5
