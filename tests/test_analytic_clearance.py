"""Clearance of whole path segments from the analytic obstacles (uam_clearance_paths_analytic / Map.path_clearance).

CPU: the numpy restatement (analytic_clearance_reference) against the exact oracle on hand cases and random segments at
km and 1e6 scale (D2), HIT => 0 on the reference's golden waypoint collisions (D1), and the form check.
GPU: the kernel against the restatement bit for bit over maps, path lengths, caps and the shape_grid option (D3); D1
against the sweep; batch independence; the lists' invalidation; the error codes; a one-sided cross-check with the raster.
"""
import ctypes as C
import math

import mpmath
import numpy as np
import pytest

from analytic_clearance_reference import (BOX_FORM, DISC_FORM, ELLIPSE_FORM, POLYGON_FORM, Unsupported, clearance_reference,
                                          delta, exact_distance, obstacle_form, pair_distance)
from analytic_sweep_reference import HIT, INVALID, segment_hits, sweep_reference
from conftest import build_product_map, full_paths
from oracle import uam_oracle as orc
from test_analytic_sweep import (ELLIPSE, LINE, _c2_like_map, _c4_like_map, _disc, _map_from_records, _mixed_map,
                                 _oshape_records, _paths, _poly, _records, _square)


def _D(recs, seg):
    return float(pair_distance(recs, *(np.array([v]) for v in seg))[0])


def _check_d2(recs, seg):
    """D2 for a non-HIT pair, D1's D = 0 for a HIT pair; returns D."""
    D = _D(recs, seg)
    if bool(segment_hits(recs, *(np.array([v]) for v in seg))[0]):
        assert D == 0.0
        return D
    ex = exact_distance(recs, *seg)
    assert D > 0.0
    assert abs(mpmath.mpf(D) - ex) <= delta(recs, *seg, float(ex)), (seg, D, ex)
    return D


TRI = [[0.0, 0.0], [4.0, 0.0], [1.0, 3.0]]
HAND = [
    # (records, segment, expected distance or None)
    (_poly(TRI), (-2.0, -1.0, -1.0, -2.0), None),                          # a vertex is closest
    (_poly(TRI), (2.0, -1.0, 3.0, -5.0), 1.0),                              # a path endpoint is closest to an edge
    (_poly(TRI), (-1.0, -0.5, 5.0, -0.5), 0.5),                             # parallel to an edge
    (_poly(TRI, -1), (-1.0, -0.5, 5.0, -0.5), 0.5),
    (_square(0.0, 0.0, 1.0, 2.0), (3.0, -5.0, 3.0, 5.0), 2.0),              # box, parallel to a side
    (_square(0.0, 0.0, 1.0), (2.0, 3.0, 4.0, 1.0), None),                   # box corner
    (_disc(0.0, 0.0, 2.0, 0.5), (-3.0, 1.5, 3.0, 1.5), 1.0),                # ellipse tangent, foot inside [0, 1]
    (_disc(0.0, 0.0, 2.0, 0.5), (1.0, 1.5, 5.0, 1.5), None),                # ... foot outside: an endpoint is nearest
    (_disc(0.0, 0.0, 0.5, 2.0), (3.0, -1.0, 4.0, 1.0), None),               # r2 > r1
    (_disc(1.0, 1.0, 1.0), (-5.0, 4.0, 5.0, 4.0), 2.0),                     # a disc
    (_disc(0.0, 0.0, 2.0, 0.5), (3.0, 0.0, 3.0, 0.0), 1.0),                 # zero-length, on the major axis
    (_poly(TRI), (5.0, 5.0, 5.0, 5.0), None),                               # zero-length segment
    (_square(0.0, 0.0, 1.0), (1.0, -3.0, 1.0, 3.0), 0.0),                   # touching at distance 0: a HIT
    (_disc(0.0, 0.0, 1.0), (-3.0, 1.0, 3.0, 1.0), 0.0),
    (_poly(TRI), (4.0, 0.0, 6.0, 1.0), 0.0),
]


@pytest.mark.parametrize('case', range(len(HAND)))
def test_hand_cases_against_exact_oracle(case):
    recs, seg, expected = HAND[case]
    D = _check_d2(recs, seg)
    if expected is not None:
        assert D == pytest.approx(expected, rel=1e-14, abs=0.0)


SHAPES = {'disc': _disc(3.0, 4.0, 1.5), 'ellipse': _disc(-2.0, 1.0, 2.0, 0.7), 'ellipse_tall': _disc(0.5, -1.0, 0.4, 1.9),
          'box': _square(1.0, -2.0, 1.2, 0.4), 'quad': _poly([[0.0, 0.0], [3.0, -1.0], [4.0, 2.0], [1.0, 3.0]]),
          'tri': _poly([[0.0, 0.0], [3.0, -1.0], [4.0, 2.0]], -1)}


@pytest.mark.parametrize('scale', [1.0, 1e6])
@pytest.mark.parametrize('name', sorted(SHAPES))
def test_random_segments_d2(name, scale):
    rng = np.random.default_rng(hash((name, scale)) % 2 ** 32)
    recs = SHAPES[name].copy()
    off = np.array([scale, -0.5 * scale]) if scale > 1 else np.zeros(2)
    for r in recs:                                              # move the shape to the scale's neighbourhood
        if int(r[0]) == LINE or int(r[0]) == ELLIPSE:
            r[1:3] += off
        elif int(r[1]) == 0:
            r[3] += off[0]
        else:
            r[3] += off[1]
    n_hit = n_far = 0
    for _ in range(60):
        a, b = rng.uniform(-6, 8, 2) + off, rng.uniform(-6, 8, 2) + off
        if rng.random() < 0.3:
            b = a + rng.normal(0, 0.05, 2)
        D = _check_d2(recs, (*a, *b))
        n_hit += D == 0.0
        n_far += D > 0.0
    assert n_hit > 0 and n_far > 0


def test_hit_implies_zero_on_golden_waypoint_collisions(fixture_spec, golden):
    omap = orc.OMap(fixture_spec)
    recs = [_oshape_records(s) for s in omap.obstacles]
    n = 0
    for key in [k for k in golden.files if (k.startswith('arc_N') and k.endswith('_collide')) or k == 'jit_collide']:
        col = golden[key].astype(bool)
        Zf = full_paths(fixture_spec, golden[key.replace('_collide', '_x')])
        f, c, k, o = clearance_reference(Zf, recs, 0.5)
        fs, ks, os_ = sweep_reference(Zf, recs)
        assert np.array_equal(f, fs)
        hit = (f & HIT) != 0
        assert np.all(hit[col.any(axis=1)])
        assert np.all(c[hit] == 0.0) and np.array_equal(k[hit], ks[hit]) and np.array_equal(o[hit], os_[hit])
        assert np.all(c[~hit] > 0.0)
        n += int(col.sum())
    assert n > 0


def test_form_detection():
    import uam_path_planning_b200 as uam
    from uam_path_planning_b200 import mapio
    assert obstacle_form(uam.polygon([0.0, 0.0], [2.0, 0.0], [2.0, 1.0], [0.5, 2.0]).records())[0] == POLYGON_FORM
    assert obstacle_form(uam.polygon([0.0, 0.0], [1.0, 2.0], [2.0, 0.0]).records())[0] == POLYGON_FORM
    assert obstacle_form(uam.square([1.0, 2.0], 0.5, 1.5).records())[0] == BOX_FORM
    assert obstacle_form(uam.ball([1.0, 2.0], 0.5).records())[0] == DISC_FORM
    assert obstacle_form(uam.ball([1.0, 2.0], 0.5, 0.7).records())[0] == ELLIPSE_FORM
    text = ("vertices = [polygon([0, 0], [4, 0], [4, 3]), ball([10, 10], 2), ball([5, -5], 1, 3), square([-4, 4], 1),"
            " polygon([20.5, 1.25], [22.0, 1.0], [23.0, 4.0], [21.0, 5.0])]")
    forms = [obstacle_form(s.records())[0] for s in mapio.parse_shapes(text)]
    assert forms == [POLYGON_FORM, DISC_FORM, ELLIPSE_FORM, BOX_FORM, POLYGON_FORM]
    mixed = np.concatenate([_disc(0.0, 0.0, 2.0), np.array([[LINE, 0.0, -5.0, 0.0, 10.0, 1.0, 0, 0]])])
    bad = {'mixed': mixed, 'two_lines': _poly(TRI)[:2], 'three_boxes': _square(0, 0, 1)[:3],
           'open_polygon': np.array([[LINE, 0, 0, 4, 0, 1, 0, 0], [LINE, 4, 0, -3, 3, 1, 0, 0], [LINE, 1, 3, 0, -2, 1, 0, 0]]),
           'outward_sign': _poly(TRI) * np.array([1, 1, 1, 1, 1, -1, 1, 1]),
           'empty_box': np.array([[2, 0, 1, 0.0, -2.0, 0, 0, 0], [2, 0, -1, 0.0, 1.0, 0, 0, 0],
                                  [2, 1, 1, 0.0, 1.0, 0, 0, 0], [2, 1, -1, 0.0, 1.0, 0, 0, 0]])}
    for name, recs in bad.items():
        with pytest.raises(Unsupported):
            obstacle_form(recs)


def test_reference_outputs_on_small_batch():
    recs = [_square(0.0, 0.0, 1.0), _disc(5.0, 0.0, 1.0)]
    Z = np.array([[-3.0, 0.0, 3.0, 0.0, 6.0, 0.0],             # hits the square on segment 0
                  [-3.0, 3.0, 3.0, 3.0, 5.0, 3.0],             # 2 above the square, then 2 above the disc
                  [-3.0, 5.0, np.nan, 5.0, 5.0, 0.0],
                  [-3.0, 50.0, 3.0, 50.0, 5.0, 50.0]])         # beyond cap
    f, c, k, o = clearance_reference(Z, recs, 10.0)
    assert f.tolist() == [HIT, 0, INVALID, 0]
    assert c[0] == 0.0 and c[1] == 2.0 and math.isnan(c[2]) and c[3] == 10.0
    assert k.tolist() == [0, 0, -1, -1] and o.tolist() == [0, 0, -1, -1]
    f, c, k, o = clearance_reference(Z[1:2], recs[::-1], 10.0)              # tie: smallest k first
    assert (c[0], k[0], o[0]) == (2.0, 0, 1)


# ---- GPU ------------------------------------------------------------------------------------------------------------
def _uam():
    import uam_path_planning_b200 as uam
    return uam


def _assert_same(got, ref):
    for g, r, name in zip(got, ref, ('flags', 'clearance', 'nearest_segment', 'nearest_obstacle')):
        g = np.asarray(g)
        if name == 'clearance':
            assert np.array_equal(g.view(np.int64), np.asarray(r).view(np.int64)), name
        else:
            assert np.array_equal(g, r), name


def _map(which, fixture_spec):
    return {'main': lambda: build_product_map(fixture_spec), 'c2': _c2_like_map, 'c4': _c4_like_map, 'mixed': _mixed_map}[which]()


@pytest.mark.gpu
@pytest.mark.parametrize('which', ['main', 'c2', 'c4', 'mixed'])
def test_device_matches_restatement(which, fixture_spec):
    m = _map(which, fixture_spec)
    lo, hi = {'c2': (0.0, 64.0), 'c4': (0.0, 128.0), 'mixed': (0.0, 32.0)}.get(which, (0.0, 0.0))
    if which == 'main':
        pts = fixture_spec['x_start'] + fixture_spec['x_goal']
        lo, hi = float(np.min(pts)) - 5, float(np.max(pts)) + 5
    recs = _records(m)
    eng = m.engine()
    rng = np.random.default_rng({'main': 201, 'c2': 202, 'c4': 204, 'mixed': 205}[which])
    n_hit = n_near = 0
    for Wp in (2, 3, 33, 64, 132):
        B = 64 if Wp == 132 else 128
        Z = _paths(rng, B, Wp, lo, hi, 0.3 * (hi - lo) / Wp)
        sweep = sweep_reference(Z, recs)
        for cap in (1e-3, 0.5, 1e3):
            ref = clearance_reference(Z, recs, cap)
            assert np.array_equal(ref[0], sweep[0])
            for grid in (1, 0):
                eng.set_option('shape_grid', grid)
                got = m.path_clearance(Z, cap)
                _assert_same(got, ref)
                f, k, o = m.sweep_paths(Z)                      # D1 against the device sweep
                hit = (f & HIT) != 0
                assert np.array_equal(got[0], f)
                assert np.all(got[1][hit] == 0.0) and np.array_equal(got[2][hit], k[hit]) and np.array_equal(got[3][hit], o[hit])
                assert np.all(got[1][~hit] > 0.0)
            eng.set_option('shape_grid', 1)
            n_hit += int((ref[0] == HIT).sum())
            n_near += int(((ref[2] >= 0) & (ref[0] == 0)).sum())
    assert n_hit > 0 and n_near > 0


@pytest.mark.gpu
def test_batch_independence_and_interfaces():
    import torch
    m = _mixed_map()
    recs = _records(m)
    rng = np.random.default_rng(31)
    Z = _paths(rng, 600, 40, 0, 32, 0.5)
    Z[5, 7] = np.nan
    Z[13] = Z[13] + 5e3                        # far outside the grid box: every obstacle is tested
    Z[15, 2] = 2e99
    Z[17, 4] = -1e100
    ref = clearance_reference(Z, recs, 2.0)
    keep = Z.copy()
    got = m.path_clearance(Z, 2.0)
    assert np.array_equal(Z, keep, equal_nan=True)
    _assert_same(got, ref)
    perm = rng.permutation(Z.shape[0])
    _assert_same(m.path_clearance(Z[perm], 2.0), tuple(r[perm] for r in ref))
    _assert_same(m.path_clearance(Z[:1], 2.0), tuple(r[:1] for r in ref))
    T = torch.from_numpy(Z).cuda()
    tg = m.path_clearance(T, 2.0)
    assert all(t.is_cuda for t in tg)
    _assert_same(tuple(t.cpu().numpy() for t in tg), ref)
    f, c, k, o = m.engine().clearance_analytic(Z, 38, 2.0, want_nearest=False)
    assert k is None and o is None and np.array_equal(f, ref[0])
    assert np.array_equal(c.view(np.int64), ref[1].view(np.int64))
    empty = _map_from_records([])
    f, c, k, o = empty.path_clearance(Z, 2.0)
    assert np.all(c[f == 0] == 2.0) and np.all(k == -1) and np.all(o == -1)


@pytest.mark.gpu
def test_lists_rebuilt_when_shapes_or_cap_change():
    uam = _uam()
    m = _c2_like_map(seed=1)
    rng = np.random.default_rng(4)
    Z = _paths(rng, 500, 20, 0, 64, 1.0)
    for cap in (0.05, 3.0, 0.05):
        _assert_same(m.path_clearance(Z, cap), clearance_reference(Z, _records(m), cap))
    for _ in range(8):
        m.add_obstacle(uam.ball(rng.uniform(2, 62, 2).tolist(), 2.0))
    m.obstacles[0] = uam.square([30.0, 30.0], 5.0)
    _assert_same(m.path_clearance(Z, 0.05), clearance_reference(Z, _records(m), 0.05))
    _assert_same(m.path_clearance(Z, 3.0), clearance_reference(Z, _records(m), 3.0))


@pytest.mark.gpu
def test_error_codes_in_order():
    uam = _uam()
    import torch
    eng = uam.Engine()
    lib, h = eng._lib, eng._h
    zt = torch.zeros((4, 6), dtype=torch.float64, device='cuda')
    ft = torch.zeros(4, dtype=torch.uint8, device='cuda')
    ct = torch.zeros(4, dtype=torch.float64, device='cuda')
    zp, fp, cp = C.c_void_p(zt.data_ptr()), C.c_void_p(ft.data_ptr()), C.c_void_p(ct.data_ptr())

    def call(zz, B, N, cap, ff):
        return lib.uam_clearance_paths_analytic(h, zz, B, N, cap, ff, cp, None, None, None)
    assert lib.uam_clearance_paths_analytic(None, zp, 4, 1, 1.0, fp, None, None, None, None) == -1
    for B, N, cap in ((-1, 1, 1.0), (4, -1, 1.0), (4, (1 << 28) + 1, 1.0), (0, 1, 0.0), (0, 1, -1.0), (0, 1, math.nan),
                      (0, 1, 1.1e100), (0, 1, math.inf)):
        assert call(None, B, N, cap, None) == -1, (B, N, cap)
    assert call(None, 0, 1, 1e100, None) == 0                      # B = 0 is a no-op
    assert call(None, 4, 1, 1.0, fp) == -1
    assert call(zp, 4, 1, 1.0, None) == -1
    assert call(zp, 4, 1, 1.0, fp) == -4                           # no shapes
    disc = _map_from_records([_disc(0, 0, 1)]).obstacles[0]
    mk = (lambda recs: uam.QuadraticObstacle(*[uam.shapes.Inequality(r) for r in recs]))
    mixed = np.concatenate([_disc(0.0, 0.0, 2.0), np.array([[LINE, 0.0, -5.0, 0.0, 10.0, 1.0, 0, 0]])])
    for name, recs, sweep_rc in (('nan', [[ELLIPSE, np.nan, 0, 1, 1, 0, 0, 0]], -5), ('mixed', mixed, 0),
                                 ('three_boxes', _square(0, 0, 1)[:3], 0)):
        eng.set_shapes([disc, mk(recs)], [])
        n0 = eng.launch_count()
        assert call(zp, 4, 1, 1.0, fp) == -5, name
        assert eng.launch_count() == n0
        assert 'obstacle 1' in lib.uam_last_error(h).decode(), name
        assert call(zp, 4, -1, 1.0, fp) == -1
        assert lib.uam_sweep_paths_analytic(h, zp, 4, 1, fp, None, None, None) == sweep_rc, name
    eng.set_shapes([], [[mk(mixed)]])                              # region shapes are not measured
    assert call(zp, 4, 1, 1.0, fp) == 0
    torch.cuda.synchronize()
    assert ft.cpu().tolist() == [0] * 4 and ct.cpu().tolist() == [1.0] * 4


@pytest.mark.gpu
def test_raster_clearance_is_an_upper_bound():
    """On C2's map at 4096^2, for paths neither check flags: sqrt(d2min) cell >= analytic clearance - 0.72 cell (a touched
    cell's centre lies within sqrt(2)/2 cell of the segment, an occupied centre inside the obstacle)."""
    uam = _uam()
    import torch
    m = _c2_like_map()
    res, km = 4096, 64.0
    cell = km / res
    rm = uam.RasterMap.from_map(m, res, res, (0.0, cell, 0.0, cell), clearance=True)
    rng = np.random.default_rng(41)
    Z = torch.from_numpy(_paths(rng, 4000, 32, 2, 62, 0.5)).cuda()
    fr, _, d2 = (t.cpu().numpy() for t in rm.sweep_paths(Z))
    fa, ca, _, _ = (t.cpu().numpy() for t in m.path_clearance(Z, 1e3))
    ok = (fr == 0) & (fa == 0) & (d2 >= 0) & (d2 < 65535)
    assert ok.sum() > 100
    assert np.all(np.sqrt(d2[ok].astype(np.float64)) * cell >= ca[ok] - 0.72 * cell)
