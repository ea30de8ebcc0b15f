"""Swept check of whole path segments against the analytic obstacles (uam_sweep_paths_analytic / Map.sweep_paths).

CPU: the numpy restatement (analytic_sweep_reference) against the exact rational oracle on hand-made cases and random
segments (G1: no missed hit; G3: no hit beyond eta), and G2 on the reference's own golden waypoint collisions.
GPU: the kernel against the restatement bit for bit over maps, path lengths and the shape_grid option (G4); G2 against
Problem.score at scale; batch independence; the cell lists' invalidation; the error codes.
"""
import ctypes as C
import math

import numpy as np
import pytest

from analytic_sweep_reference import HIT, INVALID, exact_meets, segment_hits, sweep_reference
from conftest import build_product_map, full_paths
from oracle import uam_oracle as orc

LINE, ELLIPSE, BOX = 0, 1, 2


def _disc(cx, cy, r1, r2=None):
    return np.array([[ELLIPSE, cx, cy, r1, r1 if r2 is None else r2, 0, 0, 0]], dtype=np.float64)


def _square(cx, cy, r1, r2=None):
    r2 = r1 if r2 is None else r2
    return np.array([[BOX, 0, +1, cx, r1, 0, 0, 0], [BOX, 0, -1, cx, r1, 0, 0, 0],
                     [BOX, 1, +1, cy, r2, 0, 0, 0], [BOX, 1, -1, cy, r2, 0, 0, 0]], dtype=np.float64)


def _poly(verts, orientation=1):
    """Convex polygon records from vertices in order; orientation -1 lists them the other way round (sgn flips)."""
    V = np.asarray(verts, dtype=np.float64)
    if orientation < 0:
        V = V[::-1]
    n = len(V)
    out = []
    for a in range(n):
        A, Bv = V[a], V[(a + 1) % n]
        P = V[(a + 2) % n]
        side = (Bv[1] - A[1]) * (P[0] - A[0]) - (Bv[0] - A[0]) * (P[1] - A[1])
        out.append([LINE, A[0], A[1], Bv[0] - A[0], Bv[1] - A[1], float(np.sign(side)), 0, 0])
    return np.array(out, dtype=np.float64)


def _oshape_records(s):
    rows = []
    for e in s.edges:
        if e[0] == 'line':
            _, Ax, Ay, Bx, By, sgn = e
            rows.append([LINE, Ax, Ay, Bx - Ax, By - Ay, sgn, 0, 0])
        elif e[0] == 'ellipse':
            rows.append([ELLIPSE, e[1], e[2], e[3], e[4], 0, 0, 0])
        else:
            rows.append([BOX, e[1], e[2], e[3], e[4], 0, 0, 0])
    return np.array(rows, dtype=np.float64).reshape(-1, 8)


def _check_g1_g3(recs, seg):
    ax, ay, bx, by = seg
    got = bool(segment_hits(recs, np.array([ax]), np.array([ay]), np.array([bx]), np.array([by]))[0])
    if exact_meets(recs, ax, ay, bx, by):
        assert got, f'G1: missed hit {seg}'
    if got:
        assert exact_meets(recs, ax, ay, bx, by, relax=True), f'G3: hit beyond eta {seg}'
    return got


# ---- hand cases -----------------------------------------------------------------------------------------------------
SQ = _square(0.0, 0.0, 1.0)
TRI = np.array([[0.0, 0.0], [4.0, 0.0], [1.0, 3.0]])
HAND = [
    # (records, segment, expected HIT or None = only G1 / G3)
    (_disc(0.0, 0.0, 1.0), (-3.0, 1.0, 3.0, 1.0), True),                    # tangent to a disc
    (_disc(0.0, 0.0, 2.0, 0.5), (-3.0, 0.5, 3.0, 0.5), True),               # tangent to an ellipse, r1 != r2
    (_disc(0.0, 0.0, 2.0, 0.5), (2.0, -3.0, 2.0, 3.0), True),               # ... on its other axis
    (_disc(0.0, 0.0, 1.0), (-3.0, 1.0 + 1e-12, 3.0, 1.0 + 1e-12), False),    # missing by 1e-12 km
    (_poly(TRI), (-1.0, -1.0, 1.0, 1.0), True),                              # through a vertex
    (_poly(TRI), (-1.0, 1.0, 1.0, -1.0), True),                              # grazing a vertex
    (_poly(TRI, -1), (-1.0, 1.0, 1.0, -1.0), True),                          # ... other orientation
    (_poly(TRI), (-1.0, 0.0, 5.0, 0.0), True),                               # along an edge
    (_poly(TRI, -1), (-1.0, 0.0, 5.0, 0.0), True),
    (_poly(TRI), (-1.0, -1e-12, 5.0, -1e-12), False),                        # parallel, 1e-12 km off the edge
    (SQ, (0.0, 2.0, 2.0, 0.0), True),                                        # through a square's corner
    (SQ, (0.0, 2.0 + 1e-12, 2.0 + 1e-12, 0.0), False),
    (SQ, (-3.0, 1.0 + 1e-13, 3.0, 1.0 + 1e-13), False),                      # just more than eta above the top side
    (SQ, (-3.0, 1.0 + 1e-14, 3.0, 1.0 + 1e-14), True),                       # on K_o's own tolerance
    (SQ, (1.0, 1.0, 5.0, 5.0), True),                                        # endpoint with h exactly 0
    (_disc(0.0, 0.0, 1.0), (0.6, 0.8, 3.0, 3.0), None),                      # endpoint on the circle (h ~ 0)
    (SQ, (0.5, 0.5, 0.5, 0.5), True),                                        # zero-length inside
    (SQ, (1.5, 0.5, 1.5, 0.5), False),                                       # zero-length outside
    (_disc(0.0, 0.0, 1.0), (1.0, 0.0, 1.0, 0.0), True),                      # zero-length on the boundary
    (_disc(5.0, 7.0, 0.3), (-50.0, -50.0, 60.0, 70.0), None),                # across the whole map
    (_disc(5.0, 10.0, 0.3), (-50.0, -50.0, 60.0, 70.0), True),
    (_poly([[0.0, 0.0], [10.0, 0.0], [10.0, 1e-9]]), (5.0, -1.0, 5.0, 1.0), True),          # thin sliver
    (_poly([[0.0, 0.0], [10.0, 0.0], [10.0, 1e-9]]), (11.0, -1.0, 11.0, 1.0), False),
    (_disc(0.0, 0.0, 1e-6, 5.0), (-1.0, 0.0, 1.0, 0.0), True),               # thin ellipse
    (_disc(0.0, 0.0, 1e-6, 5.0), (-1.0, 5.0 + 1e-9, 1.0, 5.0 + 1e-9), None),   # S = 3e6: within eta
    (_square(0.0, 0.0, 1e-9, 3.0), (-2.0, 2.9, 2.0, -2.9), True),            # thin box
]


@pytest.mark.parametrize('case', range(len(HAND)))
def test_hand_cases_against_exact_oracle(case):
    recs, seg, expected = HAND[case]
    got = _check_g1_g3(recs, seg)
    if expected is not None:
        assert got == expected


def test_random_segments_g1_g3():
    rng = np.random.default_rng(9)
    shapes = [_disc(3.0, 4.0, 1.5), _disc(-2.0, 1.0, 2.0, 0.7), _square(1.0, -2.0, 1.2, 0.4),
              _poly([[0.0, 0.0], [3.0, -1.0], [4.0, 2.0], [1.0, 3.0]]), _poly([[0.0, 0.0], [3.0, -1.0], [4.0, 2.0]], -1)]
    for recs in shapes:
        n_hit = 0
        for _ in range(120):
            a, b = rng.uniform(-6, 8, 2), rng.uniform(-6, 8, 2)
            if rng.random() < 0.3:                 # short segments near the boundary
                b = a + rng.normal(0, 0.05, 2)
            n_hit += _check_g1_g3(recs, (*a, *b))
        assert 0 < n_hit < 120


def test_mixed_records_in_one_obstacle():
    # a disc cut by a half-plane: one ellipse record and one line record in the same obstacle
    recs = np.concatenate([_disc(0.0, 0.0, 2.0), np.array([[LINE, 0.0, -5.0, 0.0, 10.0, 1.0, 0, 0]])])
    rng = np.random.default_rng(3)
    for _ in range(200):
        a, b = rng.uniform(-4, 4, 2), rng.uniform(-4, 4, 2)
        _check_g1_g3(recs, (*a, *b))


def test_invalid_rows_and_short_paths():
    recs = [SQ, _disc(5.0, 0.0, 1.0)]
    Z = np.array([[-3.0, 0.0, 3.0, 0.0, 6.0, 0.0],           # hits the square on segment 0
                  [-3.0, 5.0, 3.0, 5.0, 5.0, 3.0],           # clean
                  [-3.0, 5.0, np.nan, 5.0, 5.0, 0.0],
                  [-3.0, 5.0, np.inf, 5.0, 5.0, 0.0],
                  [-3.0, 5.0, 1e100, 5.0, 5.0, 0.0],
                  [4.0, 0.0, 4.0, 0.0, 4.0, 0.0]])           # repeated waypoints inside the disc
    f, k, o = sweep_reference(Z, recs)
    assert f.tolist() == [HIT, 0, INVALID, INVALID, INVALID, HIT]
    assert k.tolist() == [0, -1, -1, -1, -1, 0]
    assert o.tolist() == [0, -1, -1, -1, -1, 1]
    f, k, o = sweep_reference(np.array([[0.0, 0.0, 5.0, 0.0]]), recs)      # N = 0: one segment, both shapes
    assert (f[0], k[0], o[0]) == (HIT, 0, 0)


# ---- G2 on the reference's own data ----------------------------------------------------------------------------------
def _segment_any_hit(Zfull, recs_list):
    P = Zfull.reshape(Zfull.shape[0], -1, 2)
    A, Bp = P[:, :-1], P[:, 1:]
    out = np.zeros(A.shape[:2], dtype=bool)
    for recs in recs_list:
        out |= segment_hits(recs, A[..., 0], A[..., 1], Bp[..., 0], Bp[..., 1])
    return out


def test_g2_on_golden_waypoint_collisions(fixture_spec, golden):
    omap = orc.OMap(fixture_spec)
    recs = [_oshape_records(s) for s in omap.obstacles]
    n_col = 0
    for key in [k for k in golden.files if (k.startswith('arc_N') and k.endswith('_collide')) or k == 'jit_collide']:
        X = golden[key.replace('_collide', '_x')]
        col = golden[key].astype(bool)                         # (B, N + 2) per waypoint
        Zf = full_paths(fixture_spec, X)
        assert np.array_equal(col, omap.collides(Zf.reshape(-1, 2)).reshape(col.shape))
        seg = _segment_any_hit(Zf, recs)
        for j in range(col.shape[1]):
            if j > 0:
                assert np.all(seg[col[:, j], j - 1])
            if j < col.shape[1] - 1:
                assert np.all(seg[col[:, j], j])
        f, _, _ = sweep_reference(Zf, recs)
        assert np.all(f[col.any(axis=1)] & HIT)
        n_col += int(col.sum())
    assert n_col > 0


def _c2_like_spec(rng, n_obs=32, km=64.0):
    return {'obstacles': [{'kind': 'ball', 'center': rng.uniform(2, km - 2, 2).tolist(), 'r1': float(rng.uniform(0.3, 1.5))}
                          for _ in range(n_obs)], 'regions': []}


def test_g2_random_paths_on_c2_like_map():
    rng = np.random.default_rng(11)
    spec = _c2_like_spec(rng)
    omap = orc.OMap(spec)
    recs = [_oshape_records(s) for s in omap.obstacles]
    B, Wp = 400, 64
    s, e = rng.uniform(0, 64, (B, 1, 2)), rng.uniform(0, 64, (B, 1, 2))
    Z = (s + np.linspace(0, 1, Wp).reshape(1, Wp, 1) * (e - s) + rng.normal(0, 0.5, (B, Wp, 2))).reshape(B, 2 * Wp)
    col = omap.collides(Z.reshape(-1, 2)).reshape(B, Wp)
    f, _, _ = sweep_reference(Z, recs)
    assert col.any(axis=1).sum() > 10
    assert np.all(f[col.any(axis=1)] == HIT)
    assert (f == HIT).sum() > col.any(axis=1).sum()            # the sweep sees hits between waypoints
    # G1 / G3 on segments that pass near an obstacle
    P = Z.reshape(B, Wp, 2)
    checked = 0
    for b in range(0, B, 7):
        for k in range(0, Wp - 1, 5):
            for o, sh in enumerate(omap.obstacles):
                c = np.array([sh.edges[0][1], sh.edges[0][2]])
                if np.linalg.norm(P[b, k] - c) < 3.0:
                    _check_g1_g3(recs[o], (*P[b, k], *P[b, k + 1]))
                    checked += 1
    assert checked > 20


# ---- GPU ------------------------------------------------------------------------------------------------------------
def _uam():
    import uam_path_planning_b200 as uam
    return uam


def _records(m):
    return [o.records() for o in m.obstacles]


def _map_from_records(recs_list, regions=()):
    uam = _uam()
    m = uam.RegionMap()
    for recs in recs_list:
        m.add_obstacle(uam.QuadraticObstacle(*[uam.shapes.Inequality(r) for r in recs]))
    for name, shapes in regions:
        m.new_region(name, 'red')
        m.add_shapes_to_region(name, *shapes)
    return m


def _c2_like_map(seed=20260101):
    uam = _uam()
    rng = np.random.default_rng(seed)
    m = uam.RegionMap()
    m.new_region('Risk', 'r')
    for _ in range(64):
        m.add_shape_to_region('Risk', uam.ball(rng.uniform(2, 62, 2).tolist(), float(rng.uniform(0.5, 3))))
    for _ in range(32):
        m.add_obstacle(uam.ball(rng.uniform(2, 62, 2).tolist(), float(rng.uniform(0.3, 1.5))))
    m.x_start, m.x_goal = [6.0, 7.0], [57.0, 55.0]
    return m


def _c4_like_map(n=512, km=128.0, seed=20260104):
    uam = _uam()
    rng = np.random.default_rng(seed)
    m = uam.RegionMap()
    for _ in range(n):
        c, a = rng.uniform(1, km - 1, 2), rng.uniform(0, np.pi)
        hw, hh = rng.uniform(0.05, 0.6, 2)
        R = np.array([[np.cos(a), -np.sin(a)], [np.sin(a), np.cos(a)]])
        m.add_obstacle(uam.polygon(*(c + np.array([[-hw, -hh], [hw, -hh], [hw, hh], [-hw, hh]]) @ R.T).tolist()))
    return m


def _mixed_map(seed=5):
    uam = _uam()
    rng = np.random.default_rng(seed)
    m = uam.RegionMap()
    for i in range(24):
        c = rng.uniform(2, 30, 2)
        if i % 3 == 0:
            m.add_obstacle(uam.ball(c.tolist(), float(rng.uniform(0.3, 2)), float(rng.uniform(0.3, 2))))
        elif i % 3 == 1:
            m.add_obstacle(uam.square(c.tolist(), float(rng.uniform(0.2, 1.5)), float(rng.uniform(0.2, 1.5))))
        else:
            ang = np.sort(rng.uniform(0, 2 * np.pi, 5))
            r = rng.uniform(0.5, 2)
            m.add_obstacle(uam.polygon(*(c + r * np.stack([np.cos(ang), np.sin(ang)], 1)).tolist()))
    return m


def _paths(rng, B, Wp, lo, hi, jitter):
    s, e = rng.uniform(lo, hi, (B, 1, 2)), rng.uniform(lo, hi, (B, 1, 2))
    Z = s + np.linspace(0, 1, Wp).reshape(1, Wp, 1) * (e - s) + rng.normal(0, jitter, (B, Wp, 2))
    return np.ascontiguousarray(Z.reshape(B, 2 * Wp))


def _assert_same(got, ref):
    for g, r, name in zip(got, ref, ('flags', 'first_hit', 'first_obstacle')):
        assert np.array_equal(np.asarray(g), r), name


@pytest.mark.gpu
@pytest.mark.parametrize('which', ['main', 'c2', 'c4', 'mixed'])
def test_device_matches_restatement(which, fixture_spec):
    m = {'main': lambda: build_product_map(fixture_spec), 'c2': _c2_like_map, 'c4': _c4_like_map, 'mixed': _mixed_map}[which]()
    lo, hi = {'main': (-5.0, 30.0), 'c2': (0.0, 64.0), 'c4': (0.0, 128.0), 'mixed': (0.0, 32.0)}[which]
    if which == 'main':
        lo, hi = float(np.min(fixture_spec['x_start'] + fixture_spec['x_goal'])) - 5, float(np.max(fixture_spec['x_start'] + fixture_spec['x_goal'])) + 5
    recs = _records(m)
    eng = m.engine()
    rng = np.random.default_rng({'main': 101, 'c2': 102, 'c4': 104, 'mixed': 105}[which])
    n_hit = 0
    for Wp in (2, 3, 33, 64, 130):
        B = 96 if Wp == 130 else 160
        Z = _paths(rng, B, Wp, lo, hi, 0.3 * (hi - lo) / Wp)
        ref = sweep_reference(Z, recs)
        for grid in (1, 0):
            eng.set_option('shape_grid', grid)
            _assert_same(m.sweep_paths(Z), ref)
        eng.set_option('shape_grid', 1)
        n_hit += int((ref[0] == HIT).sum())
    assert n_hit > 0


@pytest.mark.gpu
def test_device_few_obstacles_and_no_obstacles():
    uam = _uam()
    rng = np.random.default_rng(2)
    recs = [_disc(1.0, 1.0, 0.5), _square(3.0, 0.0, 0.4)]
    m = _map_from_records(recs, regions=[('R', [uam.ball([2.0, 2.0], 1.0)])])
    Z = _paths(rng, 200, 9, -1, 5, 0.3)
    _assert_same(m.sweep_paths(Z), sweep_reference(Z, recs))
    empty = _map_from_records([], regions=[('R', [uam.ball([2.0, 2.0], 1.0)])])
    Z[3, 4] = np.nan
    f, k, o = empty.sweep_paths(Z)
    assert f.tolist() == [0, 0, 0, INVALID] + [0] * 196
    assert np.all(k == -1) and np.all(o == -1)


@pytest.mark.gpu
def test_g2_problem_score_collide_implies_hit():
    uam = _uam()
    import torch
    m = _c2_like_map()
    rng = np.random.default_rng(17)
    B, Wp = 8192, 64
    Z = torch.from_numpy(_paths(rng, B, Wp, 0, 64, 2 * 64 / 4096)).cuda()
    prob = uam.Problem(m, Wp - 2, {'length_smooth': True, 'obstacle_smooth': True})
    prob.params.update(maxratio=1.04, maxalpha=np.pi / 80, enlargement=0)
    prob.set_weight('Risk', 5000.0)
    _, col, _ = prob.score(Z)
    f, k, o = m.sweep_paths(Z)
    col, f = col.cpu().numpy().astype(bool), f.cpu().numpy()
    assert col.sum() > 100
    assert np.all(f[col] == HIT)
    assert (f == HIT).sum() > col.sum()


@pytest.mark.gpu
def test_batch_independence_and_interfaces():
    import torch
    m = _mixed_map()
    recs = _records(m)
    rng = np.random.default_rng(23)
    Z = _paths(rng, 600, 40, 0, 32, 0.5)
    Z[5, 7] = np.nan
    Z[9, 0] = np.inf
    Z[11, 3] = -np.inf
    Z[13] = Z[13] + 5e3                        # far outside the grid box: every obstacle is tested
    Z[15, 2] = 2e99                            # valid, and beyond the lists' magnitude bound
    Z[17, 4] = -1e100                          # the first magnitude that is INVALID
    ref = sweep_reference(Z, recs)
    assert (ref[0] == INVALID).sum() == 4 and ref[0][13] != INVALID and ref[0][15] != INVALID
    keep = Z.copy()
    got = m.sweep_paths(Z)
    assert np.array_equal(Z, keep, equal_nan=True)
    _assert_same(got, ref)
    perm = rng.permutation(Z.shape[0])
    _assert_same(m.sweep_paths(Z[perm]), tuple(r[perm] for r in ref))
    _assert_same(m.sweep_paths(Z[:1]), tuple(r[:1] for r in ref))
    T = torch.from_numpy(Z).cuda()
    Tk = T.clone()
    tg = m.sweep_paths(T)
    assert all(t.is_cuda for t in tg)
    assert torch.equal(torch.nan_to_num(T, 7.0), torch.nan_to_num(Tk, 7.0))
    _assert_same(tuple(t.cpu().numpy() for t in tg), ref)
    eng = m.engine()
    f, k, o = eng.sweep_analytic(Z, 38, want_first_hit=False, want_first_obstacle=False)
    assert k is None and o is None and np.array_equal(f, ref[0])


@pytest.mark.gpu
def test_lists_rebuilt_when_shapes_change():
    uam = _uam()
    m = _c2_like_map(seed=1)
    rng = np.random.default_rng(4)
    Z = _paths(rng, 500, 20, 0, 64, 1.0)
    _assert_same(m.sweep_paths(Z), sweep_reference(Z, _records(m)))
    for _ in range(8):
        m.add_obstacle(uam.ball(rng.uniform(2, 62, 2).tolist(), 2.0))
    m.obstacles[0] = uam.square([30.0, 30.0], 5.0)
    _assert_same(m.sweep_paths(Z), sweep_reference(Z, _records(m)))


@pytest.mark.gpu
def test_error_codes_in_order():
    uam = _uam()
    from uam_path_planning_b200 import _lib
    eng = uam.Engine()
    lib, h = eng._lib, eng._h
    z = np.zeros((4, 6))
    fl = np.zeros(4, dtype=np.uint8)
    import torch
    zt = torch.zeros((4, 6), dtype=torch.float64, device='cuda')
    ft = torch.zeros(4, dtype=torch.uint8, device='cuda')
    zp, fp = C.c_void_p(zt.data_ptr()), C.c_void_p(ft.data_ptr())
    call = lambda zz, B, N, ff: lib.uam_sweep_paths_analytic(h, zz, B, N, ff, None, None, None)   # noqa: E731
    assert lib.uam_sweep_paths_analytic(None, zp, 4, 1, fp, None, None, None) == -1
    assert call(zp, 4, -1, fp) == -1
    assert call(zp, -1, 1, fp) == -1
    assert call(None, 0, 1, None) == 0                              # B = 0 is a no-op
    assert call(None, 4, 1, fp) == -1
    assert call(zp, 4, 1, None) == -1
    assert call(zp, 4, 1, fp) == -4                                 # no shapes
    assert call(zp, 4, (1 << 28) + 1, fp) == -1                     # N too large: an argument error, before the state
    bad = {'nan': [[ELLIPSE, np.nan, 0, 1, 1, 0, 0, 0]], 'huge': [[BOX, 0, 1, 2e100, 1, 0, 0, 0]],
           'radius0': [[ELLIPSE, 0, 0, 0.0, 1, 0, 0, 0]], 'two_ellipses': [[ELLIPSE, 0, 0, 1, 1, 0, 0, 0], [ELLIPSE, 1, 0, 1, 1, 0, 0, 0]]}
    for name, recs in bad.items():
        eng.set_shapes([_map_from_records([_disc(0, 0, 1)]).obstacles[0],
                        uam.QuadraticObstacle(*[uam.shapes.Inequality(r) for r in recs])], [])
        n0 = eng.launch_count()
        assert call(zp, 4, 1, fp) == -5, name
        assert eng.launch_count() == n0
        assert call(zp, 4, -1, fp) == -1                             # argument errors come first
    # the same records in a region shape are not tested
    eng.set_shapes([], [[uam.QuadraticObstacle(*[uam.shapes.Inequality(r) for r in bad['nan']])]])
    assert call(zp, 4, 1, fp) == 0
    torch.cuda.synchronize()
    assert ft.cpu().tolist() == [0, 0, 0, 0]
    del z, fl, _lib
