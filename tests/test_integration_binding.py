"""INTEGRATION.md section 2 executed: integration/gpu_backend.py (the file a maintainer adds to the reference) binds
libuam_b200.so with plain ctypes from the reference's own classes.

CPU part: the tables gpu_backend.extract_tables reads out of closures laid out like the reference's equal the frozen
tests/golden/reference_tables.npz (what it read from the reference's own objects, tests/golden/make_reference_tables.py)
and, bit for bit, the tables the product's own constructors build.
GPU part: the raw binding, fed with the frozen tables, reproduces the reference's golden costs / constraint vectors.
"""
import os
import sys
from types import SimpleNamespace

import numpy as np
import pytest

from conftest import build_product_map, full_paths

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, 'integration'))
GOLD = os.path.join(ROOT, 'tests', 'golden')


def _tables():
    t = np.load(os.path.join(GOLD, 'reference_tables.npz'))
    return {k: t[k] for k in t.files}


# The reference's objects as gpu_backend sees them: a shape has `.inequalities` (`Function`s whose `.f` is a closure over
# the shape's numbers, with the reference's variable names) and `.center`; a map has `.obstacles`, `.regions[name]['shapes']`
# and `.region_names()`; a problem has `.map`, `.params`, `.weights`, `.options`.
def _function(f):
    return SimpleNamespace(f=f)


def _polygon_edge(Pa_F, Pb_F, sgn_F):                          # polygon.py:66-98
    def line_F(x):
        return (Pb_F[1, 0] - Pa_F[1, 0]) * (x[0] - Pa_F[0, 0]) - (Pb_F[0, 0] - Pa_F[0, 0]) * (x[1] - Pa_F[1, 0])
    return _function(lambda x: -sgn_F * line_F(x))


def _ellipse(center, r1, r2):                                  # ball.py:33-37
    def func(x):
        return ((x[0] - center[0]) / r1) ** 2 + ((x[1] - center[1]) / r2) ** 2 - 1
    return _function(func)


def _square_sides(center, r1, r2):                             # square.py:29-51: right, left, top, bottom
    return [_function(lambda x: x[0] - center[0] - r1), _function(lambda x: -x[0] + center[0] - r1),
            _function(lambda x: x[1] - center[1] - r2), _function(lambda x: -x[1] + center[1] - r2)]


def _reference_layout_shape(s):
    """a product shape (vertex order and edge signs of its constructor) -> the same numbers in the reference's closures"""
    R = s.records()
    if s.kind == 'polygon':
        P = [r[1:3].reshape(2, 1) for r in R]                  # hull vertices in edge order: edge k runs P[k] -> P[k + 1]
        ineq = [_polygon_edge(P[k], P[(k + 1) % len(P)], r[5]) for k, r in enumerate(R)]
    else:
        assert s.kind == 'ball'
        ineq = [_ellipse(R[0, 1:3].copy(), R[0, 3], R[0, 4])]
    return SimpleNamespace(inequalities=ineq, center=s.center)


def _reference_layout_problem(spec, N=80):
    m = build_product_map(spec)
    names = [name for name, _ in spec['regions']]
    regions = {n: {'shapes': [_reference_layout_shape(s) for s in shapes]} for n, shapes in zip(names, m._region_lists())}
    rm = SimpleNamespace(obstacles=[_reference_layout_shape(s) for s in m.obstacles], regions=regions,
                         region_names=lambda: list(regions), x_start=spec['x_start'], x_goal=spec['x_goal'])
    return SimpleNamespace(map=rm, N=N, options=dict(spec['options']), weights=dict(zip(names, spec['weights'])),
                           params={'maxratio': spec['maxratio'], 'maxalpha': spec['maxalpha'], 'enlargement': spec['enlargement']})


def test_tables_from_reference_closures(fixture_spec):
    import gpu_backend as gb
    pr = _reference_layout_problem(fixture_spec)
    g = gb.GpuProblem.__new__(gb.GpuProblem)                    # no device context: only the host-side packing
    g.p = pr
    got, frozen = gb.extract_tables(pr.map), _tables()
    for k in ('edges', 'off', 'region', 'center'):
        assert np.array_equal(got[k], frozen[k]), k
    assert int(got['n_regions']) == int(frozen['n_regions']) == 3
    sq = np.array([gb.inequality_record(f) for f in _square_sides(np.array([1.0, 1.0]), 0.5, 0.25)])
    assert np.array_equal(sq, frozen['square_records'])          # the box sides are told apart by probing f
    got = dict(got, p=g.parameter_vector(), flags=g.flags())
    # ... and they are the tables the product's constructors build from the same numbers
    from uam_path_planning_b200.shapes import flatten_shapes
    m = build_product_map(fixture_spec)
    edges, off, reg, cen = flatten_shapes(m.obstacles, m._region_lists())
    assert np.array_equal(edges, frozen['edges']) and np.array_equal(off, frozen['off'])
    assert np.array_equal(reg, frozen['region']) and np.array_equal(cen, frozen['center'])
    # parameter vector / flags in the reference's order (solver.py:60-68, problem.py:12-17)
    f = fixture_spec
    assert np.array_equal(got['p'], np.array([*f['x_start'], *f['x_goal'], f['maxratio'], f['maxalpha'], f['enlargement'], *f['weights']]))
    assert int(got['flags']) == 0b0111


def test_frozen_tables_match_product_tables(fixture_spec):
    """runs everywhere: the frozen reference tables == the product's tables (incl. the box-side records of square())"""
    import uam_path_planning_b200 as uam
    from uam_path_planning_b200.shapes import flatten_shapes
    t = _tables()
    m = build_product_map(fixture_spec)
    edges, off, reg, cen = flatten_shapes(m.obstacles, m._region_lists())
    assert np.array_equal(edges, t['edges']) and np.array_equal(off, t['off'])
    assert np.array_equal(reg, t['region']) and np.array_equal(cen, t['center'])
    assert np.array_equal(uam.square([1.0, 1.0], 0.5, 0.25).records(), t['square_records'])


@pytest.mark.gpu
@pytest.mark.parametrize('N', [80, 62, 5])
def test_raw_ctypes_binding_matches_reference_goldens(fixture_spec, golden, N):
    import gpu_backend as gb
    from uam_path_planning_b200 import build
    f = fixture_spec
    sc = gb.GpuScorer(_tables(), lib=gb.load_library(build.OUT))
    p = np.array([*f['x_start'], *f['x_goal'], f['maxratio'], f['maxalpha'], f['enlargement'], *f['weights']])
    Z = full_paths(f, golden[f'arc_N{N}_x'])
    cost, col, g = sc.score(Z, N, p, 0b0111, want_g=True)
    np.testing.assert_allclose(cost, golden[f'arc_N{N}_cost'], rtol=1e-12)
    assert np.array_equal(col, golden[f'arc_N{N}_collide'].any(axis=1))
    np.testing.assert_allclose(g, golden[f'arc_N{N}_g'], rtol=1e-9, atol=1e-300)
    assert np.array_equal(g == 0, golden[f'arc_N{N}_g'] == 0)
    sc.close()
