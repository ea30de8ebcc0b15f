"""Swept check of whole path segments against the raster (uam_sweep_paths_raster / RasterMap.sweep_paths).

CPU: the numpy restatement (raster_sweep_reference) on hand-made cases, and the property that ties the sweep to the
scorer: for a path inside the raster rectangle, the sampled collide flag of oracle.score_paths_raster implies HIT.
GPU: the kernel against the restatement bit for bit over texel forms, layouts, path lengths and row kinds; the d^2 field
against oracle.edt_sq; batch independence; the caches; errors; the property on the device scorer at scale.
"""
import ctypes as C

import numpy as np
import pytest

from oracle import uam_oracle as orc
from raster_sweep_reference import HIT, INVALID, OUTSIDE, sweep_reference, touched_cells
from test_raster_gradient import _random_paths, _random_raster

Q = 1 << 16
GEO_PIX = (-0.5, 1.0, -0.5, 1.0)            # world = pixel coordinates, exactly
GEO = (3.0, 0.25, 40.0, -0.25)              # cell edges and vertices are exact in world coordinates too


def _world(UV, geo):
    """pixel coordinates (..., 2) -> world coordinates"""
    x0, dx, y0, dy = geo
    UV = np.asarray(UV, dtype=np.float64)
    return np.stack([x0 + (UV[..., 0] + 0.5) * dx, y0 + (UV[..., 1] + 0.5) * dy], axis=-1)


def _cells(u0, v0, u1, v1, H=6, W=8):
    q = lambda x: int(np.rint(x * Q))          # noqa: E731
    ii, jj = touched_cells(q(u0), q(v0), q(u1), q(v1), H, W)
    return set(zip(ii.tolist(), jj.tolist()))


def _paths_from_pixels(rows, geo):
    return np.ascontiguousarray(np.stack([_world(r, geo).reshape(-1) for r in rows]))


def _mixed_rows(rng, Wp, H, W, geo, n_random=24):
    """Polylines of Wp waypoints in pixel coordinates of every kind the definition singles out, as world paths."""
    def line(p, q):
        t = np.linspace(0.0, 1.0, Wp)[:, None]
        return np.asarray(p, dtype=np.float64) + t * (np.asarray(q, dtype=np.float64) - np.asarray(p, dtype=np.float64))

    rows = []
    for _ in range(6):                     # along a cell edge, both axes
        i, j = int(rng.integers(0, H)), int(rng.integers(0, W))
        a, b = sorted(rng.uniform(-0.5, W - 0.5, 2))
        rows.append(line((a, i + 0.5), (b, i + 0.5)))
        a, b = sorted(rng.uniform(-0.5, H - 0.5, 2))
        rows.append(line((j - 0.5, a), (j - 0.5, b)))
    for _ in range(4):                     # diagonals through grid vertices
        i, j = int(rng.integers(1, H - 1)), int(rng.integers(1, W - 1))
        t = rng.uniform(0.3, 4.0)
        rows.append(line((j + 0.5 - t, i + 0.5 - t), (j + 0.5 + t, i + 0.5 + t)))
        rows.append(line((j + 0.5 + t, i + 0.5 - 2 * t), (j + 0.5 - t, i + 0.5 + 2 * t)))
    for p in [(2.0, 3.0), (2.5, 3.0), (2.5, 2.5), (-0.5, -0.5), (W - 0.5, H - 0.5)]:    # zero-length segments only
        rows.append(np.tile(np.asarray(p, dtype=np.float64), (Wp, 1)))
    r = line((1.0, 1.0), (W - 2.0, H - 2.0))      # repeated waypoints inside a path
    r[1::3] = r[0::3][:len(r[1::3])]
    rows.append(r)
    rows.append(line((-1.0e7, 0.3 * H), (1.0e7, 0.6 * H)))           # from far outside, across the raster
    rows.append(line((0.4 * W, 2.0e9), (0.5 * W, -2.0e9)))
    rows.append(line((-3.0 * W, -2.0 * H), (-W, 3.0 * H)))            # outside all the way
    rows.append(line((0.5 * W, -1.7), (0.5 * W, H + 0.7)))
    for bad in [np.nan, np.inf, -np.inf, 2.0 ** 31, -2.0 ** 31 - 1.0]:  # INVALID rows
        r = line((1.0, 1.0), (W - 2.0, H - 2.0))
        r[min(1, Wp - 1), int(rng.integers(0, 2))] = bad
        rows.append(r)
    Zs = _paths_from_pixels(rows, geo)
    Zr = _random_paths(rng, n_random, Wp, geo, H, W, spill=0.1)
    return np.ascontiguousarray(np.concatenate([Zs, Zr]))


# ------------------------------------------------------------------------------------------------------------------
# CPU: the restatement
# ------------------------------------------------------------------------------------------------------------------
def test_segment_on_a_cell_edge_touches_both_sides():
    assert _cells(0.5, 2.5, 4.5, 2.5) == {(i, j) for i in (2, 3) for j in range(0, 6)}
    assert _cells(3.5, 0.0, 3.5, 2.0) == {(i, j) for i in range(0, 3) for j in (3, 4)}
    # a quantum off the edge: one side only (the dilation is one quantum, the segment two away)
    assert _cells(1.0, 2.5 + 2.0 / Q, 3.0, 2.5 + 2.0 / Q) == {(3, j) for j in range(1, 4)}


def test_diagonal_through_a_vertex_touches_four_cells():
    assert _cells(2.0, 2.0, 3.0, 3.0) == {(2, 2), (2, 3), (3, 2), (3, 3)}
    assert _cells(3.0, 2.0, 2.0, 3.0) == {(2, 2), (2, 3), (3, 2), (3, 3)}
    # the anti-diagonal through the same vertex touches the two others only at the vertex
    assert _cells(2.0, 3.0, 3.0, 2.0) == {(2, 2), (2, 3), (3, 2), (3, 3)}


def test_zero_length_segment_touches_the_cells_around_its_point():
    assert _cells(2.0, 3.0, 2.0, 3.0) == {(3, 2)}
    assert _cells(2.5, 3.0, 2.5, 3.0) == {(3, 2), (3, 3)}
    assert _cells(2.5, 2.5, 2.5, 2.5) == {(2, 2), (2, 3), (3, 2), (3, 3)}
    assert _cells(-0.5, -0.5, -0.5, -0.5) == {(0, 0)}
    assert _cells(-0.6, 1.0, -0.6, 1.0) == set()


def test_segment_from_far_outside_crossing_the_raster():
    # v rises 0.7 cell over 2e8 cells: inside the raster it is 2.55 + ~1e-8, off every row edge but 2.5's by 0.05
    assert _cells(-1.0e8, 2.2, 1.0e8, 2.9) == {(3, j) for j in range(8)}
    assert _cells(-1.0e9, -1.0e9, 1.0e9, 1.0e9) == {(i, j) for i in range(6) for j in range(8) if abs(i - j) <= 1}
    occ = np.zeros((6, 8), dtype=np.uint8)
    occ[3, 6] = 1
    Z = _paths_from_pixels([np.array([[-1.0e8, 2.2], [1.0e8, 2.9]])], GEO_PIX)
    flags, first, d2min = sweep_reference(occ, GEO_PIX, Z, orc.edt_sq(occ))
    assert flags[0] == HIT | OUTSIDE and first[0] == 0 and d2min[0] == 0


def test_invalid_rows():
    occ = np.zeros((6, 8), dtype=np.uint8)
    occ[2, 0] = 1
    good = np.array([[0.0, 0.0], [2.0, 2.0], [5.0, 4.0]])
    rows = []
    for c, bad in [(0, np.nan), (1, np.inf), (0, -np.inf), (1, 2.0 ** 31), (0, -2.0 ** 31), (1, 2.0 ** 31 - 2.0 ** -20)]:
        r = good.copy()
        r[1, c] = bad
        rows.append(r)
    flags, first, d2min = sweep_reference(occ, GEO_PIX, _paths_from_pixels(rows, GEO_PIX), orc.edt_sq(occ))
    assert list(flags[:5]) == [INVALID] * 5 and list(first[:5]) == [-1] * 5 and list(d2min[:5]) == [-1] * 5
    # just below 2^31 is valid: the path leaves the raster and crosses occupied (2, 0) on its way out
    assert flags[5] == HIT | OUTSIDE and first[5] == 0


def test_paths_with_no_occupied_cell():
    rng = np.random.default_rng(3)
    occ = np.zeros((30, 40), dtype=np.uint8)
    Z = _random_paths(rng, 12, 9, GEO, 30, 40, spill=0.05)
    flags, first, d2min = sweep_reference(occ, GEO, Z, orc.edt_sq(occ))
    assert not np.any(flags & HIT) and np.all(first == -1)
    assert np.all((d2min == 65535) | ((d2min == -1) & (flags == OUTSIDE))) and np.sum(d2min == 65535) >= 8


def test_d2_clips_at_65535():
    H, W = 300, 310
    occ = np.zeros((H, W), dtype=np.uint8)
    occ[:3, :3] = 1
    d2 = orc.edt_sq(occ)
    assert d2.max() > 65535
    far = np.array([[W - 2.0, H - 2.0], [W - 30.0, H - 20.0]])        # every touched cell is > 256 cells away
    near = np.array([[200.0, 200.0], [150.0, 150.0]])                    # reaches 148^2 + 148^2 < 65535
    flags, first, d2min = sweep_reference(occ, GEO_PIX, _paths_from_pixels([far, near], GEO_PIX), d2)
    assert d2min[0] == 65535 and d2min[1] == 2 * 148 ** 2
    assert not np.any(flags & HIT)


@pytest.mark.parametrize('spc', [0.0, 0.37, 1.0])
def test_sampled_collide_implies_hit(spc):
    rng = np.random.default_rng(int(spc * 100) + 5)
    H, W = 70, 90
    lay, occ = _random_raster(rng, 1, H, W)
    Z = _random_paths(rng, 160, 10, GEO, H, W, spill=0.0, jitter=3.0)
    _, col, _ = orc.score_paths_raster(lay, occ, GEO, Z, [1.0], spc)
    flags, first, _ = sweep_reference(occ, GEO, Z)
    inside = (flags & OUTSIDE) == 0
    assert inside.sum() >= 100 and col[inside].sum() >= 10
    hit = (flags & HIT) != 0
    assert not np.any(col & inside & ~hit)
    assert hit.sum() >= col[inside].sum()
    assert np.array_equal(first >= 0, hit)


# ------------------------------------------------------------------------------------------------------------------
# GPU: the kernel against the restatement
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


_REF = {}


def _case(Wp):
    """(lay, occ, Z, reference outputs) of one path length, shared by the texel forms and layouts"""
    if Wp not in _REF:
        rng = np.random.default_rng(100 + Wp)
        H, W = 70, 90
        lay, occ = _random_raster(rng, 3, H, W)
        Z = _mixed_rows(rng, Wp, H, W, GEO)
        _REF[Wp] = (lay, occ, Z, sweep_reference(occ, GEO, Z, orc.edt_sq(occ)))
    return _REF[Wp]


@pytest.mark.gpu
@pytest.mark.parametrize('Wp', [2, 3, 5, 33, 64, 130])
@pytest.mark.parametrize('layout', [0, 1])
@pytest.mark.parametrize('L', [1, 3])
def test_kernel_equals_reference(uam, torch, L, layout, Wp):
    lay, occ, Z, (f_ref, h_ref, d_ref) = _case(Wp)
    rm = uam.RasterMap.from_arrays(lay[:L], GEO, occ, options={'raster_layout': layout})
    flags, first, d2min = rm.sweep_paths(Z)
    assert np.array_equal(flags, f_ref) and np.array_equal(first, h_ref) and np.array_equal(d2min, d_ref)
    assert np.any(f_ref == INVALID) and np.any(f_ref & HIT) and np.any(f_ref & OUTSIDE)
    # flags and first hit without the clearance (the walk may stop at the first hit)
    f2, h2, d2 = rm.engine.sweep_raster(Z, Wp - 2, True, False)
    assert d2 is None and np.array_equal(f2, f_ref) and np.array_equal(h2, h_ref)
    f3, h3, _ = rm.engine.sweep_raster(Z, Wp - 2, False, False)
    assert h3 is None and np.array_equal(f3, f_ref)


@pytest.mark.gpu
def test_kernel_equals_reference_off_grid_geometry(uam, torch):
    rng = np.random.default_rng(7)
    H, W, geo = 61, 47, (3.0, 0.3, 40.0, -0.2)
    lay, occ = _random_raster(rng, 1, H, W)
    Z = _mixed_rows(rng, 17, H, W, geo, n_random=64)
    rm = uam.RasterMap.from_arrays(lay, geo, occ)
    ref = sweep_reference(occ, geo, Z, orc.edt_sq(occ))
    got = rm.sweep_paths(Z)
    for a, b in zip(got, ref):
        assert np.array_equal(a, b)


@pytest.mark.gpu
def test_d2min_beyond_the_clip(uam, torch):
    rng = np.random.default_rng(11)
    H, W = 300, 320
    occ = np.zeros((H, W), dtype=np.uint8)
    occ[5:9, 4:12] = 1
    occ[20, 30] = 1
    lay = rng.uniform(size=(1, H, W)).astype(np.float32)
    d2 = orc.edt_sq(occ)
    assert d2.max() > 65535
    Z = np.concatenate([_random_paths(rng, 40, 6, GEO, H, W, spill=0.05, jitter=20.0),
                        _mixed_rows(rng, 6, H, W, GEO, n_random=0)])
    ref = sweep_reference(occ, GEO, Z, d2)
    assert np.any(ref[2] == 65535) and np.any((ref[2] >= 0) & (ref[2] < 65535))
    got = uam.RasterMap.from_arrays(lay, GEO, occ).sweep_paths(Z)
    for a, b in zip(got, ref):
        assert np.array_equal(a, b)


@pytest.mark.gpu
@pytest.mark.parametrize('layout', [0, 1])
def test_d2_field_equals_edt(uam, torch, layout):
    """One zero-length path per cell centre touches that cell alone: d2min is the field."""
    rng = np.random.default_rng(5)
    H, W = 37, 53
    lay, occ = _random_raster(rng, 3, H, W)
    ii, jj = np.mgrid[0:H, 0:W]
    P = np.stack([jj.ravel(), ii.ravel()], axis=-1).astype(np.float64)
    Z = _world(np.stack([P, P], axis=1), GEO).reshape(-1, 4)
    rm = uam.RasterMap.from_arrays(lay, GEO, occ, options={'raster_layout': layout})
    flags, first, d2min = rm.sweep_paths(Z)
    assert np.array_equal(d2min.reshape(H, W), np.minimum(orc.edt_sq(occ), 65535))
    assert np.array_equal(flags.reshape(H, W), occ.astype(np.uint8) * HIT)


@pytest.mark.gpu
def test_batch_independence_and_numpy_tensor_paths(uam, torch):
    lay, occ, Z, _ = _case(33)
    rm = uam.RasterMap.from_arrays(lay, GEO, occ)
    flags, first, d2min = rm.sweep_paths(Z)
    perm = np.random.default_rng(0).permutation(Z.shape[0])
    f2, h2, d2 = rm.sweep_paths(Z[perm])
    assert np.array_equal(f2, flags[perm]) and np.array_equal(h2, first[perm]) and np.array_equal(d2, d2min[perm])
    sub = perm[:7]
    f3, h3, d3 = rm.sweep_paths(Z[sub])
    assert np.array_equal(f3, flags[sub]) and np.array_equal(h3, first[sub]) and np.array_equal(d3, d2min[sub])
    Zt = torch.from_numpy(Z).cuda()
    ft, ht, dt = rm.sweep_paths(Zt)
    assert ft.is_cuda and ft.dtype == torch.uint8 and ht.dtype == torch.int32 and dt.dtype == torch.int32
    assert np.array_equal(ft.cpu().numpy(), flags) and np.array_equal(ht.cpu().numpy(), first)
    assert np.array_equal(dt.cpu().numpy(), d2min)


@pytest.mark.gpu
def test_reupload_invalidates_both_fields(uam, torch):
    rng = np.random.default_rng(9)
    H, W = 50, 60
    lay, occ = _random_raster(rng, 1, H, W)
    Z = _random_paths(rng, 64, 8, GEO, H, W, spill=0.05)
    rm = uam.RasterMap.from_arrays(lay, GEO, occ)
    first = rm.sweep_paths(Z)
    for a, b in zip(first, sweep_reference(occ, GEO, Z, orc.edt_sq(occ))):
        assert np.array_equal(a, b)
    occ2 = np.ascontiguousarray(occ[::-1, ::-1])
    rm.engine.set_raster(lay, GEO, occ2)
    got = rm.sweep_paths(Z)
    ref2 = sweep_reference(occ2, GEO, Z, orc.edt_sq(occ2))
    assert not np.array_equal(ref2[2], first[2])
    for a, b in zip(got, ref2):
        assert np.array_equal(a, b)
    # a scoring call that builds the quad texels in between (bit-plane form) leaves the sweep's answers unchanged
    rm.engine.set_raster(lay, GEO, occ)
    Zs = _random_paths(rng, 4096, 66, GEO, H, W)
    rm.score_paths(Zs, [-1.0], 1.0)
    for a, b in zip(rm.sweep_paths(Z), first):
        assert np.array_equal(a, b)


@pytest.mark.gpu
def test_errors(uam, torch):
    from uam_path_planning_b200 import _lib
    eng = uam.Engine()
    lib, h = eng._lib, eng._h
    Z = torch.zeros((4, 6), dtype=torch.float64, device='cuda')
    fl = torch.empty(4, dtype=torch.uint8, device='cuda')
    p = C.c_void_p
    assert lib.uam_sweep_paths_raster(h, p(Z.data_ptr()), 4, 1, p(fl.data_ptr()), None, None, None) == -4       # no raster
    assert lib.uam_sweep_paths_raster(h, p(Z.data_ptr()), 0, 1, p(fl.data_ptr()), None, None, None) == 0        # B = 0
    assert lib.uam_sweep_paths_raster(h, p(Z.data_ptr()), 4, -1, p(fl.data_ptr()), None, None, None) == -1
    assert lib.uam_sweep_paths_raster(h, None, 4, 1, p(fl.data_ptr()), None, None, None) == -1
    assert lib.uam_sweep_paths_raster(h, p(Z.data_ptr()), 4, 1, None, None, None, None) == -1
    # over 23170 cells per side: flags and first hit work, the clearance is refused
    H, W = 3, 23171
    occ = np.zeros((H, W), dtype=np.uint8)
    occ[1, 20000] = 1
    eng.set_raster(np.ones((1, H, W), dtype=np.float32), GEO_PIX, occ)
    Zp = _paths_from_pixels([np.array([[0.0, 1.0], [23170.0, 1.0]]), np.array([[0.0, 0.0], [100.0, 0.0]])], GEO_PIX)
    with pytest.raises(_lib.UamError, match='UNSUPPORTED'):
        eng.sweep_raster(Zp, 0, True, True)
    flags, first, d2min = eng.sweep_raster(Zp, 0, True, False)
    assert list(flags) == [HIT, 0] and list(first) == [0, -1] and d2min is None


@pytest.mark.gpu
@pytest.mark.parametrize('spc', [0.0, 1.0])
def test_device_collide_implies_hit_before_and_after_refine(uam, torch, spc):
    import bench
    n = 2048
    layers, occ, geo = bench.make_raster(torch, 'cuda:0', n)
    rm = uam.RasterMap.from_arrays(layers, geo, occ)
    Z = bench.make_paths(torch, 'cuda:0', 8192, seed=3, n=n)
    for Zc in (Z, rm.refine_paths(Z, bench.WEIGHTS, spc)[0]):
        _, col = rm.score_paths(Zc, bench.WEIGHTS, spc)
        flags, first, _ = rm.sweep_paths(Zc, clearance=False)
        inside = (flags & OUTSIDE) == 0
        hit = (flags & HIT) != 0
        assert int(inside.sum()) > 7000 and int((col.bool() & inside).sum()) > 0
        assert int((col.bool() & inside & ~hit).sum()) == 0
        assert torch.equal(first >= 0, hit)
