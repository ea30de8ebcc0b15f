"""Launches of the raster refinements (RasterMap.refine_paths, refine_paths_swept, refine_paths_keepout).

Once the quad texels and the check's fields are built, a refine of K trips enqueues the evaluation of the batch (one
gradient call's g launches, then c launches of its check: 0 without one, 1 for the raster sweep or the analytic sweep or
clearance) once at the start and once per trip, and one uam_k_refine_step per evaluation: (K + 1)(g + c + 1) launches.
K = 0 enqueues the first evaluation only: g + c.
"""
import numpy as np
import pytest

from test_raster_gradient import _random_paths, _random_raster
from test_raster_refine_keepout import GEO, _obstacle_records, _shape_map


@pytest.fixture(scope='module')
def uam():
    import uam_path_planning_b200 as u
    return u


@pytest.fixture(scope='module')
def torch():
    import torch as t
    assert t.cuda.is_available()
    return t


@pytest.mark.gpu
@pytest.mark.parametrize('spc', [0.0, 1.0])
@pytest.mark.parametrize('mode,arg', [('plain', None), ('swept', 0), ('swept', 4), ('keepout', 0.0), ('keepout', 0.5)])
def test_refine_launches_per_trip(uam, torch, spc, mode, arg):
    rng = np.random.default_rng(900)
    H, W = 150, 230
    lay, occ = _random_raster(rng, 3, H, W)
    rm = uam.RasterMap.from_arrays(lay, GEO, occ)
    rm.set_obstacles(_shape_map(uam, _obstacle_records(rng, GEO, H, W, n=18)))
    Z = torch.from_numpy(_random_paths(rng, 64, 9, GEO, H, W)).cuda()
    N = Z.shape[1] // 2 - 2
    w = [200.0, 15000.0, 27000.0]
    eng = rm.engine
    if mode == 'plain':
        def refine(K):
            return rm.refine_paths(Z, w, spc, K)

        def check():
            pass
    elif mode == 'swept':
        def refine(K):
            return rm.refine_paths_swept(Z, w, spc, K, min_d2=arg)

        def check():
            eng.sweep_raster(Z, N, False, arg > 0)
    else:
        def refine(K):
            return rm.refine_paths_keepout(Z, w, spc, K, margin=arg)

        def check():
            if arg > 0:
                eng.clearance_analytic(Z, N, arg, False)
            else:
                eng.sweep_analytic(Z, N, False, False)

    def launches(f):
        n0 = eng.launch_count()
        f()
        return eng.launch_count() - n0

    refine(1)           # builds the quad texels, the bit-plane, the d^2 field, the obstacle tables and lists
    g = launches(lambda: rm.cost_gradient(Z, w, spc))
    c = launches(check)
    assert g >= 1 and c == (0 if mode == 'plain' else 1)
    assert launches(lambda: refine(0)) == g + c
    for K in (1, 2, 3):
        assert launches(lambda: refine(K)) == (K + 1) * (g + c + 1), K
