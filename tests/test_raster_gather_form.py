"""The gather layer against the bit-plane quads.

Large batches sample the weight-folded layer C = sum_l w_l layer_l.  With combine_layers = 1 it is read by tex2Dgather
from a 2-D CUDA array of 4-byte texels (the value negated on occupied cells); combine_layers = 2 reads 16-byte quad
texels plus an occupancy bit-plane.  Both forms hold the same values, so cost, collision flags and sample counts must
agree bit for bit: in the binned pipeline (integral mode) and in the waypoint kernel.  The gradient's slopes agree to
rounding: the slope arithmetic on sign-packed values (|value| operands) may contract into fused multiply-adds in another
order than on the bit-plane form's plain values, as it already did with the sign-packed quads.
"""
import numpy as np
import pytest


@pytest.fixture(scope='module')
def uam():
    import uam_path_planning_b200 as u
    return u


@pytest.fixture(scope='module')
def torch():
    import torch as t
    assert t.cuda.is_available()
    return t


def _raster(rng, L, H, W):
    """Values in [0, 3) with cells that are zero in every layer (some occupied: -0.0 in the gather layer) and cells whose
    folded value is a float32 denormal."""
    lay = rng.uniform(0.0, 3.0, (L, H, W)).astype(np.float32)
    zero = rng.uniform(size=(H, W)) < 0.2
    tiny = ~zero & (rng.uniform(size=(H, W)) < 0.2)
    lay[:, zero] = 0.0
    lay[:, tiny] = 0.0
    lay[0, tiny] = np.float32(3e-39)              # denormal, and so is the folded 0.5 * 3e-39
    occ = (rng.uniform(size=(H, W)) < 0.3).astype(np.uint8)
    occ[zero & (rng.uniform(size=(H, W)) < 0.5)] = 1
    return lay, occ


def _paths(rng, H, W, geo):
    """4400 x 64 waypoints (281 600 segments: the large-batch pipelines), most of them outside the raster."""
    x0, dx, y0, dy = geo
    B, Wp = 4400, 64
    lo = np.array([x0 - 0.6 * W * dx, y0 - 1.6 * H * abs(dy)])
    hi = np.array([x0 + 1.6 * W * dx, y0 + 0.6 * H * abs(dy)])
    s = lo + rng.uniform(size=(B, 1, 2)) * (hi - lo)
    g = lo + rng.uniform(size=(B, 1, 2)) * (hi - lo)
    t = np.linspace(0, 1, Wp).reshape(1, Wp, 1)
    return np.ascontiguousarray((s + t * (g - s) + rng.normal(0, 0.2, (B, Wp, 2))).reshape(B, 2 * Wp))


def _same(rm_a, rm_b, Zt, w):
    for spc in (1.0, 3.0, 0.0):
        ca, ka, na = rm_a.score_paths(Zt, w, spc, True, None, want_nsamples=True)
        cb, kb, nb = rm_b.score_paths(Zt, w, spc, True, None, want_nsamples=True)
        assert np.array_equal(ca.cpu().numpy().view(np.uint32), cb.cpu().numpy().view(np.uint32)), spc
        assert np.array_equal(ka.cpu().numpy(), kb.cpu().numpy()) and np.array_equal(na.cpu().numpy(), nb.cpu().numpy())
        ca, ka, ga = rm_a.cost_gradient(Zt, w, spc, True, None)
        cb, kb, gb = rm_b.cost_gradient(Zt, w, spc, True, None)
        assert np.array_equal(ca.cpu().numpy().view(np.uint32), cb.cpu().numpy().view(np.uint32)), spc
        assert np.array_equal(ka.cpu().numpy(), kb.cpu().numpy())
        ga, gb = ga.cpu().numpy(), gb.cpu().numpy()
        scale = np.maximum(np.abs(gb).max(axis=1, keepdims=True), 1e-300)
        assert np.all(np.abs(ga - gb) <= 1e-6 * scale), (spc, float((np.abs(ga - gb) / scale).max()))


@pytest.mark.gpu
@pytest.mark.parametrize('H,W', [(2, 2), (65, 129)])
@pytest.mark.parametrize('layout', [0, 1])
@pytest.mark.parametrize('L', [1, 2, 3])
def test_gather_layer_matches_bit_plane_quads(uam, torch, L, layout, H, W):
    rng = np.random.default_rng(1000 * L + 100 * layout + H)
    geo = (-1.0, 0.5, 7.0, -0.25)
    lay, occ = _raster(rng, L, H, W)
    Zt = torch.from_numpy(_paths(rng, H, W, geo)).cuda()
    opts = {'raster_layout': layout, 'integral_variant': -1}
    rm_g = uam.RasterMap.from_arrays(lay, geo, occ, options={**opts, 'combine_layers': 1})
    rm_q = uam.RasterMap.from_arrays(lay, geo, occ, options={**opts, 'combine_layers': 2})
    w = [0.5, 0.25, 11.0][:L]
    _same(rm_g, rm_q, Zt, w)
    # a weight change and back: the folded layer follows the weights
    _same(rm_g, rm_q, Zt, [7.0, 3.0, 0.5][:L])
    c0 = rm_g.score_paths(Zt, w, 1.0, True, None)[0].cpu().numpy()
    _same(rm_g, rm_q, Zt, w)
    assert np.array_equal(rm_g.score_paths(Zt, w, 1.0, True, None)[0].cpu().numpy().view(np.uint32), c0.view(np.uint32))
    # a negative weight: the folded values (L = 2..3) or the partial sums (L = 1) go negative, their sign bits cannot
    # carry the occupancy flags (L = 2..3 then fall back to the bit-plane quads)
    _same(rm_g, rm_q, Zt, [5.0, -40.0, 1.0][:L] if L > 1 else [-40.0])
    _same(rm_g, rm_q, Zt, w)
    # a re-upload with other dimensions: the gather layer is remade at the new size
    H2, W2 = H + 37, W + 3
    lay2, occ2 = _raster(rng, L, H2, W2)
    Z2 = torch.from_numpy(_paths(rng, H2, W2, geo)).cuda()
    rm_g.engine.set_raster(lay2, geo, occ2)
    rm_q2 = uam.RasterMap.from_arrays(lay2, geo, occ2, options={**opts, 'combine_layers': 2})
    _same(rm_g, rm_q2, Z2, w)
