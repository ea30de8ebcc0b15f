"""Raster side of the hot path: rebuild cost / occupancy rasters from the map on the GPU and score candidate
paths against them.

Raster layout is rasterio's band layout as the reference reads it (map_generation/data_manager.py:13):
``(L, H, W)`` float32 C-order, row <-> y, col <-> x, affine ``geo = (x0, dx, y0, dy)``, cell centre
``(x0 + (j + 1/2) dx, y0 + (i + 1/2) dy)``; occupancy ``(H, W)`` uint8.  Layer l is the *unweighted* penalty
field of region l (problem.py:72-80), so the region weights stay a run-time parameter (solver.py:68).
"""
from __future__ import annotations

from typing import Optional, Sequence, Tuple

import numpy as np

from . import _lib
from .engine import Engine, _is_tensor
from .region_map import RegionMap


def load_dem_mask(image, threshold: float = 0.0, engine: Optional[Engine] = None):
    """mask = image > threshold (image == -9999 for threshold == -9999): the raster op of
    ``DataManager.load_dem_polygons_from_geotiff`` (map_generation/data_manager.py:14-17) on a float32 CUDA
    tensor (or a numpy array, copied to the GPU and back)."""
    import torch
    eng = engine or Engine()
    if _is_tensor(image):
        return eng.dem_mask(image.contiguous(), threshold)
    t = torch.from_numpy(np.ascontiguousarray(image, dtype=np.float32)).to(f'cuda:{eng.device}')
    return eng.dem_mask(t, threshold).cpu().numpy().astype(bool)


class RasterMap:
    """Cost layers + occupancy of a ``RegionMap`` on one GPU, and the raster path scorer on top of them."""

    def __init__(self, H: int, W: int, geo: Tuple[float, float, float, float], device: Optional[int] = None,
                 options: Optional[dict] = None):
        self.H, self.W = int(H), int(W)
        self.geo = tuple(float(v) for v in geo)
        self.engine = Engine(device)
        for k, v in (options or {}).items():
            self.engine.set_option(k, v)
        self.layers = None        # (L,H,W) float32 CUDA tensor
        self.occupancy = None     # (H,W) uint8 CUDA tensor
        self.clearance = None     # (H,W) float32 CUDA tensor (distance to the nearest occupied cell)
        self.dist2 = None

    # ---- build ---------------------------------------------------------------------------------------------
    @classmethod
    def from_map(cls, m: RegionMap, H: int, W: int, geo, enlargement: float = 0.0, device: Optional[int] = None,
                 clearance: bool = False, options: Optional[dict] = None) -> 'RasterMap':
        """Rasterise the map's regions and obstacles at the cell centres (map rebuild, config 4)."""
        rm = cls(H, W, geo, device, options)
        eng = rm.engine
        eng.set_shapes(m.obstacles, m._region_lists())
        rm.occupancy = eng.rasterize_occupancy(rm.H, rm.W, rm.geo)
        rm.layers = eng.rasterize_layers(rm.H, rm.W, rm.geo, enlargement)
        if clearance:
            rm.dist2, rm.clearance = eng.edt(rm.occupancy, abs(rm.geo[1]))
        eng.set_raster(rm.layers, rm.geo, rm.occupancy)
        return rm

    @classmethod
    def from_arrays(cls, layers, geo, occupancy=None, device: Optional[int] = None,
                    options: Optional[dict] = None) -> 'RasterMap':
        """Adopt existing rasters (numpy or CUDA tensors)."""
        L, H, W = layers.shape
        rm = cls(H, W, geo, device, options)
        rm.engine.set_raster(layers, rm.geo, occupancy)
        if _is_tensor(layers):
            rm.layers, rm.occupancy = layers, occupancy
        return rm

    # ---- score ---------------------------------------------------------------------------------------------
    def parameter_vector(self, weights: Sequence[float], x_start=None) -> np.ndarray:
        xs = np.zeros(2) if x_start is None else np.asarray(x_start, dtype=np.float64).ravel()
        return np.concatenate([xs, [0.0, 0.0, np.nan, np.nan, 0.0], np.asarray(weights, dtype=np.float64)])

    def score_paths(self, Z, weights: Sequence[float], samples_per_cell: float = 0.0, length_smooth: bool = True,
                    x_start=None, want_nsamples: bool = False, out=None):
        """Cost + collision flag of each path of Z (B, 2(N+2)) float64 (numpy or CUDA tensor).

        cost = (N+1) * L + (1/N) * sum of sampled penalties, with L the reference's length term
        (problem.py:38-44,130-146; ``x_start`` = map.x_start, None = each path's own start) and the penalty
        P(x) = sum_l w_l * bilinear(layer_l, x).  samples_per_cell = 0 samples the N+2 waypoints like the
        reference; > 0 integrates along every segment."""
        N = Z.shape[1] // 2 - 2
        flags = (_lib.UAM_LENGTH_SMOOTH if length_smooth else 0) | (_lib.UAM_OWN_START if x_start is None else 0)
        p = self.parameter_vector(weights, x_start)
        return self.engine.score_raster(Z, N, p, flags, samples_per_cell, want_nsamples, out)

    def cost_gradient(self, Z, weights: Sequence[float], samples_per_cell: float = 0.0, length_smooth: bool = True,
                      x_start=None):
        """(cost, collide, grad) of score_paths' cost for Z (B, 2(N+2)) float64 (numpy or CUDA tensor), arguments as in
        score_paths.  cost / collide are score_paths' bits; grad (B, 2(N+2)) float64 is d cost / d Z with the per-segment
        sample counts held fixed (columns 2 .. 2N+1 are the free waypoints; include/uam_b200.h has the definition)."""
        N = Z.shape[1] // 2 - 2
        flags = (_lib.UAM_LENGTH_SMOOTH if length_smooth else 0) | (_lib.UAM_OWN_START if x_start is None else 0)
        return self.engine.grad_raster(Z, N, self.parameter_vector(weights, x_start), flags, samples_per_cell)

    def refine_paths(self, Z, weights: Sequence[float], samples_per_cell: float = 0.0, iterations: int = 20,
                     length_smooth: bool = True, x_start=None, step_cells: float = 1.0, max_step_cells: float = 64.0,
                     min_step_cells: float = 1.0 / 256):
        """Refine every path of Z (B, 2(N+2)) float64 by monotone descent on score_paths' cost, arguments as in
        score_paths -> (Z_out, cost, collide, accepted).

        Per path and trip: a trial moves the free waypoints (columns 2 .. 2N+1) along -grad (cost_gradient) so that the
        largest move is tau cells; it is kept iff it collides no more and costs strictly less (tau doubles, up to
        max_step_cells), otherwise tau halves; a path stops once tau < min_step_cells.  A path's (collide, cost) never
        gets worse, and cost / collide are score_paths(Z_out)'s bits; accepted counts the kept trips.  The cost layers
        carry no obstacle term, so a colliding path is not steered out of its obstacle.  include/uam_b200.h
        (uam_refine_paths_raster) has the exact rule.  numpy in -> numpy out; a CUDA tensor in -> new CUDA tensors out
        (Z itself is not modified).

        Defaults: 20 trips from a 1-cell step, at most 64 cells, down to 1/256 cell -- the best of the settings tried on
        the C3 shard (bench_raster_refine.py --sweep, NVIDIA B200 at 1000 W): median cost reduction 23.0 % against 16.6 %
        with at most 16 cells and 9.2 % with at most 4; a first step of 1/4 or 4 cells, or a floor of 1/16 cell, moved
        it by less than 1 point."""
        N = Z.shape[1] // 2 - 2
        flags = (_lib.UAM_LENGTH_SMOOTH if length_smooth else 0) | (_lib.UAM_OWN_START if x_start is None else 0)
        return self.engine.refine_raster(Z, N, self.parameter_vector(weights, x_start), flags, samples_per_cell, iterations,
                                         step_cells, max_step_cells, min_step_cells)

    def sweep_paths(self, Z, clearance: bool = True):
        """Check every cell each segment of Z (B, 2(N+2)) float64 crosses against the occupancy -> (flags, first_hit,
        d2min); numpy in -> numpy out, a CUDA tensor in -> CUDA tensors out.  score_paths only looks at its samples.

        Segment k runs from z_k to z_{k+1} (k = 0 .. N).  In pixel coordinates U = (x - x0)/dx - 0.5, V = (y - y0)/dy - 0.5
        (fp64, the scorer's), quantised to 2^-16 cell, a raster cell is touched by a segment iff the closed segment meets
        the cell's closed square dilated by one quantum (exact integer test: a segment along a cell edge touches both
        sides, one through a grid vertex all four cells, a zero-length one the cells around its point).
          flags (uint8): 1 = some segment touches an occupied cell (HIT), 2 = some waypoint lies outside the raster
                         rectangle [-1/2, W-1/2] x [-1/2, H-1/2] (only raster cells are judged), 4 = a coordinate is not
                         finite or |U| or |V| >= 2^31 (INVALID: nothing else is evaluated, first_hit = d2min = -1);
          first_hit (int32): the first segment that touches an occupied cell, -1 if none;
          d2min (int32, None unless clearance): min over the touched cells of min(d2, 65535), d2 the squared distance in
                         cells to the nearest occupied cell's centre (0 on an occupied cell, 65535 = 256 cells or more);
                         -1 when no raster cell is touched.  The clearance in map units is sqrt(d2min) * |dx| when
                         |dx| = |dy|.
        For a path inside the raster rectangle, score_paths' collide flag (any samples_per_cell) implies HIT.  The first
        call with clearance=True after a raster upload runs an EDT of the raster (include/uam_b200.h:
        uam_sweep_paths_raster); rasters over 23170 cells per side support clearance=False only."""
        N = Z.shape[1] // 2 - 2
        return self.engine.sweep_raster(Z, N, True, clearance)

    def score_paths_best(self, Z, weights: Sequence[float], samples_per_cell: float = 0.0, length_smooth: bool = True,
                         x_start=None, global_offset: int = 0, out=None, key=None):
        """score_paths on a CUDA tensor + the best candidate's key (distributed.decode_key) in the same call; with a peer
        group attached (distributed.attach_peer_group) the key is the min over every rank's batch -- the only cross-rank
        step of the path, fused into the step's last kernel."""
        N = Z.shape[1] // 2 - 2
        flags = (_lib.UAM_LENGTH_SMOOTH if length_smooth else 0) | (_lib.UAM_OWN_START if x_start is None else 0)
        return self.engine.score_raster_best(Z, N, self.parameter_vector(weights, x_start), flags, samples_per_cell,
                                             global_offset, out, key)

    def submit(self, weights: Sequence[float], samples_per_cell: float, cost, collide, Z=None, candidates=None, N: int = None,
               jitter_sigma: float = 0.0, seed: int = 0, key=None, global_offset: int = 0, length_smooth: bool = True,
               x_start=None) -> int:
        """Queue one host-buffer batch (numpy waypoints Z, or (B, 5) candidates {xs, ys, xg, yg, displacement} that the
        device turns into paths of N interior waypoints) and return a ticket; `wait(ticket)` returns when cost / collide /
        key are filled.  Up to three batches in flight: uploads overlap the kernels of the batch before."""
        if Z is not None:
            N = Z.shape[1] // 2 - 2
        flags = (_lib.UAM_LENGTH_SMOOTH if length_smooth else 0) | (_lib.UAM_OWN_START if x_start is None else 0)
        return self.engine.submit_raster(N, self.parameter_vector(weights, x_start), flags, samples_per_cell, cost, collide,
                                         Z, candidates, jitter_sigma, seed, key, global_offset)

    def wait(self, ticket: int):
        self.engine.wait_raster(ticket)

    def score_candidates(self, candidates, N: int, weights: Sequence[float], samples_per_cell: float = 0.0,
                         jitter_sigma: float = 0.0, seed: int = 0, global_offset: int = 0, length_smooth: bool = True,
                         x_start=None):
        """The reference's flow for a whole batch (displacement -> Solver.create_x_init -> score, main.py:160-171) with 40
        bytes of input per candidate: candidates (B, 5) numpy {xs, ys, xg, yg, displacement} -> (cost, collide, key)."""
        cd = np.ascontiguousarray(candidates, dtype=np.float64)
        B = cd.shape[0]
        cost, col, key = np.empty(B, dtype=np.float32), np.empty(B, dtype=np.uint8), np.empty(1, dtype=np.uint64)
        self.wait(self.submit(weights, samples_per_cell, cost, col, candidates=cd, N=N, jitter_sigma=jitter_sigma, seed=seed,
                              key=key, global_offset=global_offset, length_smooth=length_smooth, x_start=x_start))
        return cost, col, int(key[0])
