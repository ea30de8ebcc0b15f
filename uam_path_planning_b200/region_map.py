"""``Map`` / ``RegionMap``: the planner's map container (reference: path_generation/map.py:7-97,
region_map.py:8-65), with the point queries answered by the GPU.

The container is host data (lists of shapes); an ``Engine`` with the flattened shape table is created
lazily and re-uploaded whenever the shape lists change.  Plotting / axis-limit helpers of the reference
are matplotlib-only and out of scope.
"""
from __future__ import annotations

from typing import Any, Dict, List, Optional

import numpy as np

from .shapes import QuadraticObstacle

_COLORS = {'k': [0, 0, 0], 'black': [0, 0, 0], 'b': [0, 0, 1], 'blue': [0, 0, 1], 'g': [0, 1, 0],
           'green': [0, 1, 0], 'c': [0, 1, 1], 'cyan': [0, 1, 1], 'r': [1, 0, 0], 'red': [1, 0, 0],
           'm': [1, 0, 1], 'magenta': [1, 0, 1], 'y': [1, 1, 0], 'yellow': [1, 1, 0], 'w': [1, 1, 1],
           'white': [1, 1, 1]}


def color2RGB(color):
    """utils.py:3-27: colour names -> RGB; non-strings pass through."""
    if not isinstance(color, str):
        return color
    return _COLORS.get(color.lower(), None)


class Map:
    def __init__(self, *obstacles):
        self.obstacles: List[QuadraticObstacle] = []
        self.x_goal: np.ndarray = np.zeros(2)
        self.x_start: np.ndarray = np.zeros(2)
        self._engine = None
        self._engine_sig = None
        self._sig_epoch, self._sig_lists = -1, []
        self._device: Optional[int] = None
        self.add(*obstacles)

    def add(self, *obstacles):
        """Add obstacles to the map (map.py:13-17)."""
        for obstacle in obstacles:
            assert isinstance(obstacle, QuadraticObstacle), 'Obstacle must be a QuadraticObstacle object'
            self.obstacles.append(obstacle)

    # ---- device table -----------------------------------------------------------------------------------
    def _region_lists(self):
        return []

    def _signature(self):
        """State of everything the device shape table is made from: per shape a serial number that changes with every
        assignment of its centre or of one of its inequality records (both are stored read-only, so in-place edits are
        impossible), plus the composition of the lists.  Serial numbers are never reused (unlike id())."""
        return (tuple(o.state_key() for o in self.obstacles),
                tuple(tuple(s.state_key() for s in shapes) for shapes in self._region_lists()))

    def engine(self, device: Optional[int] = None):
        """The map's Engine with the current shape table uploaded (rebuilt when the shape lists changed)."""
        from .engine import Engine
        if device is not None and device != self._device:
            self._device, self._engine = device, None
        if self._engine is None:
            self._engine = Engine(self._device)
            self._device = self._engine.device
            self._engine_sig = None
        # fast check first: no shape anywhere changed (one integer) and the lists hold the same objects (identity compare
        # at C speed; the cached copies keep the objects alive, so ids cannot be reused) -- 3 us instead of 60 for 300 shapes.
        # (Inequalities are added through QuadraticObstacle.add, as in the reference: it bumps the epoch.)
        from . import shapes as _shapes
        lists = [self.obstacles] + self._region_lists()
        if (self._engine_sig is not None and self._sig_epoch == _shapes.EPOCH[0] and len(lists) == len(self._sig_lists)
                and all(a == b for a, b in zip(lists, self._sig_lists))):
            return self._engine
        sig = self._signature()
        if sig != self._engine_sig:
            self._engine.set_shapes(self.obstacles, self._region_lists())
            self._engine_sig = sig
        self._sig_epoch = _shapes.EPOCH[0]
        self._sig_lists = [list(l) for l in lists]
        return self._engine

    # ---- queries --------------------------------------------------------------------------------------------
    def collides(self, x) -> bool:
        """Point belongs to any obstacle (map.py:41-43).  (M,2) input gives a bool array."""
        x = np.asarray(x, dtype=np.float64)
        R = len(self._region_lists())
        p = np.concatenate([[0, 0, 0, 0, 1.0, 0.0, 0.0], np.ones(R)])
        out = self.engine().eval_points(x.reshape(-1, 2), p, 0, want=('collide',))['collide'].astype(bool)
        return bool(out[0]) if x.ndim == 1 else out

    def sweep_paths(self, Z):
        """Swept check of every segment of the paths Z (B, 2(N+2)) against the hard obstacles -> (flags u8 (B,), first_hit
        i32 (B,), first_obstacle i32 (B,)); N comes from Z's width, numpy in -> numpy out, CUDA tensor in -> CUDA tensors
        out (uam_sweep_paths_analytic, include/uam_b200.h).  flags has UAM_SWEEP_HIT when some segment hits an obstacle and
        UAM_SWEEP_INVALID for a row with a coordinate that is not finite or >= 1e100 in magnitude; first_hit is the lowest
        hitting segment and first_obstacle the smallest obstacle index it hits (order of ``obstacles``), -1 if none.
        G1: a segment that meets an obstacle in exact arithmetic is always reported.
        G2: a waypoint that ``collides`` reports makes both of its segments hit, so the analytic scorer's collide flag
        implies HIT.
        G3: a reported segment comes within a few ulps of the obstacle: it meets the obstacle's inequalities relaxed by a
        bound eta_i of the record's and the endpoints' magnitudes (about 1e-12 km on the reference's maps)."""
        N = int(Z.shape[1]) // 2 - 2
        return self.engine().sweep_analytic(Z, N, True, True)

    def path_clearance(self, Z, cap):
        """How far each path of Z (B, 2(N+2)) stays from the hard obstacles, up to cap -> (flags u8 (B,), clearance f64
        (B,), nearest_segment i32 (B,), nearest_obstacle i32 (B,)); N comes from Z's width, numpy in -> numpy out, CUDA
        tensor in -> CUDA tensors out (uam_clearance_paths_analytic, include/uam_b200.h).  clearance is min(cap, the
        distance from the path's segments to the obstacles), and the nearest pair is the segment and obstacle that
        attain it (smallest segment, then smallest obstacle), -1 when nothing lies within cap.  So ``clearance >= m`` is
        the keep-out check of a margin m <= cap.  Obstacles must be polygons, boxes or ellipses, as polygon(), square()
        and ball() make them; other record combinations raise.
        D1: flags are ``sweep_paths``'s flags bit for bit; a path that hits has clearance 0 and its nearest pair is the
        sweep's first hit; any other valid path has clearance > 0.  INVALID rows get NaN and -1.
        D2: a non-hitting segment's distance is exact up to a rounding bound of a few ulps of the coordinates' magnitude
        (more for elongated ellipses: it scales with their axis ratio).
        D3: the results are deterministic, bit for bit: they do not depend on the rest of the batch, on the cell lists,
        or on cap other than through the min with cap."""
        N = int(Z.shape[1]) // 2 - 2
        return self.engine().clearance_analytic(Z, N, cap, True)

    def intersection(self, x0, direction):
        # map.py:19-39 calls QuadraticObstacle.intersection, which is commented out in the reference
        raise AttributeError("'QuadraticObstacle' object has no attribute 'intersection'")

    def __len__(self):
        return len(self.obstacles)

    def __getitem__(self, key):
        if isinstance(key, tuple):
            return self.collides(np.array(key))
        elif isinstance(key, slice):
            return self.obstacles[key]
        else:
            raise TypeError('Invalid argument type.')


class RegionMap(Map):
    def __init__(self):
        super().__init__()
        self.regions: Dict[str, Dict[str, Any]] = {}
        self.map_version = 'v1'

    def add_obstacle(self, obstacle: QuadraticObstacle):
        self.add(obstacle)

    def add_obstacles(self, *obstacles):
        self.add(*obstacles)

    def new_region(self, name: str, color):
        if self.region_exists(name):
            raise ValueError(f"Name '{name}' already in use for areas")
        self.regions[name] = {'shapes': [], 'color': color2RGB(color)}

    def add_shape_to_region(self, region: str, obstacle: QuadraticObstacle):
        if not self.region_exists(region):
            raise ValueError(f"Unknown type '{region}' of penalty obstacles. Use new_region method to define it")
        assert isinstance(obstacle, QuadraticObstacle)
        self.regions[region]['shapes'].append(obstacle)

    def add_shapes_to_region(self, region: str, *obstacles):
        for obstacle in obstacles:
            self.add_shape_to_region(region, obstacle)

    def region_names(self) -> List[str]:
        return list(self.regions.keys())

    def region_exists(self, region: str) -> bool:
        return region in self.regions

    def _region_lists(self):
        return [r['shapes'] for r in self.regions.values()]
