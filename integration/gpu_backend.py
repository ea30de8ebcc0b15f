"""path_generation/gpu_backend.py -- the file a maintainer of nomaporon/uam_path_planning adds to bind libuam_b200.so
(include/uam_b200.h) from the REFERENCE'S OWN classes with ctypes.  Shown in INTEGRATION.md section 2 and executed by
tests/test_integration_binding.py (CPU: table extraction from closures laid out like the reference's, against the tables
frozen from the reference's own objects; GPU: the raw binding below against the reference's golden costs).

Nothing here imports uam_path_planning_b200: only ctypes + numpy + the shared library.

The reference keeps a shape as a list of `Function` objects whose `.f` is a Python closure (function.py:119-120).
The numbers each closure captured are read back from its cells:
    polygon edge  f = lambda x: -sgn_F * line_F(x)      cells sgn_F, line_F -> cells Pa_F, Pb_F     polygon.py:66-98
    ellipse       f = func(x)                           cells center, r1, r2                        ball.py:33-37
    box side      f = lambda x: +-x[d] -+ center[d] - r cells center, r1 | r2 (side probed)         square.py:29-51
and packed into the 8-double inequality records of uam_map_set_shapes.
"""
import ctypes as C
import os

import numpy as np

UAM_EDGE_LINE, UAM_EDGE_ELLIPSE, UAM_EDGE_BOX = 0, 1, 2


def _cells(fn):
    return dict(zip(fn.__code__.co_freevars, (c.cell_contents for c in (fn.__closure__ or ()))))


def inequality_record(func):
    """reference `Function` -> one 8-double record (include/uam_b200.h: UAM_EDGE_*)"""
    c = _cells(func.f)
    if 'line_F' in c:                                           # polygon.py:98
        pa, pb = (np.asarray(v, dtype=np.float64).ravel() for v in (_cells(c['line_F'])['Pa_F'], _cells(c['line_F'])['Pb_F']))
        return [UAM_EDGE_LINE, pa[0], pa[1], pb[0] - pa[0], pb[1] - pa[1], float(c['sgn_F']), 0.0, 0.0]
    if 'r1' in c and 'r2' in c:                                 # ball.py:33-37
        ctr = np.asarray(c['center'], dtype=np.float64).ravel()
        return [UAM_EDGE_ELLIPSE, ctr[0], ctr[1], float(c['r1']), float(c['r2']), 0.0, 0.0, 0.0]
    ctr = np.asarray(c['center'], dtype=np.float64).ravel()     # square.py:29-51: one of right / left / top / bottom
    r = float(c['r1'] if 'r1' in c else c['r2'])
    gx = func.f(ctr + np.array([1.0, 0.0])) - func.f(ctr)       # +-1 for an x side, 0 for a y side
    gy = func.f(ctr + np.array([0.0, 1.0])) - func.f(ctr)
    axis, sign = (0, gx) if gx != 0 else (1, gy)
    return [UAM_EDGE_BOX, float(axis), float(np.sign(sign)), ctr[axis], r, 0.0, 0.0, 0.0]


def extract_tables(m):
    """reference RegionMap -> the arrays of uam_map_set_shapes: obstacles first (region -1), then the regions in
    insertion order (= the order of the weights in the parameter vector, solver.py:68,77-78)."""
    groups = [(-1, m.obstacles)] + [(r, m.regions[n]['shapes']) for r, n in enumerate(m.region_names())]
    shapes = [(r, s) for r, ss in groups for s in ss]
    edges = np.array([inequality_record(f) for _, s in shapes for f in s.inequalities], dtype=np.float64).reshape(-1, 8)
    off = np.cumsum([0] + [len(s.inequalities) for _, s in shapes]).astype(np.int32)
    reg = np.array([r for r, _ in shapes], dtype=np.int32)
    cen = np.array([np.asarray(s.center, dtype=np.float64).reshape(2) for _, s in shapes]).reshape(-1, 2)
    return {'edges': edges, 'off': off, 'region': reg, 'center': cen, 'n_regions': len(m.regions)}


def load_library(path=None):
    lib = C.CDLL(path or os.environ.get('UAM_B200_LIB', 'libuam_b200.so'))
    lib.uam_ctx_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
    lib.uam_ctx_destroy.argtypes = [C.c_void_p]
    lib.uam_last_error.argtypes = [C.c_void_p]
    lib.uam_last_error.restype = C.c_char_p
    lib.uam_map_set_shapes.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int]
    lib.uam_score_paths_analytic_host.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_int, C.c_int,
                                                  C.c_void_p, C.c_void_p, C.c_void_p]
    lib.uam_analytic_g_len.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_int64)]
    return lib


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


class GpuScorer:
    """A device context holding one shape table."""

    def __init__(self, tables, device=0, lib=None):
        self.lib, self.h = lib or load_library(), C.c_void_p()
        if self.lib.uam_ctx_create(device, C.byref(self.h)) != 0:
            raise RuntimeError('uam_ctx_create failed: no CUDA device (there is no CPU fallback)')
        t = {k: (np.ascontiguousarray(v) if isinstance(v, np.ndarray) else v) for k, v in tables.items()}
        rc = self.lib.uam_map_set_shapes(self.h, _ptr(t['edges']), len(t['edges']), _ptr(t['off']), _ptr(t['region']),
                                         _ptr(t['center']), len(t['region']), int(t['n_regions']))
        if rc != 0:
            raise RuntimeError(self.lib.uam_last_error(self.h).decode())

    def score(self, Z, N, p, flags, want_g=False):
        """rows of Z = z_ = [x_start, x, x_goal] (solver.py:64-66) -> (get_cost, any collides, get_nonlincon | None)"""
        Z = np.ascontiguousarray(Z, dtype=np.float64).reshape(-1, 2 * (N + 2))
        p = np.ascontiguousarray(p, dtype=np.float64)
        cost, col, g = np.empty(len(Z)), np.empty(len(Z), np.uint8), None
        if want_g:
            n = C.c_int64()
            self.lib.uam_analytic_g_len(self.h, N, C.byref(n))
            g = np.empty((len(Z), n.value))
        rc = self.lib.uam_score_paths_analytic_host(self.h, _ptr(Z), len(Z), N, _ptr(p), len(p), int(flags), _ptr(cost),
                                                    _ptr(col), _ptr(g) if want_g else None)
        if rc != 0:
            raise RuntimeError(self.lib.uam_last_error(self.h).decode())
        return cost, col.astype(bool), g

    def close(self):
        if self.h:
            self.lib.uam_ctx_destroy(self.h)
            self.h = C.c_void_p()


class GpuProblem:
    """Wraps a reference `Problem` (problem.py:6): same get_cost / get_nonlincon, batched over the rows of Z."""

    def __init__(self, problem, device=0, lib=None):
        self.p = problem
        self.scorer = GpuScorer(extract_tables(problem.map), device, lib)

    def parameter_vector(self):
        pr = self.p                                              # the order of solver.py:60-68
        return np.array([*pr.map.x_start, *pr.map.x_goal, pr.params['maxratio'], pr.params['maxalpha'], pr.params['enlargement'],
                         *[pr.weights[n] for n in pr.map.region_names()]], dtype=np.float64)

    def flags(self):
        o = self.p.options                                       # problem.py:12-17 -> UAM_*_SMOOTH bits
        return int(bool(o['length_smooth'])) | int(bool(o['penalty_smooth'])) << 1 | int(bool(o['obstacle_smooth'])) << 2 | \
            int(bool(o['maxratio_smooth'])) << 3

    def get_cost(self, Z):
        return self.scorer.score(Z, self.p.N, self.parameter_vector(), self.flags())[0]

    def get_nonlincon(self, Z):
        return self.scorer.score(Z, self.p.N, self.parameter_vector(), self.flags(), want_g=True)[2]
