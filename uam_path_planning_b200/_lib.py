"""ctypes binding of libuam_b200.so (the C-ABI declared in include/uam_b200.h).

There is no CPU fallback: if the shared library has not been built (``python -m
uam_path_planning_b200.build`` or ``__graft_entry__.build()``) importing works, but the first call that
needs it raises, and without a CUDA device ``uam_ctx_create`` fails with UAM_ERR_CUDA.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libuam_b200.so')

UAM_OK = 0
ERRORS = {-1: 'UAM_ERR_INVALID', -2: 'UAM_ERR_CUDA', -3: 'UAM_ERR_NOMEM', -4: 'UAM_ERR_STATE',
          -5: 'UAM_ERR_UNSUPPORTED'}

# Problem.options -> flag bits (include/uam_b200.h)
UAM_LENGTH_SMOOTH = 1 << 0
UAM_PENALTY_SMOOTH = 1 << 1
UAM_OBSTACLE_SMOOTH = 1 << 2
UAM_MAXRATIO_SMOOTH = 1 << 3
UAM_OWN_START = 1 << 4

UAM_EDGE_LINE, UAM_EDGE_ELLIPSE, UAM_EDGE_BOX = 0, 1, 2

# flag bits of uam_sweep_paths_raster / uam_sweep_paths_analytic
UAM_SWEEP_HIT, UAM_SWEEP_OUTSIDE, UAM_SWEEP_INVALID = 1, 2, 4

_vp = C.c_void_p
_i = C.c_int
_i64 = C.c_int64
_d = C.c_double

# name -> (restype, argtypes); every symbol include/uam_b200.h declares
SIGNATURES = {
    'uam_ctx_create': (_i, [_i, C.POINTER(_vp)]),
    'uam_ctx_destroy': (_i, [_vp]),
    'uam_last_error': (C.c_char_p, [_vp]),
    'uam_version': (C.c_char_p, []),
    'uam_launch_count': (_i, [_vp, C.POINTER(C.c_uint64)]),
    'uam_sync': (_i, [_vp]),
    'uam_ctx_set_option': (_i, [_vp, _i, _i64]),
    'uam_ctx_get_stat': (_i, [_vp, _i, C.POINTER(_d)]),
    'uam_map_set_shapes': (_i, [_vp, _vp, _i, _vp, _vp, _vp, _i, _i]),
    'uam_map_set_raster': (_i, [_vp, _vp, _i, _i, _i, _d, _d, _d, _d, _vp]),
    'uam_map_set_raster_device': (_i, [_vp, _vp, _i, _i, _i, _d, _d, _d, _d, _vp, _vp]),
    'uam_make_arc_paths': (_i, [_vp, _vp, _i, _vp, _i64, _vp, _vp]),
    'uam_score_paths_analytic': (_i, [_vp, _vp, _i64, _i, _vp, _i, _i, _vp, _vp, _vp, _vp]),
    'uam_score_paths_analytic_host': (_i, [_vp, _vp, _i64, _i, _vp, _i, _i, _vp, _vp, _vp]),
    'uam_grad_paths_analytic': (_i, [_vp, _vp, _i64, _i, _vp, _i, _i, _vp, _vp, _vp]),
    'uam_analytic_g_len': (_i, [_vp, _i, C.POINTER(_i64)]),
    'uam_score_paths_raster': (_i, [_vp, _vp, _i64, _i, _vp, _i, _i, _d, _vp, _vp, _vp, _vp]),
    'uam_score_paths_raster_host': (_i, [_vp, _vp, _i64, _i, _vp, _i, _i, _d, _vp, _vp]),
    'uam_grad_paths_raster': (_i, [_vp, _vp, _i64, _i, _vp, _i, _i, _d, _vp, _vp, _vp, _vp]),
    'uam_refine_paths_raster': (_i, [_vp, _vp, _i64, _i, _vp, _i, _i, _d, _i, _d, _d, _d, _vp, _vp, _vp, _vp]),
    'uam_refine_paths_raster_swept': (_i, [_vp, _vp, _i64, _i, _vp, _i, _i, _d, _i, _d, _d, _d, _i, _vp, _vp, _vp, _vp,
                                           _vp, _vp]),
    'uam_sweep_paths_raster': (_i, [_vp, _vp, _i64, _i, _vp, _vp, _vp, _vp]),
    'uam_sweep_paths_analytic': (_i, [_vp, _vp, _i64, _i, _vp, _vp, _vp, _vp]),
    'uam_eval_points': (_i, [_vp, _vp, _i64, _vp, _i, _i, _vp, _vp, _vp, _vp]),
    'uam_eval_points_host': (_i, [_vp, _vp, _i64, _vp, _i, _i, _vp, _vp, _vp]),
    'uam_eval_inequalities_host': (_i, [_vp, _vp, _i, _vp, _i64, _vp]),
    'uam_length_of': (_i, [_vp, _vp, _i64, _i, _i, _vp, _i, _vp, _vp]),
    'uam_length_of_host': (_i, [_vp, _vp, _i64, _i, _i, _vp, _i, _vp]),
    'uam_best': (_i, [_vp, _vp, _i, _i64, _i64, _vp, _i, _vp]),
    'uam_best_allreduce': (_i, [_vp, _vp, _i, _i64, _i64, _vp, _vp]),
    'uam_peer_export': (_i, [_vp, _vp]),
    'uam_peer_attach': (_i, [_vp, _i, _i, _vp]),
    'uam_peer_status': (_i, [_vp, C.POINTER(_i)]),
    'uam_make_candidates': (_i, [_vp, _vp, _i64, _i, _d, C.c_uint64, C.c_uint64, _vp, _vp]),
    'uam_score_paths_raster_best': (_i, [_vp, _vp, _i64, _i, _vp, _i, _i, _d, _vp, _vp, _i64, _vp, _vp]),
    'uam_raster_submit_paths_host': (_i, [_vp, _vp, _i64, _i, _vp, _i, _i, _d, _vp, _vp, _vp, _i64, C.POINTER(_i)]),
    'uam_raster_submit_candidates_host': (_i, [_vp, _vp, _i64, _i, _d, C.c_uint64, _vp, _i, _i, _d, _vp, _vp, _vp, _i64,
                                               C.POINTER(_i)]),
    'uam_raster_wait': (_i, [_vp, _i]),
    'uam_dem_mask': (_i, [_vp, _vp, _i64, C.c_float, _vp, _vp]),
    'uam_rasterize_occupancy': (_i, [_vp, _i, _i, _d, _d, _d, _d, _vp, _vp]),
    'uam_rasterize_layers': (_i, [_vp, _i, _i, _d, _d, _d, _d, _d, _vp, _vp]),
    'uam_edt': (_i, [_vp, _vp, _i, _i, _d, _vp, _vp, _vp]),
    'uam_label_components': (_i, [_vp, _vp, _i, _i, _i, _vp, C.POINTER(C.c_int32), _vp]),
    'uam_component_stats': (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _vp]),
    'uam_component_rects': (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _i, _d, _d, _d, _d, _vp, _vp, _vp]),
    'uam_component_submask': (_i, [_vp, _vp, _i, _i, _i, _vp, _i, _i, _i, _vp, _vp]),
    'uam_grid_search': (_i, [_vp, _vp, _vp, _i, _i, _vp, _i, _vp, _vp, _vp]),
    'uam_grid_search_goals': (_i, [_vp, _vp, _vp, _i, _i, _i, _vp, _vp, _i, _vp, _vp, _vp]),
    'uam_grid_extract_paths': (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _i, _i, _vp, _vp, _vp]),
    'uam_grid_search_bands': (_i, [_vp, _vp, _vp, _i, _i, _i, _vp, _i, _vp, _vp, _vp]),
}

_lib = None


class UamError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f'{ERRORS.get(code, code)}: {msg}')
        self.code = code


def load():
    """Load libuam_b200.so and set the prototypes.  Raises if it was not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f'{LIB_PATH} is missing: build it with `python -m uam_path_planning_b200.build` '
                           '(there is no CPU fallback)')
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib
