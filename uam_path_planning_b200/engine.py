"""Engine: one ``uam_ctx`` (one GPU) behind numpy-in / numpy-out and tensor-in / tensor-out calls.

numpy arrays go through the ``*_host`` entry points of the C-ABI (host<->device copies inside the library);
torch CUDA tensors are passed as raw device pointers on torch's current stream (torch is only the allocator).
Nothing here computes on the CPU: without libuam_b200.so or without a CUDA device every call raises.
"""
from __future__ import annotations

import ctypes as C
import operator
from typing import Optional, Sequence

import numpy as np

from . import _lib
from ._lib import UamError


def _np_ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _f64c(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.float64)


def _is_tensor(x) -> bool:
    return type(x).__module__.startswith('torch') and hasattr(x, 'data_ptr')


def _cur_stream(device_index: int):
    import torch
    return C.c_void_p(torch.cuda.current_stream(device_index).cuda_stream)


class Engine:
    def __init__(self, device: Optional[int] = None):
        self._lib = _lib.load()
        if device is None:
            device = 0
            try:
                import torch
                if torch.cuda.is_available():
                    device = torch.cuda.current_device()
            except ImportError:      # torch is optional for the numpy path
                pass
        self.device = int(device)
        h = C.c_void_p()
        rc = self._lib.uam_ctx_create(self.device, C.byref(h))
        if rc != _lib.UAM_OK:
            raise UamError(rc, f'uam_ctx_create(device={self.device}) failed: no usable CUDA device '
                               '(this framework has no CPU fallback)')
        self._h = h
        self.n_regions = 0
        self.n_obstacles = 0
        self.raster_shape = None

    # ---- plumbing -------------------------------------------------------------------------------------
    def close(self):
        if getattr(self, '_h', None):
            self._lib.uam_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != _lib.UAM_OK:
            raise UamError(rc, self._lib.uam_last_error(self._h).decode())

    def launch_count(self) -> int:
        n = C.c_uint64()
        self._check(self._lib.uam_launch_count(self._h, C.byref(n)))
        return int(n.value)

    def sync(self):
        self._check(self._lib.uam_sync(self._h))

    OPTIONS = {'raster_layout': 1, 'integral_variant': 2, 'l2_fetch_granularity': 3, 'time_kernels': 4,
               'combine_layers': 5, 'grid_delta': 6, 'host_chunks': 7, 'host_taper': 8, 'shape_grid': 9, 'rasterizer': 10, 'ccl_tiles': 11, 'grid_graph': 12, 'grid_half_cap': 13}
    STATS = {'score_kernel_ms_mean': 1, 'score_kernel_count': 2, 'grid_activations': 3, 'grid_sweeps': 4, 'grid_rounds': 5,
             'shape_grid_cells': 6, 'shape_grid_items': 7, 'grid_host_submissions': 8}

    def get_stat(self, name: str) -> float:
        v = C.c_double()
        self._check(self._lib.uam_ctx_get_stat(self._h, self.STATS[name], C.byref(v)))
        return float(v.value)

    def set_option(self, name: str, value: int):
        """Tuning knobs of include/uam_b200.h (UAM_OPT_*): raster_layout (0 row-major, 1 tiled; applies to the next
        set_raster), integral_variant (-1 auto, 0 one lane per sample, 1 lane pair, 2 binned, 3 tile-staged), l2_fetch_granularity (32/64/128)."""
        self._check(self._lib.uam_ctx_set_option(self._h, self.OPTIONS[name], int(value)))

    def _tensor_args(self, *tensors):
        import torch
        for t in tensors:
            if t is None:
                continue
            if not t.is_cuda or t.device.index != self.device:
                raise ValueError(f'tensor on {t.device}, engine on cuda:{self.device}')
            if not t.is_contiguous():
                raise ValueError('tensors must be contiguous')
        return _cur_stream(self.device)

    # ---- map ------------------------------------------------------------------------------------------------
    def set_shapes(self, obstacles: Sequence, regions: Sequence[Sequence]):
        from .shapes import flatten_shapes
        edges, off, reg, cen = flatten_shapes(obstacles, regions)
        self._check(self._lib.uam_map_set_shapes(self._h, _np_ptr(edges), edges.shape[0], _np_ptr(off), _np_ptr(reg),
                                                 _np_ptr(cen), reg.shape[0], len(regions)))
        self.n_regions = len(regions)
        self.n_obstacles = len(obstacles)

    def set_raster(self, layers, geo, occupancy=None):
        """layers (L,H,W) float32, geo = (x0, dx, y0, dy), occupancy (H,W) uint8 or None."""
        x0, dx, y0, dy = [float(v) for v in geo]
        if _is_tensor(layers):
            import torch
            assert layers.dtype == torch.float32 and layers.dim() == 3
            assert occupancy is None or (occupancy.dtype == torch.uint8 and tuple(occupancy.shape) == tuple(layers.shape[1:]))
            st = self._tensor_args(layers, occupancy)
            L, H, W = layers.shape
            self._check(self._lib.uam_map_set_raster_device(
                self._h, C.c_void_p(layers.data_ptr()), L, H, W, x0, dx, y0, dy,
                C.c_void_p(occupancy.data_ptr()) if occupancy is not None else None, st))
        else:
            layers = np.ascontiguousarray(layers, dtype=np.float32)
            assert layers.ndim == 3
            L, H, W = layers.shape
            occ = None if occupancy is None else np.ascontiguousarray(occupancy, dtype=np.uint8)
            assert occ is None or occ.shape == (H, W)
            self._check(self._lib.uam_map_set_raster(self._h, _np_ptr(layers), L, H, W, x0, dx, y0, dy, _np_ptr(occ)))
        self.raster_shape = (int(L), int(H), int(W))

    # ---- scoring ---------------------------------------------------------------------------------------------
    def g_len(self, N: int) -> int:
        n = C.c_int64()
        self._check(self._lib.uam_analytic_g_len(self._h, int(N), C.byref(n)))
        return int(n.value)

    def score_analytic(self, Z, N: int, p, flags: int, want_g: bool = False):
        """Z (B, 2(N+2)) float64 -> (cost f64 (B,), collide u8 (B,), g f64 (B, glen) | None)."""
        p = _f64c(p)
        N = int(N)
        if _is_tensor(Z):
            import torch
            assert Z.dtype == torch.float64 and Z.dim() == 2 and Z.shape[1] == 2 * (N + 2)
            st = self._tensor_args(Z)
            B = Z.shape[0]
            cost = torch.empty(B, dtype=torch.float64, device=Z.device)
            col = torch.empty(B, dtype=torch.uint8, device=Z.device)
            g = torch.empty((B, self.g_len(N)), dtype=torch.float64, device=Z.device) if want_g else None
            self._check(self._lib.uam_score_paths_analytic(
                self._h, C.c_void_p(Z.data_ptr()), B, N, _np_ptr(p), p.size, flags, C.c_void_p(cost.data_ptr()),
                C.c_void_p(col.data_ptr()), C.c_void_p(g.data_ptr()) if want_g else None, st))
            return cost, col, g
        Z = _f64c(Z)
        if Z.ndim != 2 or Z.shape[1] != 2 * (N + 2):
            raise ValueError(f'paths must be (B, {2 * (N + 2)}) for N = {N}, got {Z.shape}')
        B = Z.shape[0]
        cost = np.empty(B, dtype=np.float64)
        col = np.empty(B, dtype=np.uint8)
        g = np.empty((B, self.g_len(N)), dtype=np.float64) if want_g else None
        self._check(self._lib.uam_score_paths_analytic_host(self._h, _np_ptr(Z), B, N, _np_ptr(p), p.size, flags,
                                                            _np_ptr(cost), _np_ptr(col), _np_ptr(g)))
        return cost, col, g

    def grad_analytic(self, Z, N: int, p, flags: int):
        """Z (B, 2(N+2)) float64 -> (cost (B,), grad (B, 2(N+2))) of Problem.get_cost; numpy in -> numpy out, CUDA
        tensor in -> CUDA tensors out."""
        import torch
        p = _f64c(p)
        N = int(N)
        host = not _is_tensor(Z)
        if host:
            Z = torch.from_numpy(_f64c(Z)).to(f'cuda:{self.device}')
        assert Z.dtype == torch.float64 and Z.dim() == 2 and Z.shape[1] == 2 * (N + 2)
        st = self._tensor_args(Z)
        cost = torch.empty(Z.shape[0], dtype=torch.float64, device=Z.device)
        grad = torch.empty_like(Z)
        self._check(self._lib.uam_grad_paths_analytic(self._h, C.c_void_p(Z.data_ptr()), Z.shape[0], N, _np_ptr(p), p.size,
                                                      flags, C.c_void_p(cost.data_ptr()), C.c_void_p(grad.data_ptr()), st))
        return (cost.cpu().numpy(), grad.cpu().numpy()) if host else (cost, grad)

    def score_raster(self, Z, N: int, p, flags: int, samples_per_cell: float = 0.0, want_nsamples: bool = False,
                     out=None):
        """Z (B, 2(N+2)) float64 -> (cost f32 (B,), collide u8 (B,)[, nsamples i64 (B,)]).
        `out` = (cost, collide) preallocated buffers of the same kind as Z (optional)."""
        p = _f64c(p)
        N = int(N)
        if _is_tensor(Z):
            import torch
            assert Z.dtype == torch.float64 and Z.dim() == 2 and Z.shape[1] == 2 * (N + 2)
            B = Z.shape[0]
            cost, col = out if out is not None else (torch.empty(B, dtype=torch.float32, device=Z.device),
                                                     torch.empty(B, dtype=torch.uint8, device=Z.device))
            ns = torch.empty(B, dtype=torch.int64, device=Z.device) if want_nsamples else None
            st = self._tensor_args(Z, cost, col)
            self._check(self._lib.uam_score_paths_raster(
                self._h, C.c_void_p(Z.data_ptr()), B, N, _np_ptr(p), p.size, flags, float(samples_per_cell),
                C.c_void_p(cost.data_ptr()), C.c_void_p(col.data_ptr()), C.c_void_p(ns.data_ptr()) if want_nsamples else None,
                st))
            return (cost, col, ns) if want_nsamples else (cost, col)
        if want_nsamples:
            raise ValueError('nsamples is only available on the device-tensor path')
        if not (isinstance(Z, np.ndarray) and Z.dtype == np.float64 and Z.flags.c_contiguous):
            Z = _f64c(Z)
        if Z.ndim != 2 or Z.shape[1] != 2 * (N + 2):
            raise ValueError(f'paths must be (B, {2 * (N + 2)}) for N = {N}, got {Z.shape}')
        B = Z.shape[0]
        cost, col = out if out is not None else (np.empty(B, dtype=np.float32), np.empty(B, dtype=np.uint8))
        self._check(self._lib.uam_score_paths_raster_host(self._h, _np_ptr(Z), B, N, _np_ptr(p), p.size, flags,
                                                          float(samples_per_cell), _np_ptr(cost), _np_ptr(col)))
        return cost, col

    def grad_raster(self, Z, N: int, p, flags: int, samples_per_cell: float = 0.0):
        """Z (B, 2(N+2)) float64 -> (cost f32 (B,), collide u8 (B,), grad f64 (B, 2(N+2))) of the raster cost
        (uam_grad_paths_raster: cost / collide are score_raster's bits); numpy in -> numpy out, CUDA tensor in -> CUDA
        tensors out."""
        import torch
        p = _f64c(p)
        N = int(N)
        host = not _is_tensor(Z)
        if host:
            Z = _f64c(Z)
            if Z.ndim != 2 or Z.shape[1] != 2 * (N + 2):
                raise ValueError(f'paths must be (B, {2 * (N + 2)}) for N = {N}, got {Z.shape}')
            Z = torch.from_numpy(Z).to(f'cuda:{self.device}')
        assert Z.dtype == torch.float64 and Z.dim() == 2 and Z.shape[1] == 2 * (N + 2)
        st = self._tensor_args(Z)
        B = Z.shape[0]
        cost = torch.empty(B, dtype=torch.float32, device=Z.device)
        col = torch.empty(B, dtype=torch.uint8, device=Z.device)
        grad = torch.empty_like(Z)
        self._check(self._lib.uam_grad_paths_raster(self._h, C.c_void_p(Z.data_ptr()), B, N, _np_ptr(p), p.size, flags,
                                                    float(samples_per_cell), C.c_void_p(cost.data_ptr()),
                                                    C.c_void_p(col.data_ptr()), C.c_void_p(grad.data_ptr()), st))
        return (cost.cpu().numpy(), col.cpu().numpy(), grad.cpu().numpy()) if host else (cost, col, grad)

    def refine_raster(self, Z, N: int, p, flags: int, samples_per_cell: float, iterations: int, step_cells: float,
                      max_step_cells: float, min_step_cells: float):
        """Z (B, 2(N+2)) float64 -> (Z_out f64, cost f32 (B,), collide u8 (B,), accepted i32 (B,)) of
        uam_refine_paths_raster; numpy in -> numpy out, CUDA tensor in -> new CUDA tensors out (Z is not modified)."""
        import torch
        p = _f64c(p)
        N = int(N)
        host = not _is_tensor(Z)
        if host:
            Z = _f64c(Z)
            if Z.ndim != 2 or Z.shape[1] != 2 * (N + 2):
                raise ValueError(f'paths must be (B, {2 * (N + 2)}) for N = {N}, got {Z.shape}')
            Zo = torch.from_numpy(Z).to(f'cuda:{self.device}')
        else:
            assert Z.dtype == torch.float64 and Z.dim() == 2 and Z.shape[1] == 2 * (N + 2)
            self._tensor_args(Z)
            Zo = Z.clone()
        st = self._tensor_args(Zo)
        B = Zo.shape[0]
        cost = torch.empty(B, dtype=torch.float32, device=Zo.device)
        col = torch.empty(B, dtype=torch.uint8, device=Zo.device)
        acc = torch.empty(B, dtype=torch.int32, device=Zo.device)
        self._check(self._lib.uam_refine_paths_raster(
            self._h, C.c_void_p(Zo.data_ptr()), B, N, _np_ptr(p), p.size, flags, float(samples_per_cell), int(iterations),
            float(step_cells), float(max_step_cells), float(min_step_cells), C.c_void_p(cost.data_ptr()),
            C.c_void_p(col.data_ptr()), C.c_void_p(acc.data_ptr()), st))
        if host:
            return Zo.cpu().numpy(), cost.cpu().numpy(), col.cpu().numpy(), acc.cpu().numpy()
        return Zo, cost, col, acc

    def refine_raster_swept(self, Z, N: int, p, flags: int, samples_per_cell: float, iterations: int, step_cells: float,
                            max_step_cells: float, min_step_cells: float, min_d2: int = 0, want_d2min: bool = False):
        """Z (B, 2(N+2)) float64 -> (Z_out f64, cost f32 (B,), collide u8 (B,), accepted i32 (B,), sweep flags u8 (B,),
        d2min i32 (B,) | None) of uam_refine_paths_raster_swept; d2min is returned when want_d2min or min_d2 > 0.
        numpy in -> numpy out, CUDA tensor in -> new CUDA tensors out (Z is not modified)."""
        import torch
        p = _f64c(p)
        N = int(N)
        min_d2 = operator.index(min_d2)
        host = not _is_tensor(Z)
        if host:
            Z = _f64c(Z)
            if Z.ndim != 2 or Z.shape[1] != 2 * (N + 2):
                raise ValueError(f'paths must be (B, {2 * (N + 2)}) for N = {N}, got {Z.shape}')
            Zo = torch.from_numpy(Z).to(f'cuda:{self.device}')
        else:
            assert Z.dtype == torch.float64 and Z.dim() == 2 and Z.shape[1] == 2 * (N + 2)
            self._tensor_args(Z)
            Zo = Z.clone()
        st = self._tensor_args(Zo)
        B = Zo.shape[0]
        cost = torch.empty(B, dtype=torch.float32, device=Zo.device)
        col = torch.empty(B, dtype=torch.uint8, device=Zo.device)
        acc = torch.empty(B, dtype=torch.int32, device=Zo.device)
        sflags = torch.empty(B, dtype=torch.uint8, device=Zo.device)
        d2min = torch.empty(B, dtype=torch.int32, device=Zo.device) if want_d2min or min_d2 > 0 else None
        self._check(self._lib.uam_refine_paths_raster_swept(
            self._h, C.c_void_p(Zo.data_ptr()), B, N, _np_ptr(p), p.size, flags, float(samples_per_cell), int(iterations),
            float(step_cells), float(max_step_cells), float(min_step_cells), min_d2, C.c_void_p(cost.data_ptr()),
            C.c_void_p(col.data_ptr()), C.c_void_p(acc.data_ptr()), C.c_void_p(sflags.data_ptr()),
            None if d2min is None else C.c_void_p(d2min.data_ptr()), st))
        out = (Zo, cost, col, acc, sflags, d2min)
        if host:
            return tuple(None if t is None else t.cpu().numpy() for t in out)
        return out

    def sweep_raster(self, Z, N: int, want_first_hit: bool = True, want_d2min: bool = True):
        """Z (B, 2(N+2)) float64 -> (flags u8 (B,), first_hit i32 (B,) | None, d2min i32 (B,) | None) of
        uam_sweep_paths_raster: every cell each segment crosses checked against the raster's occupancy; numpy in -> numpy
        out, CUDA tensor in -> CUDA tensors out."""
        import torch
        N = int(N)
        host = not _is_tensor(Z)
        if host:
            Z = _f64c(Z)
            if Z.ndim != 2 or Z.shape[1] != 2 * (N + 2):
                raise ValueError(f'paths must be (B, {2 * (N + 2)}) for N = {N}, got {Z.shape}')
            Z = torch.from_numpy(Z).to(f'cuda:{self.device}')
        assert Z.dtype == torch.float64 and Z.dim() == 2 and Z.shape[1] == 2 * (N + 2)
        st = self._tensor_args(Z)
        B = Z.shape[0]
        flags = torch.empty(B, dtype=torch.uint8, device=Z.device)
        first = torch.empty(B, dtype=torch.int32, device=Z.device) if want_first_hit else None
        d2min = torch.empty(B, dtype=torch.int32, device=Z.device) if want_d2min else None
        self._check(self._lib.uam_sweep_paths_raster(self._h, C.c_void_p(Z.data_ptr()), B, N, C.c_void_p(flags.data_ptr()),
                                                     C.c_void_p(first.data_ptr()) if want_first_hit else None,
                                                     C.c_void_p(d2min.data_ptr()) if want_d2min else None, st))
        if host:
            return tuple(None if t is None else t.cpu().numpy() for t in (flags, first, d2min))
        return flags, first, d2min

    def sweep_analytic(self, Z, N: int, want_first_hit: bool = True, want_first_obstacle: bool = True):
        """Z (B, 2(N+2)) float64 -> (flags u8 (B,), first_hit i32 (B,) | None, first_obstacle i32 (B,) | None) of
        uam_sweep_paths_analytic: every segment checked against the analytic hard obstacles; numpy in -> numpy out, CUDA
        tensor in -> CUDA tensors out."""
        import torch
        N = int(N)
        host = not _is_tensor(Z)
        if host:
            Z = _f64c(Z)
            if Z.ndim != 2 or Z.shape[1] != 2 * (N + 2):
                raise ValueError(f'paths must be (B, {2 * (N + 2)}) for N = {N}, got {Z.shape}')
            Z = torch.from_numpy(Z).to(f'cuda:{self.device}')
        assert Z.dtype == torch.float64 and Z.dim() == 2 and Z.shape[1] == 2 * (N + 2)
        st = self._tensor_args(Z)
        B = Z.shape[0]
        flags = torch.empty(B, dtype=torch.uint8, device=Z.device)
        first = torch.empty(B, dtype=torch.int32, device=Z.device) if want_first_hit else None
        obst = torch.empty(B, dtype=torch.int32, device=Z.device) if want_first_obstacle else None
        self._check(self._lib.uam_sweep_paths_analytic(self._h, C.c_void_p(Z.data_ptr()), B, N, C.c_void_p(flags.data_ptr()),
                                                       C.c_void_p(first.data_ptr()) if want_first_hit else None,
                                                       C.c_void_p(obst.data_ptr()) if want_first_obstacle else None, st))
        if host:
            return tuple(None if t is None else t.cpu().numpy() for t in (flags, first, obst))
        return flags, first, obst

    def score_raster_best(self, Z, N: int, p, flags: int, samples_per_cell: float, global_offset: int = 0, out=None, key=None):
        """score_raster on a CUDA tensor + the best key of the batch -- of every rank's batch when a peer group is attached
        (attach_peers): the exchange over NVLink peer memory rides in the last kernel of the step.
        -> (cost, collide, key (1,) int64 CUDA tensor)."""
        import torch
        p = _f64c(p)
        N = int(N)
        assert _is_tensor(Z) and Z.dtype == torch.float64 and Z.dim() == 2 and Z.shape[1] == 2 * (N + 2)
        B = Z.shape[0]
        cost, col = out if out is not None else (torch.empty(B, dtype=torch.float32, device=Z.device),
                                                 torch.empty(B, dtype=torch.uint8, device=Z.device))
        if key is None:
            key = torch.empty(1, dtype=torch.int64, device=Z.device)
        st = self._tensor_args(Z, cost, col, key)
        self._check(self._lib.uam_score_paths_raster_best(
            self._h, C.c_void_p(Z.data_ptr()), B, N, _np_ptr(p), p.size, flags, float(samples_per_cell),
            C.c_void_p(cost.data_ptr()), C.c_void_p(col.data_ptr()), int(global_offset), C.c_void_p(key.data_ptr()), st))
        return cost, col, key

    def submit_raster(self, N: int, p, flags: int, samples_per_cell: float, cost, collide, Z=None, candidates=None,
                      jitter_sigma: float = 0.0, seed: int = 0, key=None, global_offset: int = 0) -> int:
        """Asynchronous host-buffer scoring (uam_raster_submit_*): queue one batch and return a ticket for wait_raster.
        Z (B, 2(N+2)) float64 numpy = the caller's waypoints, or candidates (B, 5) float64 numpy {xs, ys, xg, yg,
        displacement} generated on the device.  cost (B,) float32 / collide (B,) uint8 / key (1,) uint64 are numpy arrays
        filled by the time wait_raster(ticket) returns; every buffer must stay alive until then (pin them:
        torch.empty(...).pin_memory().numpy())."""
        p = _f64c(p)
        t = C.c_int(-1)
        for a, dt in ((cost, np.float32), (collide, np.uint8)):
            if a is not None and not (isinstance(a, np.ndarray) and a.dtype == dt and a.flags.c_contiguous):
                raise ValueError('output buffers must be contiguous numpy arrays of float32 / uint8')
        if key is not None and not (isinstance(key, np.ndarray) and key.dtype == np.uint64 and key.size >= 1):
            raise ValueError('key must be a numpy uint64 array')
        if (Z is None) == (candidates is None):
            raise ValueError('give either Z or candidates')
        if Z is not None:
            if not (isinstance(Z, np.ndarray) and Z.dtype == np.float64 and Z.flags.c_contiguous and Z.ndim == 2 and
                    Z.shape[1] == 2 * (int(N) + 2)):
                raise ValueError(f'paths must be a C-contiguous float64 array (B, {2 * (int(N) + 2)})')
            self._check(self._lib.uam_raster_submit_paths_host(
                self._h, _np_ptr(Z), Z.shape[0], int(N), _np_ptr(p), p.size, flags, float(samples_per_cell), _np_ptr(cost),
                _np_ptr(collide), _np_ptr(key), int(global_offset), C.byref(t)))
        else:
            cd = candidates
            if not (isinstance(cd, np.ndarray) and cd.dtype == np.float64 and cd.flags.c_contiguous and cd.ndim == 2 and cd.shape[1] == 5):
                raise ValueError('candidates must be a C-contiguous float64 array (B, 5): xs, ys, xg, yg, displacement')
            self._check(self._lib.uam_raster_submit_candidates_host(
                self._h, _np_ptr(cd), cd.shape[0], int(N), float(jitter_sigma), int(seed), _np_ptr(p), p.size, flags,
                float(samples_per_cell), _np_ptr(cost), _np_ptr(collide), _np_ptr(key), int(global_offset), C.byref(t)))
        return int(t.value)

    def wait_raster(self, ticket: int):
        self._check(self._lib.uam_raster_wait(self._h, int(ticket)))

    def eval_points(self, X, p, flags: int, want=('region', 'obstacle', 'collide')):
        """X (M,2) float64 -> dict(region=(M,R) weighted penalties, obstacle=(M,), collide=(M,) u8)."""
        p = _f64c(p)
        R = self.n_regions
        if _is_tensor(X):
            import torch
            assert X.dtype == torch.float64 and X.dim() == 2 and X.shape[1] == 2
            st = self._tensor_args(X)
            M = X.shape[0]
            out = {}
            if 'region' in want:
                out['region'] = torch.empty((M, R), dtype=torch.float64, device=X.device)
            if 'obstacle' in want:
                out['obstacle'] = torch.empty(M, dtype=torch.float64, device=X.device)
            if 'collide' in want:
                out['collide'] = torch.empty(M, dtype=torch.uint8, device=X.device)
            ptr = lambda k: C.c_void_p(out[k].data_ptr()) if k in out else None
            self._check(self._lib.uam_eval_points(self._h, C.c_void_p(X.data_ptr()), M, _np_ptr(p), p.size, flags,
                                                  ptr('region'), ptr('obstacle'), ptr('collide'), st))
            return out
        X = _f64c(X).reshape(-1, 2)
        M = X.shape[0]
        out = {}
        if 'region' in want:
            out['region'] = np.empty((M, R), dtype=np.float64)
        if 'obstacle' in want:
            out['obstacle'] = np.empty(M, dtype=np.float64)
        if 'collide' in want:
            out['collide'] = np.empty(M, dtype=np.uint8)
        self._check(self._lib.uam_eval_points_host(self._h, _np_ptr(X), M, _np_ptr(p), p.size, flags,
                                                   _np_ptr(out.get('region')), _np_ptr(out.get('obstacle')),
                                                   _np_ptr(out.get('collide'))))
        return out

    def length_of(self, X, N: int, x_start, x_goal, smooth: bool):
        """Problem.length_of for rows X (B, 2M) float64."""
        ends = _f64c(np.concatenate([np.ravel(x_start), np.ravel(x_goal)]))
        assert ends.size == 4
        if _is_tensor(X):
            import torch
            assert X.dtype == torch.float64 and X.dim() == 2 and X.shape[1] % 2 == 0
            st = self._tensor_args(X)
            out = torch.empty(X.shape[0], dtype=torch.float64, device=X.device)
            self._check(self._lib.uam_length_of(self._h, C.c_void_p(X.data_ptr()), X.shape[0], X.shape[1] // 2, int(N),
                                                _np_ptr(ends), int(bool(smooth)), C.c_void_p(out.data_ptr()), st))
            return out
        X = _f64c(X)
        assert X.ndim == 2 and X.shape[1] % 2 == 0
        out = np.empty(X.shape[0], dtype=np.float64)
        self._check(self._lib.uam_length_of_host(self._h, _np_ptr(X), X.shape[0], X.shape[1] // 2, int(N), _np_ptr(ends),
                                                 int(bool(smooth)), _np_ptr(out)))
        return out

    def make_arc_paths(self, x_start, x_goal, N: int, displacements):
        """Solver.create_x_init for a CUDA tensor of displacements -> (B, 2(N+2)) float64 paths incl. start and goal."""
        import torch
        assert _is_tensor(displacements) and displacements.dtype == torch.float64 and displacements.dim() == 1
        st = self._tensor_args(displacements)
        if bool((displacements.abs() > 1).any()):
            raise ValueError(f'abs(displacement) = {float(displacements.abs().max())} must be smaller than 1')
        ends = _f64c(np.concatenate([np.ravel(x_start), np.ravel(x_goal)]))
        Z = torch.empty((displacements.numel(), 2 * (int(N) + 2)), dtype=torch.float64, device=displacements.device)
        self._check(self._lib.uam_make_arc_paths(self._h, _np_ptr(ends), int(N), C.c_void_p(displacements.data_ptr()),
                                                 displacements.numel(), C.c_void_p(Z.data_ptr()), st))
        return Z

    def make_candidates(self, candidates, N: int, jitter_sigma: float = 0.0, seed: int = 0, index0: int = 0):
        """candidates (B, 5) float64 CUDA tensor {xs, ys, xg, yg, displacement} -> (B, 2(N+2)) paths: per-candidate start /
        goal, arc of Solver.create_x_init, N(0, sigma^2) jitter on the interior waypoints from the counter-based generator
        keyed by (seed, index0 + b, waypoint)."""
        import torch
        assert _is_tensor(candidates) and candidates.dtype == torch.float64 and candidates.dim() == 2 and candidates.shape[1] == 5
        st = self._tensor_args(candidates)
        if bool((candidates[:, 4].abs() > 1).any()):
            raise ValueError(f'abs(displacement) = {float(candidates[:, 4].abs().max())} must be smaller than 1')
        Z = torch.empty((candidates.shape[0], 2 * (int(N) + 2)), dtype=torch.float64, device=candidates.device)
        self._check(self._lib.uam_make_candidates(self._h, C.c_void_p(candidates.data_ptr()), candidates.shape[0], int(N),
                                                  float(jitter_sigma), int(seed), int(index0), C.c_void_p(Z.data_ptr()), st))
        return Z

    def best_allreduce(self, cost, global_offset: int = 0, key=None):
        """Engine.best with the cross-rank min built in (uam_best_allreduce): one kernel, exchange over NVLink peer memory
        when a peer group is attached, this rank's key otherwise."""
        import torch
        assert _is_tensor(cost) and cost.dtype in (torch.float32, torch.float64)
        if key is None:
            key = torch.empty(1, dtype=torch.int64, device=cost.device)
        st = self._tensor_args(cost, key)
        self._check(self._lib.uam_best_allreduce(self._h, C.c_void_p(cost.data_ptr()), int(cost.dtype == torch.float64),
                                                 cost.numel(), int(global_offset), C.c_void_p(key.data_ptr()), st))
        return key

    def peer_handle(self) -> bytes:
        """64-byte CUDA IPC handle of this engine's symmetric block (to be all-gathered over the ranks)."""
        buf = C.create_string_buffer(64)
        self._check(self._lib.uam_peer_export(self._h, buf))
        return buf.raw

    def attach_peers(self, rank: int, handles: Sequence[bytes]):
        """Map the symmetric blocks of all ranks (handles in rank order, this rank's own included)."""
        blob = b''.join(handles)
        assert len(blob) == 64 * len(handles)
        self._check(self._lib.uam_peer_attach(self._h, int(rank), len(handles), C.c_char_p(blob)))

    def peer_timed_out(self) -> bool:
        v = C.c_int(0)
        self._check(self._lib.uam_peer_status(self._h, C.byref(v)))
        return bool(v.value)

    def best(self, cost, global_offset: int = 0, key=None):
        """min over b of key(cost[b], global_offset + b) as a 1-element int64 CUDA tensor; the key (distributed.py) orders
        like (cost, index) for every float value and is a non-negative int64; an empty batch gives KEY_EMPTY."""
        import torch
        assert _is_tensor(cost) and cost.dtype in (torch.float32, torch.float64)
        reset = key is None
        if key is None:
            key = torch.empty(1, dtype=torch.int64, device=cost.device)
        st = self._tensor_args(cost, key)
        self._check(self._lib.uam_best(self._h, C.c_void_p(cost.data_ptr()), int(cost.dtype == torch.float64),
                                       cost.numel(), int(global_offset), C.c_void_p(key.data_ptr()), int(reset), st))
        return key

    # ---- map rebuild ---------------------------------------------------------------------------------------------
    def dem_mask(self, image, threshold: float = 0.0):
        """image > threshold (image == -9999 when threshold == -9999) on a float32 CUDA tensor -> uint8."""
        import torch
        assert _is_tensor(image) and image.dtype == torch.float32
        st = self._tensor_args(image)
        mask = torch.empty(image.shape, dtype=torch.uint8, device=image.device)
        self._check(self._lib.uam_dem_mask(self._h, C.c_void_p(image.data_ptr()), image.numel(), float(threshold),
                                           C.c_void_p(mask.data_ptr()), st))
        return mask

    def rasterize_occupancy(self, H: int, W: int, geo):
        import torch
        x0, dx, y0, dy = [float(v) for v in geo]
        occ = torch.empty((H, W), dtype=torch.uint8, device=f'cuda:{self.device}')
        self._check(self._lib.uam_rasterize_occupancy(self._h, H, W, x0, dx, y0, dy, C.c_void_p(occ.data_ptr()),
                                                      _cur_stream(self.device)))
        return occ

    def rasterize_layers(self, H: int, W: int, geo, enlargement: float = 0.0):
        import torch
        x0, dx, y0, dy = [float(v) for v in geo]
        lay = torch.empty((self.n_regions, H, W), dtype=torch.float32, device=f'cuda:{self.device}')
        self._check(self._lib.uam_rasterize_layers(self._h, H, W, x0, dx, y0, dy, float(enlargement),
                                                   C.c_void_p(lay.data_ptr()), _cur_stream(self.device)))
        return lay

    def edt(self, occ, cell: float = 1.0, want_clearance: bool = True):
        """Exact squared distance (cells, int32) to the nearest occupied cell + clearance = sqrt(d2)*cell."""
        import torch
        assert _is_tensor(occ) and occ.dtype == torch.uint8 and occ.dim() == 2
        st = self._tensor_args(occ)
        H, W = occ.shape
        d2 = torch.empty((H, W), dtype=torch.int32, device=occ.device)
        cl = torch.empty((H, W), dtype=torch.float32, device=occ.device) if want_clearance else None
        self._check(self._lib.uam_edt(self._h, C.c_void_p(occ.data_ptr()), H, W, float(cell), C.c_void_p(d2.data_ptr()),
                                      C.c_void_p(cl.data_ptr()) if cl is not None else None, st))
        return d2, cl

    # ---- polygon front-end (map_generation: mask -> connected regions -> minimum-area rectangles) -------------
    def label_components(self, mask, connectivity: int = 4):
        """mask (H,W) uint8 CUDA tensor -> (labels (H,W) int32, n): 0 = background, components 1..n in raster-scan order
        of their first cell (scipy.ndimage.label's numbering)."""
        import torch
        assert _is_tensor(mask) and mask.dtype == torch.uint8 and mask.dim() == 2
        st = self._tensor_args(mask)
        H, W = mask.shape
        labels = torch.empty((H, W), dtype=torch.int32, device=mask.device)
        n = C.c_int32(0)
        self._check(self._lib.uam_label_components(self._h, C.c_void_p(mask.data_ptr()), H, W, int(connectivity),
                                                   C.c_void_p(labels.data_ptr()), C.byref(n), st))
        return labels, int(n.value)

    def component_stats(self, labels, n: int):
        """labels (H,W) int32 -> (area (n,) int64 cells per component, bbox (n,4) int32 {row min, row max, col min, col max})."""
        import torch
        assert _is_tensor(labels) and labels.dtype == torch.int32 and labels.dim() == 2
        st = self._tensor_args(labels)
        H, W = labels.shape
        area = torch.empty(n, dtype=torch.int64, device=labels.device)
        bbox = torch.empty((n, 4), dtype=torch.int32, device=labels.device)
        self._check(self._lib.uam_component_stats(self._h, C.c_void_p(labels.data_ptr()), H, W, int(n),
                                                  C.c_void_p(area.data_ptr()), C.c_void_p(bbox.data_ptr()), st))
        return area, bbox

    def component_rects(self, labels, n: int, bbox, ids, geo, want_info: bool = False):
        """Minimum-area enclosing rectangle of the cell corners of the components `ids` (K distinct labels) -> (K,4,2)
        float64 world coordinates, corners consecutive around the rectangle."""
        import torch
        assert _is_tensor(labels) and labels.dtype == torch.int32 and labels.dim() == 2
        ids = torch.as_tensor(ids, dtype=torch.int32, device=labels.device).reshape(-1).contiguous()
        st = self._tensor_args(labels, bbox, ids)
        H, W = labels.shape
        K = ids.numel()
        x0, dx, y0, dy = [float(v) for v in geo]
        rect = torch.empty((K, 4, 2), dtype=torch.float64, device=labels.device)
        info = torch.empty((K, 2), dtype=torch.int32, device=labels.device) if want_info else None
        self._check(self._lib.uam_component_rects(self._h, C.c_void_p(labels.data_ptr()), H, W, int(n), C.c_void_p(bbox.data_ptr()),
                                                  C.c_void_p(ids.data_ptr()), K, x0, dx, y0, dy, C.c_void_p(rect.data_ptr()),
                                                  C.c_void_p(info.data_ptr()) if info is not None else None, st))
        return (rect, info) if want_info else rect

    def component_submask(self, labels, label: int, bbox, divisions: int, box_row: int, box_col: int):
        """Mask of one box of the large-polygon split (data_processor.py:34-53) on the grid refined `divisions` times:
        (nr, nc) uint8 CUDA tensor, nr / nc = extents of bbox = (row min, row max, col min, col max) in cells."""
        import torch
        assert _is_tensor(labels) and labels.dtype == torch.int32 and labels.dim() == 2
        st = self._tensor_args(labels)
        bb = np.ascontiguousarray(bbox, dtype=np.int32).reshape(4)
        nr, nc = int(bb[1] - bb[0] + 1), int(bb[3] - bb[2] + 1)
        mask = torch.empty((nr, nc), dtype=torch.uint8, device=labels.device)
        self._check(self._lib.uam_component_submask(self._h, C.c_void_p(labels.data_ptr()), labels.shape[0], labels.shape[1], int(label),
                                                    _np_ptr(bb), int(divisions), int(box_row), int(box_col), C.c_void_p(mask.data_ptr()), st))
        return mask

    def grid_search(self, cost, sources, blocked=None, want_parent: bool = True, goals=None):
        """Q cost-to-go sweeps on an 8-connected grid (build-defined extension, include/uam_b200.h).
        2-D: cost (H,W) uint16 CUDA tensor, sources (Q,2) int32 (row, col), blocked (H,W) uint8 or None ->
        (dist (Q,H,W) int64 with 2**62 = unreachable, parent (Q,H,W) int32 | None).
        Altitude bands: cost (bands,H,W), sources (Q,3) (band, row, col), blocked (bands,H,W) ->
        dist / parent (Q,bands,H,W), parent = flat index into (bands,H,W).
        goals (same layout as sources): start/goal queries -- each query stops once its goal's distance is final; dist /
        parent are then exact for the goal and every node closer to the source than the goal."""
        import torch
        assert _is_tensor(cost) and cost.dtype == torch.uint16 and cost.dim() in (2, 3)
        k = cost.dim()
        sources = torch.as_tensor(sources, dtype=torch.int32, device=cost.device).reshape(-1, k).contiguous()
        if blocked is not None:
            assert blocked.shape == cost.shape and blocked.dtype == torch.uint8
        st = self._tensor_args(cost, sources, blocked)
        Q = sources.shape[0]
        dist = torch.empty((Q,) + tuple(cost.shape), dtype=torch.int64, device=cost.device)
        parent = torch.empty((Q,) + tuple(cost.shape), dtype=torch.int32, device=cost.device) if want_parent else None
        pb = C.c_void_p(blocked.data_ptr()) if blocked is not None else None
        pp = C.c_void_p(parent.data_ptr()) if parent is not None else None
        if goals is not None:
            goals = torch.as_tensor(goals, dtype=torch.int32, device=cost.device).reshape(-1, k).contiguous()
            assert goals.shape == sources.shape
            Bn, (H, W) = (1 if k == 2 else cost.shape[0]), cost.shape[-2:]
            s3, g3 = self._with_band(sources), self._with_band(goals)
            self._check(self._lib.uam_grid_search_goals(self._h, C.c_void_p(cost.data_ptr()), pb, Bn, H, W, C.c_void_p(s3.data_ptr()),
                                                        C.c_void_p(g3.data_ptr()), Q, C.c_void_p(dist.data_ptr()), pp, st))
        elif k == 2:
            H, W = cost.shape
            self._check(self._lib.uam_grid_search(self._h, C.c_void_p(cost.data_ptr()), pb, H, W,
                                                  C.c_void_p(sources.data_ptr()), Q, C.c_void_p(dist.data_ptr()), pp, st))
        else:
            Bn, H, W = cost.shape
            self._check(self._lib.uam_grid_search_bands(self._h, C.c_void_p(cost.data_ptr()), pb, Bn, H, W,
                                                        C.c_void_p(sources.data_ptr()), Q, C.c_void_p(dist.data_ptr()), pp, st))
        return dist, parent

    @staticmethod
    def _with_band(rc):
        """(Q,2) (row, col) -> (Q,3) (0, row, col); (Q,3) unchanged."""
        import torch
        if rc.shape[1] == 3:
            return rc
        return torch.cat([torch.zeros((rc.shape[0], 1), dtype=torch.int32, device=rc.device), rc], dim=1).contiguous()

    def grid_paths(self, parent, sources, goals, max_len: Optional[int] = None):
        """Paths of start/goal queries from the predecessor field of grid_search: (path (Q,max_len) int32 flat node ids
        from the source to the goal, length (Q,) int32: nodes on the path, 0 = goal not reached, -k = needs k > max_len)."""
        import torch
        assert _is_tensor(parent) and parent.dtype == torch.int32 and parent.dim() in (3, 4)
        k = parent.dim() - 1
        Q = parent.shape[0]
        Bn, (H, W) = (1 if k == 2 else parent.shape[1]), parent.shape[-2:]
        s3 = self._with_band(torch.as_tensor(sources, dtype=torch.int32, device=parent.device).reshape(-1, k).contiguous())
        g3 = self._with_band(torch.as_tensor(goals, dtype=torch.int32, device=parent.device).reshape(-1, k).contiguous())
        assert s3.shape[0] == Q and g3.shape[0] == Q
        max_len = int(max_len) if max_len is not None else 4 * (H + W) + 2 * Bn
        st = self._tensor_args(parent, s3, g3)
        path = torch.full((Q, max_len), -1, dtype=torch.int32, device=parent.device)
        length = torch.empty(Q, dtype=torch.int32, device=parent.device)
        self._check(self._lib.uam_grid_extract_paths(self._h, C.c_void_p(parent.data_ptr()), Bn, H, W, C.c_void_p(s3.data_ptr()),
                                                     C.c_void_p(g3.data_ptr()), Q, max_len, C.c_void_p(path.data_ptr()),
                                                     C.c_void_p(length.data_ptr()), st))
        return path, length

    def grid_routes(self, cost, sources, goals, blocked=None, chunk: int = 16, max_len: Optional[int] = None):
        """Start/goal queries with bounded memory: the queries run `chunk` at a time through grid_search(goals=...) +
        grid_paths, the (chunk, bands, H, W) distance / predecessor fields are reused from chunk to chunk, and only what a
        planner keeps comes back: (goal_dist (Q,) int64 with 2**62 = unreachable, path (Q, max_len) int32 flat node ids
        source -> goal, length (Q,) int32).  1024 queries on 4096^2 x 8 bands need 26 GB this way instead of 1.6 TB."""
        import torch
        k = cost.dim()
        sources = torch.as_tensor(sources, dtype=torch.int32, device=cost.device).reshape(-1, k).contiguous()
        goals = torch.as_tensor(goals, dtype=torch.int32, device=cost.device).reshape(-1, k).contiguous()
        Q = sources.shape[0]
        Bn, (H, W) = (1 if k == 2 else cost.shape[0]), cost.shape[-2:]
        max_len = int(max_len) if max_len is not None else 4 * (H + W) + 2 * Bn
        gd = torch.empty(Q, dtype=torch.int64, device=cost.device)
        path = torch.empty((Q, max_len), dtype=torch.int32, device=cost.device)
        length = torch.empty(Q, dtype=torch.int32, device=cost.device)
        for q0 in range(0, Q, int(chunk)):
            q1 = min(Q, q0 + int(chunk))
            dist, parent = self.grid_search(cost, sources[q0:q1], blocked, True, goals[q0:q1])
            g = goals[q0:q1].long()
            inside = ((g >= 0) & (g < torch.tensor(cost.shape, device=cost.device))).all(dim=1)
            gc = g.clamp(min=0)
            gc = torch.minimum(gc, torch.tensor(cost.shape, device=cost.device) - 1)
            d = dist[(torch.arange(q1 - q0, device=cost.device),) + tuple(gc[:, c] for c in range(k))]
            gd[q0:q1] = torch.where(inside, d, torch.full_like(d, 2 ** 62))
            path[q0:q1], length[q0:q1] = self.grid_paths(parent, sources[q0:q1], goals[q0:q1], max_len)
            del dist, parent
        return gd, path, length

    # ---- single-shape queries (QuadraticObstacle.contains / penalty_function, Function.__call__) -----------------
    def _scratch(self) -> 'Engine':
        if getattr(self, '_scratch_engine', None) is None:
            self._scratch_engine = Engine(self.device)
        return self._scratch_engine

    def eval_single_shape(self, shape, x, want: str, smooth: bool = True, enlargement: float = 0.0):
        """contains -> bool array; psi -> unnormalised penalty prod_i min(h_i - e, 0)^2 (or the non-smooth form)."""
        from .shapes import QuadraticObstacle
        X = _f64c(x).reshape(-1, 2)
        eng = self._scratch()
        bare = QuadraticObstacle(*shape.inequalities)     # center = NaN -> no normalisation (problem.py:76-77)
        p = np.array([0, 0, 0, 0, 1.0, 0.0, float(enlargement), 1.0])
        if want == 'contains':
            eng.set_shapes([bare], [[]])
            return eng.eval_points(X, p, 0, want=('collide',))['collide'].astype(bool)
        eng.set_shapes([], [[bare]])
        flags = _lib.UAM_PENALTY_SMOOTH if smooth else 0
        return eng.eval_points(X, p, flags, want=('region',))['region'][:, 0]

    def eval_inequalities(self, records, x) -> np.ndarray:
        """h_i(x_m) for raw inequality records (n,8) at points (M,2) -> (n, M) float64 (Function.__call__)."""
        R = _f64c(records).reshape(-1, 8)
        X = _f64c(x).reshape(-1, 2)
        out = np.empty((R.shape[0], X.shape[0]), dtype=np.float64)
        self._check(self._lib.uam_eval_inequalities_host(self._h, _np_ptr(R), R.shape[0], _np_ptr(X), X.shape[0],
                                                         _np_ptr(out)))
        return out


_default: Optional[Engine] = None


def default_engine() -> Engine:
    global _default
    if _default is None:
        _default = Engine()
    return _default
