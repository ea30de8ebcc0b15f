#!/usr/bin/env python
"""bench.py -- candidate-path segment evaluations / s (cost + collision) on an 8192^2 multi-layer raster.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json configs[2], SURVEY.md 8d "C3"): synthetic 8192^2 raster with L = 3 float32 cost layers
(fractal terrain with the real DEM's statistics, building heights, noise field) + uint8 occupancy, and candidate
paths of 64 waypoints (N = 62) from the "scatter" distribution: every candidate is an independent start/goal query
(start, goal uniform in the raster, straight line) whose 62 interior waypoints carry N(0, 2 cells) jitter -- generated on
the device from 40-byte candidate rows {xs, ys, xg, yg, displacement} by the batched Solver.create_x_init
(uam_make_candidates), the reference's own flow (main.py:160-171: displacement -> create_x_init -> score).  One step =
one pass of the raster path scorer over this rank's batch in integral mode (samples_per_cell = 1: every segment is sampled
once per cell it crosses) INCLUDING the best-path reduction: the last kernel of the step finds the local argmin and, when
N > 1, exchanges the 8-byte key with the other ranks through NVLink peer memory (uam_score_paths_raster_best; `--reduce
nccl` uses an NCCL all-reduce of the key instead).  Paths shard over the ranks, the map is replicated; per-GPU work is
fixed (weak scaling).  `value` counts segment evaluations (63 per path).

Timing: device-resident inputs, CUDA events on the launching stream, barrier + synchronize on both sides, max over
ranks.  The raster (1 GiB of texels) and the path batch (1 KiB per path) are both larger than L2, so no explicit L2
flush is needed between steps.  `e2e` times the same paths through the host-buffer entry points of the C-ABI with all
copies inside the timed region: the candidate rows go up (40 B per path), costs + flags + key come back
(uam_raster_submit_candidates_host / uam_raster_wait); `e2e_host_waypoints` uploads the same paths as 1 KiB of float64
waypoints each instead (uam_raster_submit_paths_host).  `cpu_baseline` / `--impl reference` time the oracle (oracle/ --
the CPU restatement of the path; the reference itself has no raster path and cannot be installed: it needs
casadi/opengen/cargo): its C/OpenMP form on every host core, and its numpy form on one core.  `configs` carries short
runs of the other BASELINE.json configs (C2 / C4 / C5, bench_configs.py), each with its own roofline / CPU / parity figures.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark leaves the tree as it found it (no __pycache__ of the modules it imports)

RASTER = 8192
WP = 64                 # waypoints per path (N = 62 free + start + goal)
KM = 64.0               # raster spans 64 km
WEIGHTS = [200.0, 15000.0, 27000.0]       # path_generation/main.py:145
SPC = 1.0               # samples per cell (integral mode)
METRIC = 'candidate-path segment evaluations/s (cost+collision), 8192^2 3-layer raster, integral mode'


# ---------------------------------------------------------------------------------------------------------------
# synthetic workload (SURVEY.md 8d, C3)
# ---------------------------------------------------------------------------------------------------------------
def make_raster(torch, device, n=RASTER, seed=20260102):
    """(layers (3,n,n) f32, occupancy (n,n) u8, geo).  Same seed -> same map on every rank (map replicated)."""
    g = torch.Generator(device=device).manual_seed(seed)
    # terrain: 1/f^2 fractal, rescaled to the DEM statistics of merge_test.tif.aux.xml (min -12, max 557.5), 47 % sea
    f = torch.fft.fftfreq(n, device=device)
    k2 = f[:, None] ** 2 + f[None, :] ** 2
    k2[0, 0] = 1.0
    spec = torch.randn((n, n), device=device, generator=g, dtype=torch.float32) + 1j * torch.randn(
        (n, n), device=device, generator=g, dtype=torch.float32)
    t = torch.fft.ifft2(spec / k2).real
    del spec, k2
    q = torch.quantile(t.flatten()[:: max(1, t.numel() // (1 << 22))], 0.47)
    t = t - q
    land = t > 0
    terrain = torch.where(land, -12.0 + t / t.max() * 569.5, torch.zeros_like(t)).clamp_(min=0.0)
    # building height: random axis-aligned footprints x U(5,150) m
    bld = torch.zeros((n, n), device=device)
    R = torch.rand((4096, 5), generator=g, device=device).cpu().numpy()
    for r in R:
        i0, j0 = int(r[0] * (n - 64)), int(r[1] * (n - 64))
        bld[i0:i0 + 8 + int(r[2] * 56), j0:j0 + 8 + int(r[3] * 56)] = 5.0 + 145.0 * float(r[4])
    bld = bld * land
    # noise: 64 Gaussian sources (separable -> one rank-64 product)
    S = torch.rand((64, 4), generator=g, device=device)
    ax = torch.arange(n, device=device, dtype=torch.float32)[None, :]
    sig = (50.0 + 400.0 * S[:, 2:3]) * (n / 8192.0)
    gx = torch.exp(-(ax - S[:, 0:1] * n) ** 2 / (2 * sig ** 2))
    gy = torch.exp(-(ax - S[:, 1:2] * n) ** 2 / (2 * sig ** 2)) * (40.0 + 40.0 * S[:, 3:4])
    noise = gy.t() @ gx
    # normalise each layer to O(1) so the three weighted terms are comparable
    layers = torch.stack([terrain / 557.5, bld / 150.0, noise / noise.max()]).contiguous()
    occ = ((terrain + bld) > 300.0).to(torch.uint8)          # altitude band at 300 m
    dx = KM / n
    return layers, occ, (0.0, dx, 0.0, dx)


def make_paths(torch, device, B, seed, n=RASTER):
    """Scatter distribution: start/goal uniform in the raster, straight line + N(0, 2 cells) jitter."""
    g = torch.Generator(device=device).manual_seed(seed)
    cell = KM / n
    s = torch.rand((B, 1, 2), device=device, generator=g, dtype=torch.float64) * KM
    e = torch.rand((B, 1, 2), device=device, generator=g, dtype=torch.float64) * KM
    t = torch.linspace(0, 1, WP, device=device, dtype=torch.float64).reshape(1, WP, 1)
    Z = s + t * (e - s)
    Z = Z + torch.randn((B, WP, 2), device=device, generator=g, dtype=torch.float64) * (2.0 * cell)
    return Z.reshape(B, 2 * WP).contiguous()


def make_candidates_host(B, seed, n=RASTER):
    """(B, 5) float64 candidate rows {xs, ys, xg, yg, displacement = 0}: start / goal uniform in the raster (scatter)."""
    rng = np.random.default_rng(seed)
    cand = np.zeros((B, 5), dtype=np.float64)
    cand[:, :4] = rng.random((B, 4)) * KM
    return cand


JITTER_CELLS = 2.0      # sigma of the waypoint jitter in cells (SURVEY 8d: N(0, 2 cells))
JITTER_SEED = 20260103


def algorithmic_bytes(total_samples, B, L=3):
    """SURVEY.md 8(d): per segment 16 B (one new float64 waypoint) + S * (L * 4 texels * 4 B + 1 B occupancy),
    + per path 16 B (first point) + 5 B (float32 cost + uint8 flag).  total_samples includes the goal sample."""
    return (WP - 1) * B * 16 + total_samples * (L * 16 + 1) + B * (16 + 5)


# ---------------------------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock + throttle reasons while the timed loops run: NVML polled in-process every ~2 ms (a 40 ms timed region gets
    ~20 samples), `nvidia-smi -lms 10` when NVML is not importable."""
    Q = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')
    NAMES = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']

    def __init__(self, index):
        self.index, self.rows, self.proc, self.th, self.stop_flag, self.mode = index, [], None, None, False, None
        self.windows = []

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            mx = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            bits = [pynvml.nvmlClocksEventReasonHwSlowdown, pynvml.nvmlClocksEventReasonHwThermalSlowdown,
                    pynvml.nvmlClocksEventReasonSwThermalSlowdown, pynvml.nvmlClocksEventReasonSwPowerCap]

            def poll():
                while not self.stop_flag:
                    try:
                        r = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h)
                        self.rows.append([float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)), mx] +
                                         [bool(r & b) for b in bits] + [time.time()])
                    except Exception:
                        pass
                    time.sleep(0.002)
            self.mode = 'nvml 2 ms'
            self.th = threading.Thread(target=poll, daemon=True)
            self.th.start()
            return
        except Exception:
            pass
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--id={self.index}', f'--query-gpu={self.Q}',
                                          '--format=csv,noheader,nounits', '-lms', '10'], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.mode = 'nvidia-smi -lms 10'
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            c = [x.strip() for x in line.split(',')]
            if len(c) >= 6 and c[0].replace('.', '').isdigit():
                self.rows.append([float(c[0]), float(c[1])] + [x.lower().startswith('active') for x in c[2:6]] + [time.time()])

    def window(self, t0, t1):
        """a timed region: only samples taken inside the windows are kept (all of them if none fell inside)"""
        self.windows.append((t0, t1))

    def stop(self):
        if not self.th:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['no clock source (NVML and nvidia-smi unavailable)']}
        time.sleep(0.03)
        self.stop_flag = True
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()
        rows = list(self.rows)
        inside = [r for r in rows if any(a <= r[-1] <= b + 0.005 for a, b in self.windows)]
        main = [r for r in rows if self.windows and self.windows[0][0] <= r[-1] <= self.windows[0][1] + 0.005]
        rows = inside or rows
        sm = [r[0] for r in rows]
        reasons = [nm for i, nm in enumerate(self.NAMES) if any(r[2 + i] for r in rows)]
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_min_mhz': min(sm) if sm else None,
                'sm_max_mhz': max(r[1] for r in rows) if rows else None, 'reasons': reasons, 'samples': len(sm),
                'samples_in_device_timed_loop': len(main), 'source': self.mode,
                'note': 'samples taken inside the timed regions (device-resident loop + e2e loops)'}


# ---------------------------------------------------------------------------------------------------------------
# CPU arm: the oracle (oracle/ -- CPU restatement of the path; the reference itself is Python + CasADi/OpEn and cannot
# be installed here) on a bounded sample.  Two forms: the C / OpenMP restatement on every host core (the baseline that
# is reported) and the float64 numpy restatement on one core (what a direct port of the reference's Python gives).
# ---------------------------------------------------------------------------------------------------------------
def cpu_c_rate(layers, occ, geo, Z, threads=0):
    """segments/s of oracle/uam_oracle_c (C, OpenMP over paths) -> (rate, seconds, threads, (cost, collide, nsamples))."""
    from oracle import uam_oracle_c as occ_c
    th = threads or (os.cpu_count() or 1)
    t0 = time.perf_counter()
    res = occ_c.score_paths_raster(layers, occ, geo, Z, WEIGHTS, SPC, True, None, threads=th)
    dt = time.perf_counter() - t0
    return Z.shape[0] * (WP - 1) / dt, dt, th, res


def cpu_numpy_rate(layers, occ, geo, Z):
    from oracle import uam_oracle as orc
    t0 = time.perf_counter()
    res = orc.score_paths_raster(layers, occ, geo, Z, WEIGHTS, SPC, True, None)
    dt = time.perf_counter() - t0
    return Z.shape[0] * (WP - 1) / dt, dt, res


def host_paths(B, seed, n=RASTER):
    """the workload's paths made on the host by the oracle's restatement of the candidate generator (CPU arm)"""
    from oracle import uam_oracle as orc
    return orc.make_candidates(make_candidates_host(B, seed, n), WP - 2, JITTER_CELLS * KM / n, JITTER_SEED, 0)


def run_reference(args):
    """--impl reference: the CPU implementation of the path on all host cores.  Rank 0 only."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    import torch
    cores = os.cpu_count() or 1
    n = args.raster
    torch.manual_seed(0)
    layers, occ, geo = make_raster(torch, 'cpu', n)
    layers, occ = layers.numpy(), occ.numpy()
    # a step = a bounded sample of the workload: the whole per-GPU batch when few steps are asked for (the driver's 20 + 5),
    # fewer paths per step for long runs, so that the run stays at about a minute of CPU work (the rate does not depend on
    # the sample size)
    per_step = args.paths if args.steps + args.warmup <= 30 else max(2000, args.paths * 25 // (args.steps + args.warmup))
    Z = host_paths(per_step, 2000, n)                # rank 0's batch of the GPU arm (same seed)
    times = []
    for s in range(args.warmup + args.steps):
        rate, dt, th, res = cpu_c_rate(layers, occ, geo, Z, cores)
        if s >= args.warmup:
            times.append(dt)
    if args.dump_outputs:
        c, k, _ = res
        i = int(np.argmin(c))
        dump_outputs(args.dump_outputs, torch.from_numpy(c), torch.from_numpy(k), float(c[i]), i)
    T = float(np.sum(times))
    value = per_step * (WP - 1) * args.steps / T
    line = {'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': 'segment-evals/s', 'n_gpus': args.gpus,
            'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * T / args.steps, 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
            'config': workload_config(args),
            'cpu_baseline': {'value': value, 'unit': 'segment-evals/s', 'cores': cores, 'kind': 'port',
                             'sample': f'{per_step} paths per step of the same workload (rank 0\'s batch), oracle/uam_oracle_c.c (C '
                                       f'restatement of the float64 oracle, OpenMP over paths, {cores} threads), integral mode'},
            'e2e': {'value': value, 'unit': 'segment-evals/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'gpu_launches': 0}
    print(json.dumps(line))


def analytic_c1(torch, dev, args, B=100000, n_cpu=2000, with_cpu=True):
    import uam_path_planning_b200 as uam
    sys.path.insert(0, os.path.join(ROOT, 'tests'))
    from conftest import build_product_problem
    spec = json.load(open(os.path.join(ROOT, 'tests', 'golden', 'fixture_main_map.json')))
    N = 80
    prob = build_product_problem(spec, N)
    sol = uam.Solver(prob, {})
    g = torch.Generator(device=dev).manual_seed(7)
    d = torch.rand(B, device=dev, generator=g, dtype=torch.float64) * 1.8 - 0.9
    Z = sol.candidates_device(d)
    Z[:, 2:-2] += torch.randn((B, 2 * N), device=dev, generator=g, dtype=torch.float64) * 0.05
    for _ in range(3):
        cost, col, _ = prob.score(Z)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(10):
        cost, col, _ = prob.score(Z)
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / 10
    out = {'workload': f'C1: Problem.get_cost + collides on the main.py map ({len(prob.map.obstacles)} obstacles, '
                       f'{sum(len(r) for r in prob.map._region_lists())} region shapes), N = {N}, {B} arc candidates + jitter',
           'ms_per_batch': ms, 'paths_per_s': B / (ms * 1e-3), 'value': B * (N + 1) / (ms * 1e-3), 'unit': 'segment-evals/s',
           'dtype': 'f64', 'collisions': int(col.sum().item())}
    if not args.no_cpu and with_cpu:
        from oracle import uam_oracle as orc
        om = orc.OMap(spec)
        Zh = Z[:n_cpu].cpu().numpy()
        t0 = time.perf_counter()
        c_ref = orc.get_cost(om, Zh, N, spec['weights'], spec['enlargement'], spec['options'])
        k_ref = orc.path_collides(om, Zh, N)
        dt = time.perf_counter() - t0
        out['cpu_numpy_1core'] = {'paths': n_cpu, 'seconds': dt, 'paths_per_s': n_cpu / dt,
                                  'max_rel_err_gpu_vs_oracle': float(np.max(np.abs(cost[:n_cpu].cpu().numpy() - c_ref) / np.abs(c_ref))),
                                  'collide_equal': bool(np.array_equal(col[:n_cpu].cpu().numpy().astype(bool), k_ref))}
    return out


def workload_config(args):
    """the same dict on both arms (the CPU arm's bounded sample is described in its cpu_baseline.sample)"""
    return {'workload': f'C3: {args.raster}^2 raster, L=3 float32 layers + uint8 occupancy, scatter candidates (independent '
                        f'start/goal queries, straight line + N(0, {JITTER_CELLS:g} cells) jitter) x {WP} waypoints, integral mode '
                        f'samples_per_cell={SPC}',
            'raster': args.raster, 'layers': 3, 'waypoints': WP, 'paths_per_gpu_per_step': args.paths,
            'samples_per_cell': SPC, 'sharding': 'paths sharded contiguously over ranks, map replicated',
            'l2': 'inputs larger than L2 (texels 1 GiB, paths 1 KiB each); no explicit flush'}


DUMP_MAX_PATHS = 1 << 22         # 2 x 16 MiB of float32 per-path outputs at most; larger batches are sampled
DUMP_SEED = 20260104


def dump_outputs(out_dir, cost, col, best_cost, best_idx):
    """--dump-outputs: what the caller of the timed step receives (RasterMap.score_paths_best), as .npy files, so that two
    builds can be compared output for output.  The inputs are seeded, so the same arguments give the same inputs.
    cost.npy (B,) f32, collide.npy (B,) f32 0 / 1, best_cost.npy / best_index.npy (1,) f64 (the decoded best key).
    Batches of more than DUMP_MAX_PATHS paths keep a fixed seeded sample of the rows, listed in path_index.npy."""
    os.makedirs(out_dir, exist_ok=True)
    c = cost.cpu().numpy().astype(np.float32)
    k = col.cpu().numpy().astype(np.float32)
    if c.size > DUMP_MAX_PATHS:
        idx = np.sort(np.random.default_rng(DUMP_SEED).choice(c.size, DUMP_MAX_PATHS, replace=False))
        c, k = c[idx], k[idx]
        np.save(os.path.join(out_dir, 'path_index.npy'), idx.astype(np.float64))
    np.save(os.path.join(out_dir, 'cost.npy'), c)
    np.save(os.path.join(out_dir, 'collide.npy'), k)
    np.save(os.path.join(out_dir, 'best_cost.npy'), np.array([best_cost], dtype=np.float64))
    np.save(os.path.join(out_dir, 'best_index.npy'), np.array([best_idx], dtype=np.float64))


def kernel_profile(kname, B, n):
    """ncu figures of the dominant kernel for this workload, committed under profiles/ (traffic.json)"""
    try:
        tj = json.load(open(os.path.join(ROOT, 'profiles', 'traffic.json')))
        for ent in tj['entries']:
            if ent['kernel'] == kname and ent['paths'] == B and ent['raster'] == n:
                return ent
    except Exception:
        pass
    return {}


# ---------------------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    import uam_path_planning_b200 as uam
    from uam_path_planning_b200 import distributed as udist

    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py needs a CUDA device (no CPU fallback)')
    torch.cuda.set_device(local)
    dev = f'cuda:{local}'
    # stdout carries the ONE JSON line and nothing else: NCCL prints its version banner on file descriptor 1 from C, so
    # fd 1 is pointed at stderr for the whole run and the line is written to a saved copy of the real stdout
    sys.stdout.flush()
    real_stdout = os.fdopen(os.dup(1), 'w')
    os.dup2(2, 1)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=torch.device(dev))

    def allmax(vals):
        t = torch.tensor(vals, dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(v) for v in t.tolist()]

    n, B = args.raster, args.paths
    layers, occ, geo = make_raster(torch, dev, n)
    rm = uam.RasterMap.from_arrays(layers, geo, occ, device=local)
    eng = rm.engine
    offset = rank * B
    # this rank's candidates: 40-byte rows on the host (pinned), the paths generated from them on the device
    cand_h = torch.from_numpy(make_candidates_host(B, 2000 + rank, n)).pin_memory()
    sigma = JITTER_CELLS * KM / n
    Z = eng.make_candidates(cand_h.to(dev), WP - 2, sigma, JITTER_SEED, offset)
    cost = torch.empty(B, dtype=torch.float32, device=dev)
    col = torch.empty(B, dtype=torch.uint8, device=dev)
    key = torch.empty(1, dtype=torch.int64, device=dev)
    reduce_mode = 'none (1 GPU)'
    if world > 1:
        reduce_mode = 'nccl all_reduce(MIN) of the 8-byte key'
        if args.reduce == 'peer':
            try:
                udist.attach_peer_group(eng)
                reduce_mode = 'peer memory: key stored into every rank\'s symmetric block over NVLink from the tail of the step\'s last kernel'
            except Exception as exc:               # CUDA IPC not permitted on this box: the NCCL form of the same reduction
                print(f'[bench] peer group unavailable ({exc!r}); using NCCL for the key', file=sys.stderr)
        ok = allmax([0.0 if reduce_mode.startswith('peer') else 1.0])[0]
        if ok != 0.0 and reduce_mode.startswith('peer'):
            raise SystemExit('peer group attached on some ranks only')
    use_nccl = world > 1 and reduce_mode.startswith('nccl')

    def step():
        rm.score_paths_best(Z, WEIGHTS, SPC, True, None, global_offset=offset, out=(cost, col), key=key)
        if use_nccl:
            dist.all_reduce(key, op=dist.ReduceOp.MIN)

    # sample counts -> algorithmic bytes (one extra untimed call)
    _, _, ns = rm.score_paths(Z, WEIGHTS, SPC, True, None, want_nsamples=True)
    total_samples = int(ns.sum().item())
    del ns
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()              # polling already while the warm-up runs; only the samples of the timed regions are kept
    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    launches0 = eng.launch_count()
    eng.set_option('time_kernels', 1)      # CUDA events around the dominant scoring kernel, on the launching stream
    t_start, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    wall0 = time.time()
    t_start.record()
    for s in range(args.steps):
        step()
    t_end.record()
    torch.cuda.synchronize()
    clocks.window(wall0, time.time())
    if world > 1:
        dist.barrier()
    launches = eng.launch_count() - launches0
    ms_total = t_start.elapsed_time(t_end)
    k_ms = eng.get_stat('score_kernel_ms_mean')                         # the dominant kernel alone
    assert int(eng.get_stat('score_kernel_count')) == args.steps
    eng.set_option('time_kernels', 0)
    best_cost, best_idx = udist.decode_key(int(key.item()))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, cost, col, best_cost, best_idx)
    variant = int(os.environ.get('UAM_INT_VARIANT', '-1'))
    combine = int(os.environ.get('UAM_COMBINE_LAYERS', '1'))
    quad = {0: '4', 1: '8', 2: '1'}[combine]         # texel form sampled by the large-batch pipelines (8: sign-packed quads)
    kname = {0: 'uam_k_score_raster_int<4,L,0>', 1: 'uam_k_score_raster_int<4,L,1>', 3: f'uam_k_score_tiles<{quad}>'}.get(
        variant, f'uam_k_score_groups<{quad},1>')

    def timed(fn, reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(reps):
            fn(i)
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps

    # ---- secondary: the scoring call alone (no best-key tail), waypoint mode, and a weights change every step ---------
    reps2 = min(args.steps, 20)
    for _ in range(3):
        rm.score_paths(Z, WEIGHTS, 0.0, True, None, out=(cost, col))
    wp_ms = timed(lambda i: rm.score_paths(Z, WEIGHTS, 0.0, True, None, out=(cost, col)), reps2)
    # the weights are run-time parameters in the reference (p[7:], solver.py:60-68): with new weights every step the quad
    # texels (the three layers folded into one weighted layer) are rebuilt inside every step
    wsets = [WEIGHTS, [w * 1.5 for w in WEIGHTS]]
    for i in range(2):
        rm.score_paths_best(Z, wsets[i % 2], SPC, True, None, global_offset=offset, out=(cost, col), key=key)
    wchg_ms = timed(lambda i: rm.score_paths_best(Z, wsets[i % 2], SPC, True, None, global_offset=offset, out=(cost, col), key=key), reps2)
    step()                                                               # restore the integral-mode costs of WEIGHTS
    torch.cuda.synchronize()
    cost_dev = cost.cpu().numpy()
    col_dev = col.cpu().numpy()

    # ---- secondary: the reference's own function on the reference's own map (C1) ----------------------------------
    analytic = None
    if rank == 0:
        try:
            analytic = analytic_c1(torch, dev, args, with_cpu=world == 1)      # CPU legs run at N = 1 only
        except Exception as exc:              # a secondary figure must not take the headline down
            analytic = {'error': repr(exc)}

    # ---- e2e: host buffers through the C-ABI, all copies inside the timed region -----------------------------------
    # three sets of pinned output buffers (one per ring slot); two batches in flight: the upload of step s+1 overlaps the
    # kernels of step s
    pin = lambda shape, dt: torch.empty(shape, dtype=dt).pin_memory()
    outs = [(pin(B, torch.float32).numpy(), pin(B, torch.uint8).numpy(), pin(1, torch.int64).numpy().view(np.uint64)) for _ in range(3)]
    cand_np = cand_h.numpy()
    Zh = pin((B, 2 * WP), torch.float64)
    Zh.copy_(Z)
    Zh_np = Zh.numpy()
    e2e_steps = max(3, min(args.steps, args.e2e_steps))

    def e2e_loop(submit):
        for i in range(4):                                               # warm-up: every slot of the 3-deep ring allocates its staging / scratch once
            rm.wait(submit(i))
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        w0 = time.time()
        t0 = time.perf_counter()
        pending = []
        for i in range(e2e_steps):
            pending.append(submit(i))
            if len(pending) > 2:
                rm.wait(pending.pop(0))                                  # results of step i-2 are in the host buffers now
        for t in pending:
            rm.wait(t)
        torch.cuda.synchronize()
        ms = (time.perf_counter() - t0) * 1e3 / e2e_steps
        clocks.window(w0, time.time())
        return ms

    e2e_c_ms = e2e_loop(lambda i: rm.submit(WEIGHTS, SPC, outs[i % 3][0], outs[i % 3][1], candidates=cand_np, N=WP - 2,
                                            jitter_sigma=sigma, seed=JITTER_SEED, key=outs[i % 3][2], global_offset=offset))
    last = outs[(e2e_steps - 1) % 3]
    assert np.array_equal(last[0], cost_dev) and np.array_equal(last[1], col_dev), 'candidate entry point disagrees with the device entry point'
    assert int(last[2][0]) == udist.host_best_key(cost_dev, offset)
    e2e_z_ms = e2e_loop(lambda i: rm.submit(WEIGHTS, SPC, outs[i % 3][0], outs[i % 3][1], Z=Zh_np, key=outs[i % 3][2], global_offset=offset))
    assert np.array_equal(last[0], cost_dev), 'host-waypoint entry point disagrees with the device entry point'
    # one synchronous call at a time (latency of a single batch: chunked upload / score / download pipeline inside the call)
    rm.score_paths(Zh_np, WEIGHTS, SPC, True, None, out=(outs[0][0], outs[0][1]))
    t0 = time.perf_counter()
    for _ in range(3):
        rm.score_paths(Zh_np, WEIGHTS, SPC, True, None, out=(outs[0][0], outs[0][1]))
    e2e_sync_ms = (time.perf_counter() - t0) * 1e3 / 3
    clk = clocks.stop() if rank == 0 else None
    peer_late = eng.peer_timed_out() if world > 1 and not use_nccl else False

    # ---- max over ranks -----------------------------------------------------------------------------------------
    per_rank = torch.tensor([ms_total / args.steps, e2e_c_ms, e2e_z_ms], dtype=torch.float64, device=dev)
    if world > 1:
        parts = [torch.empty_like(per_rank) for _ in range(world)]
        dist.all_gather(parts, per_rank)
        per_rank = torch.stack(parts)
    per_rank = per_rank.reshape(-1, 3).cpu().numpy()
    ms_total, k_ms, e2e_c_ms, e2e_z_ms, e2e_sync_ms, wp_ms, wchg_ms, late = allmax(
        [ms_total, k_ms, e2e_c_ms, e2e_z_ms, e2e_sync_ms, wp_ms, wchg_ms, float(peer_late)])

    # ---- the other BASELINE configs, short forms (C2 / C4 on one GPU, C5 sharded over the ranks) -------------------
    configs = None
    if not args.no_configs:
        del Zh, Zh_np
        configs = other_configs(args, torch, uam, dev, rank, world, lambda x: allmax([x])[0],
                                free=lambda: None)

    if rank == 0:
        segs = B * (WP - 1)
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
        except Exception:
            pass
        peak = float(peaks.get('hbm_gbs', 6650.0))
        abytes = algorithmic_bytes(total_samples, B)
        achieved = abytes / (k_ms * 1e-3) / 1e9
        prof = kernel_profile(kname, B, n)
        traffic = prof.get('dram_bytes_per_launch')
        model_bytes = total_samples * 16 + B * WP * 16 + B * WP * (4 + 4 + 1)    # quad taps + waypoints + ids / partials
        wp_bytes = (WP - 1) * B * 16 + B * WP * 49 + B * 21
        line = {
            'metric': METRIC, 'value': segs * world * args.steps / (ms_total * 1e-3), 'unit': 'segment-evals/s',
            'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms_total / args.steps,
            'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32 (fp64 coordinates)',
            'data': 'synthetic', 'config': workload_config(args),
            'samples_per_step_per_gpu': total_samples,
            'samples_per_s': total_samples * world * args.steps / (ms_total * 1e-3),
            'best_reduction': reduce_mode, 'peer_wait_timed_out': bool(late),
            'ms_per_step_per_rank': {'device_resident': [round(float(v), 4) for v in per_rank[:, 0]],
                                     'e2e': [round(float(v), 4) for v in per_rank[:, 1]],
                                     'e2e_host_waypoints': [round(float(v), 4) for v in per_rank[:, 2]]},
            'roofline': {
                'bound': 'hbm', 'achieved': achieved, 'peak': peak, 'unit': 'GB/s', 'frac': achieved / peak,
                'traffic': traffic, 'traffic_source': prof.get('source'),
                'kernel': kname, 'kernel_ms': k_ms, 'algorithmic_bytes_per_launch': abytes,
                # what the kernel physically does with memory, next to the contract's algorithmic figure:
                'hbm_frac': (traffic / (k_ms * 1e-3) / 1e9 / peak) if traffic else None,
                'model_bytes_per_launch': model_bytes, 'model_GBps': model_bytes / (k_ms * 1e-3) / 1e9,
                'model_frac': model_bytes / (k_ms * 1e-3) / 1e9 / peak,
                'limiter': prof.get('limiter'), 'limiter_unit': prof.get('limiter_unit'), 'limiter_frac': prof.get('limiter_frac'),
                'l2_to_l1_bytes_per_launch': prof.get('l2_to_l1_bytes_per_launch'),
                'l2_to_l1_over_useful': prof.get('l2_to_l1_over_useful'),
                'note': 'achieved / frac follow the contract: SURVEY 8(d) algorithmic bytes (16 B per segment + (L x 16 + 1) B per '
                        'sample) / event-timed kernel duration.  They exceed the HBM peak because the kernel does not move those '
                        'bytes: the L layers are folded into one weighted layer (linearity), a tap is one 16-B quad texel '
                        '(model_bytes: 16 B per tap, model_frac of the HBM peak if they came from DRAM), and the binned order serves '
                        'the taps from L2 -- hbm_frac is the physical DRAM traffic (ncu) / time / peak.  The kernel is bound by the '
                        'L1 load/store data pipe (limiter_frac of its wavefront peak, ncu), not by HBM',
                'peak_source': 'MEASURED_PEAKS.json hbm_gbs (measured)' if 'hbm_gbs' in peaks else 'fallback 6650 GB/s'},
            'e2e': {'value': segs * world / (e2e_c_ms * 1e-3), 'unit': 'segment-evals/s',
                    'h2d_bytes_per_step': B * 5 * 8, 'd2h_bytes_per_step': B * 5 + 8, 'ms_per_step': e2e_c_ms,
                    'api': 'RasterMap.submit(candidates=(B,5) numpy) / wait -> uam_raster_submit_candidates_host / uam_raster_wait: '
                           'candidate rows {start, goal, displacement} up (the input of Solver.create_x_init, main.py:160-171), paths '
                           'generated on the device, costs + flags + best key down; 2 batches in flight', 'steps': e2e_steps},
            'e2e_host_waypoints': {'value': segs * world / (e2e_z_ms * 1e-3), 'unit': 'segment-evals/s',
                                   'h2d_bytes_per_step': B * 2 * WP * 8, 'd2h_bytes_per_step': B * 5 + 8, 'ms_per_step': e2e_z_ms,
                                   'api': 'RasterMap.submit(Z=(B,128) numpy) / wait -> uam_raster_submit_paths_host: the same paths '
                                          'uploaded as float64 waypoints (1 KiB per path; PCIe / host-memory bound), 2 batches in flight',
                                   'single_call_ms': e2e_sync_ms,
                                   'single_call_api': 'RasterMap.score_paths(numpy) -> uam_score_paths_raster_host (one synchronous call)'},
            'weights_changed_every_step': {'ms_per_step': wchg_ms, 'value': segs * world / (wchg_ms * 1e-3), 'unit': 'segment-evals/s',
                                           'note': 'new layer weights (p[7:]) in every step: the quad texels are rebuilt inside the step'},
            'waypoint_mode': {'ms_per_step': wp_ms, 'value': segs * world / (wp_ms * 1e-3), 'unit': 'segment-evals/s',
                              'algorithmic_GBps': wp_bytes / (wp_ms * 1e-3) / 1e9, 'frac': wp_bytes / (wp_ms * 1e-3) / 1e9 / peak,
                              'note': 'samples_per_cell = 0 (one sample per waypoint, the reference sampling), same batch; '
                                      'a DRAM-latency-bound gather, reported, not the roofline claim'},
            'gpu_launches': launches, 'clocks': clk,
            'best': {'cost': best_cost, 'index': best_idx},
            'analytic_mode': analytic,
            'configs': configs,
        }
        if world == 1 and not args.no_cpu:
            Lh, Oh = layers.cpu().numpy(), occ.cpu().numpy()
            nb = min(B, args.cpu_sample)
            Zs = Z[:nb].cpu().numpy()
            rate, dt, th, (c_ref, col_ref, ns_ref) = cpu_c_rate(Lh, Oh, geo, Zs)
            c_gpu = cost_dev[:nb].astype(np.float64)
            err = float(np.max(np.abs(c_gpu - c_ref) / np.abs(c_ref)))
            n1 = min(nb, args.numpy_sample)
            rate1, dt1, (c_np, col_np, _) = cpu_numpy_rate(Lh, Oh, geo, Zs[:n1])
            Zo = host_paths(min(nb, 2000), 2000 + rank, n)                 # the generator itself against the oracle's restatement
            line['cpu_baseline'] = {
                'value': rate, 'unit': 'segment-evals/s', 'cores': th, 'kind': 'port',
                'sample': f'first {nb} paths of the same batch, oracle/uam_oracle_c.c (C restatement of the float64 oracle, '
                          f'OpenMP over paths, {th} threads), integral mode, {dt:.1f} s',
                'max_rel_err_gpu_vs_oracle': err, 'paths_compared': nb,
                'collide_equal': bool(np.array_equal(col_dev[:nb].astype(bool), col_ref)),
                'candidate_generator_max_abs_diff_vs_oracle_km': float(np.max(np.abs(Zo - Zs[:len(Zo)]))),
                'numpy_1core': {'value': rate1, 'paths': n1, 'seconds': dt1,
                                'max_rel_diff_c_vs_numpy': float(np.max(np.abs(c_np - c_ref[:n1]) / np.abs(c_np)))}}
        real_stdout.write(json.dumps(line) + '\n')
        real_stdout.flush()
    if world > 1:
        dist.destroy_process_group()


def other_configs(args, torch, uam, dev, rank, world, reduce_max, free):
    """Short runs of BASELINE.json's other configs inside the driver's run (bench_configs.py has the long forms):
    C2 and C4 are single-GPU configs (rank 0 of an N = 1 run), C5's queries shard over the ranks."""
    import types
    import bench_configs as bc
    a = types.SimpleNamespace(c4_size=args.c4_size, reps=3, no_cpu=args.no_cpu, c5_size=4096, c5_queries=args.c5_queries,
                              c5_queries_bands=args.c5_queries_bands, c5_reps=1, c5_routes=args.c5_routes,
                              c5_cpu_bands=False)      # one 8-band CPU Dijkstra takes 18 s: bench_configs.py times it
    out = {}
    torch.cuda.empty_cache()
    if world == 1:
        for name, fn in (('C2', bc.run_c2), ('C4', bc.run_c4)):
            try:
                out[name] = fn(a, torch, uam, dev)
            except Exception as exc:          # a secondary figure must not take the headline down
                out[name] = {'error': repr(exc)}
            torch.cuda.empty_cache()
    try:
        out['C5'] = bc.run_c5(a, torch, uam, dev, rank, world, reduce_max)
    except Exception as exc:
        out['C5'] = {'error': repr(exc)}
        if world > 1:
            raise                             # a rank that stops here would leave the others in a collective
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=200)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--raster', type=int, default=RASTER)
    ap.add_argument('--paths', type=int, default=125000, help='candidate paths per GPU per step (C3: 1M over 8 GPUs)')
    ap.add_argument('--reduce', default='peer', choices=['peer', 'nccl'], help='N > 1: how the 8-byte best key crosses the ranks')
    ap.add_argument('--cpu-sample', type=int, default=125000, help='paths of the batch the cpu_baseline leg scores and compares (C/OpenMP oracle)')
    ap.add_argument('--numpy-sample', type=int, default=1024, help='paths the 1-core numpy oracle scores')
    ap.add_argument('--e2e-steps', type=int, default=20)
    ap.add_argument('--no-cpu', action='store_true')
    ap.add_argument('--no-configs', action='store_true', help='skip the short C2 / C4 / C5 runs')
    ap.add_argument('--c4-size', type=int, default=16384)
    ap.add_argument('--c5-queries', type=int, default=16, help='C5: queries per GPU, 1 altitude band')
    ap.add_argument('--c5-queries-bands', type=int, default=4, help='C5: full sweeps per GPU, 8 altitude bands')
    ap.add_argument('--c5-routes', type=int, default=128, help='C5: start/goal queries per GPU (128 x 8 GPUs = the 1024 of BASELINE config 5)')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='after the timed steps, write the outputs of the last one (rank 0: per-path cost and collision flag, '
                         'best cost and index) as DIR/<name>.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    args.warmup = max(args.warmup, 3) if args.impl == 'ours' else args.warmup
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_ours(args)


if __name__ == '__main__':
    main()
