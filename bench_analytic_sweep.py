"""Swept check against the analytic obstacles (uam_sweep_paths_analytic / Map.sweep_paths) against one analytic scoring
call (Problem.score) of the same batch:
  - C2's map (bench_configs.run_c2: 192 risk polygons, 64 risk discs, 32 obstacle discs = 288 shapes, 64 km), its
    10 000-path corridor and scatter batches of 64 waypoints;
  - C4's 4096 rectangular footprints as obstacles on a 128 km map, a 125 000 x 64 scatter batch.
Times are medians of CUDA-event-timed steps, score and sweep alternated; the first call after an upload (which builds the
cell lists) is timed separately.  Counts: paths whose waypoints are clean (Problem.score collide = 0) but which sweep
HIT, and on C2's map rasterised at 4096^2 and 8192^2 the paths on which RasterMap.sweep_paths and this sweep disagree,
each way.  --profile adds a torch.profiler run of its own for the kernel times.

    python bench_analytic_sweep.py [--steps 20] [--warmup 3] [--profile] [--out profiles/r07_bench_analytic_sweep.json]

Writes one JSON line to --out (and prints it).
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


def card():
    """(name, power limit) of GPU 0 as nvidia-smi reports them (read-only query)."""
    try:
        out = subprocess.run(['nvidia-smi', '--id=0', '--query-gpu=name,power.limit', '--format=csv,noheader'],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [s.strip() for s in out.split(',')]
        return name, power
    except Exception as e:
        import torch
        return torch.cuda.get_device_name(0), f'unknown ({e})'


def c2_map(uam, rng):
    """bench_configs.run_c2's map, drawn from the same seed in the same order."""
    m = uam.RegionMap()
    m.new_region('Risk', 'r')
    for _ in range(192):
        c, a = rng.uniform(2, 62, 2), rng.uniform(0, np.pi)
        hw, hh = rng.uniform(0.25, 2.0, 2)
        R = np.array([[np.cos(a), -np.sin(a)], [np.sin(a), np.cos(a)]])
        m.add_shape_to_region('Risk', uam.polygon(*(c + np.array([[-hw, -hh], [hw, -hh], [hw, hh], [-hw, hh]]) @ R.T).tolist()))
    for _ in range(64):
        m.add_shape_to_region('Risk', uam.ball(rng.uniform(2, 62, 2).tolist(), float(rng.uniform(0.5, 3))))
    for _ in range(32):
        m.add_obstacle(uam.ball(rng.uniform(2, 62, 2).tolist(), float(rng.uniform(0.3, 1.5))))
    m.x_start, m.x_goal = [6.0, 7.0], [57.0, 55.0]
    return m


def c4_map(uam, rng, n=4096, km=128.0):
    """C4-like footprints: n rotated rectangles (minAreaRect-like, 30 - 600 m half sides) as hard obstacles."""
    m = uam.RegionMap()
    for _ in range(n):
        c, a = rng.uniform(1, km - 1, 2), rng.uniform(0, np.pi)
        hw, hh = rng.uniform(0.03, 0.6, 2)
        R = np.array([[np.cos(a), -np.sin(a)], [np.sin(a), np.cos(a)]])
        m.add_obstacle(uam.polygon(*(c + np.array([[-hw, -hh], [hw, -hh], [hw, hh], [-hw, hh]]) @ R.T).tolist()))
    m.x_start, m.x_goal = [2.0, 2.0], [km - 2, km - 2]
    return m


def scatter(rng, B, Wp, km, jitter):
    s, e = rng.uniform(0, km, (B, 1, 2)), rng.uniform(0, km, (B, 1, 2))
    return (s + np.linspace(0, 1, Wp).reshape(1, Wp, 1) * (e - s) + rng.normal(0, jitter, (B, Wp, 2))).reshape(B, 2 * Wp)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--steps', type=int, default=20, help='timed (score, sweep) pairs per batch')
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--profile', action='store_true', help='also run torch.profiler (separate run) for kernel times')
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'r07_bench_analytic_sweep.json'))
    args = ap.parse_args()
    import torch
    import uam_path_planning_b200 as uam
    from uam_path_planning_b200 import _lib

    assert torch.cuda.is_available(), 'bench_analytic_sweep.py needs a CUDA device'
    dev = 'cuda:0'
    torch.cuda.set_device(0)
    HIT = _lib.UAM_SWEEP_HIT

    def ev():
        return torch.cuda.Event(enable_timing=True)

    def alternate(fns):
        for _ in range(args.warmup):
            for f in fns:
                f()
        ts = [[] for _ in fns]
        for _ in range(args.steps):
            for i, f in enumerate(fns):
                a, b = ev(), ev()
                a.record()
                f()
                b.record()
                torch.cuda.synchronize()
                ts[i].append(a.elapsed_time(b))
        return [float(np.median(t)) for t in ts]

    def first_call(m, Z):
        eng = m.engine()
        eng.set_shapes(m.obstacles, m._region_lists())        # a fresh upload: the next sweep builds the cell lists
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        m.sweep_paths(Z)
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) * 1e3

    def problem(m, Wp, risk=True):
        prob = uam.Problem(m, Wp - 2, {'length_smooth': True, 'obstacle_smooth': True})
        prob.params.update(maxratio=1.04, maxalpha=np.pi / 80, enlargement=0)
        if risk:
            prob.set_weight('Risk', 5000.0)
        return prob

    def measure(m, prob, Zh):
        Z = torch.from_numpy(np.ascontiguousarray(Zh)).to(dev)
        t_first = first_call(m, Z)
        ms_score, ms_sweep = alternate([lambda: prob.score(Z), lambda: m.sweep_paths(Z)])
        _, col, _ = prob.score(Z)
        f, k, o = m.sweep_paths(Z)
        col, f = col.cpu().numpy().astype(bool), f.cpu().numpy()
        hit = (f & HIT) != 0
        assert not np.any(col & ~hit), 'collide without HIT'
        return Z, {'paths': int(Z.shape[0]), 'waypoints': int(Z.shape[1] // 2), 'ms_score': ms_score, 'ms_sweep': ms_sweep,
                   'sweep_over_score': ms_sweep / ms_score, 'ms_first_sweep_incl_lists': t_first,
                   'collide': int(col.sum()), 'hit': int(hit.sum()), 'clean_waypoints_but_hit': int((hit & ~col).sum())}

    out = {}
    rng = np.random.default_rng(20260101)
    m2 = c2_map(uam, rng)
    Wp, B, KM, n = 64, 10000, 64.0, 4096
    prob2 = problem(m2, Wp)
    cell = KM / n
    Zc = uam.Solver(prob2, {}).candidates(rng.uniform(-0.9, 0.9, B), jitter=0.25 * cell, rng=rng)
    s, e = rng.uniform(0, KM, (B, 1, 2)), rng.uniform(0, KM, (B, 1, 2))
    Zs = (s + np.linspace(0, 1, Wp).reshape(1, Wp, 1) * (e - s) + rng.normal(0, 2 * cell, (B, Wp, 2))).reshape(B, 2 * Wp)
    eng2 = m2.engine()
    c2 = {}
    batches = {}
    for name, Zh in (('corridor', Zc), ('scatter', Zs)):
        batches[name], c2[name] = measure(m2, prob2, Zh)
        for grid in (0, 1):                     # the lists on and off give the same bits
            eng2.set_option('shape_grid', grid)
            torch.cuda.synchronize()
            r = [t.cpu().numpy() for t in m2.sweep_paths(batches[name])]
            if grid == 0:
                ref = r
            else:
                assert all(np.array_equal(a, b) for a, b in zip(r, ref))
        eng2.set_option('shape_grid', 0)
        c2[name]['ms_sweep_every_obstacle'] = alternate([lambda: m2.sweep_paths(batches[name])])[0]
        eng2.set_option('shape_grid', 1)
    # certification error of the raster sweep, as a number
    for res in (4096, 8192):
        rm = uam.RasterMap.from_map(m2, res, res, (0.0, KM / res, 0.0, KM / res))
        for name, Z in batches.items():
            fr = rm.sweep_paths(Z, clearance=False)[0].cpu().numpy()
            fa = m2.sweep_paths(Z)[0].cpu().numpy()
            hr, ha = (fr & HIT) != 0, (fa & HIT) != 0
            c2[name][f'raster_{res}_hit_analytic_clean'] = int((hr & ~ha).sum())
            c2[name][f'raster_{res}_clean_analytic_hit'] = int((~hr & ha).sum())
        del rm
    out['c2'] = dict(c2, shapes=288, obstacles=32, map_km=KM)

    rng4 = np.random.default_rng(20260104)
    m4 = c4_map(uam, rng4)
    prob4 = problem(m4, 64, risk=False)
    Z4 = scatter(rng4, 125000, 64, 128.0, 2 * 128.0 / 8192)
    _, out['c4'] = measure(m4, prob4, Z4)
    out['c4'].update(obstacles=4096, map_km=128.0)

    if args.profile:
        from torch.profiler import ProfilerActivity, profile
        Z = batches['corridor']
        Z4t = torch.from_numpy(np.ascontiguousarray(Z4)).to(dev)
        kern = {}
        for tag, m, prob, ZZ in (('c2_corridor', m2, prob2, Z), ('c4_scatter', m4, prob4, Z4t)):
            for _ in range(3):
                prob.score(ZZ)
                m.sweep_paths(ZZ)
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as p:
                for _ in range(10):
                    prob.score(ZZ)
                    m.sweep_paths(ZZ)
                torch.cuda.synchronize()
            for e in p.key_averages():
                if e.key.startswith('_Z') or 'uam_k' in e.key:
                    name = 'uam_k_sweep_analytic' if 'sweep_analytic' in e.key else (
                        'uam_k_score_analytic' if 'score_analytic' in e.key else None)
                    if name:
                        t = getattr(e, 'device_time_total', None) or getattr(e, 'cuda_time_total', 0.0)
                        kern[f'{tag}_{name}_ms'] = t / 1e3 / max(e.count, 1)
        out['kernel_ms_profiler'] = kern

    name, power = card()
    out.update(steps=args.steps, warmup=args.warmup, gpu=name, power_limit=power)
    line = json.dumps(out)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as fh:
        fh.write(line + '\n')


if __name__ == '__main__':
    main()
