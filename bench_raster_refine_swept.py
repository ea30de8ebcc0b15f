"""Refinement under the swept check on the C3 shard (bench.py's workload: 125 000 paths x 64 waypoints, 8192^2 3-layer
raster, integral mode at 1 sample per cell, bench.py's weights and seeds): time of a refine call of K trips in three modes
alternated in one process -- refine_paths, refine_paths_swept with min_d2 = 0 and with min_d2 = 4 -- against the gradient
call; per-kernel times; and what each mode does to the batch: cost reduction, and the paths that gain a sweep HIT or lose
capped clearance.

    python bench_raster_refine_swept.py [--paths 125000] [--iterations 20] [--steps 6] [--warmup 2]

Prints one JSON line.  Writes nothing.
"""
import argparse
import json
import os
import subprocess
import sys

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

MIN_D2 = 4          # clearance of the third mode: 2 cells


def card():
    """(name, power limit) of GPU 0 as nvidia-smi reports them (read-only query)."""
    try:
        out = subprocess.run(['nvidia-smi', '--id=0', '--query-gpu=name,power.limit', '--format=csv,noheader'],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [s.strip() for s in out.split(',')]
        return name, power
    except Exception as e:      # the numbers stay meaningful with the torch name alone
        import torch
        return torch.cuda.get_device_name(0), f'unknown ({e})'


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--paths', type=int, default=125000)
    ap.add_argument('--iterations', type=int, default=20, help='trips per refine call')
    ap.add_argument('--steps', type=int, default=6, help='timed rounds of (gradient, plain, swept, swept + clearance)')
    ap.add_argument('--warmup', type=int, default=2)
    args = ap.parse_args()
    import torch
    import bench
    import uam_path_planning_b200 as uam
    from uam_path_planning_b200 import _lib

    assert torch.cuda.is_available(), 'bench_raster_refine_swept.py needs a CUDA device'
    dev = 'cuda:0'
    torch.cuda.set_device(0)
    layers, occ, geo = bench.make_raster(torch, dev)
    rm = uam.RasterMap.from_arrays(layers, geo, occ)
    Z = bench.make_paths(torch, dev, args.paths, seed=1)
    B = Z.shape[0]
    K = args.iterations
    W, SPC = bench.WEIGHTS, bench.SPC

    modes = {
        'plain': lambda: rm.refine_paths(Z, W, SPC, K, True, None),
        'swept': lambda: rm.refine_paths_swept(Z, W, SPC, K, True, None, min_d2=0),
        f'swept_min_d2_{MIN_D2}': lambda: rm.refine_paths_swept(Z, W, SPC, K, True, None, min_d2=MIN_D2),
    }

    def grad():
        return rm.cost_gradient(Z, W, SPC, True, None)

    for _ in range(args.warmup):
        grad()
        for f in modes.values():
            f()
    torch.cuda.synchronize()
    # alternate the calls in one process, each bracketed by its own events
    names = ['grad'] + list(modes)
    calls = [grad] + list(modes.values())
    ev = [[(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in calls]
          for _ in range(args.steps)]
    for row in ev:
        for (e0, e1), f in zip(row, calls):
            e0.record()
            f()
            e1.record()
    torch.cuda.synchronize()
    ms = {n: float(np.median([row[i][0].elapsed_time(row[i][1]) for row in ev])) for i, n in enumerate(names)}

    # what each mode does to the batch
    c0, k0 = rm.score_paths(Z, W, SPC)
    f0, _, d0 = rm.sweep_paths(Z)
    hit0 = (f0 & _lib.UAM_SWEEP_HIT) != 0
    inside0 = (f0 & _lib.UAM_SWEEP_OUTSIDE) == 0
    outcome = {}
    for n, f in modes.items():
        Zo, c, k, acc = f()[:4]
        cs, ks = rm.score_paths(Zo, W, SPC)
        fs, _, ds = rm.sweep_paths(Zo)
        red = ((c0 - c) / c0.abs()).double().cpu().numpy()
        hit = (fs & _lib.UAM_SWEEP_HIT) != 0
        outcome[n] = {
            'call_ms': round(ms[n], 3), 'ms_per_trip': round((ms[n] - ms['grad']) / max(K, 1), 4),
            'median_rel_reduction': round(float(np.median(red)), 6), 'mean_rel_reduction': round(float(red.mean()), 6),
            'improved': round(float((c < c0).float().mean()), 5), 'mean_accepted': round(float(acc.float().mean()), 3),
            'cost_collide_equal_to_scorer': bool(torch.equal(cs, c) and torch.equal(ks, k)),
            'gained_hit': int((hit & ~hit0).sum()), 'gained_hit_inside': int((hit & ~hit0 & inside0).sum()),
            'gained_any_sweep_flag': int(((fs & ~f0) != 0).sum()),
            f'lost_clearance_capped_{MIN_D2}': int((torch.clamp(ds, max=MIN_D2) < torch.clamp(d0, max=MIN_D2)).sum()),
            'collide0_but_hit': int(((k == 0) & hit).sum()), 'collide_after': int(k.sum())}
    counts = {'paths': B, 'collide_before': int(k0.sum()), 'hit_before': int(hit0.sum()),
              'collide0_but_hit_before': int(((k0 == 0) & hit0).sum()),
              f'clearance_below_{MIN_D2}_before': int((d0 < MIN_D2).sum())}

    # per-kernel device times, in a run of their own: gradient kernels, sweep, step
    from torch.profiler import ProfilerActivity, profile
    kernels = {}
    for n in (f'swept_min_d2_{MIN_D2}', 'swept'):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(2):
                modes[n]()
            torch.cuda.synchronize()
        split = {'sweep': 0.0, 'refine_step': 0.0, 'gradient_and_rest': 0.0}
        for a in prof.key_averages():
            t = getattr(a, 'device_time_total', None)
            if t is None:
                t = a.cuda_time_total
            if t <= 0:
                continue
            t = t / 2 / 1000.0                               # ms per refine call
            if 'uam_k_sweep_paths' in a.key:
                split['sweep'] += t
            elif 'uam_k_refine_step' in a.key:
                split['refine_step'] += t
            else:
                split['gradient_and_rest'] += t
        kernels[n] = {k_: round(v, 3) for k_, v in split.items()}
        kernels[n]['sweep_ms_per_launch'] = round(split['sweep'] / (K + 1), 4)

    name, power = card()
    print(json.dumps({
        'workload': f'C3 shard: {B} paths x {bench.WP} waypoints, {bench.RASTER}^2 x 3 layers, spc = {SPC}; {K} trips',
        'grad_call_ms': round(ms['grad'], 4), 'modes': outcome, 'kernels_ms_per_call': kernels, 'counts': counts,
        'steps': args.steps, 'gpu': name, 'power_limit': power}))


if __name__ == '__main__':
    main()
