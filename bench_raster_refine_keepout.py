"""Refinement under the analytic obstacle check on C2's map: bench_analytic_sweep.c2_map (32 obstacle discs among 288
shapes, 64 km) rasterised with RasterMap.from_map at 8192^2 (L = 1, Risk weight 5000), its 10 000-path corridor batch
of 64 waypoints, integral mode at 1 sample per cell, K trips.  Four arms alternated in one process, each call bracketed
by CUDA events: refine_paths, refine_paths_swept (raster sweep, min_d2 = 0), refine_paths_keepout with margin = 0 and
with margin = 0.5 km; and the gradient call they all start with.  Per arm: the time per trip, the median cost
reduction, and what the arm does to the batch against the shapes themselves: paths that gain an analytic HIT, paths
whose clearance capped at 0.5 km drops, paths with collide = 0 yet an analytic HIT.  --profile adds a torch.profiler run
of its own for the per-launch kernel times of the keep-out arms.

    python bench_raster_refine_keepout.py [--iterations 20] [--steps 10] [--warmup 2] [--profile]
                                          [--out profiles/r09_bench_raster_refine_keepout.json]

Writes one JSON line to --out (and prints it).
"""
import argparse
import json
import os
import sys

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

MARGIN = 0.5        # km: the margin of the fourth arm and the cap of the clearance counts


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--iterations', type=int, default=20, help='trips per refine call')
    ap.add_argument('--steps', type=int, default=10, help='timed rounds of (gradient, four arms)')
    ap.add_argument('--warmup', type=int, default=2)
    ap.add_argument('--raster', type=int, default=8192)
    ap.add_argument('--profile', action='store_true', help='also run torch.profiler (separate run) for kernel times')
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'r09_bench_raster_refine_keepout.json'))
    args = ap.parse_args()
    import torch
    import uam_path_planning_b200 as uam
    from uam_path_planning_b200 import _lib
    from bench_analytic_sweep import c2_map, card

    assert torch.cuda.is_available(), 'bench_raster_refine_keepout.py needs a CUDA device'
    dev = 'cuda:0'
    torch.cuda.set_device(0)
    HIT = _lib.UAM_SWEEP_HIT
    rng = np.random.default_rng(20260101)
    m = c2_map(uam, rng)
    KM, n, Wp, B = 64.0, args.raster, 64, 10000
    rm = uam.RasterMap.from_map(m, n, n, (0.0, KM / n, 0.0, KM / n))
    prob = uam.Problem(m, Wp - 2, {'length_smooth': True, 'obstacle_smooth': True})
    prob.params.update(maxratio=1.04, maxalpha=np.pi / 80, enlargement=0)
    prob.set_weight('Risk', 5000.0)
    Zh = uam.Solver(prob, {}).candidates(rng.uniform(-0.9, 0.9, B), jitter=0.25 * KM / 4096, rng=rng)   # C2's corridor
    Z = torch.from_numpy(np.ascontiguousarray(Zh)).to(dev)
    K, W, SPC = args.iterations, [5000.0], 1.0

    arms = {
        'plain': lambda: rm.refine_paths(Z, W, SPC, K),
        'raster_swept': lambda: rm.refine_paths_swept(Z, W, SPC, K, min_d2=0),
        'keepout_margin_0': lambda: rm.refine_paths_keepout(Z, W, SPC, K, margin=0.0),
        f'keepout_margin_{MARGIN:g}': lambda: rm.refine_paths_keepout(Z, W, SPC, K, margin=MARGIN),
    }

    def grad():
        return rm.cost_gradient(Z, W, SPC)

    names = ['grad'] + list(arms)
    calls = [grad] + list(arms.values())
    for _ in range(args.warmup):
        for f in calls:
            f()
    torch.cuda.synchronize()
    ev = [[(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in calls]
          for _ in range(args.steps)]
    for row in ev:
        for (e0, e1), f in zip(row, calls):
            e0.record()
            f()
            e1.record()
    torch.cuda.synchronize()
    ms = {nm: float(np.median([row[i][0].elapsed_time(row[i][1]) for row in ev])) for i, nm in enumerate(names)}

    c0, k0 = rm.score_paths(Z, W, SPC)
    f0 = m.sweep_paths(Z)[0]
    cl0 = m.path_clearance(Z, MARGIN)[1]
    hit0 = (f0 & HIT) != 0
    outcome = {}
    for nm, f in arms.items():
        Zo, c, k, acc = f()[:4]
        cs, ks = rm.score_paths(Zo, W, SPC)
        fa = m.sweep_paths(Zo)[0]
        cl = m.path_clearance(Zo, MARGIN)[1]
        red = ((c0 - c) / c0.abs()).double().cpu().numpy()
        hit = (fa & HIT) != 0
        outcome[nm] = {
            'call_ms': round(ms[nm], 3), 'ms_per_trip': round((ms[nm] - ms['grad']) / max(K, 1), 4),
            'median_rel_reduction': round(float(np.median(red)), 6), 'mean_rel_reduction': round(float(red.mean()), 6),
            'improved': round(float((c < c0).float().mean()), 5), 'mean_accepted': round(float(acc.float().mean()), 3),
            'cost_collide_equal_to_scorer': bool(torch.equal(cs, c) and torch.equal(ks, k)),
            'gained_analytic_hit': int((hit & ~hit0).sum()),
            f'clearance_capped_{MARGIN:g}_dropped': int((cl < cl0).sum()),
            'collide0_but_analytic_hit': int(((k == 0) & hit).sum()), 'collide_after': int(k.sum())}
    counts = {'paths': B, 'waypoints': Wp, 'collide_before': int(k0.sum()), 'analytic_hit_before': int(hit0.sum()),
              'collide0_but_analytic_hit_before': int(((k0 == 0) & hit0).sum()),
              f'clean_within_{MARGIN:g}_before': int((~hit0 & (cl0 < MARGIN)).sum())}

    kernels = {}
    if args.profile:
        from torch.profiler import ProfilerActivity, profile
        for nm in ('keepout_margin_0', f'keepout_margin_{MARGIN:g}', 'plain'):
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(2):
                    arms[nm]()
                torch.cuda.synchronize()
            split = {'analytic_check': 0.0, 'refine_step': 0.0, 'gradient_and_rest': 0.0}
            for a in prof.key_averages():
                t = getattr(a, 'device_time_total', None)
                if t is None:
                    t = a.cuda_time_total
                if t <= 0:
                    continue
                t = t / 2 / 1000.0                               # ms per refine call
                if 'uam_k_sweep_analytic' in a.key or 'uam_k_clearance_analytic' in a.key:
                    split['analytic_check'] += t
                elif 'uam_k_refine_step' in a.key:
                    split['refine_step'] += t
                else:
                    split['gradient_and_rest'] += t
            kernels[nm] = {k_: round(v, 3) for k_, v in split.items()}
            kernels[nm]['analytic_ms_per_launch'] = round(split['analytic_check'] / (K + 1), 4)

    name, power = card()
    out = {'workload': f'C2 corridor: {B} paths x {Wp} waypoints, from_map {n}^2 (L = 1), spc = {SPC}; {K} trips',
           'grad_call_ms': round(ms['grad'], 4), 'arms': outcome, 'counts': counts, 'kernels_ms_per_call': kernels,
           'steps': args.steps, 'warmup': args.warmup, 'gpu': name, 'power_limit': power}
    line = json.dumps(out)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as fh:
        fh.write(line + '\n')


if __name__ == '__main__':
    main()
