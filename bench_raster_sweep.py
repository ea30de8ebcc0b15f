"""Swept segment check on the C3 shard (bench.py's workload: 125 000 paths x 64 waypoints, 8192^2 3-layer raster, bench.py's
weights and seeds): time of the sweep with flags and first hit, and with the clearance, against one scoring step; the
first-call builds of the bit-plane and the d^2 field; per-kernel times; and how many paths the sampled collide flag misses.

    python bench_raster_sweep.py [--paths 125000] [--steps 20] [--warmup 3]

Prints one JSON line.  Writes nothing.
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
    except Exception as e:      # the numbers stay meaningful with the torch name alone
        import torch
        return torch.cuda.get_device_name(0), f'unknown ({e})'


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--paths', type=int, default=125000)
    ap.add_argument('--steps', type=int, default=20, help='timed (score, sweep, sweep with clearance) triples')
    ap.add_argument('--warmup', type=int, default=3)
    args = ap.parse_args()
    import torch
    import bench
    import uam_path_planning_b200 as uam
    from uam_path_planning_b200 import _lib

    assert torch.cuda.is_available(), 'bench_raster_sweep.py needs a CUDA device'
    dev = 'cuda:0'
    torch.cuda.set_device(0)
    layers, occ, geo = bench.make_raster(torch, dev)
    rm = uam.RasterMap.from_arrays(layers, geo, occ)
    Z = bench.make_paths(torch, dev, args.paths, seed=1)
    B, N = Z.shape[0], Z.shape[1] // 2 - 2
    W, SPC = bench.WEIGHTS, bench.SPC
    eng = rm.engine
    key = torch.empty(1, dtype=torch.int64, device=dev)
    cost = torch.empty(B, dtype=torch.float32, device=dev)
    col = torch.empty(B, dtype=torch.uint8, device=dev)

    def score():
        rm.score_paths_best(Z, W, SPC, True, None, out=(cost, col), key=key)

    def sweep():
        return eng.sweep_raster(Z, N, True, False)

    def sweep_d2():
        return eng.sweep_raster(Z, N, True, True)

    # first calls after the upload: the bit-plane build (flags), then the d^2 field build (clearance), host clock around
    # work that ends in a synchronise
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    sweep()
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    sweep_d2()
    torch.cuda.synchronize()
    t2 = time.perf_counter()
    first_flags_ms, first_d2_ms = (t1 - t0) * 1e3, (t2 - t1) * 1e3

    for _ in range(args.warmup):
        score()
        sweep()
        sweep_d2()
    torch.cuda.synchronize()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(6)] for _ in range(args.steps)]
    for e in ev:
        e[0].record()
        score()
        e[1].record()
        e[2].record()
        sweep()
        e[3].record()
        e[4].record()
        sweep_d2()
        e[5].record()
    torch.cuda.synchronize()
    score_ms = float(np.median([e[0].elapsed_time(e[1]) for e in ev]))
    sweep_ms = float(np.median([e[2].elapsed_time(e[3]) for e in ev]))
    sweep_d2_ms = float(np.median([e[4].elapsed_time(e[5]) for e in ev]))

    # what the sampled collide flag misses
    flags, first, d2min = sweep_d2()
    hit = (flags & _lib.UAM_SWEEP_HIT) != 0
    inside = (flags & _lib.UAM_SWEEP_OUTSIDE) == 0
    counts = {'paths': B, 'inside_raster': int(inside.sum()), 'hit': int(hit.sum()), 'hit_inside': int((hit & inside).sum())}
    for spc in (0.0, 1.0):
        _, c = rm.score_paths(Z, W, spc)
        c = c.bool()
        counts[f'collide_spc{spc:g}'] = int(c.sum())
        counts[f'collide_spc{spc:g}_inside'] = int((c & inside).sum())
        counts[f'collide_spc{spc:g}_not_hit_inside'] = int((c & inside & ~hit).sum())     # must be 0
        counts[f'hit_inside_not_collide_spc{spc:g}'] = int((hit & inside & ~c).sum())
    Zr, _, kr, _ = rm.refine_paths(Z, W, SPC)
    fr, _, _ = eng.sweep_raster(Zr, N, True, False)
    hr = (fr & _lib.UAM_SWEEP_HIT) != 0
    ir = (fr & _lib.UAM_SWEEP_OUTSIDE) == 0
    kr = kr.bool()
    counts['refined_collide_spc1'] = int(kr.sum())
    counts['refined_clean_but_hit'] = int((~kr & hr).sum())
    counts['refined_clean_but_hit_inside'] = int((~kr & hr & ir).sum())
    counts['refined_collide_not_hit_inside'] = int((kr & ir & ~hr).sum())            # must be 0
    dm = d2min[d2min >= 0].double()
    clearance = {'d2min_median': float(dm.median()), 'd2min_zero': int((d2min == 0).sum()),
                 'd2min_clip': int((d2min == 65535).sum()), 'no_cell_touched': int((d2min < 0).sum())}

    # per-kernel device times, in a run of their own
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(4):
            score()
            sweep()
            sweep_d2()
        torch.cuda.synchronize()
    kernels = {}
    for a in prof.key_averages():
        t = getattr(a, 'device_time_total', None)
        if t is None:
            t = a.cuda_time_total
        if t > 0:
            kernels[a.key[:90]] = round(t / 4 / 1000.0, 4)       # ms per step
    kernels = dict(sorted(kernels.items(), key=lambda kv: -kv[1])[:10])

    name, power = card()
    print(json.dumps({
        'workload': f'C3 shard: {B} paths x {bench.WP} waypoints, {bench.RASTER}^2 x 3 layers; scoring at spc = {SPC}',
        'score_best_ms': round(score_ms, 4), 'sweep_flags_first_hit_ms': round(sweep_ms, 4),
        'sweep_with_d2min_ms': round(sweep_d2_ms, 4),
        'first_call_flags_ms': round(first_flags_ms, 3), 'first_call_d2min_ms': round(first_d2_ms, 3),
        'kernels_ms_per_step': kernels, 'counts': counts, 'clearance': clearance,
        'steps': args.steps, 'gpu': name, 'power_limit': power}))


if __name__ == '__main__':
    main()
