"""Raster refinement on the C3 shard (bench.py's workload: 125 000 paths x 64 waypoints, 8192^2 3-layer raster,
integral mode at 1 sample per cell, bench.py's weights and seeds): time of a refine call of K trips against the gradient
call, per-kernel times, and what the refinement does to the batch.

    python bench_raster_refine.py [--paths 125000] [--iterations 20] [--steps 10] [--warmup 2] [--sweep]

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
    ap.add_argument('--steps', type=int, default=10, help='timed refine / gradient call pairs')
    ap.add_argument('--warmup', type=int, default=2)
    ap.add_argument('--sweep', action='store_true', help='also report the outcome for a few (step, max, min) settings')
    args = ap.parse_args()
    import torch
    import bench
    import uam_path_planning_b200 as uam

    assert torch.cuda.is_available(), 'bench_raster_refine.py needs a CUDA device'
    dev = 'cuda:0'
    torch.cuda.set_device(0)
    layers, occ, geo = bench.make_raster(torch, dev)
    rm = uam.RasterMap.from_arrays(layers, geo, occ)
    Z = bench.make_paths(torch, dev, args.paths, seed=1)
    B = Z.shape[0]
    K = args.iterations
    W, SPC = bench.WEIGHTS, bench.SPC

    def refine(**kw):
        return rm.refine_paths(Z, W, SPC, K, True, None, **kw)

    def grad():
        return rm.cost_gradient(Z, W, SPC, True, None)

    for _ in range(args.warmup):
        refine()
        grad()
    torch.cuda.synchronize()
    # alternate the two calls in one process, each bracketed by its own events
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(args.steps)]
    for e in ev:
        e[0].record()
        refine()
        e[1].record()
        e[2].record()
        grad()
        e[3].record()
    torch.cuda.synchronize()
    refine_ms = float(np.median([e[0].elapsed_time(e[1]) for e in ev]))
    grad_ms = float(np.median([e[2].elapsed_time(e[3]) for e in ev]))

    # what the refinement does, and whether cost / collide are the scorer's bits for the returned paths
    key = torch.empty(1, dtype=torch.int64, device=dev)
    c0 = torch.empty(B, dtype=torch.float32, device=dev)
    k0 = torch.empty(B, dtype=torch.uint8, device=dev)
    rm.score_paths_best(Z, W, SPC, True, None, out=(c0, k0), key=key)
    best0 = float(c0.min())
    Zo, c, k, acc = refine()
    cs = torch.empty_like(c)
    ks = torch.empty_like(k)
    rm.score_paths_best(Zo, W, SPC, True, None, out=(cs, ks), key=key)
    torch.cuda.synchronize()
    same_bits = bool(torch.equal(cs, c) and torch.equal(ks, k))
    red = ((c0 - c) / c0.abs()).double().cpu().numpy()

    def outcome(c_, k_, acc_):
        r = ((c0 - c_) / c0.abs()).double().cpu().numpy()
        return {'improved': round(float((c_ < c0).float().mean()), 5), 'median_rel_reduction': round(float(np.median(r)), 6),
                'mean_rel_reduction': round(float(r.mean()), 6), 'mean_accepted': round(float(acc_.float().mean()), 3),
                'worse': int((c_ > c0).sum()), 'new_collisions': int(((k0 == 0) & (k_ != 0)).sum())}

    sweep = {}
    if args.sweep:
        for step, mx, mn in [(0.25, 16.0, 1 / 256), (1.0, 16.0, 1 / 256), (4.0, 16.0, 1 / 256), (1.0, 4.0, 1 / 256),
                             (1.0, 64.0, 1 / 256), (1.0, 16.0, 1 / 16)]:
            _, c_, k_, a_ = refine(step_cells=step, max_step_cells=mx, min_step_cells=mn)
            sweep[f'step {step}, max {mx}, min {mn:g}'] = outcome(c_, k_, a_)

    # per-kernel device times, in a run of their own
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(2):
            refine()
        torch.cuda.synchronize()
    kernels = {}
    for a in prof.key_averages():
        t = getattr(a, 'device_time_total', None)
        if t is None:
            t = a.cuda_time_total
        if t > 0:
            kernels[a.key[:90]] = round(t / 2 / 1000.0, 4)       # ms per refine call
    step_ms = sum(v for kk, v in kernels.items() if 'uam_k_refine_step' in kk)
    kernels = dict(sorted(kernels.items(), key=lambda kv: -kv[1])[:8])

    name, power = card()
    res = {
        'workload': f'C3 shard: {B} paths x {bench.WP} waypoints, {bench.RASTER}^2 x 3 layers, spc = {SPC}; {K} trips',
        'refine_call_ms': round(refine_ms, 3), 'refine_ms_per_trip': round((refine_ms - grad_ms) / max(K, 1), 4),
        'grad_call_ms': round(grad_ms, 4), 'refine_step_kernel_ms_per_launch': round(step_ms / (K + 1), 4),
        'refine_kernels_ms_per_call': kernels,
        'cost_collide_equal_to_scorer': same_bits,
        'improved': round(float((c < c0).float().mean()), 5), 'median_rel_reduction': round(float(np.median(red)), 6),
        'mean_rel_reduction': round(float(red.mean()), 6), 'mean_accepted': round(float(acc.float().mean()), 3),
        'worse': int((c > c0).sum()), 'collide_before': int(k0.sum()), 'collide_after': int(k.sum()),
        'best_cost_before': best0, 'best_cost_after': float(c.min()),
        'defaults': {'step_cells': 1.0, 'max_step_cells': 64.0, 'min_step_cells': 1 / 256},
        'gpu': name, 'power_limit': power}
    if sweep:
        res['sweep'] = sweep
    print(json.dumps(res))


if __name__ == '__main__':
    main()
