"""Raster cost gradient on the C3 shard (bench.py's workload: 125 000 paths x 64 waypoints, 8192^2 3-layer raster,
integral mode at 1 sample per cell, bench.py's weights and seeds): step time of the gradient call against the scoring
step (score_paths_best), per-kernel times, and the gradient of 256 seeded paths against the float64 oracle.

    python bench_raster_grad.py [--paths 125000] [--steps 50] [--warmup 5]

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
    ap.add_argument('--steps', type=int, default=50)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--check', type=int, default=256, help='seeded paths compared with the oracle gradient')
    args = ap.parse_args()
    import torch
    import bench
    import uam_path_planning_b200 as uam
    sys.path.insert(0, os.path.join(ROOT, 'tests'))
    from raster_gradient_oracle import score_paths_raster_gradient

    assert torch.cuda.is_available(), 'bench_raster_grad.py needs a CUDA device'
    dev = 'cuda:0'
    torch.cuda.set_device(0)
    layers, occ, geo = bench.make_raster(torch, dev)
    rm = uam.RasterMap.from_arrays(layers, geo, occ)
    Z = bench.make_paths(torch, dev, args.paths, seed=1)
    B = Z.shape[0]
    cost = torch.empty(B, dtype=torch.float32, device=dev)
    col = torch.empty(B, dtype=torch.uint8, device=dev)
    key = torch.empty(1, dtype=torch.int64, device=dev)

    def score():
        rm.score_paths_best(Z, bench.WEIGHTS, bench.SPC, True, None, out=(cost, col), key=key)

    def grad():
        return rm.cost_gradient(Z, bench.WEIGHTS, bench.SPC, True, None)

    for _ in range(args.warmup):
        score()
        grad()
    torch.cuda.synchronize()
    # alternate the two calls in one process, each bracketed by its own events
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(args.steps)]
    for e in ev:
        e[0].record()
        score()
        e[1].record()
        e[2].record()
        grad()
        e[3].record()
    torch.cuda.synchronize()
    score_ms = float(np.median([e[0].elapsed_time(e[1]) for e in ev]))
    grad_ms = float(np.median([e[2].elapsed_time(e[3]) for e in ev]))

    # cost / collide are the scorer's bits
    c_g, k_g, g = grad()
    score()
    torch.cuda.synchronize()
    same_bits = bool(torch.equal(c_g, cost) and torch.equal(k_g, col))

    # per-kernel device times, in a run of their own
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(5):
            grad()
        torch.cuda.synchronize()
    kernels = {}
    for a in prof.key_averages():
        t = getattr(a, 'device_time_total', None)
        if t is None:
            t = a.cuda_time_total
        if t > 0:
            kernels[a.key[:90]] = round(t / 5 / 1000.0, 4)       # ms per gradient call
    kernels = dict(sorted(kernels.items(), key=lambda kv: -kv[1])[:8])

    # 256 seeded paths against the float64 oracle
    idx = np.sort(np.random.default_rng(20260105).choice(B, args.check, replace=False))
    Zc = Z[idx].cpu().numpy()
    _, _, _, g_ref = score_paths_raster_gradient(layers.cpu().numpy(), occ.cpu().numpy(), geo, Zc, bench.WEIGHTS,
                                                 bench.SPC, True, None)
    gd = g.cpu().numpy()[idx]
    err = np.abs(gd - g_ref).max(axis=1) / np.abs(g_ref).max(axis=1)
    name, power = card()
    print(json.dumps({
        'workload': f'C3 shard: {B} paths x {bench.WP} waypoints, {bench.RASTER}^2 x 3 layers, spc = {bench.SPC}',
        'score_step_ms': round(score_ms, 4), 'grad_step_ms': round(grad_ms, 4), 'grad_over_score': round(grad_ms / score_ms, 3),
        'grad_kernels_ms': kernels, 'cost_collide_equal_to_scorer': same_bits,
        'grad_rel_err_vs_oracle_max': float(err.max()), 'grad_rel_err_vs_oracle_median': float(np.median(err)),
        'checked_paths': int(args.check), 'gpu': name, 'power_limit': power}))


if __name__ == '__main__':
    main()
