"""Count the 128-byte lines and 32-byte sectors of quad texels that one 32-sample gather of the binned group loop touches, with
one tiled copy of the quads and with a transposed second copy read by steep segments (CPU only, no GPU).  The second copy is
modelled here only: built, it cut the count by 13-15 % and ran slower (DESIGN 4.1, profiles/r03_ab_quad_copies.txt).

The batch is a seeded sample of bench.py's C3 shard (8192^2 raster, 64 waypoints per path, samples_per_cell 1).  Per segment:
the oracle's sample arithmetic (U = (x - x0) / dx - 1/2, S = max(1, ceil(|dz|_pixels * spc)), step dU / S, plus the goal
pseudo-segment), the bin of uam_k_bin_hist (Morton id of the midpoint's 128-cell bin; with two copies the direction class
first), groups of 32 consecutive records, their samples concatenated, windows of 32 consecutive samples.  A sample reads the
quad of cell (floor v, floor u) (clamped like the kernel): copy 0 at uam_tex_row<4, 1>(i, rs0) + uam_tex_col<4, 1>(j), copy 1
(steep records: |SU| < |SV|) at n0 + uam_tex_row<4, 1>(j, rs1) + uam_tex_col<4, 1>(i); 8 quads per line, 2 per sector.

  python tools/gather_lines.py [--paths 2000] [--seed 2000]
"""
import argparse
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True


def tex_row(i, rs):
    return (i >> 1) * rs + ((i & 1) << 1)


def tex_col(j):
    return 2 * j - (j & 1)


def part1by1(x):
    x = x & 0xffff
    x = (x | (x << 8)) & 0x00ff00ff
    x = (x | (x << 4)) & 0x0f0f0f0f
    x = (x | (x << 2)) & 0x33333333
    return (x | (x << 1)) & 0x55555555


def records(Z, n, spc, dx):
    """per segment (path-major, goal pseudo-segment last): U, V, SU, SV, S and the float midpoint pixel coordinate"""
    B = Z.shape[0]
    P = Z.reshape(B, -1, 2)
    U = P[..., 0] / dx - 0.5
    V = P[..., 1] / dx - 0.5
    dU, dV = U[:, 1:] - U[:, :-1], V[:, 1:] - V[:, :-1]
    S = np.maximum(1.0, np.ceil(np.sqrt(dU * dU + dV * dV) * spc))
    z = np.zeros((B, 1))
    SU = np.concatenate([dU / S, z], 1)
    SV = np.concatenate([dV / S, z], 1)
    S = np.concatenate([S, z + 1], 1).astype(np.int64)
    Pn = np.concatenate([P[:, 1:], P[:, -1:]], 1)
    mu = np.clip(((P[..., 0] + Pn[..., 0]) * (0.5 / dx) - 0.5).astype(np.float32), 0, n - 1)
    mv = np.clip(((P[..., 1] + Pn[..., 1]) * (0.5 / dx) - 0.5).astype(np.float32), 0, n - 1)
    f = lambda a: a.reshape(-1)
    return f(U), f(V), f(SU), f(SV), f(S), f(mu), f(mv)


def count(U, V, SU, SV, S, order, two, n, n0, rs0, rs1):
    """mean distinct lines and sectors per 32-sample window, windows restarting at every group of 32 records"""
    U, V, SU, SV, S = U[order], V[order], SU[order], SV[order], S[order]
    rec = np.repeat(np.arange(len(S)), S)
    start = np.concatenate([[0], np.cumsum(S)[:-1]])
    s = np.arange(len(rec)) - start[rec]
    group = rec >> 5
    gstart = np.concatenate([[0], np.cumsum(np.add.reduceat(S, np.arange(0, len(S), 32)))[:-1]])
    window = (np.arange(len(rec)) - gstart[group]) >> 5
    wid = group.astype(np.int64) * (1 << 20) + window
    u = U[rec] + s * SU[rec]
    v = V[rec] + s * SV[rec]
    j = np.clip(np.floor(u), 0, n - 2).astype(np.int64)
    i = np.clip(np.floor(v), 0, n - 2).astype(np.int64)
    addr = tex_row(i, rs0) + tex_col(j)
    if two:
        steep = (np.abs(SU) < np.abs(SV))[rec]
        addr = np.where(steep, n0 + tex_row(j, rs1) + tex_col(i), addr)
    nw = len(np.unique(wid))
    lines = len(np.unique(np.stack([wid, addr >> 3], 1), axis=0))
    sectors = len(np.unique(np.stack([wid, addr >> 1], 1), axis=0))
    return lines / nw, sectors / nw, nw


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    ap.add_argument('--paths', type=int, default=2000, help='paths of the seeded sample of the C3 batch')
    ap.add_argument('--seed', type=int, default=2000, help="candidate seed (bench.py: rank 0's batch)")
    args = ap.parse_args()
    import bench
    n, spc, shift = bench.RASTER, bench.SPC, 7
    dx = bench.KM / n
    Z = bench.host_paths(args.paths, args.seed, n)
    U, V, SU, SV, S, mu, mv = records(Z, n, spc, dx)
    nsp_side = n >> shift
    morton = part1by1(mu.astype(np.int64) >> shift) | (part1by1(mv.astype(np.int64) >> shift) << 1)
    P = Z.reshape(Z.shape[0], -1, 2)
    Pn = np.concatenate([P[:, 1:], P[:, -1:]], 1)
    d = (Pn - P).reshape(-1, 2).astype(np.float32)
    steep_bin = np.abs(d[:, 0]) < np.abs(d[:, 1])
    rs0 = rs1 = ((n + 3) // 4) * 8
    n0 = ((n + 3) // 4) * ((n + 1) // 2) * 8
    print(f'{args.paths} paths x {P.shape[1] - 1} segments + goal, {int(S.sum())} samples; '
          f'{np.mean(np.abs(SU) < np.abs(SV)):.3f} of the segments steep')
    one = count(U, V, SU, SV, S, np.argsort(morton, kind='stable'), False, n, n0, rs0, rs1)
    key2 = morton + steep_bin.astype(np.int64) * nsp_side * nsp_side
    two = count(U, V, SU, SV, S, np.argsort(key2, kind='stable'), True, n, n0, rs0, rs1)
    print(f'{"layout":46s} lines/window  sectors/window  windows')
    print(f'{"one copy (Morton bins)":46s} {one[0]:12.2f}  {one[1]:14.2f}  {one[2]}')
    print(f'{"+ transposed copy for steep (class-major bins)":46s} {two[0]:12.2f}  {two[1]:14.2f}  {two[2]}')
    print(f'change: lines {100 * (two[0] / one[0] - 1):+.1f} %, sectors {100 * (two[1] / one[1] - 1):+.1f} %')


if __name__ == '__main__':
    main()
