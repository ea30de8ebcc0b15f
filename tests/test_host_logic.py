"""CPU-side tests: host logic of the product (shape tables, candidates, map file reader, sharding, key
packing), the C-ABI export list, and the no-CPU-fallback behaviour.  No kernel runs here."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import uam_path_planning_b200 as uam
from uam_path_planning_b200 import _lib, distributed as udist
from uam_path_planning_b200.shapes import flatten_shapes
from oracle import uam_oracle as orc
from conftest import ROOT, build_product_map, have_gpu


def _h_from_records(R, P):
    """Evaluate inequality records with the ORACLE's formulas (checker only)."""
    out = np.empty((R.shape[0], P.shape[0]))
    for i, r in enumerate(R):
        k = int(r[0])
        if k == _lib.UAM_EDGE_LINE:
            e = ('line', r[1], r[2], r[1] + r[3], r[2] + r[4], r[5])
            # the record stores Bx-Ax / By-Ay exactly; rebuild the oracle's op order from them
            line = r[4] * (P[:, 0] - r[1]) - r[3] * (P[:, 1] - r[2])
            out[i] = -r[5] * line
        elif k == _lib.UAM_EDGE_ELLIPSE:
            out[i] = orc.OShape('b', [('ellipse', r[1], r[2], r[3], r[4])], None, 0).h(P)[0]
        else:
            out[i] = orc.OShape('s', [('box', int(r[1]), r[2], r[3], r[4])], None, 0).h(P)[0]
    return out


def test_shape_tables_match_reference(fixture_spec, golden):
    """Edge order, signs and coefficients of every shape of the main.py map: evaluating the product's records
    reproduces the reference's h_i(x) bit for bit; centers and areas match."""
    m = build_product_map(fixture_spec)
    shapes = list(m.obstacles) + [s for r in m._region_lists() for s in r]
    off, P = golden['h_offsets'], golden['h_points']
    assert len(shapes) == len(off) - 1
    for k, s in enumerate(shapes):
        R = s.records()
        assert R.shape == (off[k + 1] - off[k], 8)
        assert np.array_equal(_h_from_records(R, P), golden['h_values'][off[k]:off[k + 1]]), k
        np.testing.assert_array_equal(np.asarray(s.center, dtype=float), golden['shape_centers'][k])
        assert s.area == pytest.approx(golden['shape_areas'][k], rel=1e-14)
    sp = uam.polygon(*golden['shuffled_poly_verts'].tolist())
    assert np.array_equal(_h_from_records(sp.records(), P), golden['shuffled_poly_h'])
    np.testing.assert_array_equal(sp.center, golden['shuffled_poly_center'])


def test_flatten_orders_obstacles_then_regions(fixture_spec):
    m = build_product_map(fixture_spec)
    edges, off, reg, cen = flatten_shapes(m.obstacles, m._region_lists())
    assert edges.shape == (143, 8) and off[0] == 0 and off[-1] == 143
    assert reg.tolist() == [-1] * 5 + [0] * 4 + [1] * 29 + [2]
    assert cen.shape == (39, 2) and not np.isnan(cen).any()
    bare = uam.QuadraticObstacle(*m.obstacles[0].inequalities)
    assert np.isnan(bare.center_or_nan()).all()


def test_constructor_errors(golden_meta):
    c = golden_meta['constructors']['errors']
    cases = {'two_vertices': [[0., 0.], [1., 1.]], 'aligned': [[0., 0.], [1., 0.], [2., 0.], [1., 1.]],
             'nonconvex': [[0., 0.], [2., 0.], [0.5, 0.5], [0., 2.]]}
    for name, pts in cases.items():
        with pytest.raises(ValueError) as ei:
            uam.polygon(*pts)
        assert str(ei.value) == c[name][1]
    with pytest.raises(Exception):              # integer first vertex + float vertices: numpy casting error (Q6)
        uam.polygon([0, 0], [1.5, 0.], [1., 1.])
    sq = uam.square([1, 1], 0.5)
    assert sq.area == 1.0 and len(sq.inequalities) == 4 and len(sq) == 4 and len(uam.ball(1.0)) == 1
    bl = uam.ball([1, 1], 2, 1)
    assert bl.area == pytest.approx(golden_meta['constructors']['ball_area'])
    assert uam.ball(3.0).records()[0].tolist() == [1, 0, 0, 3, 3, 0, 0, 0]


@pytest.mark.parametrize('N', [80, 62, 64, 5])
def test_create_x_init(fixture_spec, golden, golden_meta, N):
    m = build_product_map(fixture_spec)
    sol = uam.Solver(uam.Problem(m, N), {})
    for i, d in enumerate(golden['arc_disp']):
        np.testing.assert_allclose(sol.create_x_init(float(d)), golden[f'arc_N{N}_x'][i], rtol=1e-15, atol=1e-15)
    with pytest.raises(ValueError) as ei:
        sol.create_x_init(1.5)
    assert str(ei.value) == golden_meta['constructors']['errors']['x_init_1.5'][1]
    Z = sol.candidates([-0.5, 0.0, 0.5])
    assert Z.shape == (3, 2 * (N + 2)) and Z.flags.c_contiguous
    np.testing.assert_array_equal(Z[:, :2], np.tile(fixture_spec['x_start'], (3, 1)))
    np.testing.assert_array_equal(Z[:, -2:], np.tile(fixture_spec['x_goal'], (3, 1)))
    with pytest.raises(NotImplementedError):
        sol.solve(None, None)
    assert sol.get_error_code_explanation(3003) == 'Vector `parameter` has wrong length'
    assert sol.get_error_code_explanation(7) == 'Error code not found'


def test_region_map_container():
    m = uam.RegionMap()
    m.new_region('A', 'Red')
    with pytest.raises(ValueError) as ei:
        m.new_region('A', 'b')
    assert str(ei.value) == "Name 'A' already in use for areas"
    with pytest.raises(ValueError) as ei:
        m.add_shape_to_region('B', uam.ball(1.0))
    assert 'Unknown type' in str(ei.value)
    m.add_shapes_to_region('A', uam.ball(1.0), uam.square([0, 0], 1))
    m.add_obstacle(uam.ball([3, 3], 1))
    assert m.region_names() == ['A'] and len(m) == 1 and m.regions['A']['color'] == [1, 0, 0]
    assert m[0:1] == m.obstacles
    with pytest.raises(TypeError):
        m['x']
    prob = uam.Problem(m, 4)
    assert prob.weights == {'A': 1} and prob.options['penalty_smooth'] and not prob.options['length_smooth']
    prob.params.update(maxratio=1.1, maxalpha=0.1, enlargement=0.5)
    prob.set_weight('A', 7)
    np.testing.assert_array_equal(prob.parameter_vector(), [0, 0, 0, 0, 1.1, 0.1, 0.5, 7])
    assert prob.flags() == _lib.UAM_PENALTY_SMOOTH
    prob.params['enlargement'] = None
    with pytest.raises(TypeError):
        prob.parameter_vector()


def test_map_file_reader(tmp_path):
    txt = ('vertices = [polygon([16.0, 11.0], [11.5, -6.25], [30.25, -30.5], [32.0, -16.0], [28.5, 1.0]),\n'
           'polygon([0, 0], [2, 0], [2, 1], [0, 1]),\nball([1.0, -2.0], 3),\nsquare([1, 1], 0.5, 2)]\n')
    f = tmp_path / 'area.txt'
    f.write_text(txt)
    shapes = uam.get_var_from_file(str(f), 'vertices')
    assert [s.kind for s in shapes] == ['polygon', 'polygon', 'ball', 'square']
    assert len(shapes[0].inequalities) == 5 and shapes[1].area == 2.0
    o = orc.make_polygon([[16.0, 11.0], [11.5, -6.25], [30.25, -30.5], [32.0, -16.0], [28.5, 1.0]])
    P = np.random.default_rng(0).uniform(-40, 40, (32, 2))
    assert np.array_equal(_h_from_records(shapes[0].records(), P), o.h(P))
    for bad in ['import os\nvertices = []', 'vertices = [__import__("os").system("true")]',
                'vertices = [polygon([1, 2], [3, open("x")], [5, 6])]', 'vertices = 3']:
        with pytest.raises((ValueError, SyntaxError)):
            uam.parse_shapes(bad)
    with pytest.raises(KeyError):
        uam.parse_shapes('other = []')


def test_shard_range_and_keys():
    for total, world in [(1_000_000, 8), (10, 3), (5, 8), (0, 2)]:
        spans = [udist.shard_range(total, r, world) for r in range(world)]
        assert spans[0][0] == 0 and spans[-1][1] == total
        assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
        sizes = [e - b for b, e in spans]
        assert max(sizes) - min(sizes) <= 1
    with pytest.raises(ValueError):
        udist.shard_range(10, 3, 3)
    cost = np.array([5.0, 2.5, 2.5, 9.0], dtype=np.float32)
    k = udist.host_best_key(cost, 100)
    assert udist.decode_key(k) == (2.5, 101)          # tie -> smaller index
    assert udist.encode_key(2.5, 101) == k and 0 <= k < 2 ** 63
    assert udist.host_best_key(np.zeros(0)) == udist.KEY_EMPTY
    assert udist.global_best(k) == (2.5, 101)          # no process group: identity
    # the argmin shortcut and the image keys agree, also with zeros / negatives / NaN / inf in the vector (key order =
    # float order, -inf < negative < -0 < +0 < positive < inf < NaN, ties to the smaller index)
    rng = np.random.default_rng(3)

    def ref_key(c, off):
        order = sorted(range(c.size), key=lambda i: (np.isnan(c[i]), 0.0 if np.isnan(c[i]) else float(c[i]),
                                                     0 if np.isnan(c[i]) else (not np.signbit(c[i])), i))
        return order[0] + off
    for special in ([], [0.0], [np.nan], [np.inf, np.nan], [0.0, 0.0, np.nan], [-1.5, -1.5, 0.0], [-np.inf, -3.0],
                    [-0.0, 0.0], [-2.0, np.nan, -2.5]):
        c = rng.random(257).astype(np.float32) + np.float32(0.25)
        c[rng.choice(257, len(special), replace=False)] = special
        k = udist.host_best_key(c, 7)
        assert 0 <= k < udist.KEY_EMPTY
        cost_k, idx_k = udist.decode_key(k)
        assert idx_k == ref_key(c, 7), special
        assert cost_k == c[idx_k - 7] and np.signbit(cost_k) == np.signbit(c[idx_k - 7])
    assert udist.decode_key(udist.host_best_key(np.array([np.nan, 3.0, 1.0], dtype=np.float32)))[1] == 2
    # every key is a non-negative int64 below KEY_EMPTY, so an empty shard can never win a signed MIN reduction, and a
    # negative cost beats a positive one (ADVICE r1: the old bit-pattern key ranked negatives last and an empty shard first)
    assert udist.host_best_key(np.array([-1.0, 2.0], dtype=np.float32)) < udist.host_best_key(np.array([2.0], dtype=np.float32))
    assert udist.host_best_key(np.array([np.nan], dtype=np.float32)) < udist.KEY_EMPTY
    assert min(udist.KEY_EMPTY, udist.host_best_key(np.array([7.0], dtype=np.float32), 3)) != udist.KEY_EMPTY
    assert np.isnan(udist.decode_key(udist.KEY_EMPTY)[0])
    with pytest.raises(ValueError):
        udist.host_best_key(np.zeros(4, dtype=np.float32), 2 ** 31 - 2)


_GLOO_WORKER = r'''
import os, sys
import numpy as np, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from uam_path_planning_b200 import distributed as ud
dist.init_process_group('gloo', init_method='tcp://127.0.0.1:' + sys.argv[2], rank=int(sys.argv[3]), world_size=2)
rank = dist.get_rank()
rng = np.random.default_rng(7)
cost = rng.uniform(1, 100, 1001).astype(np.float32)      # the same global vector on both ranks
cost[[17, 700]] = 0.5                                     # tie across the two shards
b, e = ud.shard_range(cost.size, rank, 2)
key = torch.tensor([ud.host_best_key(cost[b:e], b)], dtype=torch.int64)
c, i = ud.global_best(key)
full = ud.gather_costs(torch.from_numpy(np.pad(cost[b:e], (0, 501 - (e - b)))))
assert (c, i) == (0.5, 17), (c, i)
assert full.numel() == 1002
# one rank with an empty shard (fewer units than ranks) and a negative cost on the other: the empty key must lose
one = np.array([-3.25], dtype=np.float32)
b, e = ud.shard_range(1, rank, 2)
key = torch.tensor([ud.host_best_key(one[b:e], b)], dtype=torch.int64)
assert ud.global_best(key) == (-3.25, 0)
# peer-group plumbing (the CUDA IPC handles are plain bytes): every rank ends up with all handles in rank order
class FakeEngine:
    def peer_handle(self): return bytes([rank]) * 64
    def attach_peers(self, r, handles): self.got = (r, list(handles))
fe = FakeEngine()
assert ud.attach_peer_group(fe) == 2
assert fe.got == (rank, [bytes([0]) * 64, bytes([1]) * 64])
print('ok', rank)
'''


def test_global_best_two_ranks_gloo(tmp_path):
    """world_size 2 over gloo: shard a cost vector, min-reduce the packed key, same answer on both ranks."""
    import socket
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    port = str(s.getsockname()[1])
    s.close()
    script = tmp_path / 'w.py'
    script.write_text(_GLOO_WORKER)
    procs = [subprocess.Popen([sys.executable, str(script), ROOT, port, str(r)], stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT, text=True) for r in range(2)]
    outs = [p.communicate(timeout=240)[0] for p in procs]
    for r, (p, o) in enumerate(zip(procs, outs)):
        assert p.returncode == 0 and f'ok {r}' in o, o


def test_c_abi_exports_every_declared_symbol():
    from uam_path_planning_b200 import build
    build.build()
    lib = _lib.load()
    hdr = open(os.path.join(ROOT, 'include', 'uam_b200.h')).read()
    declared = set(re.findall(r'\b(uam_[a-z0-9_]+)\s*\(', hdr))
    assert len(declared) >= 20
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    for name in declared:
        assert hasattr(lib, name), name
    assert b'sm_100a' in lib.uam_version()


def test_option_and_stat_tables_match_the_header():
    """Engine.OPTIONS / Engine.STATS are the enum values of include/uam_b200.h (UAM_OPT_* / UAM_STAT_*): every enumerator has
    its name in the Python table with the same number, and nothing else is in the tables."""
    import re
    from uam_path_planning_b200.engine import Engine
    hdr = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'include', 'uam_b200.h')).read()
    hdr = re.sub(r'/\*.*?\*/', ' ', hdr, flags=re.S)
    opts = {m.group(1).lower(): int(m.group(2)) for m in re.finditer(r'UAM_OPT_([A-Z0-9_]+)\s*=\s*(\d+)', hdr)}
    stats = {m.group(1).lower(): int(m.group(2)) for m in re.finditer(r'UAM_STAT_([A-Z0-9_]+)\s*=\s*(\d+)', hdr)}
    assert opts == Engine.OPTIONS, set(opts.items()) ^ set(Engine.OPTIONS.items())
    assert {k.replace('score_kernel_ms_mean', 'score_kernel_ms_mean'): v for k, v in stats.items()} == Engine.STATS, \
        set(stats.items()) ^ set(Engine.STATS.items())
    assert len(set(opts.values())) == len(opts) and len(set(stats.values())) == len(stats)


def test_no_cpu_fallback():
    """Without a GPU the product refuses to work: ctx creation fails and every evaluation raises.  On a machine with a GPU
    the same checks run in a child process that sees no device (CUDA_VISIBLE_DEVICES empty)."""
    if not have_gpu():
        _check_no_cpu_fallback()
        return
    code = 'import conftest, test_host_logic as t; t._check_no_cpu_fallback(); print("ok")'
    r = subprocess.run([sys.executable, '-c', code], cwd=os.path.dirname(os.path.abspath(__file__)), capture_output=True,
                       text=True, timeout=300, env=dict(os.environ, CUDA_VISIBLE_DEVICES=''))
    assert r.returncode == 0 and r.stdout.strip().endswith('ok'), r.stdout[-3000:] + r.stderr[-3000:]


def _check_no_cpu_fallback():
    lib = _lib.load()
    h = ctypes.c_void_p()
    assert lib.uam_ctx_create(0, ctypes.byref(h)) == -2 and not h.value
    with pytest.raises(uam.UamError):
        uam.Engine()
    with pytest.raises(uam.UamError):
        uam.ball(1.0).contains([0.0, 0.0])
    m = uam.RegionMap()
    with pytest.raises(uam.UamError):
        m.collides([0.0, 0.0])


def test_map_file_writer_round_trip_and_reference_file(tmp_path):
    """save_polygons writes the reference's format (data_manager.py:56-72); the reader takes it back bit for bit.  The
    text below is the head of the reference's data/processed/populated_area.txt."""
    ref_head = ('vertices = [polygon([28.836, -32.708], [29.607, -36.124], [32.53, -35.464], [31.759, -32.048]),\n'
                'polygon([29.185, -27.687], [29.35, -29.043], [32.001, -28.719], [31.835, -27.362])\n]')
    metres = [[(28836, -32708), (29607, -36124), (32530, -35464), (31759, -32048), (28836, -32708)],
              [(29185, -27687), (29350, -29043), (32001, -28719), (31835, -27362)]]
    f = tmp_path / 'populated_area.txt'
    uam.save_polygons(metres, str(f))
    assert f.read_text() == ref_head
    shapes = uam.get_var_from_file(str(f), 'vertices')
    assert len(shapes) == 2 and all(s.kind == 'polygon' and len(s.inequalities) == 4 for s in shapes)
    uam.save_polygons([], str(f))
    assert uam.get_var_from_file(str(f)) == []


def test_result_export_conventions():
    """main.py:103-116: km -> m (x1000), start / goal points prepended / appended, EPSG:2443 axis order."""
    x = [30.5, -20.25, 28.0, -5.0]
    pts = uam.result_points(x)
    assert pts.shape == (4, 2)
    assert pts[0].tolist() == [35590.685, -27711.422] and pts[-1].tolist() == [26478.673, 9564.082]
    assert pts[1].tolist() == [30500.0, -20250.0] and pts[2].tolist() == [28000.0, -5000.0]
    assert uam.result_wkt(x, [1, 2], [3, 4]) == 'LINESTRING (1.0 2.0, 30500.0 -20250.0, 28000.0 -5000.0, 3.0 4.0)'
    assert uam.result_wkt([], [1, 2], [3, 4], kind='points') == 'MULTIPOINT ((1.0 2.0), (3.0 4.0))'
    with pytest.raises(ValueError):
        uam.result_points([1.0, 2.0, 3.0])


def test_seed_from_grid_path_and_rect_area():
    """Host-side helpers around the grid search and the polygon front-end (no GPU involved): a grid route resampled into
    the flat (2N,) vector Solver.create_x_init returns (solver.py:103-136), the shoelace area used for the
    `p.area > min_approx_polygon_area` filter (map_generation/data_processor.py:34)."""
    m = uam.RegionMap()
    geo = (100.0, 2.0, -50.0, 2.0)                  # cell centres at x0 + (j + 1/2) dx, y0 + (i + 1/2) dy
    H, W = 40, 60
    # an L-shaped route on a 2-band grid: along row 5 from column 3 to 30, a band change, then down column 30 to row 25
    nodes = [5 * W + j for j in range(3, 31)] + [H * W + 5 * W + 30] + [H * W + i * W + 30 for i in range(6, 26)]
    m.x_start = [geo[0] + 3.5 * geo[1], geo[2] + 5.5 * geo[3]]
    m.x_goal = [geo[0] + 30.5 * geo[1], geo[2] + 25.5 * geo[3]]
    N = 46
    sol = uam.Solver(uam.Problem(m, N, {}), {})
    x = sol.seed_from_grid_path(nodes, (2, H, W), geo).reshape(N, 2)
    full = np.concatenate([[m.x_start], x, [m.x_goal]])
    steps = np.sqrt(((full[1:] - full[:-1]) ** 2).sum(1))
    route = 27 * 2.0 + 20 * 2.0                     # 27 cells east, 20 cells south
    assert np.all(steps <= route / (N + 1) + 1e-9)
    on_first_leg = np.isclose(x[:, 1], m.x_start[1])
    on_second_leg = np.isclose(x[:, 0], m.x_goal[0])
    assert np.all(on_first_leg | on_second_leg) and on_first_leg.sum() >= 20 and on_second_leg.sum() >= 15
    assert np.all(np.diff(x[on_first_leg, 0]) > 0) and np.all(np.diff(x[on_second_leg & ~on_first_leg, 1]) > 0)
    assert sol.seed_from_grid_path(nodes, (2, H, W), geo).shape == sol.create_x_init(0.0).shape
    # source == goal: every point is the start
    m.x_goal = m.x_start
    assert np.allclose(sol.seed_from_grid_path([5 * W + 3], (H, W), geo).reshape(N, 2), m.x_start)
    r = np.array([[[0, 0], [4, 0], [4, 3], [0, 3]], [[0, 0], [2, 2], [0, 4], [-2, 2]]], dtype=np.float64)
    assert np.allclose(uam.mapgen.rect_area(r), [12.0, 8.0])


def test_map_signature_follows_content(fixture_spec):
    """ADVICE r1: the cached device shape table must be re-uploaded after a shape changes and must not be confused by rebuilt
    lists whose objects reuse ids.  Centres and inequality records are stored read-only (an in-place edit raises), so every
    change is an assignment, and every assignment takes a fresh serial number that the signature carries."""
    from conftest import build_product_map
    m = build_product_map(fixture_spec)
    s0 = m._signature()
    assert s0 == m._signature()
    assert s0 != build_product_map(fixture_spec)._signature()          # other objects: re-upload (cheap, and always safe)
    with pytest.raises(ValueError):
        m.obstacles[0].center[0] = 1.0                                  # read-only
    with pytest.raises(ValueError):
        m.obstacles[1].inequalities[0].record[3] += 0.5                 # read-only
    m.obstacles[0].center = np.array([1.0, 2.0])
    s1 = m._signature()
    assert s1 != s0
    rec = m.obstacles[1].inequalities[0].record.copy()
    rec[3] += 0.5
    m.obstacles[1].inequalities[0].record = rec
    s2 = m._signature()
    assert s2 not in (s0, s1)
    m.regions['Land']['shapes'].pop()
    assert m._signature() not in (s0, s1, s2)
    import timeit
    assert timeit.timeit(m._signature, number=200) / 200 < 2e-3        # cheap enough to check on every call
