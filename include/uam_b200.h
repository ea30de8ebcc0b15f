/*
 * uam_b200.h -- C-ABI of the B200-native path scorer for nomaporon/uam_path_planning.
 *
 * The reference has no FFI of its own (it is pure Python); this header is the boundary a
 * maintainer binds with ctypes from the reference's Python classes (see INTEGRATION.md).  Each
 * entry point names the reference interface it replaces; file:line are relative to
 * geo_simulation_project/ in the reference tree.
 *
 * Conventions
 *   - plain C: pointers, sizes, doubles.  No C++ / torch types.
 *   - every call returns int: 0 = UAM_OK, negative = error; never throws, never aborts.
 *     uam_last_error(ctx) gives the message of the last failing call on that ctx.
 *   - pointers named d_* are DEVICE pointers owned by the caller (e.g. torch tensor data_ptr());
 *     pointers named h_* (and all small parameter tables) are HOST pointers.
 *   - `stream` is the caller's cudaStream_t passed as void* (NULL = CUDA's default stream, as in
 *     every CUDA API).  Device-pointer calls are asynchronous and stream-ordered; host-buffer
 *     calls (*_host) run on the ctx's own streams and return when the results are in the
 *     caller's host buffers.
 *   - a ctx is bound to one GPU and is not thread-safe.  No global state.  There is no CPU
 *     fallback: without a CUDA device uam_ctx_create fails with UAM_ERR_CUDA.
 *
 * Layouts (kept from the reference)
 *   paths   z_  : (B, 2*(N+2)) float64, C-contiguous, interleaved [xs,ys,x1,y1,...,xN,yN,xg,yg]
 *                 = start + N free waypoints + goal      (path_generation/solver.py:59-66)
 *   params  p   : [ms_x, ms_y, mg_x, mg_y, maxratio, maxalpha, enlargement, w_0 .. w_{R-1}]
 *                 (solver.py:60-68; p[0:4] = map.x_start / map.x_goal as used by
 *                 Problem.length_of, problem.py:137-140; weights in region insertion order)
 *   rasters     : (L, H, W) float32 C-order, row <-> y, col <-> x, affine (x0, dx, y0, dy),
 *                 cell centre (x0 + (j+1/2) dx, y0 + (i+1/2) dy); occupancy (H, W) uint8
 *                 (rasterio band layout as read at map_generation/data_manager.py:13)
 */
#ifndef UAM_B200_H
#define UAM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct uam_ctx uam_ctx;

enum {
    UAM_OK = 0,
    UAM_ERR_INVALID = -1,      /* bad argument */
    UAM_ERR_CUDA = -2,         /* CUDA runtime error (message in uam_last_error) */
    UAM_ERR_NOMEM = -3,
    UAM_ERR_STATE = -4,        /* required map state missing (no shapes / no raster uploaded) */
    UAM_ERR_UNSUPPORTED = -5
};

/* option flags = Problem.options (path_generation/problem.py:12-17) */
enum {
    UAM_LENGTH_SMOOTH   = 1 << 0,
    UAM_PENALTY_SMOOTH  = 1 << 1,
    UAM_OBSTACLE_SMOOTH = 1 << 2,
    UAM_MAXRATIO_SMOOTH = 1 << 3,
    /* the length term's first pair is (map.x_start, z_0) (problem.py:137-145).  With this flag the
     * scorer uses each path's own z_0 instead of p[0:2], i.e. the term is 0 -- for batches of
     * independent start/goal queries. */
    UAM_OWN_START       = 1 << 4
};

/* inequality record kinds of uam_map_set_shapes: 8 doubles per record, rec[0] = kind */
enum {
    UAM_EDGE_LINE = 0,     /* rec = {0, Ax, Ay, Bx-Ax, By-Ay, sgn, 0, 0}   h = -sgn*((By-Ay)(x-Ax) - (Bx-Ax)(y-Ay))
                              path_generation/polygon.py:69-71,98 */
    UAM_EDGE_ELLIPSE = 1,  /* rec = {1, cx, cy, r1, r2, 0, 0, 0}           h = ((x-cx)/r1)^2 + ((y-cy)/r2)^2 - 1
                              path_generation/ball.py:33-37 */
    UAM_EDGE_BOX = 2       /* rec = {2, axis, sign, c, r, 0, 0, 0}         h = sign>0 ? x_d - c - r : -x_d + c - r
                              path_generation/square.py:29-51 */
};

/* ---- context ------------------------------------------------------------------------------- */
int uam_ctx_create(int device, uam_ctx** ctx);
int uam_ctx_destroy(uam_ctx* ctx);
const char* uam_last_error(const uam_ctx* ctx);
const char* uam_version(void);
/* number of kernels this ctx has launched since creation (bench.py's gpu_launches) */
int uam_launch_count(const uam_ctx* ctx, uint64_t* n);
/* wait for the ctx's own streams */
int uam_sync(uam_ctx* ctx);
/* tuning knobs (defaults are the measured-best settings; see DESIGN.md) */
enum {
    UAM_OPT_RASTER_LAYOUT = 1,        /* texel layout used by the next uam_map_set_raster*: 0 row-major, 1 tiled */
    UAM_OPT_INTEGRAL_VARIANT = 2,     /* integral mode: -1 auto (default: 2 for batches of >= 2^18 segments, else 0),
                                         0 warp per path / lane per sample, 1 lane pair per sample,
                                         2 segments binned by raster tile, warp per 32 sorted segments,
                                         3 segments cut at 64 x 64-cell tile boundaries, pieces sorted by tile, the
                                           tile staged in shared memory by one bulk async copy (cp.async.bulk) */
    UAM_OPT_L2_FETCH_GRANULARITY = 3, /* cudaLimitMaxL2FetchGranularity for this device: 32, 64 or 128 bytes */
    UAM_OPT_TIME_KERNELS = 4,         /* 1: bracket the dominant raster-scoring kernel of every device-pointer call with
                                         CUDA events on the caller's stream (resets the statistics) */
    UAM_OPT_GRID_DELTA = 6,           /* grid search: width of the distance window relaxed per round (0 = automatic: the cost
                                         of crossing one 32-cell tile at the mean cell cost); ordering only, same results */
    UAM_OPT_COMBINE_LAYERS = 5,       /* 1 (default): large-batch integral mode (and waypoint mode) samples the layers folded
                                         into ONE layer sum_l w_l * layer_l (the penalty is linear in the layers).  First
                                         choice is the "gather layer": 4 bytes per cell in a 2-D CUDA array, occupancy in
                                         the sign bits, a tap is one tex2Dgather of the 2 x 2 bilinear footprint.  Integral
                                         variant 3, rasters beyond the device's gather limits and folded values < 0 use
                                         "quad texels" instead: every cell stores its footprint as one float4, a tap is one
                                         16-byte load; occupancy flags ride in the sign bits when all values are >= 0, else
                                         in a bit-plane.  Rebuilt when the weights or the raster change.  2: always the
                                         quad texels with the bit-plane.  0: always sample every layer texel by texel */
    UAM_OPT_HOST_CHUNKS = 7,          /* uam_score_paths_raster_host: chunks per call flowing through the copy / score
                                         pipeline (0 = default 4) */
    UAM_OPT_HOST_TAPER = 8,           /* ... chunk sizes change linearly from the first to the last chunk: t > 0 the last chunk
                                         is t percent smaller than the first, t < 0 the first is |t| percent smaller than the
                                         last, 0 (default) equal chunks; -95 .. 95 */
    UAM_OPT_RASTERIZER = 10,          /* 1 (default): uam_rasterize_occupancy / uam_rasterize_layers find, per raster row and shape, the
                                         interval of cells inside the shape by bisection with the exact fp64 predicate (the value of
                                         an inequality along a row is monotone in the column) and only touch those cells; 0: every
                                         cell of every surviving tile is evaluated (round-1 kernels); 2: as 1 with the tile form of the
                                         layer kernel (row intervals by bisection inside 16 x 64 tiles); 3: as 1 with the sampled row
                                         form of the layer kernel (coarse spans from 32 sample columns per row).  Same bits in every mode */
    UAM_OPT_CCL_TILES = 11,           /* 1 (default): uam_label_components labels 32 x 32-cell tiles in shared memory first and unites only
                                         the pairs across tile borders in HBM; 0: global union-find over all cells (round 1).  Same labels */
    UAM_OPT_GRID_GRAPH = 12,          /* 1 (default): the relaxation rounds of uam_grid_search* are looped on the device -- one CUDA graph
                                         with a WHILE conditional node whose body is a round (min key, selection, tile relaxation) and a
                                         one-thread kernel that re-arms the loop while tiles are pending; 0: the host enqueues the rounds
                                         and reads the active count back every 8 rounds.  Same results */
    UAM_OPT_GRID_HALF_CAP = 13,       /* grid search: half sweeps (32 row steps) a tile activation may run before the tile is handed to the
                                         next round with what it has (default 4 = two double sweeps; 0: to the fixed point).  Scheduling
                                         only, same results */
    UAM_OPT_SHAPE_GRID = 9            /* 1 (default): the analytic scorer / point queries look up per-cell candidate lists over
                                         the shapes (a shape with one inequality > max(e, 1e-14) on a whole cell contributes
                                         exact zeros there and is left out; same bits).  0: every shape at every point */
};
/* statistics of UAM_OPT_TIME_KERNELS: mean device time (ms) of the dominant scoring kernel (uam_k_score_tiles / uam_k_score_groups /
 * uam_k_score_raster_int / uam_k_score_raster_wp) over the timed calls, and their number */
enum { UAM_STAT_SCORE_KERNEL_MS_MEAN = 1, UAM_STAT_SCORE_KERNEL_COUNT = 2,
       /* counted work of the last uam_grid_search*: tile activations, double sweeps (one = 64 row steps of 32 cells, each
          relaxing the 8 in-plane edges of its cells), relaxation rounds */
       UAM_STAT_GRID_ACTIVATIONS = 3, UAM_STAT_GRID_SWEEPS = 4, UAM_STAT_GRID_ROUNDS = 5,
       /* shape grid of the analytic scorer (UAM_OPT_SHAPE_GRID) as last built: cells (0 = none) and list entries in all */
       UAM_STAT_SHAPE_GRID_CELLS = 6, UAM_STAT_SHAPE_GRID_ITEMS = 7,
       /* what the host enqueued for the last uam_grid_search*: kernel launches + memsets + graph launches (UAM_OPT_GRID_GRAPH) */
       UAM_STAT_GRID_HOST_SUBMISSIONS = 8 };
int uam_ctx_get_stat(uam_ctx* ctx, int stat, double* value);
int uam_ctx_set_option(uam_ctx* ctx, int option, int64_t value);

/* ---- map: shape tables ------------------------------------------------------------------------
 * Replaces the object graph RegionMap / Map / QuadraticObstacle / Function
 * (path_generation/region_map.py:8-61, map.py:7-43, quadratic_obstacle.py:8-39, function.py:119).
 *   h_edges        n_edges x 8 doubles, inequality records in reference order
 *   h_shape_off    n_shapes+1 prefix into h_edges
 *   h_shape_region n_shapes: -1 = hard obstacle (map.obstacles), else region index (insertion order)
 *   h_shape_center n_shapes x 2: QuadraticObstacle.center; NaN = none (penalty not normalised,
 *                  problem.py:76-77)
 * Obstacles keep insertion order among themselves (it is the order of get_nonlincon's blocks). */
int uam_map_set_shapes(uam_ctx* ctx, const double* h_edges, int n_edges, const int32_t* h_shape_off,
                       const int32_t* h_shape_region, const double* h_shape_center, int n_shapes,
                       int n_regions);

/* ---- map: rasters -------------------------------------------------------------------------------
 * Upload L float32 cost layers + uint8 occupancy; the library re-lays them out on the device
 * (texel-interleaved).  L in [1,3].  Host and device-pointer forms. */
int uam_map_set_raster(uam_ctx* ctx, const float* h_layers, int L, int H, int W, double x0, double dx,
                       double y0, double dy, const uint8_t* h_occupancy);
int uam_map_set_raster_device(uam_ctx* ctx, const float* d_layers, int L, int H, int W, double x0,
                              double dx, double y0, double dy, const uint8_t* d_occupancy, void* stream);

/* ---- candidates ---------------------------------------------------------------------------------------
 * Solver.create_x_init (path_generation/solver.py:103-136) for B displacements at once: d_z (B, 2(N+2)) float64
 * receives [start, arc through start and goal with sagitta d_b |goal-start|/2 (straight line for d_b = 0), goal].
 * h_ends = [x_start(2), x_goal(2)]; |d_b| <= 1 is the caller's check (the reference raises ValueError). */
int uam_make_arc_paths(uam_ctx* ctx, const double* h_ends, int N, const double* d_displacement, int64_t B,
                       double* d_z, void* stream);

/* The general form: row b of d_cand = {xs, ys, xg, yg, displacement} -- every candidate its own start / goal (a batch of
 * independent start/goal queries, 40 bytes each) -- and, for jitter_sigma > 0, N(0, sigma^2) added to both coordinates of
 * the N interior waypoints (start and goal stay fixed, as in the reference's flow create_x_init -> solve, main.py:160-171).
 * The normals come from a counter-based generator keyed by (seed, index0 + b, waypoint): a candidate depends on its global
 * index only, not on the batch split or the number of GPUs. */
int uam_make_candidates(uam_ctx* ctx, const double* d_cand, int64_t B, int N, double jitter_sigma, uint64_t seed,
                        uint64_t index0, double* d_z, void* stream);

/* ---- path scoring: analytic shapes -------------------------------------------------------------
 * Replaces, batched over B paths:
 *   d_cost[b]    = Problem.get_cost(z_)                      path_generation/problem.py:38-44
 *                  (length term incl. the dropped-last-segment behaviour of problem.py:39,140-145)
 *   d_collide[b] = any_j Map.collides(z_j)                   map.py:41-43, quadratic_obstacle.py:89-94
 *   d_g[b,:]     = Problem.get_nonlincon(z_)  (nullable)     problem.py:84-114, length 3N + n_obs(N+2)
 * All fp64 in the reference's operation order (no FMA contraction): inequalities, collision flags
 * and the zero pattern of g are bit-exact; costs differ from the reference only through the order
 * in which the per-waypoint terms are summed (warp-shuffle tree), ~1e-15 relative.
 * uam_analytic_g_len gives the row length of d_g for this map and N. */
int uam_score_paths_analytic(uam_ctx* ctx, const double* d_z, int64_t B, int N, const double* h_p,
                             int n_p, int flags, double* d_cost, uint8_t* d_collide, double* d_g,
                             void* stream);
int uam_score_paths_analytic_host(uam_ctx* ctx, const double* h_z, int64_t B, int N, const double* h_p,
                                  int n_p, int flags, double* h_cost, uint8_t* h_collide, double* h_g);
int uam_analytic_g_len(const uam_ctx* ctx, int N, int64_t* len);

/* Gradient of Problem.get_cost with respect to every waypoint: d_grad (B, 2(N+2)) float64, same layout as d_z
 * (columns 2 .. 2N+1 are the solver's decision variables z_1..z_N, solver.py:59); d_cost nullable.  The reference gets
 * this derivative from CasADi's algorithmic differentiation inside OpEn (solver.py:82-101); here it is analytic, fp64.
 * Needs UAM_PENALTY_SMOOTH.  The length term follows get_cost (last segment absent, problem.py:39,140-145). */
int uam_grad_paths_analytic(uam_ctx* ctx, const double* d_z, int64_t B, int N, const double* h_p, int n_p, int flags,
                            double* d_cost, double* d_grad, void* stream);

/* Problem.length_of(x, smooth) (problem.py:130-146) for B rows of M points each (x is (B, 2M) float64):
 * y = [map.x_start; x; map.x_goal], out = sum of nrm(y_{k+1} - y_k) over the FIRST N+1 pairs (N <= M).
 * M = N reproduces Solver.solve's call (solver.py:49), M = N+2 the call inside get_cost (problem.py:39).
 * h_ends = [x_start(2), x_goal(2)]. */
int uam_length_of(uam_ctx* ctx, const double* d_x, int64_t B, int M, int N, const double* h_ends, int smooth,
                  double* d_out, void* stream);
int uam_length_of_host(uam_ctx* ctx, const double* h_x, int64_t B, int M, int N, const double* h_ends,
                       int smooth, double* h_out);

/* ---- path scoring: rasters ----------------------------------------------------------------------
 * Same cost functional with P(x) = sum_l w_l * bilinear(layer_l, x) and collision = occupancy of
 * the nearest cell.  samples_per_cell == 0: one sample per waypoint (the reference's sampling,
 * problem.py:42-43).  > 0: every segment is sampled S_k = max(1, ceil(|dz_k|_cells * samples_per_cell))
 * times (left-endpoint rule, mean per segment; S_k capped at 2^20) -- build-defined line-integral
 * extension.  p[7:] are the L layer weights.  World->pixel coordinates, S_k and sample positions are
 * fp64 (same cells and sample counts as the oracle, bit for bit); texel arithmetic and the penalty
 * sum are fp32; the length term is fp64; d_cost is float32.  d_nsamples (nullable, int64 per path)
 * receives the number of raster samples taken for the path. */
int uam_score_paths_raster(uam_ctx* ctx, const double* d_z, int64_t B, int N, const double* h_p, int n_p,
                           int flags, double samples_per_cell, float* d_cost, uint8_t* d_collide,
                           int64_t* d_nsamples, void* stream);
int uam_score_paths_raster_host(uam_ctx* ctx, const double* h_z, int64_t B, int N, const double* h_p,
                                int n_p, int flags, double samples_per_cell, float* h_cost,
                                uint8_t* h_collide);

/* Gradient of the raster cost with respect to every waypoint: d_grad (B, 2(N+2)) float64, same layout as d_z (columns
 * 2 .. 2N+1 are the solver's variables z_1..z_N).  d_cost / d_collide (nullable) receive the same bits as
 * uam_score_paths_raster for the same inputs and options, so the gradient is that of the function being scored:
 *   - the sample counts S_k are held fixed: S_k is piecewise constant in z and the cost jumps where it changes; the
 *     gradient is that of the piece the path is on;
 *   - dP/du on the cell the scorer samples, at its fp32 fractions: sum_l w_l ((1-fy)(t01-t00) + fy(t11-t10)) (dP/dv
 *     likewise), 0 in a coordinate whose clamp to [0, W-1] / [0, H-1] is active; du/dx = 1/dx, dv/dy = 1/dy;
 *   - sample s of segment k moves with weight 1 - s/S_k with z_k and s/S_k with z_{k+1}; the goal sample with z_{N+1};
 *   - the length part is uam_grad_paths_analytic's (fp64, pairs (m_s, z_0) unless UAM_OWN_START, last segment absent;
 *     2 d with UAM_LENGTH_SMOOTH, else d / |d| with the zero subgradient at |d| = 0), times N+1.
 * Penalty slopes are summed in fp32 like the cost, in an order fixed per path: a path's gradient has the same bits
 * whatever else the batch holds.  Same kernel choice as the scorer (waypoint kernel; integral mode: variant -1 / 0 / 2,
 * quad texels where the scorer uses them); a forced integral variant 1 or 3 gives UAM_ERR_UNSUPPORTED. */
int uam_grad_paths_raster(uam_ctx* ctx, const double* d_z, int64_t B, int N, const double* h_p, int n_p, int flags,
                          double samples_per_cell, float* d_cost, uint8_t* d_collide, double* d_grad, void* stream);

/* Refine every path of d_z in place by monotone descent on the raster cost of uam_grad_paths_raster (same p, flags and
 * samples_per_cell), each path with its own step.  "Evaluate Z" below is one gradient launch on the whole batch:
 * (c f32, k u8, g f64), c / k being uam_score_paths_raster's bits.  Per path, with h = min(|dx|, |dy|) of the raster:
 *   start: tau = step_cells, accepted = 0, (c, k, g) = evaluate(Z);
 *   each of the `iterations` trips:
 *     1. m = max |g| over the free columns 2 .. 2N+1; the path is active iff tau >= min_step_cells, every free g is
 *        finite, m > 0 and c is finite;
 *     2. trial Zt: free columns Z - r g with r = (tau h) / m (fp64, rounded multiply, divide, subtract: no waypoint
 *        moves more than tau cells) for an active path, Zt = Z otherwise; columns 0, 1, 2N+2, 2N+3 are never written;
 *     3. (ct, kt, gt) = evaluate(Zt) for the whole batch;
 *     4. accept iff active and kt <= k and ct < c (float32; a NaN ct rejects): Z, c, k, g <- Zt, ct, kt, gt,
 *        tau <- min(2 tau, max_step_cells), accepted += 1; an active path that is not accepted halves tau.
 * On return d_z, d_cost and d_collide hold the final Z, c and k (c / k = uam_score_paths_raster's bits for the returned
 * paths), d_accepted (int32, nullable) the accepted trips.  So a path's (collide, cost) never gets worse, a path that did
 * not collide never starts to, and a row with NaN or inf in its gradient is left as it was.  The penalty layers carry no
 * obstacle term: refinement does not steer a colliding path out of an obstacle.  S_k may change along the way (the cost
 * is piecewise smooth); the accept test uses the scored cost.  Everything after the quad texels are built (see
 * uam_raster_precompute: the first call for a raster / weights may synchronise) is ordered on `stream`: iterations + 1
 * gradient launches and as many uam_k_refine_step launches, no host read-back.  Scratch: 48 (N + 2) + 18 bytes per path,
 * kept by the ctx.  B = 0 is a no-op; iterations < 0, step sizes that are not finite or break
 * 0 < min_step_cells <= step_cells <= max_step_cells, or a NULL pointer (d_accepted excepted) give UAM_ERR_INVALID; no
 * raster UAM_ERR_STATE; a forced integral variant 1 or 3 UAM_ERR_UNSUPPORTED, as for the gradient. */
int uam_refine_paths_raster(uam_ctx* ctx, double* d_z, int64_t B, int N, const double* h_p, int n_p, int flags,
                            double samples_per_cell, int iterations, double step_cells, double max_step_cells,
                            double min_step_cells, float* d_cost, uint8_t* d_collide, int32_t* d_accepted,
                            void* stream);

/* uam_refine_paths_raster with the swept check (uam_sweep_paths_raster, below) in its accept test, so that refinement
 * never moves a path into an occupied cell between the scorer's samples, and, with min_d2 > 0, never closer than
 * sqrt(min_d2) cells to an obstacle.  The rule is exactly uam_refine_paths_raster's (steps 1 - 4 above) with two
 * additions:
 *   - "evaluate Z" also runs the swept check on the whole batch: f = its flags (UAM_SWEEP_HIT | OUTSIDE | INVALID) and,
 *     when the clearance is used (min_d2 > 0 or a non-NULL d_d2min), d2 = its d2min; these are uam_sweep_paths_raster's
 *     bits;
 *   - step 4 becomes: accept iff active and kt <= k and ct < c and (ft & ~f) == 0 and
 *     (min_d2 == 0 or min(d2t, min_d2) >= min(d2, min_d2)) (signed int32: d2 = -1, no raster cell touched, is the
 *     worst); on accept also f, d2 <- ft, d2t.
 * So a trial never adds a swept flag the path did not have: a path inside the raster that sweeps clean stays clean,
 * inside and valid.  A path that is already HIT may still be accepted into collide = 0 while it crosses an occupied
 * cell: it gains no flag.  With min_d2 > 0 a path's clearance capped at min_d2, min(d2min, min_d2), never decreases: a path
 * that starts at least sqrt(min_d2) cells from every occupied cell ends so too.  Every trial this call accepts,
 * uam_refine_paths_raster would have accepted as well; when the swept conditions never reject a trial, the outputs
 * are bit-identical to it.  On return d_cost / d_collide hold uam_score_paths_raster's bits for the returned paths, as
 * there, and d_sweep_flags (uint8, required) / d_d2min (int32, nullable) uam_sweep_paths_raster's flags / d2min.
 * min_d2 is in squared cells, the unit of d2min, in 0 .. 65535.  With d_d2min NULL and min_d2 > 0 the clearance is kept
 * in scratch; with d_d2min NULL and min_d2 == 0 no clearance is computed.  Each trip adds one sweep launch of the trial
 * batch after its gradient launch, on `stream`, no host read-back.  The occupancy bit-plane, the d^2 field (clearance
 * only) and the quad texels are built first when missing (each may synchronise).  Scratch: that of
 * uam_refine_paths_raster + 1 byte per path, + 4 with the clearance, + 4 more when d_d2min is NULL.  Errors: those of
 * uam_refine_paths_raster in the same order (min_d2 out of range is UAM_ERR_INVALID with the step sizes, a NULL
 * d_sweep_flags with the other pointers); then UAM_ERR_UNSUPPORTED for the clearance on a raster over 23170 cells per
 * side or an N too large for the sweep's shared-memory table (N <= 3656), both before anything is built or reserved. */
int uam_refine_paths_raster_swept(uam_ctx* ctx, double* d_z, int64_t B, int N, const double* h_p, int n_p, int flags,
                                  double samples_per_cell, int iterations, double step_cells, double max_step_cells,
                                  double min_step_cells, int min_d2, float* d_cost, uint8_t* d_collide,
                                  int32_t* d_accepted, uint8_t* d_sweep_flags, int32_t* d_d2min, void* stream);

/* uam_refine_paths_raster with the analytic check (uam_sweep_paths_analytic and uam_clearance_paths_analytic, below) in
 * its accept test, so that refinement never moves a path into a no-fly shape, between the raster's cell centres as
 * well, and, with margin > 0, never closer than margin (map units, km) to one.  The shapes are those of the last
 * uam_map_set_shapes.  The rule is exactly uam_refine_paths_raster's (steps 1 - 4 above) with two additions:
 *   - "evaluate Z" also computes, for the whole batch, f = the flags of uam_sweep_paths_analytic (UAM_SWEEP_HIT |
 *     INVALID) and, with margin > 0, cl = the clearance of uam_clearance_paths_analytic at cap = margin; these are those
 *     calls' bits;
 *   - step 4 becomes: accept iff active and kt <= k and ct < c and (ft & ~f) == 0 and (margin == 0 or clt >= cl) (fp64;
 *     a NaN compares false and rejects); on accept also f, cl <- ft, clt.
 *   K1 (no new hit): a trial never adds HIT or INVALID: a path that sweeps clean against the shapes stays clean, with
 *      G1's "never misses" carried over;
 *   K2 (keep-out): with margin > 0, min(clearance, margin) never drops: a path that starts at least margin from every
 *      obstacle (up to the clearance's delta, D2) ends so, and one that starts closer never gets closer;
 *   K3 (refines no further than the plain call): every trial this call accepts, uam_refine_paths_raster would have
 *      accepted as well; when the new terms never reject a trial (for example a map without obstacles, or with
 *      obstacles far from every path), the outputs are bit-identical to it;
 *   K4 (outputs): on return d_cost / d_collide hold uam_score_paths_raster's bits for the returned paths, as there;
 *      d_sweep_flags (uint8, required) uam_sweep_paths_analytic's flags; d_clearance (float64, nullable, only with
 *      margin > 0) uam_clearance_paths_analytic's clearance at cap = margin.
 * A path that is already HIT may still be accepted into collide = 0 while it cuts a shape: that trial adds no flag.  With
 * margin > 0 a path whose clearance is NaN (INVALID) takes no trial.  margin is in [0, 1e100]; margin = 0 uses the sweep
 * only.  Each trip adds one launch of the analytic sweep (margin = 0) or of the analytic clearance (margin > 0) of the
 * trial batch after its gradient launch, on `stream`, no host read-back.  The record checks and the sweep's cell lists,
 * the clearance's lists for cap = margin (both cached: per upload, and per upload and cap) and the quad texels are built
 * first when missing (each may synchronise).  Scratch: that of uam_refine_paths_raster + 1 byte per path, + 8 with
 * margin > 0, + 8 more when d_clearance is NULL.  Errors, in this order: those of uam_refine_paths_raster in the same
 * order (margin out of range or N > 2^28 is UAM_ERR_INVALID with the step sizes; a NULL d_sweep_flags, or a non-NULL
 * d_clearance with margin = 0, UAM_ERR_INVALID with the other pointers); no shapes uploaded UAM_ERR_STATE; the sweep's
 * record checks, then with margin > 0 the clearance's form checks, UAM_ERR_UNSUPPORTED; all before any quad build or
 * scratch reservation. */
int uam_refine_paths_raster_keepout(uam_ctx* ctx, double* d_z, int64_t B, int N, const double* h_p, int n_p, int flags,
                                    double samples_per_cell, int iterations, double step_cells, double max_step_cells,
                                    double min_step_cells, double margin, float* d_cost, uint8_t* d_collide,
                                    int32_t* d_accepted, uint8_t* d_sweep_flags, double* d_clearance, void* stream);

/* Swept check of whole path segments against the raster's occupancy, and each path's clearance.  The scorer above only
 * looks at its samples; this call looks at every cell a segment crosses.  For every path of d_z (B, 2(N+2)) and every
 * segment k = 0 .. N (z_k -> z_{k+1}):
 *   1. pixel coordinates U = (x - x0)/dx - 0.5, V = (y - y0)/dy - 0.5 in fp64, in the scorer's order (round-to-nearest
 *      divide, then subtract, no FMA): oracle.pixel_coords before its clamp.  Cell (i, j) has its centre at (U, V) = (j, i)
 *      and its square is [j - 1/2, j + 1/2] x [i - 1/2, i + 1/2].
 *   2. fixed point: Uq = rint(U 2^16), Vq = rint(V 2^16) (int64, ties to even).  A path with a non-finite coordinate or with
 *      |U| or |V| >= 2^31 gets flags = UAM_SWEEP_INVALID and nothing else is evaluated for it: first hit = -1, d2min = -1.
 *   3. a raster cell (0 <= i < H, 0 <= j < W) is touched by a segment iff the closed quantised segment meets the cell's
 *      closed square dilated by one quantum: in fixed-point units the box [(2j-1) 2^15 - 1, (2j+1) 2^15 + 1] in u, likewise
 *      in v.  Exact integer arithmetic (128-bit products of 48-bit differences): a zero-length segment touches the cells
 *      around its point, a segment along a cell edge touches both sides, one through a grid vertex all four cells.
 *   4. per path:
 *      d_flags (uint8):         UAM_SWEEP_HIT: some segment touches an occupied cell;
 *                               UAM_SWEEP_OUTSIDE: some waypoint lies outside the closed raster rectangle
 *                               [-1/2, W-1/2] x [-1/2, H-1/2] (only raster cells are ever tested, the part outside is not
 *                               judged); UAM_SWEEP_INVALID: see 2.
 *      d_first_hit (int32, nullable): the lowest k whose segment touches an occupied cell, -1 if none.
 *      d_d2min (int32, nullable):     min over all touched cells of min(d2, 65535), d2 = squared distance in cells from the
 *                               cell's centre to the nearest occupied cell's centre (uam_edt's d_dist2: 0 on occupied
 *                               cells); -1 when no raster cell is touched.  65535 means "at least 256 cells".  In map units
 *                               the clearance is sqrt(d2min) |dx| when |dx| = |dy|.
 * The one-quantum dilation covers the scorer's rounding (quantisation moves an endpoint by <= 2^-17 cell, the scorer's fp64
 * samples lie within ~1e-11 cell of the segment, its nearest-cell choice on an fp32 fraction is off by <= 2^-24), so for a
 * path inside the raster rectangle uam_score_paths_raster's collide flag (any samples_per_cell) implies UAM_SWEEP_HIT.
 * Stream-ordered on `stream`, no host read-back; a path's outputs do not depend on the rest of the batch.  Uses the ctx's
 * current raster: the occupancy bit-plane (flags, first hit) and, for d_d2min only, a uint16 field of min(d2, 65535) made
 * with uam_edt (2 B per cell kept, ~26 B per cell of scratch while it is built) are built on the first call after each
 * raster upload and kept; that first call may synchronise.  B = 0 is a no-op; N < 0 or a NULL d_z / d_flags give
 * UAM_ERR_INVALID; no raster UAM_ERR_STATE; d_d2min on a raster over 23170 cells per side UAM_ERR_UNSUPPORTED (uam_edt's
 * limit; flags and first hit work at any size). */
enum { UAM_SWEEP_HIT = 1, UAM_SWEEP_OUTSIDE = 2, UAM_SWEEP_INVALID = 4 };
int uam_sweep_paths_raster(uam_ctx* ctx, const double* d_z, int64_t B, int N, uint8_t* d_flags, int32_t* d_first_hit,
                           int32_t* d_d2min, void* stream);

/* Swept check of whole path segments against the analytic hard obstacles (the shapes Map.collides tests, uploaded with
 * uam_map_set_shapes; region shapes are not tested).  uam_score_paths_analytic's collide flag, like map.py:41-43, looks at
 * the N + 2 waypoints only; this call asks whether any segment enters an obstacle between them.
 * Definition.  For every path of d_z (B, 2(N+2)) float64, segment k = 0 .. N from z_k to z_{k+1}, z(t) = z_k + t (z_{k+1}
 * - z_k), and hard obstacle o (obstacle order = insertion order = device order): let h_i^R be the formula of record i of
 * o (uam_h_exact: lines and boxes are affine in (x, y), an ellipse is a convex quadratic) in exact real arithmetic on the
 * record's doubles, and K_o = { x : h_i^R(x) <= 1e-14 for every i of o } (`contains`, quadratic_obstacle.py:89-94, in
 * exact arithmetic).  The segment meets K_o when some t in [0, 1] has z(t) in K_o.  The device decides HIT(k, o) in fp64:
 *   G1 (never misses): if the real segment meets K_o, then HIT(k, o);
 *   G2 (agrees with the waypoint check): if the fp64 `contains` is true at z_k or z_{k+1} (uam_psi's `inside`, the bits of
 *      Map.collides and of uam_score_paths_analytic's collide flag), then HIT(k, o); so for every path that is not
 *      INVALID, the analytic scorer's collide flag implies UAM_SWEEP_HIT;
 *   G3 (bounded false alarm): if HIT(k, o), the real segment meets K_o^eta = { x : h_i^R(x) <= 1e-14 + eta_i for every i },
 *      with A = z_k, B = z_{k+1}, u = 2^-53 and
 *        line  (rec {0, Ax', Ay', dx', dy', sgn}):  eta_i = 2^-46 (M_i(A) + M_i(B)) + 2^-990,
 *                                                   M_i(x, y) = |sgn| (|dy'| (|x| + |Ax'|) + |dx'| (|y| + |Ay'|));
 *        box   (rec {2, axis, sign, c, r}):         eta_i = 2^-46 (M_i(A) + M_i(B)) + 2^-990,  M_i = |x_axis| + |c| + |r|;
 *        ellipse (rec {1, cx, cy, r1, r2}):         eta_i = 2^-44 (2 + S) + 2^-94 S^2 + 2^-990,
 *                                                   S = (|Ax - cx| + |Bx - Ax|) / |r1| + (|Ay - cy| + |By - Ay|) / |r2|,
 *                                                   for S <= 2^40 (a segment within 2^40 radii of the ellipse);
 *      M_i bounds the fp64 evaluation error of the formula, 3.01 u M_i,, which eta_i exceeds 16-fold, as G2 needs; S is
 *      the segment's extent in the ellipse's scaled coordinates (DESIGN.md 9g derives both);
 *   G4 (deterministic): the outputs are those of the numpy restatement in tests/analytic_sweep_reference.py, bit for bit,
 *      in the same fp64 operation order; a path's outputs depend on that path and the map only, not on the rest of the
 *      batch nor on UAM_OPT_SHAPE_GRID.
 * Per path:
 *   d_flags (uint8):                UAM_SWEEP_HIT: HIT(k, o) for some k and o; UAM_SWEEP_INVALID: a coordinate is not
 *                                   finite or |coordinate| >= 1e100 (uam_psi's bound), nothing else is evaluated for the
 *                                   path (first hit and first obstacle -1); UAM_SWEEP_OUTSIDE is never set.
 *   d_first_hit (int32, nullable):  the lowest k with a hit, -1 if none;
 *   d_first_obstacle (int32, nullable): the smallest o with HIT(first_hit, o), -1 if none.
 * Cell lists: a G x G grid (G = 32 .. 256) over the obstacles' bounding box lists per cell the obstacles that may meet the
 * cell at tolerance 1e-14; a segment tests only the obstacles listed in the cells it crosses.  They are built on the
 * first call after each uam_map_set_shapes (that call synchronises) and kept; with UAM_OPT_SHAPE_GRID = 0, or fewer than 4
 * obstacles, every segment tests every obstacle.  Stream-ordered on `stream` otherwise, no host read-back.
 * Errors, in this order: B < 0, N < 0 or N > 2^28 UAM_ERR_INVALID; then B = 0 is a no-op; a NULL d_z / d_flags
 * UAM_ERR_INVALID; no shapes uploaded UAM_ERR_STATE;
 * then, before anything is launched, UAM_ERR_UNSUPPORTED for an obstacle record with a field that is not finite or beyond
 * 1e100 in magnitude, an ellipse radius below 1e-50 in magnitude (0 included), or an obstacle with two ellipse records:
 * the error bounds above do not hold for them.  A map without obstacles gives flags 0 (INVALID rows excepted) and -1. */
int uam_sweep_paths_analytic(uam_ctx* ctx, const double* d_z, int64_t B, int N, uint8_t* d_flags, int32_t* d_first_hit,
                             int32_t* d_first_obstacle, void* stream);

/* Clearance of whole path segments from the analytic hard obstacles: how far each path stays from the obstacles, and
 * which segment and obstacle come closest.  Paths, segments and obstacle order as in uam_sweep_paths_analytic.
 * The set P_o of obstacle o, by the form of its records (the forms polygon(), square() and ball() make):
 *   polygon: >= 3 line records; P_o is the convex hull of their origins (Ax, Ay).  Checked on the host: each direction
 *            ends at the next origin, |A_i + d_i - A_{i+1}| <= 2^-50 (|A_i| + |A_{i+1}|) per component, cyclically, and
 *            every origin but the record's own two lies strictly inside it (fp64 h < 0): a strictly convex polygon in
 *            hull order with inward signs;
 *   box:     exactly 4 box records, one per (axis, sign); P_o is the rectangle [c- - r-, c+ + r+] per axis (fp64), not empty;
 *   ellipse: exactly one ellipse record; P_o is the filled ellipse (a disc when |r1| == |r2|, measured in closed form).
 * Any other obstacle (for example line records with an ellipse record) gives UAM_ERR_UNSUPPORTED naming it, before
 * anything is launched; uam_sweep_paths_analytic does not look at forms.
 * The distance of segment k and obstacle o: D(k, o) = 0 iff HIT(k, o) (the sweep's own decision); otherwise the fp64
 * distance from the segment to P_o, at least 2^-1022:
 *   polygon, box: the minimum of the point-to-segment distances of each vertex to the segment and of A and B to each edge;
 *   disc:         (distance from the centre to the segment) - r;
 *   ellipse:      the minimum of the point-to-ellipse distances of A and B (Eberly's bisection, run until its midpoint
 *                 repeats an end) and of the distances from the segment to the two boundary points whose normal is
 *                 perpendicular to it, each counted when its foot on the segment's line falls in [0, 1].
 * Per path: d_clearance (float64, nullable) = min(cap, min over k, o of D(k, o)); d_nearest_segment / d_nearest_obstacle
 * (int32, nullable): the pair that attains it, the smallest k and then the smallest o, both -1 when the clearance equals
 * cap (nothing lies within cap); d_flags (uint8, required): UAM_SWEEP_HIT and UAM_SWEEP_INVALID as the sweep sets them.
 * An INVALID row gets clearance NaN and -1.  So clearance >= m is the keep-out check of a margin m <= cap.
 *   D1 (agrees with the sweep): d_flags equals uam_sweep_paths_analytic's flags bit for bit; a HIT path has clearance 0,
 *      nearest segment = first hit and nearest obstacle = first obstacle; a path neither HIT nor INVALID has clearance > 0.
 *   D2 (error bound): for a pair that is not HIT, |D(k, o) - dist(segment k, P_o)| <= delta, with A, B the segment's ends,
 *      D the exact distance, u = 2^-53, M the largest coordinate magnitude of A, B and the obstacle (polygon: its
 *      vertices; box: its rectangle's bounds; disc and ellipse: |cx| + e0, |cy| + e0, e0 >= e1 the semi-axes):
 *        polygon, box, disc: delta = 2^-48 M + 4 u D + 2^-1000;
 *        ellipse:            delta = 2^-40 (e0 / e1) M + 4 u D + 2^-1000.
 *      For a HIT pair the segment meets K_o^eta (G3), whose points lie within eps of P_o: box eps = sum over the two
 *      axes of max_i (1e-14 + eta_i); ellipse eps = e0 (1e-14 + eta) / 2; polygon eps = max_i (1e-14 + eta_i) /
 *      (|sgn_i| |d_i|) / cos(phi / 2), phi the largest exterior angle (DESIGN.md 9h).
 *   D3 (deterministic): the outputs are those of the numpy restatement in tests/analytic_clearance_reference.py, bit for
 *      bit; a path's outputs depend on that path and the map only, not on the rest of the batch nor on
 *      UAM_OPT_SHAPE_GRID, and on cap only through the min with cap.
 * Cell lists: the sweep's cells, listing also every obstacle whose box lies within cap (1 + 2^-40) of the cell (plus a
 * margin above delta).  They are built on the first call after each uam_map_set_shapes or change of cap (that call
 * synchronises) and kept; with UAM_OPT_SHAPE_GRID = 0, where the sweep has no lists, or where the lists would hold over
 * 3/4 of all (cell, obstacle) pairs, every segment tests every obstacle.  Stream-ordered on `stream` otherwise.
 * Errors, in this order: B < 0, N < 0, N > 2^28, or cap not in (0, 1e100] UAM_ERR_INVALID; then B = 0 is a no-op; a NULL
 * d_z / d_flags UAM_ERR_INVALID; no shapes UAM_ERR_STATE; the sweep's record checks, then the form checks above,
 * UAM_ERR_UNSUPPORTED.  A map without obstacles gives clearance = cap and -1 (INVALID rows excepted). */
int uam_clearance_paths_analytic(uam_ctx* ctx, const double* d_z, int64_t B, int N, double cap, uint8_t* d_flags,
                                 double* d_clearance, int32_t* d_nearest_segment, int32_t* d_nearest_obstacle,
                                 void* stream);

/* Scoring + best candidate in one call: as uam_score_paths_raster, and *d_key receives the best key (see uam_best) of the
 * batch -- of ALL ranks' batches when a peer group is attached (uam_peer_attach): the last kernel of the step finds the
 * local min, pushes it into every peer's symmetric block over NVLink and waits for theirs (no separate collective).
 * Every rank of the group must make the same sequence of *_best / uam_best_allreduce calls (B == 0 is allowed). */
int uam_score_paths_raster_best(uam_ctx* ctx, const double* d_z, int64_t B, int N, const double* h_p, int n_p,
                                int flags, double samples_per_cell, float* d_cost, uint8_t* d_collide,
                                int64_t global_offset, uint64_t* d_key, void* stream);

/* Asynchronous host-buffer scoring: a ring of 3 slots (stream + staging each).  submit queues upload -> (candidate
 * generation ->) whole-batch scoring -> download on the slot's stream and returns a ticket at once; uam_raster_wait(ticket)
 * returns when the results are in h_cost / h_collide / *h_key (nullable; *h_key = this rank's best key with
 * global_offset + b as index).  With two tickets in flight the upload of batch s+1 overlaps the kernels of batch s.  The
 * host buffers must stay valid (and should be pinned) until the wait; a 4th submission first waits for the oldest ticket.
 *   uam_raster_submit_paths_host       h_z (B, 2(N+2)) float64: the caller's waypoints (1 KiB per path at N = 62)
 *   uam_raster_submit_candidates_host  h_cand (B, 5) float64 {xs, ys, xg, yg, displacement}: the candidates are generated on
 *                                      the device (uam_make_candidates with index0 = global_offset), 40 bytes per path --
 *                                      the reference's own flow (displacement -> create_x_init -> score, main.py:160-171) */
int uam_raster_submit_paths_host(uam_ctx* ctx, const double* h_z, int64_t B, int N, const double* h_p, int n_p,
                                 int flags, double samples_per_cell, float* h_cost, uint8_t* h_collide,
                                 uint64_t* h_key, int64_t global_offset, int* ticket);
int uam_raster_submit_candidates_host(uam_ctx* ctx, const double* h_cand, int64_t B, int N, double jitter_sigma,
                                      uint64_t seed, const double* h_p, int n_p, int flags, double samples_per_cell,
                                      float* h_cost, uint8_t* h_collide, uint64_t* h_key, int64_t global_offset,
                                      int* ticket);
int uam_raster_wait(uam_ctx* ctx, int ticket);

/* ---- point queries --------------------------------------------------------------------------------
 * Replaces Problem.get_penalty_function(region)(x) (problem.py:59-82), get_total_penalty_function
 * (:49-56) and Map.collides(x) (map.py:41-43) for M points x (M,2) float64.  Outputs nullable:
 *   d_region_pen (M, R) float64 weighted per-region penalties; d_obst_pen (M) float64 =
 *   get_penalty_function(None)(x); d_collide (M) uint8.  All fp64 (this is the exact path). */
int uam_eval_points(uam_ctx* ctx, const double* d_x, int64_t M, const double* h_p, int n_p, int flags,
                    double* d_region_pen, double* d_obst_pen, uint8_t* d_collide, void* stream);
int uam_eval_points_host(uam_ctx* ctx, const double* h_x, int64_t M, const double* h_p, int n_p, int flags,
                         double* h_region_pen, double* h_obst_pen, uint8_t* h_collide);

/* Function.__call__ (function.py:119-120): h_i(x_m) of n_rec raw inequality records (8 doubles each, the
 * record kinds above) at M points, h_out[i*M + m]; fp64, bit-exact with the reference's closures
 * (polygon.py:69-71,98; ball.py:33-37; square.py:29-51). */
int uam_eval_inequalities_host(uam_ctx* ctx, const double* h_records, int n_rec, const double* h_x, int64_t M,
                               double* h_out);

/* ---- best candidate --------------------------------------------------------------------------------
 * Replaces the running min of path_generation/main.py:162-180.  *d_key = min over b of
 *     key(cost[b], global_offset + b) = (img(float32 cost) << 31) | index        (63 bits, index < 2^31)
 * img = order-preserving image of the float32 bit pattern (all bits flipped for a negative value, top bit set otherwise;
 * NaN -> 0xffffffff), so the unsigned order of the keys is the float order of the costs for EVERY value (negative costs
 * are reachable through negative layer weights), a NaN never wins, ties resolve to the smaller index (the strict `<` of
 * main.py:175) and the key is a non-negative int64: the caller min-reduces it across ranks with a signed or unsigned min
 * alike (NCCL).  An empty batch leaves 2^63 - 1.  d_key must be pre-set (to 2^63 - 1) by the caller or by passing
 * reset != 0.  d_cost is float32 (raster scorer) or float64 (analytic scorer, rounded to float32 for the key) according
 * to cost_is_f64. */
int uam_best(uam_ctx* ctx, const void* d_cost, int cost_is_f64, int64_t B, int64_t global_offset,
             uint64_t* d_key, int reset, void* stream);

/* The same with the cross-rank exchange built in: *d_key = min over the attached peer group (or this rank alone when no
 * group is attached) of the batch keys; B == 0 takes part with "no candidate".  One kernel: local min + push / wait over
 * NVLink peer memory in its last CTA. */
int uam_best_allreduce(uam_ctx* ctx, const void* d_cost, int cost_is_f64, int64_t B, int64_t global_offset,
                       uint64_t* d_key, void* stream);
/* Peer group of the ranks of one box (one process per GPU).  uam_peer_export writes the 64-byte CUDA IPC handle of this
 * ctx's symmetric block; the caller all-gathers the handles (torch.distributed, any backend) and passes all `world` of them
 * (rank order, 64 bytes each) to uam_peer_attach, which maps the peers' blocks.  uam_peer_status: *timed_out != 0 if a
 * wait for the peers ever gave up (2 s; the key of that step is then a partial min). */
int uam_peer_export(uam_ctx* ctx, void* h_handle64);
int uam_peer_attach(uam_ctx* ctx, int rank, int world, const void* h_handles);
int uam_peer_status(uam_ctx* ctx, int* timed_out);

/* ---- map rebuild (map_generation) --------------------------------------------------------------------
 * uam_dem_mask: mask = image > threshold, or image == -9999 when threshold == -9999
 *               (map_generation/data_manager.py:14-17).
 * uam_rasterize_occupancy: occ[i,j] = Map.collides(cell centre)  (map.py:41-43), fp64, bit-exact.
 * uam_rasterize_layers: layer[l,i,j] = float32(sum_{s in region l} psi_s(xc;e)/psi_s(c_s;e)), unweighted
 *               (problem.py:72-80 without w; quadratic_obstacle.py:33-35).
 * uam_edt: exact squared Euclidean distance (cells) to the nearest occupied cell and clearance =
 *               sqrt(d2)*cell (build-defined extension; no reference counterpart). */
int uam_dem_mask(uam_ctx* ctx, const float* d_image, int64_t n, float threshold, uint8_t* d_mask,
                 void* stream);
int uam_rasterize_occupancy(uam_ctx* ctx, int H, int W, double x0, double dx, double y0, double dy,
                            uint8_t* d_occ, void* stream);
int uam_rasterize_layers(uam_ctx* ctx, int H, int W, double x0, double dx, double y0, double dy,
                         double enlargement, float* d_layers, void* stream);
int uam_edt(uam_ctx* ctx, const uint8_t* d_occ, int H, int W, double cell, int32_t* d_dist2,
            float* d_clearance, void* stream);

/* ---- polygon front-end of map_generation (SURVEY.md 8f item 3) ------------------------------------------------
 * The data-parallel core of DataManager.load_dem_polygons_from_geotiff (map_generation/data_manager.py:11-19: one polygon
 * per connected region of the mask, as rasterio.features.shapes yields them with its default 4-connectivity) and of
 * DataProcessor.process_polygons (map_generation/data_processor.py:16-34,67-71: area filter + cv2.minAreaRect of each
 * polygon's exterior ring).
 * uam_label_components: d_mask (H,W) uint8 -> d_labels (H,W) int32: 0 = background, components numbered 1..n in raster-scan
 *                       order of their first cell (scipy.ndimage.label's numbering); connectivity 4 or 8; *h_n_components
 *                       (host) receives n.  Synchronises `stream`.
 * uam_component_stats:  d_area (n) int64 = cells per component (polygon.area / cell area); d_bbox (n,4) int32 =
 *                       {row min, row max, col min, col max}.  Synchronises `stream`.
 * uam_component_rects:  minimum-area enclosing rectangle of the cell corners of each listed component (d_ids: K distinct
 *                       labels) = of the polygon's exterior ring; d_rect (K,4,2) float64 world coordinates of the corners
 *                       (x0 + col*dx, y0 + row*dy at cell corners), consecutive around the rectangle, the first two on the
 *                       line of the chosen hull edge; d_info (K,2) int32 (nullable) = {hull vertices, chosen edge}.  Exact:
 *                       every hull edge is tried with integer extents and a 128-bit area comparison, ties to the first
 *                       edge.  Needs square cells and H, W <= 32766.  Synchronises `stream`. */
int uam_label_components(uam_ctx* ctx, const uint8_t* d_mask, int H, int W, int connectivity, int32_t* d_labels,
                         int32_t* h_n_components, void* stream);
int uam_component_stats(uam_ctx* ctx, const int32_t* d_labels, int H, int W, int n_components, int64_t* d_area,
                        int32_t* d_bbox, void* stream);
int uam_component_rects(uam_ctx* ctx, const int32_t* d_labels, int H, int W, int n_components, const int32_t* d_bbox,
                        const int32_t* d_ids, int K, double x0, double dx, double y0, double dy, double* d_rect,
                        int32_t* d_info, void* stream);

/* Large-polygon split of DataProcessor._divide_and_approximate_polygon (map_generation/data_processor.py:34-53): mask of
 * box (box_row, box_col) of the divisions x divisions box grid over component `label`'s bounding box h_bbox = {row min, row
 * max, col min, col max} (host), on the grid refined `divisions` times: d_mask (nr, nc) uint8 with nr, nc = the bounding
 * box's extents in cells.  Sub-cell (r, c) has the corners (col min + (box_col nc + c) / divisions, row min + (box_row nr +
 * r) / divisions) .. + 1 / divisions in cell units.  The box edges are sub-cell boundaries, so the 4-connected regions of the
 * mask (uam_label_components) are the pieces of polygon.intersection(box) and uam_component_rects on them, with the affine of
 * the refined grid, gives each piece's minimum-area rectangle. */
int uam_component_submask(uam_ctx* ctx, const int32_t* d_labels, int H, int W, int label, const int32_t* h_bbox,
                          int divisions, int box_row, int box_col, uint8_t* d_mask, void* stream);

/* ---- grid search / cost-to-go (build-defined extension; the reference has none: SURVEY.md section 0) ----------
 * Q independent single-source cost-to-go sweeps on an 8-connected H x W grid, optionally stacked in `bands` altitude
 * bands, with integer edge costs: in-plane step(u,v) * (cost[b,u] + cost[b,v]), step = 2 (axis) / 3 (diagonal); band
 * change at a fixed cell 2 * (cost[b,v] + cost[b+-1,v]); blocked cells (nullable) are impassable.
 * uam_grid_search:       d_cost (H,W) uint16, d_sources (Q,2) int32 (row, col); d_dist (Q,H,W) int64 (2^62 =
 *                        unreachable); d_parent (Q,H,W) int32 (nullable): flat index of the best predecessor, ties to
 *                        the lowest neighbour slot in the order (-1,-1),(-1,0),(-1,1),(0,-1),(0,1),(1,-1),(1,0),(1,1);
 *                        parent[source] = source, unreachable = -1.
 * uam_grid_search_bands: d_cost / d_blocked (bands,H,W), d_sources (Q,3) int32 (band, row, col); d_dist / d_parent
 *                        (Q,bands,H,W); parent = flat index into (bands,H,W); two more predecessor slots after the eight
 *                        in-plane ones: band below (8), band above (9).
 * Frontier-parallel tile relaxation (warp per 32 x 32 tile, Gauss-Seidel row sweeps with (min,+) warp scans); results
 * are bit-identical to Dijkstra.  Synchronises `stream` internally (the number of rounds is data dependent).
 * Precondition for predecessors: every passable cell has cost >= 1 (a weight-0 edge between two cost-0 cells would let
 * them choose each other); with d_parent != NULL a grid with passable cost-0 cells is refused (UAM_ERR_UNSUPPORTED),
 * with d_parent == NULL distances are computed as usual (they stay exact for weights >= 0). */
/* uam_grid_search_goals: start/goal queries.  As uam_grid_search_bands (bands >= 1; d_sources and d_goals are (Q,3) int32
 *                        {band, row, col}), but a query stops as soon as nothing pending can lower its goal's distance:
 *                        dist is exact for the goal and for every node closer to the source than the goal (nodes farther
 *                        away hold upper bounds or 2^62), and the predecessors of those nodes are the ones of the full
 *                        search (edge weights are positive for cost >= 1), so the extracted path is the same.  A goal
 *                        outside the grid leaves the query unbounded.
 * uam_grid_extract_paths: one path per query from d_parent (Q,bands,H,W): d_path (Q,max_len) int32 flat node ids from the
 *                        source to the goal, d_len (Q) = nodes on the path, 0 = goal not reached, -k = the path has
 *                        k > max_len nodes (nothing written). */
int uam_grid_search_goals(uam_ctx* ctx, const uint16_t* d_cost, const uint8_t* d_blocked, int bands, int H, int W,
                          const int32_t* d_sources, const int32_t* d_goals, int Q, int64_t* d_dist, int32_t* d_parent,
                          void* stream);
int uam_grid_extract_paths(uam_ctx* ctx, const int32_t* d_parent, int bands, int H, int W, const int32_t* d_sources,
                           const int32_t* d_goals, int Q, int max_len, int32_t* d_path, int32_t* d_len, void* stream);
int uam_grid_search(uam_ctx* ctx, const uint16_t* d_cost, const uint8_t* d_blocked, int H, int W,
                    const int32_t* d_sources, int Q, int64_t* d_dist, int32_t* d_parent, void* stream);
int uam_grid_search_bands(uam_ctx* ctx, const uint16_t* d_cost, const uint8_t* d_blocked, int bands, int H, int W,
                          const int32_t* d_sources, int Q, int64_t* d_dist, int32_t* d_parent, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* UAM_B200_H */
