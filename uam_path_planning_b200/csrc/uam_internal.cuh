// Internal declarations shared by the translation units of libuam_b200.so (sm_100a).
// Public surface: include/uam_b200.h.
#pragma once

#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "uam_b200.h"

#define UAM_MAX_REGIONS 16
#define UAM_WARPS_PER_CTA 8
#define UAM_CTA_THREADS (UAM_WARPS_PER_CTA * 32)
#define UAM_HOST_PIPE_DEPTH 3
#define UAM_INTERNAL_FINITE_EDGES (1 << 30)   // UamParams.flags, set by the library: psi products may stop at their first zero

// ---- device table records ---------------------------------------------------------------------
// Inequality record, same 8-double layout as the C-ABI (rec[0] = kind).
struct __align__(16) UamEdge {
    double kind, p0, p1, p2, p3, p4, p5, p6;
};

// One shape = a run of inequality records.  Device order: hard obstacles first (insertion order),
// then region shapes, region-major in insertion order.
struct __align__(16) UamShape {
    double cx, cy;            // QuadraticObstacle.center (NaN = none)
    int e0, e1;               // edge range [e0, e1)
    int region;               // -1 = hard obstacle
    int has_center;
};

struct UamParams {
    double ms_x, ms_y;        // map.x_start (first pair of the length term, problem.py:137-145)
    double maxratio, mincos, e;
    double w[UAM_MAX_REGIONS];
    int flags;
    int n_regions;
};

// Cell lists over the shapes for the analytic scorer (uam_shape_grid.cu): cell (cy, cx) of a G x G grid over the shapes'
// bounding box holds, in ascending device order, every shape that can contribute a non-zero penalty / constraint term or
// contain a point anywhere in the cell; all other shapes contribute exact zeros there.  G == 0: no grid (evaluate all).
struct UamShapeGrid {
    double gx0, gy0, inv_cw, inv_ch;
    int G;
    int obs_values;       // 1: the obstacles' psi values may come from the lists too (obstacle_smooth); 0: only `contains`
    const int* start;     // G * G + 1 offsets into items
    const int* items;
};

// Cell lists over the hard obstacles for the swept analytic check (uam_sweep_analytic.cu): cell (cy, cx) of a G x G grid
// lists, in ascending obstacle order, every obstacle no single record of which is > 1e-14 (with the margin of
// uam_edge_excludes_tile) on the cell's box widened by 1/1000 of a cell; the boxes of the border cells reach out to
// +-ext.  Only segments whose four coordinates are all within [-qmax, qmax] use the lists (see the bound in the .cu).
struct UamObsGrid {
    double gx0, gy0, inv_cw, inv_ch;
    double qmax;
    int G;
    const int* start;     // G * G + 1 offsets into items
    const int* items;
};

// Form of a hard obstacle for the clearance (uam_clearance_paths_analytic), decided on the host from its records
enum { UAM_FORM_POLYGON = 0, UAM_FORM_ELLIPSE = 1, UAM_FORM_BOX = 2, UAM_FORM_DISC = 3 };
struct UamObsGeom {
    double x0, x1, y0, y1;        // box: the rectangle [x0, x1] x [y0, y1] (fp64 c - r, c + r of its records)
    double bx0, bx1, by0, by1;    // a box that contains the obstacle (P_o), rounded outward
    double rho;                   // the factor of the distance's error bound: 1, or e0 / e1 for an ellipse (DESIGN.md 9h)
    int form;
    int pad;
};

struct UamRasterGeo {
    double x0, dx, y0, dy;
    int H, W, L;
    int texel_floats;         // 2 (L == 1: layer, occupancy) or 4 (L in 2..3: l0, l1, l2, occupancy)
    int layout;               // 0 = row-major texels, 1 = tiled (see uam_tex_index)
    int tiles_x;              // tiled: tiles per tile-row (tile = 4 x 2 texels for float4, 4 x 4 for float2)
    int tiles_y;
};

// What the raster kernels of one API call read (uam_score_raster.cu): made by uam_raster_prepare from the call's
// arguments, completed by uam_raster_precompute.
struct UamRasterParams {
    double x0, dx, y0, dy;
    double ms_x, ms_y;
    double spc;
    int H, W;
    unsigned row_stride;  // tiled layout: texels per tile-row (tiles_x * texels per tile); row-major: W (of the quads if combined)
    float w0, w1, w2;     // combined with L = 2..3: {1, 0, 0}, the weights are inside the quads
    int flags;
    int variant;          // integral-mode kernel, decided once per API call from the call's whole batch
    int combined;         // score on the weight-folded layer: 1 = quad texels (ctx->d_tex_comb) + bit-plane, 2 = sign-packed
                          // quad texels, 3 = sign-packed gather layer (gather_tex)
    const unsigned* occ_bits;   // quad mode: occupancy bit-plane (uam_occ_word / uam_occ_bit)
    unsigned occ_blocks_x;      // 32 x 32-cell blocks per block-row of the bit-plane
    unsigned long long gather_tex;   // combined == 3: texture object of ctx->gather_arr
};

// ---- best-candidate exchange between the ranks of one box (uam_best.cu) -------------------------------------------
// One-sided min-reduce of the 8-byte best key over NVLink peer memory: every rank owns a small "symmetric block"
// (cudaMalloc + CUDA IPC, mapped into every peer process); the tail of the scoring step stores this rank's key into its
// own column of every peer's block, raises an epoch-tagged flag behind a system-scope fence, then waits until the flags
// of all ranks carry the epoch and takes the min -- the all-reduce is part of the step's last kernel, no NCCL launch.
#define UAM_MAX_PEERS 16
#define UAM_PEER_RING 4        // epochs in flight: a rank cannot be more than one epoch ahead of a peer (it waits for all)
struct UamPeerBlock {
    unsigned long long keys[UAM_PEER_RING][UAM_MAX_PEERS];
    unsigned flags[UAM_PEER_RING][UAM_MAX_PEERS];      // = epoch of the key in the same cell (monotone, never reset)
};
struct UamBestTail {
    unsigned long long* local;     // [0] running min of this launch, [1] CTAs done (both restored by the last CTA)
    unsigned long long* out;       // where the (global) best key goes (device, nullable)
    unsigned* status;              // != 0: the wait for the peers timed out
    UamPeerBlock* peer[UAM_MAX_PEERS];
    unsigned long long offset;     // global index of this launch's first path
    int world, rank;               // world <= 1: no exchange
    unsigned epoch;
    int combine;                   // 1: *out = min(*out, key) (uam_best's accumulate form), 0: *out = key
};

// ---- context --------------------------------------------------------------------------------------
struct uam_ctx {
    int device = 0;
    int sm_count = 148;
    cudaStream_t stream = nullptr;                       // own stream
    cudaStream_t pipe_stream[UAM_HOST_PIPE_DEPTH] = {};  // host-buffer pipeline
    cudaEvent_t pipe_event[UAM_HOST_PIPE_DEPTH] = {};
    std::string err;
    uint64_t launches = 0;
    // tuning knobs (uam_ctx_set_option / environment at ctx creation)
    int raster_layout = 1;    // layout used by the next uam_map_set_raster*
    int host_chunks = 0;      // *_host raster scoring: pipeline chunks per call (0 = default)
    int host_taper = 0;       // ... and by how many percent the last chunk is smaller (> 0) / the first chunk is smaller (< 0)
    int ccl_tiles = 1;        // UAM_OPT_CCL_TILES: 1 = tile-local labelling in shared memory first, 0 = global union-find only
    int rasterizer_scan = 1;  // UAM_OPT_RASTERIZER: 1 = scanline rasterisers (row intervals), 0 = per-cell evaluation
    int int_variant = -1;     // integral mode: -1 = auto; 0 = warp per path, lane per sample; 1 = lane pair per sample;
                              // 2 = segments binned by raster tile (L2-resident raster); 3 = pieces sorted by tile, tile staged in smem

    // device shape tables
    UamEdge* d_edges = nullptr;
    UamShape* d_shapes = nullptr;
    double* d_psic = nullptr;           // psi_s(center_s; e) per shape, made by uam_k_shape_norm
    int n_shapes = 0, n_edges = 0, n_regions = 0, n_obs = 0;
    int region_begin[UAM_MAX_REGIONS + 1] = {};  // shape index range of each region
    bool has_shapes = false;
    bool edges_finite = false;          // every inequality record is finite: the psi product may stop at its first zero
    double edges_max_abs = 0.0;         // largest magnitude in the records (finite ones)
    int max_edges_per_shape = 0;
    bool psic_valid = false;
    bool shape_grid_built = false;      // the analytic scorer's cell lists exist for the current (e, flags)
    double psic_e = 0.0;
    int psic_flags = -1;
    // shape grid of the analytic scorer (rebuilt with psic: it depends on the enlargement)
    int shape_grid_opt = 1;             // UAM_OPT_SHAPE_GRID
    double shape_bbox[4] = {};          // x0, x1, y0, y1 of all shapes (host, from the records); x0 > x1: none
    int* d_grid_start = nullptr;
    int* d_grid_items = nullptr;
    size_t grid_start_bytes = 0, grid_items_bytes = 0;
    UamShapeGrid shape_grid = {};       // G == 0 until built / when disabled
    int grid_items_total = 0;

    // raster
    void* d_tex = nullptr;              // float2 / float4 texels, row-major (H, W)
    size_t tex_bytes = 0;
    UamRasterGeo geo = {};
    bool has_raster = false;

    // staging for the *_host entry points
    void* d_stage_in[UAM_HOST_PIPE_DEPTH] = {};
    size_t stage_in_bytes[UAM_HOST_PIPE_DEPTH] = {};
    void* d_stage_out[UAM_HOST_PIPE_DEPTH] = {};
    size_t stage_out_bytes[UAM_HOST_PIPE_DEPTH] = {};
    void* h_stage_out[UAM_HOST_PIPE_DEPTH] = {};   // pinned
    size_t h_stage_out_bytes[UAM_HOST_PIPE_DEPTH] = {};
    void* d_cull_scratch = nullptr;     // rasteriser: coarse (supertile) shape lists
    size_t cull_scratch_bytes = 0;
    void* d_cull0_scratch = nullptr;    // ... and the lists of the 2048-cell blocks above them
    size_t cull0_scratch_bytes = 0;
    void* d_scratch = nullptr;          // EDT, grid search
    size_t scratch_bytes = 0;
    // optional CUDA-event timing of the dominant scoring kernel (UAM_OPT_TIME_KERNELS), read by uam_ctx_get_stat
    int time_kernels = 0;
    // ring of event pairs: the timed kernel's begin / end are recorded on the launching stream and read back only when
    // the ring is full or a statistic is asked for, so a timed loop never makes the host wait for the device
    static constexpr int kTimeRing = 128;
    cudaEvent_t time_ev[2 * kTimeRing] = {};
    int time_pending = 0;
    double time_sum_ms = 0.0;
    uint64_t time_count = 0;
    long long grid_delta = 0;           // UAM_OPT_GRID_DELTA (0 = automatic)
    int grid_half_cap = 4;              // half sweeps per activation before a tile is handed to the next round (UAM_GRID_HALF_CAP; 0: none)
    int grid_graph = 1;                 // UAM_OPT_GRID_GRAPH: relaxation rounds looped on the device (CUDA graph WHILE node)
    int bin_chunk = 8192;               // ... segments per CTA of the histogram / scatter kernels (UAM_BIN_CHUNK, A/B runs only)
    int bin_pt = 2;                     // ... paths a warp of the histogram kernel works on at a time (UAM_BIN_PT: 1, 2, 4)
    int bin_shift = 7;                  // binned raster scorer: bin side = 2^bin_shift cells (UAM_BIN_SHIFT, A/B runs only)
    double grid_activations = 0, grid_sweeps = 0, grid_rounds = 0;   // counted work of the last uam_grid_search*
    double grid_host_submissions = 0;   // ... and what the host enqueued for it (kernel launches + memsets + graph launches)
    void* d_bin_scratch[UAM_HOST_PIPE_DEPTH + 1] = {};   // binned raster scorer: [0] caller stream, [1..] pipeline stages
    size_t bin_scratch_bytes[UAM_HOST_PIPE_DEPTH + 1] = {};
    // tile-staged raster scorer (variant 3): tile-major copy of the texels (built on first use) + piece scratch
    void* d_tiles = nullptr;
    size_t tiles_bytes = 0;
    bool tiles_valid = false;
    uint64_t tiles_key = 0;             // which texel array the tile copy was made from
    // quad texels (weight-combined layer, 2 x 2 footprint per cell) + occupancy bit-plane for the large-batch
    // integral pipelines, per (raster, weights)
    void* d_tex_comb = nullptr;
    size_t tex_comb_bytes = 0;
    bool comb_valid = false;
    void* d_occ_bits = nullptr;         // 4 words (uam_build_quads_t's flag) + the bit-plane (uam_ensure_occ_bits)
    size_t occ_bits_bytes = 0;
    bool occ_bits_valid = false;
    bool comb_packed = false;           // quads carry the occupancy flags in their sign bits
    // gather layer: the folded layer, 4 bytes per cell (sign bit = occupancy), in a 2-D CUDA array read by tex2Dgather;
    // made instead of the quads when the raster fits gather_max_w x gather_max_h and the folded values are >= 0
    cudaArray_t gather_arr = nullptr;
    cudaTextureObject_t gather_tex = 0;
    int gather_w = 0, gather_h = 0;     // dimensions of gather_arr
    int gather_max_w = 0, gather_max_h = 0;   // cudaDevAttrMaxTexture2DGatherWidth / Height of the device
    bool comb_gather = false;           // the valid folded form is the gather layer (else the quads)
    bool comb_want_gather = false;      // ... and it was built for a call that asked for the gather layer
    int no_sign_pack = 0;               // UAM_NO_SIGN_PACK=1 forces the bit-plane form (tests)
    float comb_w[3] = {};
    uint64_t comb_gen = 0, raster_gen = 0;
    int combine_layers = 1;             // UAM_OPT_COMBINE_LAYERS
    void* d_piece_scratch[UAM_HOST_PIPE_DEPTH + 1] = {};
    size_t piece_scratch_bytes[UAM_HOST_PIPE_DEPTH + 1] = {};
    // best-candidate tail / peer exchange (uam_best.cu)
    unsigned long long* d_best_local = nullptr;      // {running min, CTAs done, status} x (1 + UAM_HOST_PIPE_DEPTH) slots
    UamPeerBlock* d_peer_own = nullptr;              // this rank's symmetric block
    UamPeerBlock* peer_ptr[UAM_MAX_PEERS] = {};      // every rank's block as mapped here ([rank] = d_peer_own)
    int peer_world = 0, peer_rank = 0;
    unsigned peer_epoch = 0;
    // asynchronous host-buffer scoring (uam_raster_submit_* / uam_raster_wait): one ticket per pipeline slot
    int ring_next = 0;
    int ring_last = -1;                                  // slot of the latest submission (its pipe_event marks its kernels' end)
    bool ring_busy[UAM_HOST_PIPE_DEPTH] = {};
    void* d_ring_cand[UAM_HOST_PIPE_DEPTH] = {};
    size_t ring_cand_bytes[UAM_HOST_PIPE_DEPTH] = {};
    unsigned long long* d_ring_key[UAM_HOST_PIPE_DEPTH] = {};
    // raster refinement (uam_refine.cu): trial paths, both gradients and the per-path step state
    void* d_refine_scratch = nullptr;
    size_t refine_scratch_bytes = 0;
    // swept path check (uam_sweep.cu): min(EDT d^2, 65535) per cell (H, W) uint16 of the raster of generation sweep_d2_gen
    void* d_sweep_d2 = nullptr;
    size_t sweep_d2_bytes = 0;
    uint64_t sweep_d2_gen = 0;          // 0: none (raster_gen counts uploads from 1)
    // swept check against the analytic obstacles (uam_sweep_analytic.cu): the obstacles' records checked on the host and
    // their cell lists, both for the shape table of generation obs_gen (shapes_gen counts uploads from 1)
    uint64_t shapes_gen = 0;
    uint64_t obs_gen = 0;
    int obs_rc = UAM_OK;                // UAM_ERR_UNSUPPORTED when the records break the sweep's error bounds
    std::string obs_err;
    UamObsGrid obs_grid = {};           // G == 0: no lists (fewer than 4 obstacles, or the bounds do not allow them)
    int* d_obs_grid = nullptr;          // G * G + 1 offsets (+ G * G counts while they are built)
    int* d_obs_items = nullptr;
    size_t obs_grid_bytes = 0, obs_items_bytes = 0;
    // clearance (same file): the obstacles' forms and boxes, checked with the records above, and cell lists dilated by
    // the cap of generation clr_gen (clr_cap)
    int clr_rc = UAM_OK;                // UAM_ERR_UNSUPPORTED when an obstacle is none of the forms the clearance measures
    std::string clr_err;
    UamObsGeom* d_obs_geom = nullptr;
    size_t obs_geom_bytes = 0;
    std::vector<UamObsGeom> h_obs_geom;
    double obs_cw = 0.0, obs_ch = 0.0, obs_ext = 0.0;   // the sweep grid's cell sides and border reach
    uint64_t clr_gen = 0;
    double clr_cap = 0.0;
    UamObsGrid clr_grid = {};           // G == 0: every segment tests every obstacle
    int* d_clr_grid = nullptr;
    int* d_clr_items = nullptr;
    size_t clr_grid_bytes = 0, clr_items_bytes = 0;
};

int uam_fail(uam_ctx* ctx, int code, const char* fmt, ...);
int uam_cuda_fail(uam_ctx* ctx, cudaError_t e, const char* what);
int uam_reserve(uam_ctx* ctx, void** ptr, size_t* cur, size_t need);
int uam_reserve_pinned(uam_ctx* ctx, void** ptr, size_t* cur, size_t need);
int uam_make_params(uam_ctx* ctx, const double* h_p, int n_p, int flags, UamParams* out);
int uam_ensure_shape_norm(uam_ctx* ctx, const UamParams& prm, cudaStream_t st, bool want_grid = true);
int uam_build_shape_grid(uam_ctx* ctx, double e, int flags, cudaStream_t st);
// the shape grid's exclusive prefix sum: start[0..n] of counts[0..n) (one CTA on `st`)
int uam_shape_grid_scan(uam_ctx* ctx, const int* counts, int n, int* start, cudaStream_t st);
// the grid to use for a call with these parameters (G == 0 when culling would not be exact for them)
UamShapeGrid uam_pick_shape_grid(const uam_ctx* ctx, const UamParams& prm);
cudaStream_t uam_pick_stream(uam_ctx* ctx, void* stream);
int uam_time_collect(uam_ctx* ctx);
int uam_time_begin(uam_ctx* ctx, cudaStream_t st);
int uam_time_end(uam_ctx* ctx, cudaStream_t st);
// best-candidate tail (uam_best.cu): the tail descriptor for a launch that starts at global index `offset` (slot = which
// {running min, counter} pair of the ctx: 0 for caller-stream calls, 1.. for the host pipeline slots); with_peers: exchange
// with the attached ranks (advances the epoch); and the stand-alone kernel for scorers without a fused tail
int uam_best_tail(uam_ctx* ctx, int slot, unsigned long long offset, unsigned long long* d_out, bool with_peers, bool combine,
                  UamBestTail* tail);
int uam_best_launch(uam_ctx* ctx, const void* d_cost, int cost_is_f64, int64_t B, const UamBestTail& tail, cudaStream_t st);
int uam_make_candidates_launch(uam_ctx* ctx, const double* d_cand, const double* h_ends, const double* d_disp, int N, int64_t B,
                               double jitter_sigma, uint64_t seed, uint64_t index0, double* d_z, cudaStream_t st);
// Raster scorer (uam_score_raster.cu), in the three steps of a call: uam_raster_prepare checks the arguments and fills
// the parameters; uam_raster_precompute builds the quad texels when a batch of this B and N samples them (may
// synchronise); uam_raster_grad_enqueue then enqueues one gradient launch (uam_grad_paths_raster's kernels) of a batch of
// the same B and N on `st`, without host synchronisation.  d_cost / d_collide are nullable, d_z and d_grad are not.
// uam_raster_grad_supported refuses the integral variants without a gradient form (1 and 3); a gradient call checks it
// before uam_raster_precompute.
int uam_raster_prepare(uam_ctx* ctx, int64_t B, int N, const double* h_p, int n_p, int flags, double spc, UamRasterParams* rp);
int uam_raster_grad_supported(uam_ctx* ctx, const UamRasterParams& rp);
int uam_raster_precompute(uam_ctx* ctx, UamRasterParams* rp, int64_t B, int N, cudaStream_t st);
int uam_raster_grad_enqueue(uam_ctx* ctx, const UamRasterParams& rp, const double* d_z, int64_t B, int N, float* d_cost,
                            uint8_t* d_collide, double* d_grad, cudaStream_t st);

// Occupancy bit-plane of the current raster: one bit per cell, a 32-bit word = 8 x 4 cells, a 128-byte line = 4 x 8 words
// = a 32 x 32-cell block (8192^2 cells = 8 MiB: L2-resident, mostly L1-resident along a path).  It sits at word 4 of
// ctx->d_occ_bits.  uam_ensure_occ_bits builds it from the texels on first use after each raster upload and synchronises
// `st` when it does, so every stream may read it afterwards (quad texels of the scorer, uam_sweep_paths_raster).
int uam_ensure_occ_bits(uam_ctx* ctx, cudaStream_t st);
inline unsigned uam_occ_words(int H, int W) { return (unsigned)((W + 31) / 32) * (unsigned)((H + 31) / 32) * 32u; }
__host__ __device__ __forceinline__ unsigned uam_occ_word(unsigned i, unsigned j, unsigned blocks_x) {
    return ((i >> 5) * blocks_x + (j >> 5)) * 32u + ((i >> 2) & 7u) * 4u + ((j >> 3) & 3u);
}
__host__ __device__ __forceinline__ unsigned uam_occ_bit(unsigned i, unsigned j) { return (i & 3u) * 8u + (j & 7u); }

// Swept check (uam_sweep.cu), in the steps of a call: uam_sweep_supported refuses an N whose segment table does not fit
// in shared memory and, with the clearance, a raster beyond uam_edt's limit; uam_ensure_occ_bits and, with the
// clearance, uam_sweep_ensure_d2 build the fields (both may synchronise: call them before enqueueing work that must
// stay ordered); uam_sweep_enqueue then enqueues one uam_k_sweep_paths launch on `st`, without host synchronisation.
// d_first_hit / d_d2min are nullable; d_d2min needs the d^2 field.
int uam_sweep_supported(uam_ctx* ctx, int N, bool clearance);
int uam_sweep_ensure_d2(uam_ctx* ctx, cudaStream_t st);
int uam_sweep_enqueue(uam_ctx* ctx, const double* d_z, int64_t B, int N, uint8_t* d_flags, int32_t* d_first_hit,
                      int32_t* d_d2min, cudaStream_t st);

// Analytic sweep and clearance (uam_sweep_analytic.cu), in the steps of a call once the shapes are known to be uploaded:
// uam_ensure_obs_tables checks the obstacles' records and forms and builds the sweep's cell lists on the first call
// after each upload; uam_obs_supported then returns the record checks' verdict and, with the clearance, the form
// checks' (UAM_ERR_UNSUPPORTED naming the obstacle); uam_ensure_clr_lists builds the clearance's lists for `cap` when
// they are missing (shape_grid option on).  Both builds synchronise the device when they run: call them before
// enqueueing work that must stay ordered.  uam_sweep_analytic_enqueue / uam_clearance_analytic_enqueue then enqueue one
// launch on `st`, without host synchronisation; the clearance's needs uam_ensure_clr_lists for the same cap first.
int uam_ensure_obs_tables(uam_ctx* ctx, cudaStream_t st);
int uam_obs_supported(uam_ctx* ctx, bool clearance);
int uam_ensure_clr_lists(uam_ctx* ctx, double cap, cudaStream_t st);
int uam_sweep_analytic_enqueue(uam_ctx* ctx, const double* d_z, int64_t B, int N, uint8_t* d_flags, int32_t* d_first_hit,
                               int32_t* d_first_obstacle, cudaStream_t st);
int uam_clearance_analytic_enqueue(uam_ctx* ctx, const double* d_z, int64_t B, int N, double cap, uint8_t* d_flags,
                                   double* d_clearance, int32_t* d_nearest_segment, int32_t* d_nearest_obstacle,
                                   cudaStream_t st);

// NVTX range over the rest of the enclosing scope (host side; a no-op costing a few ns when no profiler is attached):
// upload / bin / score / reduce / exchange phases show up by name on an Nsight Systems timeline
struct UamNvtxRange {
    explicit UamNvtxRange(const char* name) { nvtxRangePushA(name); }
    ~UamNvtxRange() { nvtxRangePop(); }
};
#define UAM_NVTX_CAT2(a, b) a##b
#define UAM_NVTX_CAT(a, b) UAM_NVTX_CAT2(a, b)
#define UAM_NVTX(name) UamNvtxRange UAM_NVTX_CAT(uam_nvtx_, __LINE__)(name)

#define UAM_CUDA(ctx, call)                                             \
    do {                                                                \
        cudaError_t _e = (call);                                        \
        if (_e != cudaSuccess) return uam_cuda_fail((ctx), _e, #call);  \
    } while (0)

#define UAM_CHECK_LAUNCH(ctx, name)                                     \
    do {                                                                \
        cudaError_t _e = cudaGetLastError();                            \
        if (_e != cudaSuccess) return uam_cuda_fail((ctx), _e, name);   \
        (ctx)->launches++;                                              \
    } while (0)

#define UAM_TRY(expr)                 \
    do {                              \
        int _rc = (expr);             \
        if (_rc != UAM_OK) return _rc; \
    } while (0)

#ifdef __CUDACC__
// ---- device helpers: exact fp64 inequality evaluation ----------------------------------------------
// Explicit round-to-nearest intrinsics keep nvcc from contracting a*b+c into an FMA, so the result
// has the same bits as the reference's numpy float64 arithmetic.
__device__ __forceinline__ double uam_h_exact(const UamEdge& r, double x, double y) {
    const int kind = (int)r.kind;
    if (kind == UAM_EDGE_LINE) {
        // -sgn * ((By-Ay)*(x-Ax) - (Bx-Ax)*(y-Ay))      polygon.py:69-71,98
        const double t1 = __dmul_rn(r.p3, __dsub_rn(x, r.p0));
        const double t2 = __dmul_rn(r.p2, __dsub_rn(y, r.p1));
        return __dmul_rn(-r.p4, __dsub_rn(t1, t2));
    } else if (kind == UAM_EDGE_ELLIPSE) {
        // ((x-cx)/r1)^2 + ((y-cy)/r2)^2 - 1             ball.py:33-37
        const double a = __ddiv_rn(__dsub_rn(x, r.p0), r.p2);
        const double b = __ddiv_rn(__dsub_rn(y, r.p1), r.p3);
        return __dsub_rn(__dadd_rn(__dmul_rn(a, a), __dmul_rn(b, b)), 1.0);
    } else {
        // x_d - c - r   |   -x_d + c - r                square.py:29-51
        const double xd = ((int)r.p0 == 0) ? x : y;
        if (r.p1 > 0) return __dsub_rn(__dsub_rn(xd, r.p2), r.p3);
        return __dsub_rn(__dadd_rn(-xd, r.p2), r.p3);
    }
}

// true if inequality r is > thr everywhere on the box [xa,xb] x [ya,yb] (with a rounding margin): used to cull shapes
// per raster tile (uam_map_rebuild.cu) and per cell of the shape grid (uam_shape_grid.cu)
__device__ __forceinline__ bool uam_edge_excludes_tile(const UamEdge& r, double xa, double xb, double ya, double yb,
                                                       double thr) {
    const int kind = (int)r.kind;
    double hmin, scale;
    if (kind == UAM_EDGE_ELLIPSE) {
        const double px = fmin(fmax(r.p0, xa), xb), py = fmin(fmax(r.p1, ya), yb);
        hmin = uam_h_exact(r, px, py);
        scale = fabs(hmin) + 2.0;
    } else {
        const double h0 = uam_h_exact(r, xa, ya), h1 = uam_h_exact(r, xb, ya);
        const double h2 = uam_h_exact(r, xa, yb), h3 = uam_h_exact(r, xb, yb);
        hmin = fmin(fmin(h0, h1), fmin(h2, h3));
        if (kind == UAM_EDGE_LINE) {
            const double mx = fmax(fabs(xa - r.p0), fabs(xb - r.p0)), my = fmax(fabs(ya - r.p1), fabs(yb - r.p1));
            scale = fabs(r.p3) * mx + fabs(r.p2) * my;
        } else {
            scale = fmax(fabs(xa), fabs(xb)) + fmax(fabs(ya), fabs(yb)) + fabs(r.p2) + fabs(r.p3);
        }
    }
    return hmin > thr + 1e-9 * scale + 1e-300;
}

__device__ __forceinline__ UamEdge uam_load_edge(const UamEdge* __restrict__ p) {
    // 4 x 16-byte read-only loads; every lane reads the same record (broadcast, L1-resident)
    const double2* q = reinterpret_cast<const double2*>(p);
    const double2 a = __ldg(q), b = __ldg(q + 1), c = __ldg(q + 2), d = __ldg(q + 3);
    UamEdge r;
    r.kind = a.x; r.p0 = a.y; r.p1 = b.x; r.p2 = b.y; r.p3 = c.x; r.p4 = c.y; r.p5 = d.x; r.p6 = d.y;
    return r;
}

// psi_s(x; e) = prod_i min(h_i - e, 0)^2 (smooth) | prod_i min(e - h_i, 0)   quadratic_obstacle.py:27-39
// `inside` (nullable) gets all_i h_i <= 1e-14                                  quadratic_obstacle.py:89-94
// `early_exit`: stop at the first zero of the running product.  Exact: with finite inequality records (checked at
// upload) and |x|, |y| < 1e100 every later factor is finite, so the reference's full product is the same 0 (a product
// that overflowed to inf before the zero gives NaN in both); when `inside` is wanted the loop also needs some
// h_i > 1e-14 before it may stop.
__device__ __forceinline__ double uam_psi(const UamEdge* __restrict__ edges, int e0, int e1, double x,
                                          double y, bool smooth, double e, bool* inside, bool early_exit = false) {
    double res = 1.0;
    bool in = true;
    const bool fast = early_exit && fabs(x) < 1e100 && fabs(y) < 1e100;
    for (int i = e0; i < e1; ++i) {
        const UamEdge r = uam_load_edge(edges + i);
        const double h = uam_h_exact(r, x, y);
        in = in && (h <= 1e-14);
        if (smooth) {
            const double m = fmin(__dsub_rn(h, e), 0.0);
            res = __dmul_rn(res, __dmul_rn(m, m));
        } else {
            res = __dmul_rn(res, fmin(__dsub_rn(e, h), 0.0));
        }
        if (fast && res == 0.0 && (!inside || !in)) break;
    }
    if (inside) *inside = in;
    return res;
}

// cell of (x, y) in the shape grid, -1 when there is no grid or the point is outside it (or not finite)
__device__ __forceinline__ int uam_shape_grid_cell(const UamShapeGrid& sg, double x, double y) {
    if (sg.G == 0) return -1;
    const double fx = __dmul_rn(__dsub_rn(x, sg.gx0), sg.inv_cw), fy = __dmul_rn(__dsub_rn(y, sg.gy0), sg.inv_ch);
    const double g = (double)sg.G;
    if (!(fx >= 0.0 && fx < g && fy >= 0.0 && fy < g)) return -1;
    return (int)fy * sg.G + (int)fx;
}

// Best-candidate key (uam_best, the fused tail of the raster scorer): 63 bits, (order-preserving image of the float32 cost)
// << 31 | global index (31 bits).  The image flips all bits of a negative cost and sets the top bit of a non-negative one,
// so unsigned order = float order for EVERY value (negative costs are reachable through negative layer weights), NaN maps
// to the largest image (a NaN never wins), and the key is a non-negative int64: the unsigned device min and the signed
// min of the cross-rank all-reduce agree.  Empty batch = 2^63 - 1 = distributed.KEY_EMPTY.
#define UAM_KEY_EMPTY 0x7fffffffffffffffull
__device__ __forceinline__ unsigned long long uam_best_key(float c, unsigned long long index) {
    unsigned bits = __float_as_uint(c);
    bits = (c != c) ? 0xffffffffu : ((bits & 0x80000000u) ? ~bits : (bits | 0x80000000u));
    return ((unsigned long long)bits << 31) | (index & 0x7fffffffull);
}

// ---- tail of a best-candidate launch -----------------------------------------------------------------------------------
// Every CTA calls it once with its own min key (thread 0's value counts); the last CTA to arrive owns the launch's min, and
// its first warp exchanges it with the peers: lane r stores the key into column `rank` of rank r's block, fences, raises
// the flag, then waits (bounded: ~2 s) for column r of its own block and the warp takes the min.  Must be reached by all
// threads of the CTA (it synchronises).
__device__ __forceinline__ unsigned long long uam_globaltimer() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
__device__ __forceinline__ void uam_best_tail_cta(const UamBestTail& tl, unsigned long long cta_key) {
    __shared__ int s_last;
    if (threadIdx.x == 0) {
        if (cta_key != UAM_KEY_EMPTY) atomicMin(tl.local, cta_key);
        __threadfence();
        const unsigned long long t = atomicAdd(tl.local + 1, 1ull);
        s_last = (t == (unsigned long long)gridDim.x - 1);
    }
    __syncthreads();
    if (!s_last || threadIdx.x >= 32) return;
    const int lane = threadIdx.x;
    __threadfence();
    unsigned long long key = *((volatile unsigned long long*)tl.local);
    if (lane == 0) {                       // ready for the next launch on this slot
        tl.local[0] = UAM_KEY_EMPTY;
        tl.local[1] = 0ull;
    }
    if (tl.world > 1) {
        const int ring = (int)(tl.epoch % UAM_PEER_RING);
        if (lane < tl.world) {
            UamPeerBlock* pb = tl.peer[lane];
            *((volatile unsigned long long*)&pb->keys[ring][tl.rank]) = key;
            __threadfence_system();
            *((volatile unsigned*)&pb->flags[ring][tl.rank]) = tl.epoch;
        }
        unsigned long long got = UAM_KEY_EMPTY;
        bool late = false;
        if (lane < tl.world) {
            UamPeerBlock* own = tl.peer[tl.rank];
            const unsigned long long t0 = uam_globaltimer();
            while (*((volatile unsigned*)&own->flags[ring][lane]) != tl.epoch) {
                if (uam_globaltimer() - t0 > 2000000000ull) { late = true; break; }
                __nanosleep(64);
            }
            __threadfence_system();
            if (!late) got = *((volatile unsigned long long*)&own->keys[ring][lane]);
        }
        if (__any_sync(0xffffffffu, late) && lane == 0 && tl.status) atomicExch(tl.status, 1u);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const unsigned long long t = __shfl_xor_sync(0xffffffffu, got, o);
            got = t < got ? t : got;
        }
        key = got;
    }
    if (lane == 0 && tl.out) {
        if (tl.combine) atomicMin(tl.out, key);
        else *tl.out = key;
    }
}
// min over the CTA of per-thread keys (all threads call; thread 0 returns the CTA's min)
__device__ __forceinline__ unsigned long long uam_cta_min_key(unsigned long long k) {
    __shared__ unsigned long long s_k[32];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long t = __shfl_xor_sync(0xffffffffu, k, o);
        k = t < k ? t : k;
    }
    if ((threadIdx.x & 31) == 0) s_k[threadIdx.x >> 5] = k;
    __syncthreads();
    if (threadIdx.x == 0)
        for (int i = 1; i < (int)((blockDim.x + 31) >> 5); ++i) k = s_k[i] < k ? s_k[i] : k;
    return k;
}

// pixel coordinate of a world coordinate: (x - x0)/dx - 1/2 with a true division (oracle: pixel_coords); the raster scorer's
// and the swept check's
__device__ __forceinline__ double uam_pix(double x, double x0, double dx) {
    return __dsub_rn(__ddiv_rn(__dsub_rn(x, x0), dx), 0.5);
}

__device__ __forceinline__ float uam_warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double uam_warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
#endif
