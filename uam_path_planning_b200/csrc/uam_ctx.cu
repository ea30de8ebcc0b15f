// Context, error handling, map uploads (shape tables and rasters) of libuam_b200.so.
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>

#include "uam_internal.cuh"

// ---------------------------------------------------------------------------------------------------
// errors / small helpers
// ---------------------------------------------------------------------------------------------------
int uam_fail(uam_ctx* ctx, int code, const char* fmt, ...) {
    if (ctx) {
        char buf[512];
        va_list ap;
        va_start(ap, fmt);
        vsnprintf(buf, sizeof buf, fmt, ap);
        va_end(ap);
        ctx->err = buf;
    }
    return code;
}

int uam_cuda_fail(uam_ctx* ctx, cudaError_t e, const char* what) {
    return uam_fail(ctx, e == cudaErrorMemoryAllocation ? UAM_ERR_NOMEM : UAM_ERR_CUDA, "%s: %s (%s)", what,
                    cudaGetErrorString(e), cudaGetErrorName(e));
}

int uam_reserve(uam_ctx* ctx, void** ptr, size_t* cur, size_t need) {
    if (*cur >= need && *ptr) return UAM_OK;
    if (*ptr) {
        UAM_CUDA(ctx, cudaFree(*ptr));
        *ptr = nullptr;
        *cur = 0;
    }
    size_t cap = need + need / 4 + 256;
    UAM_CUDA(ctx, cudaMalloc(ptr, cap));
    *cur = cap;
    return UAM_OK;
}

int uam_reserve_pinned(uam_ctx* ctx, void** ptr, size_t* cur, size_t need) {
    if (*cur >= need && *ptr) return UAM_OK;
    if (*ptr) {
        UAM_CUDA(ctx, cudaFreeHost(*ptr));
        *ptr = nullptr;
        *cur = 0;
    }
    size_t cap = need + need / 4 + 256;
    UAM_CUDA(ctx, cudaMallocHost(ptr, cap));
    *cur = cap;
    return UAM_OK;
}

// `stream` is the caller's cudaStream_t; NULL is CUDA's (legacy) default stream, as everywhere in CUDA
cudaStream_t uam_pick_stream(uam_ctx* ctx, void* stream) {
    (void)ctx;
    return reinterpret_cast<cudaStream_t>(stream);
}

// p = [ms_x, ms_y, mg_x, mg_y, maxratio, maxalpha, enlargement, w_0..w_{R-1}]   (solver.py:60-68)
int uam_make_params(uam_ctx* ctx, const double* h_p, int n_p, int flags, UamParams* out) {
    if (!h_p) return uam_fail(ctx, UAM_ERR_INVALID, "parameter vector p is NULL");
    if (n_p < 7) return uam_fail(ctx, UAM_ERR_INVALID, "parameter vector p needs >= 7 entries, got %d", n_p);
    const int R = n_p - 7;
    if (R > UAM_MAX_REGIONS)
        return uam_fail(ctx, UAM_ERR_UNSUPPORTED, "%d region weights given, at most %d supported", R, UAM_MAX_REGIONS);
    memset(out, 0, sizeof *out);
    out->ms_x = h_p[0];
    out->ms_y = h_p[1];
    out->maxratio = h_p[4];
    out->mincos = std::cos(h_p[5]);     // cs.cos(maxalpha), problem.py:98
    out->e = h_p[6];
    for (int r = 0; r < R; ++r) out->w[r] = h_p[7 + r];
    out->flags = flags & 0xffff;          // the upper bits are the library's own (UAM_INTERNAL_*)
    out->n_regions = R;
    return UAM_OK;
}

// ---------------------------------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------------------------------
extern "C" const char* uam_version(void) { return "uam_b200 0.1 (sm_100a)"; }

extern "C" int uam_ctx_create(int device, uam_ctx** out) {
    if (!out) return UAM_ERR_INVALID;
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0 || device < 0 || device >= n) return UAM_ERR_CUDA;  // no CPU fallback
    uam_ctx* ctx = new (std::nothrow) uam_ctx();
    if (!ctx) return UAM_ERR_NOMEM;
    ctx->device = device;
    if (cudaSetDevice(device) != cudaSuccess) { delete ctx; return UAM_ERR_CUDA; }
    cudaDeviceGetAttribute(&ctx->sm_count, cudaDevAttrMultiProcessorCount, device);
    if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) { delete ctx; return UAM_ERR_CUDA; }
    for (int i = 0; i < UAM_HOST_PIPE_DEPTH; ++i) {
        if (cudaStreamCreateWithFlags(&ctx->pipe_stream[i], cudaStreamNonBlocking) != cudaSuccess ||
            cudaEventCreateWithFlags(&ctx->pipe_event[i], cudaEventDisableTiming) != cudaSuccess) {
            delete ctx;
            return UAM_ERR_CUDA;
        }
    }
    // tuning knobs from the environment (bench A/B runs); uam_ctx_set_option overrides
    if (const char* e = getenv("UAM_RASTER_LAYOUT")) ctx->raster_layout = atoi(e) ? 1 : 0;
    if (const char* e = getenv("UAM_INT_VARIANT")) ctx->int_variant = std::min(3, std::max(-1, atoi(e)));
    if (const char* e = getenv("UAM_GRID_HALF_CAP")) ctx->grid_half_cap = std::max(0, atoi(e));
    if (const char* e = getenv("UAM_GRID_GRAPH")) ctx->grid_graph = atoi(e) ? 1 : 0;
    if (const char* e = getenv("UAM_GRID_DELTA")) ctx->grid_delta = std::max(0ll, atoll(e));
    if (const char* e = getenv("UAM_BIN_CHUNK")) ctx->bin_chunk = std::min(1 << 20, std::max(1024, atoi(e)));
    if (const char* e = getenv("UAM_BIN_PT")) ctx->bin_pt = atoi(e);
    if (const char* e = getenv("UAM_BIN_SHIFT")) ctx->bin_shift = std::min(10, std::max(4, atoi(e)));
    if (const char* e = getenv("UAM_NO_SIGN_PACK")) ctx->no_sign_pack = atoi(e) ? 1 : 0;
    if (const char* e = getenv("UAM_COMBINE_LAYERS")) ctx->combine_layers = atoi(e) ? 1 : 0;
    if (const char* e = getenv("UAM_HOST_CHUNKS")) ctx->host_chunks = std::max(0, atoi(e));
    if (const char* e = getenv("UAM_HOST_TAPER")) ctx->host_taper = std::min(95, std::max(-95, atoi(e)));
    if (const char* e = getenv("UAM_L2_FETCH_GRANULARITY")) cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, (size_t)atoi(e));
    *out = ctx;
    return UAM_OK;
}

extern "C" int uam_ctx_set_option(uam_ctx* ctx, int option, int64_t value) {
    if (!ctx) return UAM_ERR_INVALID;
    switch (option) {
        case UAM_OPT_RASTER_LAYOUT:
            if (value != 0 && value != 1) return uam_fail(ctx, UAM_ERR_INVALID, "raster layout must be 0 or 1");
            ctx->raster_layout = (int)value;
            return UAM_OK;
        case UAM_OPT_INTEGRAL_VARIANT:
            if (value < -1 || value > 3) return uam_fail(ctx, UAM_ERR_INVALID, "integral variant must be -1 (auto), 0, 1, 2 or 3");
            ctx->int_variant = (int)value;
            return UAM_OK;
        case UAM_OPT_L2_FETCH_GRANULARITY:
            if (value != 32 && value != 64 && value != 128) return uam_fail(ctx, UAM_ERR_INVALID, "L2 fetch granularity must be 32, 64 or 128");
            UAM_CUDA(ctx, cudaSetDevice(ctx->device));
            UAM_CUDA(ctx, cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, (size_t)value));
            return UAM_OK;
        case UAM_OPT_GRID_DELTA:
            if (value < 0) return uam_fail(ctx, UAM_ERR_INVALID, "grid delta must be >= 0");
            ctx->grid_delta = (long long)value;
            return UAM_OK;
        case UAM_OPT_GRID_HALF_CAP:
            if (value < 0 || value > 1000000) return uam_fail(ctx, UAM_ERR_INVALID, "grid half-sweep cap must be 0 (none) .. 1000000");
            ctx->grid_half_cap = (int)value;
            return UAM_OK;
        case UAM_OPT_GRID_GRAPH:
            if (value != 0 && value != 1) return uam_fail(ctx, UAM_ERR_INVALID, "grid graph must be 0 or 1");
            ctx->grid_graph = (int)value;
            return UAM_OK;
        case UAM_OPT_COMBINE_LAYERS:
            if (value < 0 || value > 2) return uam_fail(ctx, UAM_ERR_INVALID, "combine_layers must be 0, 1 or 2");
            ctx->combine_layers = value != 0;
            ctx->no_sign_pack = value == 2;
            ctx->comb_valid = false;
            return UAM_OK;
        case UAM_OPT_HOST_CHUNKS:
            if (value < 0 || value > 64) return uam_fail(ctx, UAM_ERR_INVALID, "host chunks must be 0 (default) .. 64");
            ctx->host_chunks = (int)value;
            return UAM_OK;
        case UAM_OPT_HOST_TAPER:
            if (value < -95 || value > 95) return uam_fail(ctx, UAM_ERR_INVALID, "host taper must be -95 .. 95 percent");
            ctx->host_taper = (int)value;
            return UAM_OK;
        case UAM_OPT_SHAPE_GRID:
            if (value != 0 && value != 1) return uam_fail(ctx, UAM_ERR_INVALID, "shape grid must be 0 or 1");
            ctx->shape_grid_opt = (int)value;
            ctx->psic_valid = false;        // rebuilt (or dropped) with the next analytic call
            ctx->shape_grid = UamShapeGrid{};
            return UAM_OK;
        case UAM_OPT_CCL_TILES:
            if (value != 0 && value != 1) return uam_fail(ctx, UAM_ERR_INVALID, "ccl_tiles must be 0 or 1");
            ctx->ccl_tiles = (int)value;
            return UAM_OK;
        case UAM_OPT_RASTERIZER:
            if (value < 0 || value > 3) return uam_fail(ctx, UAM_ERR_INVALID, "rasterizer must be 0 (per cell), 1 (scanline), 2 (scanline, tile form of the layers) or 3 (scanline, sampled row form of the layers)");
            ctx->rasterizer_scan = (int)value;
            return UAM_OK;
        case UAM_OPT_TIME_KERNELS:
            UAM_CUDA(ctx, cudaSetDevice(ctx->device));
            if (value && !ctx->time_ev[0]) {
                for (int i = 0; i < 2 * uam_ctx::kTimeRing; ++i) UAM_CUDA(ctx, cudaEventCreate(&ctx->time_ev[i]));
            }
            ctx->time_kernels = value ? 1 : 0;
            ctx->time_pending = 0;
            ctx->time_sum_ms = 0.0;
            ctx->time_count = 0;
            return UAM_OK;
        default:
            return uam_fail(ctx, UAM_ERR_INVALID, "unknown option %d", option);
    }
}

// Folds the pending event pairs into the running sum (waits for the last timed kernel).  Called when the ring is full
// and before a statistic is read -- never between two launches of a timed loop shorter than the ring.
int uam_time_collect(uam_ctx* ctx) {
    for (int i = 0; i < ctx->time_pending; ++i) {
        float ms = 0.0f;
        UAM_CUDA(ctx, cudaEventSynchronize(ctx->time_ev[2 * i + 1]));
        UAM_CUDA(ctx, cudaEventElapsedTime(&ms, ctx->time_ev[2 * i], ctx->time_ev[2 * i + 1]));
        ctx->time_sum_ms += ms;
        ctx->time_count += 1;
    }
    ctx->time_pending = 0;
    return UAM_OK;
}

int uam_time_begin(uam_ctx* ctx, cudaStream_t st) {
    if (ctx->time_pending == uam_ctx::kTimeRing) UAM_TRY(uam_time_collect(ctx));
    UAM_CUDA(ctx, cudaEventRecord(ctx->time_ev[2 * ctx->time_pending], st));
    return UAM_OK;
}

int uam_time_end(uam_ctx* ctx, cudaStream_t st) {
    UAM_CUDA(ctx, cudaEventRecord(ctx->time_ev[2 * ctx->time_pending + 1], st));
    ctx->time_pending += 1;
    return UAM_OK;
}

extern "C" int uam_ctx_get_stat(uam_ctx* ctx, int stat, double* value) {
    if (!ctx || !value) return UAM_ERR_INVALID;
    UAM_CUDA(ctx, cudaSetDevice(ctx->device));
    UAM_TRY(uam_time_collect(ctx));
    switch (stat) {
        case UAM_STAT_SCORE_KERNEL_MS_MEAN:
            *value = ctx->time_count ? ctx->time_sum_ms / (double)ctx->time_count : 0.0;
            return UAM_OK;
        case UAM_STAT_SCORE_KERNEL_COUNT:
            *value = (double)ctx->time_count;
            return UAM_OK;
        case UAM_STAT_GRID_ACTIVATIONS: *value = ctx->grid_activations; return UAM_OK;
        case UAM_STAT_GRID_SWEEPS: *value = ctx->grid_sweeps; return UAM_OK;
        case UAM_STAT_GRID_ROUNDS: *value = ctx->grid_rounds; return UAM_OK;
        case UAM_STAT_GRID_HOST_SUBMISSIONS: *value = ctx->grid_host_submissions; return UAM_OK;
        case UAM_STAT_SHAPE_GRID_CELLS: *value = (double)ctx->shape_grid.G * ctx->shape_grid.G; return UAM_OK;
        case UAM_STAT_SHAPE_GRID_ITEMS: *value = ctx->shape_grid.G ? (double)ctx->grid_items_total : 0.0; return UAM_OK;
        default:
            return uam_fail(ctx, UAM_ERR_INVALID, "unknown stat %d", stat);
    }
}

extern "C" int uam_ctx_destroy(uam_ctx* ctx) {
    if (!ctx) return UAM_OK;
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    cudaFree(ctx->d_edges);
    cudaFree(ctx->d_shapes);
    cudaFree(ctx->d_psic);
    cudaFree(ctx->d_grid_start);
    cudaFree(ctx->d_grid_items);
    cudaFree(ctx->d_obs_grid);
    cudaFree(ctx->d_obs_items);
    cudaFree(ctx->d_tex);
    cudaFree(ctx->d_scratch);
    cudaFree(ctx->d_cull_scratch);
    cudaFree(ctx->d_cull0_scratch);
    for (int i = 0; i <= UAM_HOST_PIPE_DEPTH; ++i) cudaFree(ctx->d_bin_scratch[i]);
    for (int i = 0; i <= UAM_HOST_PIPE_DEPTH; ++i) cudaFree(ctx->d_piece_scratch[i]);
    cudaFree(ctx->d_tiles);
    cudaFree(ctx->d_tex_comb);
    cudaFree(ctx->d_occ_bits);
    cudaFree(ctx->d_refine_scratch);
    cudaFree(ctx->d_sweep_d2);
    for (int i = 0; i < UAM_HOST_PIPE_DEPTH; ++i) {
        cudaFree(ctx->d_stage_in[i]);
        cudaFree(ctx->d_stage_out[i]);
        cudaFreeHost(ctx->h_stage_out[i]);
        if (ctx->pipe_stream[i]) cudaStreamDestroy(ctx->pipe_stream[i]);
        if (ctx->pipe_event[i]) cudaEventDestroy(ctx->pipe_event[i]);
    }
    for (int i = 0; i < UAM_HOST_PIPE_DEPTH; ++i) {
        cudaFree(ctx->d_ring_cand[i]);
        cudaFree(ctx->d_ring_key[i]);
    }
    cudaFree(ctx->d_best_local);
    for (int r = 0; r < ctx->peer_world; ++r)
        if (r != ctx->peer_rank && ctx->peer_ptr[r]) cudaIpcCloseMemHandle(ctx->peer_ptr[r]);
    cudaFree(ctx->d_peer_own);
    for (int i = 0; i < 2 * uam_ctx::kTimeRing; ++i)
        if (ctx->time_ev[i]) cudaEventDestroy(ctx->time_ev[i]);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
    return UAM_OK;
}

extern "C" const char* uam_last_error(const uam_ctx* ctx) { return ctx ? ctx->err.c_str() : "null ctx"; }

extern "C" int uam_launch_count(const uam_ctx* ctx, uint64_t* n) {
    if (!ctx || !n) return UAM_ERR_INVALID;
    *n = ctx->launches;
    return UAM_OK;
}

extern "C" int uam_sync(uam_ctx* ctx) {
    if (!ctx) return UAM_ERR_INVALID;
    UAM_CUDA(ctx, cudaSetDevice(ctx->device));
    UAM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    for (int i = 0; i < UAM_HOST_PIPE_DEPTH; ++i) UAM_CUDA(ctx, cudaStreamSynchronize(ctx->pipe_stream[i]));
    return UAM_OK;
}

// ---------------------------------------------------------------------------------------------------
// shape tables
// ---------------------------------------------------------------------------------------------------
extern "C" int uam_map_set_shapes(uam_ctx* ctx, const double* h_edges, int n_edges, const int32_t* h_shape_off,
                                  const int32_t* h_shape_region, const double* h_shape_center, int n_shapes,
                                  int n_regions) {
    if (!ctx) return UAM_ERR_INVALID;
    UAM_NVTX("uam.map.set_shapes");
    if (n_shapes < 0 || n_edges < 0 || n_regions < 0) return uam_fail(ctx, UAM_ERR_INVALID, "negative table size");
    if (n_regions > UAM_MAX_REGIONS)
        return uam_fail(ctx, UAM_ERR_UNSUPPORTED, "%d regions, at most %d supported", n_regions, UAM_MAX_REGIONS);
    if (n_shapes > 0 && (!h_shape_off || !h_shape_region || !h_shape_center || (n_edges > 0 && !h_edges)))
        return uam_fail(ctx, UAM_ERR_INVALID, "NULL shape table");
    if (n_shapes > 0 && (h_shape_off[0] != 0 || h_shape_off[n_shapes] != n_edges))
        return uam_fail(ctx, UAM_ERR_INVALID, "shape offsets must run from 0 to n_edges");
    for (int s = 0; s < n_shapes; ++s) {
        if (h_shape_off[s + 1] < h_shape_off[s]) return uam_fail(ctx, UAM_ERR_INVALID, "shape offsets not monotone");
        if (h_shape_region[s] < -1 || h_shape_region[s] >= n_regions)
            return uam_fail(ctx, UAM_ERR_INVALID, "shape %d: region %d out of range", s, h_shape_region[s]);
    }
    for (int i = 0; i < n_edges; ++i) {
        const int k = (int)h_edges[8 * (size_t)i];
        if (k != UAM_EDGE_LINE && k != UAM_EDGE_ELLIPSE && k != UAM_EDGE_BOX)
            return uam_fail(ctx, UAM_ERR_INVALID, "inequality %d: unknown kind %d", i, k);
    }
    bool finite = true;
    double max_abs = 0.0;
    for (size_t i = 0; i < 8 * (size_t)n_edges; ++i) {
        finite = finite && std::isfinite(h_edges[i]);
        if (std::isfinite(h_edges[i])) max_abs = std::max(max_abs, std::fabs(h_edges[i]));
    }
    int max_per_shape = 0;
    for (int s = 0; s < n_shapes; ++s) max_per_shape = std::max(max_per_shape, h_shape_off[s + 1] - h_shape_off[s]);
    ctx->edges_max_abs = max_abs;
    ctx->max_edges_per_shape = max_per_shape;
    // bounding box of the shapes as far as the records tell (polygon vertices, ellipse / box extents): the extent of
    // the analytic scorer's shape grid.  Points outside it are scored with the full loops, so it only has to be sensible.
    double bx0 = INFINITY, bx1 = -INFINITY, by0 = INFINITY, by1 = -INFINITY;
    for (int i = 0; i < n_edges && finite; ++i) {
        const double* r = h_edges + 8 * (size_t)i;
        const int k = (int)r[0];
        if (k == UAM_EDGE_LINE) {
            bx0 = std::min(bx0, std::min(r[1], r[1] + r[3])); bx1 = std::max(bx1, std::max(r[1], r[1] + r[3]));
            by0 = std::min(by0, std::min(r[2], r[2] + r[4])); by1 = std::max(by1, std::max(r[2], r[2] + r[4]));
        } else if (k == UAM_EDGE_ELLIPSE) {
            bx0 = std::min(bx0, r[1] - std::fabs(r[3])); bx1 = std::max(bx1, r[1] + std::fabs(r[3]));
            by0 = std::min(by0, r[2] - std::fabs(r[4])); by1 = std::max(by1, r[2] + std::fabs(r[4]));
        } else if ((int)r[1] == 0) {
            bx0 = std::min(bx0, r[3] - std::fabs(r[4])); bx1 = std::max(bx1, r[3] + std::fabs(r[4]));
        } else {
            by0 = std::min(by0, r[3] - std::fabs(r[4])); by1 = std::max(by1, r[3] + std::fabs(r[4]));
        }
    }
    ctx->shape_bbox[0] = bx0; ctx->shape_bbox[1] = bx1; ctx->shape_bbox[2] = by0; ctx->shape_bbox[3] = by1;
    ctx->shape_grid = UamShapeGrid{};
    UAM_CUDA(ctx, cudaSetDevice(ctx->device));

    // device order: obstacles (insertion order), then regions 0..R-1 (insertion order inside each)
    std::vector<UamEdge> edges;
    std::vector<UamShape> shapes;
    edges.reserve(n_edges);
    shapes.reserve(n_shapes);
    int n_obs = 0;
    for (int pass = -1; pass < n_regions; ++pass) {
        if (pass >= 0) ctx->region_begin[pass] = (int)shapes.size();
        for (int s = 0; s < n_shapes; ++s) {
            if (h_shape_region[s] != pass) continue;
            UamShape sh;
            sh.cx = h_shape_center[2 * s];
            sh.cy = h_shape_center[2 * s + 1];
            sh.has_center = !(std::isnan(sh.cx) || std::isnan(sh.cy));   // np.isnan(obs.center).any(), problem.py:76
            sh.region = pass;
            sh.e0 = (int)edges.size();
            for (int i = h_shape_off[s]; i < h_shape_off[s + 1]; ++i) {
                UamEdge r;
                memcpy(&r, h_edges + 8 * (size_t)i, sizeof r);
                edges.push_back(r);
            }
            sh.e1 = (int)edges.size();
            shapes.push_back(sh);
            if (pass < 0) ++n_obs;
        }
    }
    ctx->region_begin[n_regions] = (int)shapes.size();

    cudaFree(ctx->d_edges);  ctx->d_edges = nullptr;
    cudaFree(ctx->d_shapes); ctx->d_shapes = nullptr;
    cudaFree(ctx->d_psic);   ctx->d_psic = nullptr;
    UAM_CUDA(ctx, cudaMalloc(&ctx->d_edges, sizeof(UamEdge) * (edges.size() + 1)));
    UAM_CUDA(ctx, cudaMalloc(&ctx->d_shapes, sizeof(UamShape) * (shapes.size() + 1)));
    UAM_CUDA(ctx, cudaMalloc(&ctx->d_psic, sizeof(double) * (shapes.size() + 1)));
    if (!edges.empty())
        UAM_CUDA(ctx, cudaMemcpy(ctx->d_edges, edges.data(), sizeof(UamEdge) * edges.size(), cudaMemcpyHostToDevice));
    if (!shapes.empty())
        UAM_CUDA(ctx, cudaMemcpy(ctx->d_shapes, shapes.data(), sizeof(UamShape) * shapes.size(), cudaMemcpyHostToDevice));
    ctx->n_shapes = (int)shapes.size();
    ctx->n_edges = (int)edges.size();
    ctx->n_regions = n_regions;
    ctx->n_obs = n_obs;
    ctx->has_shapes = true;
    ctx->shapes_gen++;
    ctx->edges_finite = finite;
    ctx->psic_valid = false;
    return UAM_OK;
}

// psi_s(center_s; e) per shape (problem.py:79), recomputed only when e / smooth flags change
__global__ void uam_k_shape_norm(const UamEdge* __restrict__ edges, const UamShape* __restrict__ shapes, int n_shapes,
                                 int flags, double e, double* __restrict__ psic) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_shapes) return;
    const UamShape sh = shapes[s];
    if (!sh.has_center) { psic[s] = 1.0; return; }
    // hard obstacles: obstacle_smooth, enlargement = params['enlargement'] (get_penalty_function(None))
    const bool smooth = sh.region < 0 ? (flags & UAM_OBSTACLE_SMOOTH) != 0 : (flags & UAM_PENALTY_SMOOTH) != 0;
    psic[s] = uam_psi(edges, sh.e0, sh.e1, sh.cx, sh.cy, smooth, e, nullptr);
}

int uam_ensure_shape_norm(uam_ctx* ctx, const UamParams& prm, cudaStream_t st, bool want_grid) {
    const int key = prm.flags & (UAM_PENALTY_SMOOTH | UAM_OBSTACLE_SMOOTH);
    if (!(ctx->psic_valid && ctx->psic_e == prm.e && ctx->psic_flags == key)) {
        if (ctx->n_shapes > 0) {
            // all streams that may still read the old table must be done before it is overwritten
            UAM_CUDA(ctx, cudaDeviceSynchronize());
            uam_k_shape_norm<<<(ctx->n_shapes + 127) / 128, 128, 0, st>>>(ctx->d_edges, ctx->d_shapes, ctx->n_shapes,
                                                                           prm.flags, prm.e, ctx->d_psic);
            UAM_CHECK_LAUNCH(ctx, "uam_k_shape_norm");
            UAM_CUDA(ctx, cudaStreamSynchronize(st));
        }
        ctx->shape_grid = UamShapeGrid{};
        ctx->shape_grid_built = false;
        ctx->psic_valid = true;
        ctx->psic_e = prm.e;
        ctx->psic_flags = key;
    }
    // the analytic scorer's cell lists are built on its first call for these parameters, not for the rasterisers (which
    // cull per raster tile): 8 ms per build on config C4's 4096 shapes
    if (want_grid && !ctx->shape_grid_built) {
        if (ctx->n_shapes > 0) {
            UAM_CUDA(ctx, cudaDeviceSynchronize());
            UAM_TRY(uam_build_shape_grid(ctx, prm.e, prm.flags, st));
        }
        ctx->shape_grid_built = true;
    }
    return UAM_OK;
}

// ---------------------------------------------------------------------------------------------------
// rasters: planar (L,H,W) float32 + (H,W) uint8  ->  interleaved texels (layer values + occupancy)
// ---------------------------------------------------------------------------------------------------
// One thread per OUTPUT texel (coalesced writes); tiled layouts are padded to whole tiles with zero texels.
template <int TF, int LAYOUT>
__global__ void uam_k_pack_texels(const float* __restrict__ layers, const uint8_t* __restrict__ occ, int L, int H, int W,
                                  int tiles_x, size_t n_out, float* __restrict__ tex) {
    const size_t n_cells = (size_t)H * W;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t o = (size_t)blockIdx.x * blockDim.x + threadIdx.x; o < n_out; o += stride) {
        int i, j;
        if (LAYOUT == 0) {
            i = (int)(o / W);
            j = (int)(o - (size_t)i * W);
        } else if (TF == 4) {
            const size_t tile = o >> 3;
            const int w = (int)(o & 7), ty = (int)(tile / tiles_x), tx = (int)(tile - (size_t)ty * tiles_x);
            i = ty * 2 + ((w >> 1) & 1);
            j = tx * 4 + ((w >> 2) & 1) * 2 + (w & 1);
        } else {
            const size_t tile = o >> 4;
            const int w = (int)(o & 15), ty = (int)(tile / tiles_x), tx = (int)(tile - (size_t)ty * tiles_x);
            i = ty * 4 + ((w >> 3) & 1) * 2 + ((w >> 1) & 1);
            j = tx * 4 + ((w >> 2) & 1) * 2 + (w & 1);
        }
        const bool in = i < H && j < W;
        const size_t c = (size_t)i * W + j;
        const float ov = (in && occ && occ[c]) ? 1.0f : 0.0f;
        if (TF == 2) {
            reinterpret_cast<float2*>(tex)[o] = make_float2(in ? layers[c] : 0.0f, ov);
        } else {
            const float l0 = in ? layers[c] : 0.0f;
            const float l1 = (in && L > 1) ? layers[n_cells + c] : 0.0f;
            const float l2 = (in && L > 2) ? layers[2 * n_cells + c] : 0.0f;
            reinterpret_cast<float4*>(tex)[o] = make_float4(l0, l1, l2, ov);
        }
    }
}

static int uam_check_raster_args(uam_ctx* ctx, const void* layers, int L, int H, int W, double dx, double dy) {
    if (!ctx) return UAM_ERR_INVALID;
    if (!layers) return uam_fail(ctx, UAM_ERR_INVALID, "layers is NULL");
    if (L < 1 || L > 3) return uam_fail(ctx, UAM_ERR_UNSUPPORTED, "L = %d cost layers, supported: 1..3", L);
    if (H < 2 || W < 2) return uam_fail(ctx, UAM_ERR_INVALID, "raster must be at least 2 x 2, got %d x %d", H, W);
    if (!(dx != 0.0) || !(dy != 0.0) || std::isnan(dx) || std::isnan(dy))
        return uam_fail(ctx, UAM_ERR_INVALID, "cell size must be non-zero");
    return UAM_OK;
}

extern "C" int uam_map_set_raster_device(uam_ctx* ctx, const float* d_layers, int L, int H, int W, double x0, double dx,
                                         double y0, double dy, const uint8_t* d_occupancy, void* stream) {
    UAM_TRY(uam_check_raster_args(ctx, d_layers, L, H, W, dx, dy));
    UAM_NVTX("uam.map.set_raster (pack texels)");
    UAM_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = uam_pick_stream(ctx, stream);
    const int tf = (L == 1) ? 2 : 4;
    const int layout = ctx->raster_layout;
    const int tile_h = (tf == 4) ? 2 : 4;
    const int tiles_x = (W + 3) / 4, tiles_y = (H + tile_h - 1) / tile_h;
    const size_t n_out = layout ? (size_t)tiles_x * tiles_y * 4 * tile_h : (size_t)H * W;
    if (n_out >= 0xffffffffull) return uam_fail(ctx, UAM_ERR_UNSUPPORTED, "raster has 2^32 or more texels");
    // the old texels may still be read by kernels queued on other streams
    UAM_CUDA(ctx, cudaDeviceSynchronize());
    UAM_TRY(uam_reserve(ctx, &ctx->d_tex, &ctx->tex_bytes, n_out * tf * sizeof(float)));
    const int grid = ctx->sm_count * 8;
    float* tex = (float*)ctx->d_tex;
    if (tf == 2 && layout) uam_k_pack_texels<2, 1><<<grid, 256, 0, st>>>(d_layers, d_occupancy, L, H, W, tiles_x, n_out, tex);
    else if (tf == 2) uam_k_pack_texels<2, 0><<<grid, 256, 0, st>>>(d_layers, d_occupancy, L, H, W, tiles_x, n_out, tex);
    else if (layout) uam_k_pack_texels<4, 1><<<grid, 256, 0, st>>>(d_layers, d_occupancy, L, H, W, tiles_x, n_out, tex);
    else uam_k_pack_texels<4, 0><<<grid, 256, 0, st>>>(d_layers, d_occupancy, L, H, W, tiles_x, n_out, tex);
    UAM_CHECK_LAUNCH(ctx, "uam_k_pack_texels");
    ctx->geo.x0 = x0; ctx->geo.dx = dx; ctx->geo.y0 = y0; ctx->geo.dy = dy;
    ctx->geo.H = H; ctx->geo.W = W; ctx->geo.L = L; ctx->geo.texel_floats = tf;
    ctx->geo.layout = layout; ctx->geo.tiles_x = tiles_x; ctx->geo.tiles_y = tiles_y;
    ctx->has_raster = true;
    ctx->tiles_valid = false;
    ctx->comb_valid = false;
    ctx->occ_bits_valid = false;
    ctx->raster_gen += 1;
    return UAM_OK;
}

extern "C" int uam_map_set_raster(uam_ctx* ctx, const float* h_layers, int L, int H, int W, double x0, double dx,
                                  double y0, double dy, const uint8_t* h_occupancy) {
    UAM_TRY(uam_check_raster_args(ctx, h_layers, L, H, W, dx, dy));
    UAM_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t n_cells = (size_t)H * W;
    float* d_layers = nullptr;
    uint8_t* d_occ = nullptr;
    UAM_CUDA(ctx, cudaMalloc(&d_layers, n_cells * L * sizeof(float)));
    cudaError_t e = cudaMemcpy(d_layers, h_layers, n_cells * L * sizeof(float), cudaMemcpyHostToDevice);
    if (e == cudaSuccess && h_occupancy) {
        e = cudaMalloc(&d_occ, n_cells);
        if (e == cudaSuccess) e = cudaMemcpy(d_occ, h_occupancy, n_cells, cudaMemcpyHostToDevice);
    }
    int rc = UAM_OK;
    if (e != cudaSuccess) rc = uam_cuda_fail(ctx, e, "raster upload");
    if (rc == UAM_OK) rc = uam_map_set_raster_device(ctx, d_layers, L, H, W, x0, dx, y0, dy, d_occ, nullptr);
    if (rc == UAM_OK) {
        cudaError_t e2 = cudaStreamSynchronize(nullptr);
        if (e2 != cudaSuccess) rc = uam_cuda_fail(ctx, e2, "raster pack");
    }
    cudaFree(d_layers);
    cudaFree(d_occ);
    return rc;
}
