// Raster path scorer: the reference's cost functional (problem.py:38-44,130-146) with the analytic penalty
// replaced by a bilinear lookup in the cost rasters, and Map.collides replaced by nearest-cell occupancy.
//
// HBM layout: one texel per cell, the L cost layers interleaved with the occupancy flag (float2 for L = 1, float4
// for L = 2..3), either row-major or tiled (uam_tex_row / uam_tex_col): one bilinear tap = 4 texel loads of 8/16 B.
//
// Sampling modes
//   waypoint mode  (samples_per_cell == 0): one sample per waypoint -- the reference's sampling; warp per path,
//                  lanes stride the N+2 waypoints.
//   integral mode  (samples_per_cell  > 0): segment k gets S_k = max(1, ceil(|dz_k|_cells * spc)) left-endpoint
//                  samples (mean per segment).  Three kernels, selected by UAM_OPT_INTEGRAL_VARIANT:
//       0  warp per path; the path's samples are flattened, lanes stride the flat sample index
//       1  as 0 with a lane PAIR per sample (kept for comparison; slower)
//       2  binned: the batch's segments are counting-sorted by raster bin, a warp scores 32 consecutive sorted
//          segments with the same flat loop, a last kernel adds the per-segment partials per path.  The warps in
//          flight then sample the same few bins and the raster streams through L2 about once per batch instead of
//          once per path corridor.
// World -> pixel coordinates, S_k and the sample positions are fp64 in a fixed operation order (identical bits to
// the oracle: same cells, same occupancy lookups, same sample counts); bilinear weights, texel arithmetic and the
// penalty sums are fp32; the length term is fp64.  Sums finish with warp-shuffle reductions in a fixed order
// (bit-reproducible; no floating-point atomics).
#include <algorithm>
#include <type_traits>

#include "uam_internal.cuh"

#define UAM_MAX_SAMPLES_PER_SEGMENT 1048576.0   // cap on S_k (a segment never spans more cells than this)
// B * (N + 2) from which a batch is large: the auto integral variant is the binned pipeline, and waypoint mode is worth
// the one-off build of the quad texels
#define UAM_LARGE_BATCH_SEGMENTS 262144ull

namespace {

template <int TF> struct UamTexel;
template <> struct UamTexel<2> { typedef float2 T; };
template <> struct UamTexel<4> { typedef float4 T; };
template <> struct UamTexel<1> { typedef float4 T; };      // quad mode: the 2 x 2 bilinear footprint of a cell in one texel
template <> struct UamTexel<8> { typedef float4 T; };      // quad mode, occupancy flags in the sign bits (values >= 0)
template <int TF> struct UamIsQuad { static const bool v = (TF == 1 || TF == 8); };

// Texel address = uam_tex_row(i) + uam_tex_col(j)  (both layouts are separable).
// LAYOUT 0: row-major (H, W).  LAYOUT 1: tiled so that one 128-byte line is a compact 2-D block and every 32-byte
// sector a 2 x 1 (float4) / 2 x 2 (float2) block:
//   float4: line = 4 wide x 2 tall:  ((i>>1) * tiles_x + (j>>2)) * 8  + ((j>>1)&1)*4 + (i&1)*2 + (j&1)
//   float2: line = 4 wide x 4 tall:  ((i>>2) * tiles_x + (j>>2)) * 16 + ((i>>1)&1)*8 + ((j>>1)&1)*4 + (i&1)*2 + (j&1)
// Texel indices are 32-bit (uam_map_set_raster refuses rasters with 2^32 or more texels).
template <int TF, int LAYOUT>
__device__ __forceinline__ unsigned uam_tex_row(unsigned i, unsigned row_stride) {
    if (LAYOUT == 0) return i * row_stride;
    if (TF == 4) return (i >> 1) * row_stride + ((i & 1u) << 1);
    return (i >> 2) * row_stride + ((i & 2u) << 2) + ((i & 1u) << 1);
}
template <int TF, int LAYOUT>
__device__ __forceinline__ unsigned uam_tex_col(unsigned j) {
    if (LAYOUT == 0) return j;
    if (TF == 4) return 2u * j - (j & 1u);                  // (j>>2)*8 + ((j>>1)&1)*4 + (j&1)
    return ((j >> 2) << 4) + ((j & 2u) << 1) + (j & 1u);
}

// Quad-texel address of cell (i, j): uam_tex_row<4, LAYOUT>(i, rs) + uam_tex_col<4, LAYOUT>(j), the same 32-bit value.  Tiled:
// 2i = 4 (i >> 1) + 2 (i & 1), so (i >> 1) rs + 2 (i & 1) + 2j - (j & 1) = (i >> 1)(rs - 4) + 2 (i + j) - (j & 1), which the
// compiler issues in 6 instructions (shift, and, add, shift-add, multiply-add, wide multiply-add) instead of 8.
template <int LAYOUT>
__device__ __forceinline__ unsigned uam_quad_index(unsigned i, unsigned j, unsigned rs) {
    if (LAYOUT == 0) return i * rs + j;
    return (i >> 1) * (rs - 4u) + ((i + j) << 1) - (j & 1u);
}

__device__ __forceinline__ double uam_norm2r(double dx, double dy) {
    return sqrt(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)));
}

__device__ __forceinline__ float uam_lerp2(float t00, float t01, float t10, float t11, float fx, float fy) {
    const float top = t00 + fx * (t01 - t00);
    const float bot = t10 + fx * (t11 - t10);
    return top + fy * (bot - top);
}

// exact (double)n for any int n without the conversion unit: 2^52 + 2^31 + n assembled as bits, minus the bias
__device__ __forceinline__ double uam_int2double(int n) {
    return __dsub_rn(__hiloint2double(0x43300000, n ^ (int)0x80000000), 4503601774854144.0);
}

// fp64 -> fp32 with clamping to [0, 1] in one conversion
__device__ __forceinline__ float uam_sat_f32(double x) {
    float r;
    asm("cvt.rn.sat.f32.f64 %0, %1;" : "=f"(r) : "d"(x));
    return r;
}

// Cell + fp32 fraction of a pixel coordinate.  Same result as the oracle's clamp(u, 0, n-1); j0 = min(floor(u),
// n-2); f = float32(u - j0): for u < 0 the cell clamps to 0 and the saturating conversion gives f = 0, for
// u > n-1 the cell clamps to n-2 and f saturates to 1.
__device__ __forceinline__ void uam_cell_frac1(double u, int n, int& j0, float& f) {
    j0 = min(max(__double2int_rd(u), 0), n - 2);
    f = uam_sat_f32(__dsub_rn(u, uam_int2double(j0)));
}
// the same for 0 <= u < n - 1 (caller's promise): neither clamp nor saturation can act, same bits.  floor(u) comes from
// one round-down add: u + 2^52 rounded towards -inf is 2^52 + floor(u) (the spacing of doubles in [2^52, 2^53) is 1), whose
// low word IS the integer -- no conversion instruction, no bit assembly of (double)j0.
__device__ __forceinline__ void uam_cell_frac1_inside(double u, int& j0, float& f) {
    const double fu = __dadd_rd(u, 4503599627370496.0);
    j0 = __double2loint(fu);
    f = (float)__dsub_rn(u, __dsub_rn(fu, 4503599627370496.0));
}

// A bilinear tap split into its load half and its arithmetic half, so that a loop can issue the loads of several
// samples before it consumes the first one.
template <int TF>
struct UamTap {
    typename UamTexel<TF>::T a, b, c, d;   // (i0,j0) (i0,j0+1) (i0+1,j0) (i0+1,j0+1)
    float fx, fy;
};
// quad mode: one 16-byte texel holds the four corner values of cell (i0, j0); occupancy of the nearest cell is one bit
template <>
struct UamTap<1> {
    float4 q;              // value at (i0,j0) (i0,j0+1) (i0+1,j0) (i0+1,j0+1)
    unsigned ow, ob;       // occupancy word and bit index of the nearest cell
    float fx, fy;
};

// sign-packed quads: every corner value is >= 0 and carries its own cell's occupancy flag in the sign bit
template <>
struct UamTap<8> {
    float4 q;
    float fx, fy;
};

template <int TF, int LAYOUT, bool CLAMP = true>
__device__ __forceinline__ void uam_tap_load(const typename UamTexel<TF>::T* __restrict__ tex, const UamRasterParams& rp,
                                             double u, double v, UamTap<TF>& t) {
    int i0, j0;
    if constexpr (CLAMP) {
        uam_cell_frac1(u, rp.W, j0, t.fx);
        uam_cell_frac1(v, rp.H, i0, t.fy);
    } else {
        uam_cell_frac1_inside(u, j0, t.fx);
        uam_cell_frac1_inside(v, i0, t.fy);
    }
    if constexpr (TF == 8) {
        t.q = __ldg(tex + uam_quad_index<LAYOUT>(i0, j0, rp.row_stride));
    } else if constexpr (TF == 1) {
        t.q = __ldg(tex + uam_quad_index<LAYOUT>(i0, j0, rp.row_stride));
        const unsigned ni = (unsigned)i0 + (t.fy >= 0.5f ? 1u : 0u), nj = (unsigned)j0 + (t.fx >= 0.5f ? 1u : 0u);
        t.ow = __ldg(rp.occ_bits + uam_occ_word(ni, nj, rp.occ_blocks_x));
        t.ob = uam_occ_bit(ni, nj);
    } else {
        const unsigned r0 = uam_tex_row<TF, LAYOUT>(i0, rp.row_stride), r1 = uam_tex_row<TF, LAYOUT>(i0 + 1, rp.row_stride);
        const unsigned c0 = uam_tex_col<TF, LAYOUT>(j0), c1 = uam_tex_col<TF, LAYOUT>(j0 + 1);
        t.a = __ldg(tex + (r0 + c0));
        t.b = __ldg(tex + (r0 + c1));
        t.c = __ldg(tex + (r1 + c0));
        t.d = __ldg(tex + (r1 + c1));
    }
}

template <int TF>
__device__ __forceinline__ void uam_tap_eval(const UamRasterParams& rp, const UamTap<TF>& t, float& pen, bool& occ) {
    if constexpr (TF == 8) {
        pen = rp.w0 * uam_lerp2(fabsf(t.q.x), fabsf(t.q.y), fabsf(t.q.z), fabsf(t.q.w), t.fx, t.fy);
        const bool right = t.fx >= 0.5f, down = t.fy >= 0.5f;
        const float o = down ? (right ? t.q.w : t.q.z) : (right ? t.q.y : t.q.x);
        occ = __float_as_int(o) < 0;
    } else if constexpr (TF == 1) {
        pen = rp.w0 * uam_lerp2(t.q.x, t.q.y, t.q.z, t.q.w, t.fx, t.fy);
        occ = ((t.ow >> t.ob) & 1u) != 0u;
    } else {
        const bool right = t.fx >= 0.5f, down = t.fy >= 0.5f;
        if constexpr (TF == 2) {
            pen = rp.w0 * uam_lerp2(t.a.x, t.b.x, t.c.x, t.d.x, t.fx, t.fy);
            const float o = down ? (right ? t.d.y : t.c.y) : (right ? t.b.y : t.a.y);
            occ = o != 0.0f;
        } else {
            pen = rp.w0 * uam_lerp2(t.a.x, t.b.x, t.c.x, t.d.x, t.fx, t.fy) + rp.w1 * uam_lerp2(t.a.y, t.b.y, t.c.y, t.d.y, t.fx, t.fy) +
                  rp.w2 * uam_lerp2(t.a.z, t.b.z, t.c.z, t.d.z, t.fx, t.fy);
            const float o = down ? (right ? t.d.w : t.c.w) : (right ? t.b.w : t.a.w);
            occ = o != 0.0f;
        }
    }
}

// Slopes of one layer's bilinear interpolant on the sampled cell, at the fp32 fractions of the tap.
__device__ __forceinline__ void uam_lerp2_grad(float t00, float t01, float t10, float t11, float fx, float fy, float& du, float& dv) {
    du = (1.0f - fy) * (t01 - t00) + fy * (t11 - t10);
    dv = (1.0f - fx) * (t10 - t00) + fx * (t11 - t01);
}

// uam_tap_eval (same pen / occ bits) + the slopes dP/du, dP/dv of the weighted penalty on the sampled cell.  The caller
// zeroes a slope whose clamp is active (the clamped coordinate does not move with the waypoint).
template <int TF>
__device__ __forceinline__ void uam_tap_grad(const UamRasterParams& rp, const UamTap<TF>& t, float& pen, bool& occ, float& du, float& dv) {
    uam_tap_eval<TF>(rp, t, pen, occ);
    if constexpr (TF == 8) {
        uam_lerp2_grad(fabsf(t.q.x), fabsf(t.q.y), fabsf(t.q.z), fabsf(t.q.w), t.fx, t.fy, du, dv);
        du *= rp.w0; dv *= rp.w0;
    } else if constexpr (TF == 1) {
        uam_lerp2_grad(t.q.x, t.q.y, t.q.z, t.q.w, t.fx, t.fy, du, dv);
        du *= rp.w0; dv *= rp.w0;
    } else {
        uam_lerp2_grad(t.a.x, t.b.x, t.c.x, t.d.x, t.fx, t.fy, du, dv);
        du *= rp.w0; dv *= rp.w0;
        if constexpr (TF == 4) {
            float u1, v1, u2, v2;
            uam_lerp2_grad(t.a.y, t.b.y, t.c.y, t.d.y, t.fx, t.fy, u1, v1);
            uam_lerp2_grad(t.a.z, t.b.z, t.c.z, t.d.z, t.fx, t.fy, u2, v2);
            du += rp.w1 * u1 + rp.w2 * u2;
            dv += rp.w1 * v1 + rp.w2 * v2;
        }
    }
}

// true where the clamp of a pixel coordinate to [0, n-1] is inactive (the sample moves with its waypoint)
__device__ __forceinline__ bool uam_free_coord(double u, int n) { return u >= 0.0 && u <= (double)(n - 1); }

// Lane-pair form: the two lanes of a pair work on the SAME sample; lane `side` (0 = left, 1 = right) fetches the
// texel column j0 + side (rows i0 and i0 + 1), lerps it in y, and the pair exchanges the column results with one
// shuffle per layer.  Must be called by all 32 lanes (shuffles); `active` masks lanes past the end.
template <int TF, int LAYOUT>
__device__ __forceinline__ void uam_sample_pair(const typename UamTexel<TF>::T* __restrict__ tex,
                                                const UamRasterParams& rp, double u, double v, int side, bool active,
                                                float& pen, bool& occ) {
    float fx = 0.0f, fy = 0.0f;
    float c0 = 0.0f, c1 = 0.0f, c2 = 0.0f, o = 0.0f;
    if (active) {
        int i0, j0;
        uam_cell_frac1(u, rp.W, j0, fx);
        uam_cell_frac1(v, rp.H, i0, fy);
        const bool down = fy >= 0.5f;
        const unsigned r0 = uam_tex_row<TF, LAYOUT>(i0, rp.row_stride), r1 = uam_tex_row<TF, LAYOUT>(i0 + 1, rp.row_stride);
        const unsigned cc = uam_tex_col<TF, LAYOUT>(j0 + side);
        if constexpr (TF == 2) {
            const float2* t2 = reinterpret_cast<const float2*>(tex);
            const float2 a = __ldg(t2 + r0 + cc), b = __ldg(t2 + r1 + cc);
            c0 = a.x + fy * (b.x - a.x);
            o = down ? b.y : a.y;
        } else {
            const float4* t4 = reinterpret_cast<const float4*>(tex);
            const float4 a = __ldg(t4 + r0 + cc), b = __ldg(t4 + r1 + cc);
            c0 = a.x + fy * (b.x - a.x);
            c1 = a.y + fy * (b.y - a.y);
            c2 = a.z + fy * (b.z - a.z);
            o = down ? b.w : a.w;
        }
    }
    const float p0 = __shfl_xor_sync(0xffffffffu, c0, 1);
    // after the exchange: (left, right) = side ? (p, c) : (c, p)
    float val = rp.w0 * (side ? p0 + fx * (c0 - p0) : c0 + fx * (p0 - c0));
    if constexpr (TF == 4) {
        const float p1 = __shfl_xor_sync(0xffffffffu, c1, 1);
        const float p2 = __shfl_xor_sync(0xffffffffu, c2, 1);
        val += rp.w1 * (side ? p1 + fx * (c1 - p1) : c1 + fx * (p1 - c1));
        val += rp.w2 * (side ? p2 + fx * (c2 - p2) : c2 + fx * (p2 - c2));
    }
    pen = val;
    // nearest cell column = j0 + (fx >= 0.5): only the lane holding that column reports occupancy
    occ = active && ((fx >= 0.5f) == (side != 0)) && (o != 0.0f);
}

// ---- shared pieces of the path kernels -----------------------------------------------------------------------
// length term of one waypoint j (reference quirk: segments 0..N-1 only + |z_0 - map.x_start|)
__device__ __forceinline__ double uam_len_term(const double2* __restrict__ zp, int j, int N, const double2 p,
                                               const UamRasterParams& rp) {
    const bool len_smooth = (rp.flags & UAM_LENGTH_SMOOTH) != 0;
    double acc = 0.0;
    if (j < N) {
        const double2 q = zp[j + 1];
        const double d = uam_norm2r(__dsub_rn(q.x, p.x), __dsub_rn(q.y, p.y));
        acc += len_smooth ? __dmul_rn(d, d) : d;
    }
    if (j == 0 && !(rp.flags & UAM_OWN_START)) {
        const double d = uam_norm2r(__dsub_rn(p.x, rp.ms_x), __dsub_rn(p.y, rp.ms_y));
        acc += len_smooth ? __dmul_rn(d, d) : d;
    }
    return acc;
}

// d(length term)/d z_j in fp64, the expressions of uam_k_grad_analytic: pairs (m_s, z_0) (unless UAM_OWN_START),
// (z_0, z_1), ..., (z_{N-1}, z_N); 2 d with UAM_LENGTH_SMOOTH, else d / |d| (zero subgradient at |d| = 0)
__device__ __forceinline__ double2 uam_len_grad(const double2* __restrict__ zp, int j, int N, const double2 p,
                                                const UamRasterParams& rp) {
    const bool len_smooth = (rp.flags & UAM_LENGTH_SMOOTH) != 0;
    double Lx = 0.0, Ly = 0.0;
    if (j <= N) {
        if (j >= 1 || !(rp.flags & UAM_OWN_START)) {
            const double2 a = j >= 1 ? zp[j - 1] : make_double2(rp.ms_x, rp.ms_y);
            const double dx = p.x - a.x, dy = p.y - a.y;
            if (len_smooth) { Lx += 2.0 * dx; Ly += 2.0 * dy; }
            else { const double n = sqrt(dx * dx + dy * dy); if (n > 0.0) { Lx += dx / n; Ly += dy / n; } }
        }
        if (j <= N - 1) {
            const double2 q = zp[j + 1];
            const double dx = q.x - p.x, dy = q.y - p.y;
            if (len_smooth) { Lx -= 2.0 * dx; Ly -= 2.0 * dy; }
            else { const double n = sqrt(dx * dx + dy * dy); if (n > 0.0) { Lx -= dx / n; Ly -= dy / n; } }
        }
    }
    return make_double2(Lx, Ly);
}

// Per-segment gradient sums -> the segment's share of its two waypoints' penalty gradient (pixel units, fp32).
// In: su = {sum dP/du, sum s dP/du, sum dP/dv, sum s dP/dv} over the segment's samples s = 0..S-1, is = 1/S.  Sample s
// sits at (1 - s/S) z_k + (s/S) z_{k+1} and carries weight 1/S: out = {z_k: du, dv, z_{k+1}: du, dv}.
__device__ __forceinline__ float4 uam_seg_grad(float4 su, float is) {
    return make_float4(is * (su.x - is * su.y), is * (su.z - is * su.w), is * (is * su.y), is * (is * su.w));
}

// Gradient of waypoint j: (N+1) d(length)/dz_j + (1/N) dP/dz_j, with (pu, pv) the penalty part in pixel units
__device__ __forceinline__ double2 uam_grad_point(double2 lg, float pu, float pv, int N, const UamRasterParams& rp) {
    const double dN1 = (double)(N + 1), dN = (double)N;
    return make_double2(dN1 * lg.x + (double)pu / rp.dx / dN, dN1 * lg.y + (double)pv / rp.dy / dN);
}

// sample count of a segment with pixel-space extent (dU, dV)
__device__ __forceinline__ double uam_seg_samples(double dU, double dV, double spc) {
    double Sd = fmax(1.0, ceil(__dmul_rn(uam_norm2r(dU, dV), spc)));
    if (!(Sd <= UAM_MAX_SAMPLES_PER_SEGMENT)) Sd = UAM_MAX_SAMPLES_PER_SEGMENT;
    return Sd;
}

// Per-warp segment table in shared memory, walked by the flat sample loop.
struct UamSegTable {
    double* U;
    double* V;
    double* SU;
    double* SV;
    int* P;          // exclusive prefix of the sample counts, n + 1 entries
    float* IS;       // 1 / S_k
};
__host__ __device__ inline size_t uam_seg_table_bytes(int n) {
    size_t b = (size_t)n * 8 * 4 + (size_t)(n + 1) * 4 + (size_t)n * 4;
    return (b + 15) & ~(size_t)15;
}
__device__ __forceinline__ UamSegTable uam_seg_table(unsigned char* base, int n) {
    UamSegTable t;
    t.U = reinterpret_cast<double*>(base);
    t.V = t.U + n;
    t.SU = t.V + n;
    t.SV = t.SU + n;
    t.P = reinterpret_cast<int*>(t.SV + n);
    t.IS = reinterpret_cast<float*>(t.P + n + 1);
    return t;
}

// ---- waypoint mode ----------------------------------------------------------------------------------------
// GRAD: also the gradient (uam_grad_paths_raster): every waypoint is its own segment's only sample (weight 1), so
// waypoint j's gradient is its own tap's slopes + its length part, written by the lane that holds it.
template <int TF, int LAYOUT, bool GRAD = false>
__global__ void __launch_bounds__(UAM_CTA_THREADS)
uam_k_score_raster_wp(const double2* __restrict__ z, long long B, int Wp, UamRasterParams rp,
                      const typename UamTexel<TF>::T* __restrict__ tex, float* __restrict__ cost,
                      uint8_t* __restrict__ collide, long long* __restrict__ nsamp, double2* __restrict__ grad) {
    const int lane = threadIdx.x & 31;
    const long long warp0 = (long long)blockIdx.x * UAM_WARPS_PER_CTA + (threadIdx.x >> 5);
    const long long nwarps = (long long)gridDim.x * UAM_WARPS_PER_CTA;
    const int N = Wp - 2;
    for (long long path = warp0; path < B; path += nwarps) {
        const double2* zp = z + path * Wp;
        float pen_sum = 0.0f;
        double len_sum = 0.0;
        bool col = false;
        // two waypoints per lane per trip: 8 texel gathers in flight before the first lerp (DRAM-latency bound)
        for (int j = lane; j < Wp; j += 64) {
            const int j2 = j + 32;
            const bool two = j2 < Wp;
            const double2 p = zp[j];
            const double2 q = zp[two ? j2 : j];
            UamTap<TF> ta, tb;
            uam_tap_load<TF, LAYOUT>(tex, rp, uam_pix(p.x, rp.x0, rp.dx), uam_pix(p.y, rp.y0, rp.dy), ta);
            uam_tap_load<TF, LAYOUT>(tex, rp, uam_pix(q.x, rp.x0, rp.dx), uam_pix(q.y, rp.y0, rp.dy), tb);
            len_sum += uam_len_term(zp, j, N, p, rp);
            if (two) len_sum += uam_len_term(zp, j2, N, q, rp);
            float pen;
            bool occ;
            if constexpr (GRAD) {
                float du, dv;
                uam_tap_grad<TF>(rp, ta, pen, occ, du, dv);
                pen_sum += pen;
                col = col || occ;
                const double pu = uam_pix(p.x, rp.x0, rp.dx), pv = uam_pix(p.y, rp.y0, rp.dy);
                grad[path * Wp + j] = uam_grad_point(uam_len_grad(zp, j, N, p, rp), uam_free_coord(pu, rp.W) ? du : 0.0f,
                                                     uam_free_coord(pv, rp.H) ? dv : 0.0f, N, rp);
                uam_tap_grad<TF>(rp, tb, pen, occ, du, dv);
                if (two) {
                    pen_sum += pen;
                    col = col || occ;
                    const double qu = uam_pix(q.x, rp.x0, rp.dx), qv = uam_pix(q.y, rp.y0, rp.dy);
                    grad[path * Wp + j2] = uam_grad_point(uam_len_grad(zp, j2, N, q, rp), uam_free_coord(qu, rp.W) ? du : 0.0f,
                                                          uam_free_coord(qv, rp.H) ? dv : 0.0f, N, rp);
                }
            } else {
                uam_tap_eval<TF>(rp, ta, pen, occ);
                pen_sum += pen;
                col = col || occ;
                uam_tap_eval<TF>(rp, tb, pen, occ);
                if (two) {
                    pen_sum += pen;
                    col = col || occ;
                }
            }
        }
        pen_sum = uam_warp_sum(pen_sum);
        len_sum = uam_warp_sum(len_sum);
        col = __any_sync(0xffffffffu, col);
        if (lane == 0) {
            if (cost) cost[path] = (float)((double)(N + 1) * len_sum + (double)pen_sum / (double)N);
            if (collide) collide[path] = col ? 1 : 0;
            if (nsamp) nsamp[path] = Wp;
        }
    }
}

// ---- integral mode, warp per path (variants 0 and 1) --------------------------------------------------------------
// The path's samples are flattened (segment k owns flat indices [P_k, P_{k+1})), lanes stride the flat index, so 32
// consecutive samples of one polyline -- a compact footprint in the raster -- are fetched together and no lane
// idles on short segments.  Total samples per path are capped at 2^31 - 1 by the host-side S_k cap.
// GRAD (PAIR = 0 only): also the gradient.  One sample per lane per trip and all lanes run every trip; per window of 32
// consecutive samples the lanes of each segment's run combine their {dP/du, s dP/du, dP/dv, s dP/dv} with a segmented
// shuffle sum keyed by the segment, and the run's last lane adds the result to the segment's sums in shared memory (one
// writer per segment and window, windows in order: the bits depend on the path alone).  The per-lane penalty sums see
// the same samples in the same order as the scorer's two-per-trip loop, so cost and collide are the scorer's bits.
template <int TF, int LAYOUT, int PAIR, bool GRAD = false>
__global__ void __launch_bounds__(UAM_CTA_THREADS)
uam_k_score_raster_int(const double2* __restrict__ z, long long B, int Wp, UamRasterParams rp,
                       const typename UamTexel<TF>::T* __restrict__ tex, float* __restrict__ cost,
                       uint8_t* __restrict__ collide, long long* __restrict__ nsamp, double2* __restrict__ grad) {
    extern __shared__ __align__(128) unsigned char uam_smem[];
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int wpc = blockDim.x >> 5;
    unsigned char* const wbase = uam_smem + (size_t)warp * (uam_seg_table_bytes(Wp) + (GRAD ? (size_t)Wp * sizeof(float4) : 0));
    const UamSegTable tb = uam_seg_table(wbase, Wp);
    float4* const gs = reinterpret_cast<float4*>(wbase + uam_seg_table_bytes(Wp));     // GRAD: per-segment sums
    const long long warp0 = (long long)blockIdx.x * wpc + warp;
    const long long nwarps = (long long)gridDim.x * wpc;
    const int N = Wp - 2;

    for (long long path = warp0; path < B; path += nwarps) {
        const double2* zp = z + path * Wp;
        double len_sum = 0.0;
        // A: pixel coordinates of the waypoints
        for (int j = lane; j < Wp; j += 32) {
            const double2 p = zp[j];
            tb.U[j] = uam_pix(p.x, rp.x0, rp.dx);
            tb.V[j] = uam_pix(p.y, rp.y0, rp.dy);
            len_sum += uam_len_term(zp, j, N, p, rp);
        }
        __syncwarp();
        // B: per-segment sample count, step and exclusive prefix; pseudo-segment Wp-1 = the goal waypoint
        int carry = 0;
        for (int b0 = 0; b0 < Wp; b0 += 32) {
            const int k = b0 + lane;
            int S = 0;
            if (k < Wp - 1) {
                const double dU = __dsub_rn(tb.U[k + 1], tb.U[k]), dV = __dsub_rn(tb.V[k + 1], tb.V[k]);
                const double Sd = uam_seg_samples(dU, dV, rp.spc);
                S = (int)Sd;
                tb.SU[k] = __ddiv_rn(dU, Sd);
                tb.SV[k] = __ddiv_rn(dV, Sd);
                tb.IS[k] = (float)(1.0 / Sd);
            } else if (k == Wp - 1) {
                S = 1;
                tb.SU[k] = 0.0;
                tb.SV[k] = 0.0;
                tb.IS[k] = 1.0f;
            }
            int incl = S;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int t = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += t;
            }
            if (k < Wp) tb.P[k] = carry + incl - S;
            carry += __shfl_sync(0xffffffffu, incl, 31);
        }
        if (lane == 0) tb.P[Wp] = carry;
        __syncwarp();
        // C: flat sample loop
        const int T = carry;
        float acc = 0.0f;
        bool col = false;
        int k = 0, p1 = tb.P[1];
        double kU = tb.U[0], kV = tb.V[0], kSU = tb.SU[0], kSV = tb.SV[0];
        float kIS = tb.IS[0];
        if constexpr (GRAD) {
            for (int j = lane; j < Wp; j += 32) gs[j] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
            __syncwarp();
            double sd = (double)lane;
            for (int t0 = 0; t0 < T; t0 += 32) {
                const int t = t0 + lane;
                float4 g = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
                int kk = Wp;                      // lanes past the end: a key no segment has
                if (t < T) {
                    if (t >= p1) {
                        do { ++k; p1 = tb.P[k + 1]; } while (t >= p1);
                        sd = (double)(t - tb.P[k]);
                        kU = tb.U[k]; kV = tb.V[k]; kSU = tb.SU[k]; kSV = tb.SV[k]; kIS = tb.IS[k];
                    }
                    const double u = __dadd_rn(kU, __dmul_rn(sd, kSU));
                    const double v = __dadd_rn(kV, __dmul_rn(sd, kSV));
                    const float s = (float)sd;
                    sd += 32.0;
                    UamTap<TF> a;
                    uam_tap_load<TF, LAYOUT>(tex, rp, u, v, a);
                    float pen, du, dv;
                    bool occ;
                    uam_tap_grad<TF>(rp, a, pen, occ, du, dv);
                    acc += pen * kIS;
                    col = col || occ;
                    if (!uam_free_coord(u, rp.W)) du = 0.0f;
                    if (!uam_free_coord(v, rp.H)) dv = 0.0f;
                    g = make_float4(du, s * du, dv, s * dv);
                    kk = k;
                }
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const int ko = __shfl_up_sync(0xffffffffu, kk, o);
                    const float x = __shfl_up_sync(0xffffffffu, g.x, o), y = __shfl_up_sync(0xffffffffu, g.y, o);
                    const float zz = __shfl_up_sync(0xffffffffu, g.z, o), w = __shfl_up_sync(0xffffffffu, g.w, o);
                    if (lane >= o && ko == kk) { g.x += x; g.y += y; g.z += zz; g.w += w; }
                }
                const int kn = __shfl_down_sync(0xffffffffu, kk, 1);
                if (kk < Wp && (lane == 31 || kn != kk)) {
                    float4 c = gs[kk];
                    c.x += g.x; c.y += g.y; c.z += g.z; c.w += g.w;
                    gs[kk] = c;
                }
                __syncwarp();
            }
            for (int j = lane; j < Wp; j += 32) {
                const float4 a = uam_seg_grad(gs[j], tb.IS[j]);
                float pu = a.x, pv = a.y;
                if (j >= 1) {
                    const float4 b = uam_seg_grad(gs[j - 1], tb.IS[j - 1]);
                    pu += b.z;
                    pv += b.w;
                }
                grad[path * Wp + j] = uam_grad_point(uam_len_grad(zp, j, N, zp[j], rp), pu, pv, N, rp);
            }
        } else if (PAIR) {
            const int side = lane & 1;
            double sd = (double)(lane >> 1);
            for (int tb0 = 0; tb0 < T; tb0 += 16) {
                const int t = tb0 + (lane >> 1);
                const bool active = t < T;
                double u = 0.0, v = 0.0;
                if (active) {
                    if (t >= p1) {
                        do { ++k; p1 = tb.P[k + 1]; } while (t >= p1);
                        sd = (double)(t - tb.P[k]);
                        kU = tb.U[k]; kV = tb.V[k]; kSU = tb.SU[k]; kSV = tb.SV[k]; kIS = tb.IS[k];
                    }
                    u = __dadd_rn(kU, __dmul_rn(sd, kSU));
                    v = __dadd_rn(kV, __dmul_rn(sd, kSV));
                    sd += 16.0;
                }
                float pen;
                bool occ;
                uam_sample_pair<TF, LAYOUT>(tex, rp, u, v, side, active, pen, occ);
                if (active && side == 0) acc += pen * kIS;
                col = col || occ;
            }
        } else {
            // two samples per lane per trip (t and t + 32): all 8 texel loads are issued before the first lerp, which
            // doubles the bytes each warp keeps in flight (the kernel is DRAM-latency bound on scattered paths)
            double sd = (double)lane;
            for (int t = lane; t < T; t += 64) {
                if (t >= p1) {
                    do { ++k; p1 = tb.P[k + 1]; } while (t >= p1);
                    sd = (double)(t - tb.P[k]);
                    kU = tb.U[k]; kV = tb.V[k]; kSU = tb.SU[k]; kSV = tb.SV[k]; kIS = tb.IS[k];
                }
                const double u0 = __dadd_rn(kU, __dmul_rn(sd, kSU));
                const double v0 = __dadd_rn(kV, __dmul_rn(sd, kSV));
                const float is0 = kIS;
                sd += 32.0;
                const int t2 = t + 32;
                const bool two = t2 < T;
                double u1 = u0, v1 = v0;
                if (two) {
                    if (t2 >= p1) {
                        do { ++k; p1 = tb.P[k + 1]; } while (t2 >= p1);
                        sd = (double)(t2 - tb.P[k]);
                        kU = tb.U[k]; kV = tb.V[k]; kSU = tb.SU[k]; kSV = tb.SV[k]; kIS = tb.IS[k];
                    }
                    u1 = __dadd_rn(kU, __dmul_rn(sd, kSU));
                    v1 = __dadd_rn(kV, __dmul_rn(sd, kSV));
                    sd += 32.0;
                }
                UamTap<TF> a, b;
                uam_tap_load<TF, LAYOUT>(tex, rp, u0, v0, a);
                uam_tap_load<TF, LAYOUT>(tex, rp, u1, v1, b);
                float pen;
                bool occ;
                uam_tap_eval<TF>(rp, a, pen, occ);
                acc += pen * is0;
                col = col || occ;
                uam_tap_eval<TF>(rp, b, pen, occ);
                if (two) {
                    acc += pen * kIS;
                    col = col || occ;
                }
            }
        }
        acc = uam_warp_sum(acc);
        len_sum = uam_warp_sum(len_sum);
        col = __any_sync(0xffffffffu, col);
        if (lane == 0) {
            if (cost) cost[path] = (float)((double)(N + 1) * len_sum + (double)acc / (double)N);
            if (collide) collide[path] = col ? 1 : 0;
            if (nsamp) nsamp[path] = T;
        }
        __syncwarp();
    }
}

// ---- integral mode, binned (variant 2) -------------------------------------------------------------------------
// With candidates scattered over a raster much larger than L2 every path drags its own corridor of texels through
// DRAM and every texel is fetched many times per batch by different paths.  The binned pipeline reorders the WORK
// instead of the data: the batch's segments (one unit = one polyline segment, plus one pseudo-segment for the goal
// waypoint) are counting-sorted by the raster bin (64 x 64 cells or larger, Morton order) of their midpoint; the
// sort writes a 48-byte record per segment at its sorted position; a warp then scores 32 consecutive records with
// the flat sample loop (per-segment partial sums in shared memory), and a last warp-per-path kernel adds the
// per-segment partials in a fixed order.
//   uam_k_bin_hist -> uam_k_bin_scan -> uam_k_bin_scatter -> uam_k_score_groups -> uam_k_reduce_paths
struct UamBinGeo {
    int shift;        // bin side = 1 << shift cells
    int nbins;        // Morton id space (power of 4)
    float hx, ox, hy, oy;   // float32 pixel coordinate of a segment's midpoint: u = (p.x + q.x) * hx + ox (ordering only)
};

struct __align__(16) UamSegRec {
    double U, V, SU, SV;   // first sample (pixel coordinates) and per-sample step
    int S;                 // samples
    float IS;              // 1 / S
    unsigned id;           // b * Wp + k
    unsigned pad;
};

__device__ __forceinline__ unsigned uam_part1by1(unsigned x) {
    x &= 0x0000ffffu;
    x = (x | (x << 8)) & 0x00ff00ffu;
    x = (x | (x << 4)) & 0x0f0f0f0fu;
    x = (x | (x << 2)) & 0x33333333u;
    x = (x | (x << 1)) & 0x55555555u;
    return x;
}

// segment id = b * Wp + k; k < Wp-1: segment z_k -> z_{k+1}; k == Wp-1: the goal waypoint alone
__device__ __forceinline__ UamSegRec uam_make_segment(const double2* __restrict__ z, unsigned long long id, int Wp,
                                                      const UamRasterParams& rp) {
    const unsigned long long b = id / (unsigned)Wp;
    const int k = (int)(id - b * (unsigned)Wp);
    const double2 p = z[b * Wp + k];
    UamSegRec r;
    r.U = uam_pix(p.x, rp.x0, rp.dx);
    r.V = uam_pix(p.y, rp.y0, rp.dy);
    r.SU = 0.0; r.SV = 0.0; r.S = 1; r.IS = 1.0f;
    r.id = (unsigned)id;
    r.pad = 0;
    if (k < Wp - 1) {
        const double2 q = z[b * Wp + k + 1];
        const double dU = __dsub_rn(uam_pix(q.x, rp.x0, rp.dx), r.U), dV = __dsub_rn(uam_pix(q.y, rp.y0, rp.dy), r.V);
        const double Sd = uam_seg_samples(dU, dV, rp.spc);
        r.S = (int)Sd;
        r.SU = __ddiv_rn(dU, Sd);
        r.SV = __ddiv_rn(dV, Sd);
        r.IS = (float)(1.0 / Sd);
    }
    return r;
}

// The raster bin of a segment (uam_k_bin_hist) is the Morton id of the bin that holds its midpoint (the goal waypoint for the
// pseudo-segment k = Wp - 1), clamped into the raster (NaN -> 0).  The bin only decides the ORDER the segments are scored in
// (locality), never a result, so it is computed with two multiplications per coordinate -- no sample count, no divisions.
#define UAM_BIN_CHUNK 8192     // segments per CTA in the histogram / scatter kernels (rounded down to whole paths)

// One pass over the waypoints: bin id of every segment + per-CTA histogram, and -- the waypoints being in registers anyway --
// the path's length term (same lane assignment and shuffle tree as uam_k_reduce_paths used to run, same bits), so the last
// kernel of the step no longer re-reads the 1 KiB of waypoints per path.  A CTA owns `ppc` consecutive paths, a warp one path
// at a time, lanes stride its waypoints: path and waypoint index are loop counters (the id -> (path, k) form of this kernel
// spent its time in a 64-bit division per segment: ncu r02, issue-bound at 78 %).
template <int PT>
__global__ void __launch_bounds__(1024)
uam_k_bin_hist(const double2* __restrict__ z, long long B, int Wp, int ppc, UamRasterParams rp, UamBinGeo bg,
               unsigned short* __restrict__ seg_bin, unsigned* __restrict__ hist, double* __restrict__ len_path) {
    extern __shared__ int s_hist[];
    for (int i = threadIdx.x; i < bg.nbins; i += blockDim.x) s_hist[i] = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long p0 = (long long)blockIdx.x * ppc;
    const long long p1 = p0 + ppc < B ? p0 + ppc : B;
    // bin coordinate in float32 (ordering only): u = (mid_x - x0) / dx - 0.5 with mid_x = (p.x + q.x) / 2
    const float hx = bg.hx, hy = bg.hy, ox = bg.ox, oy = bg.oy;
    const float wl = (float)(rp.W - 1), hl = (float)(rp.H - 1);
    const int N = Wp - 2;
    const bool len_smooth = (rp.flags & UAM_LENGTH_SMOOTH) != 0;
    const bool map_start = !(rp.flags & UAM_OWN_START);
    // a warp works on PT paths at a time: 2 x PT 16-byte loads in flight per lane, PT interleaved shuffle trees
    for (long long pb = p0 + (long long)warp * PT; pb < p1; pb += 32 * PT) {
        const double2* zb = z + pb * Wp;
        const int np = (int)(p1 - pb < PT ? p1 - pb : PT);
        // the term |z_0 - map start| of uam_len_term (added to waypoint 0's own term): lane t computes path t's
        double d_start = 0.0;
        if (map_start && lane < np) {
            const double2 p = zb[(size_t)lane * Wp];
            const double d = uam_norm2r(__dsub_rn(p.x, rp.ms_x), __dsub_rn(p.y, rp.ms_y));
            d_start = len_smooth ? __dmul_rn(d, d) : d;
        }
        double len_sum[PT], ds[PT];
#pragma unroll
        for (int t = 0; t < PT; ++t) {
            len_sum[t] = 0.0;
            ds[t] = __shfl_sync(0xffffffffu, d_start, t);
        }
        for (int j0 = 0; j0 < Wp; j0 += 32) {
            const int j = j0 + lane;
            double2 p[PT], q[PT];
            bool ok[PT];
#pragma unroll
            for (int t = 0; t < PT; ++t) {
                ok[t] = j < Wp && t < np;
                const double2* zp = zb + (size_t)t * Wp;
                p[t] = ok[t] ? zp[j] : make_double2(0.0, 0.0);
                q[t] = (ok[t] && j < Wp - 1) ? zp[j + 1] : p[t];
            }
#pragma unroll
            for (int t = 0; t < PT; ++t) {
                if (ok[t]) {
                    const float u = fminf(fmaxf(fmaf((float)(p[t].x + q[t].x), hx, ox), 0.0f), wl);
                    const float v = fminf(fmaxf(fmaf((float)(p[t].y + q[t].y), hy, oy), 0.0f), hl);
                    const int bin = (int)(uam_part1by1((unsigned)((int)u >> bg.shift)) | (uam_part1by1((unsigned)((int)v >> bg.shift)) << 1));
                    seg_bin[(size_t)(pb + t) * Wp + j] = (unsigned short)bin;
                    atomicAdd(&s_hist[bin], 1);
                    // uam_len_term: acc = 0; j < N: acc += d(z_j, z_j+1); j == 0: acc += d(z_0, map start); len_sum += acc
                    double acc = 0.0;
                    if (j < N) {
                        const double d = uam_norm2r(__dsub_rn(q[t].x, p[t].x), __dsub_rn(q[t].y, p[t].y));
                        acc += len_smooth ? __dmul_rn(d, d) : d;
                    }
                    if (j == 0 && map_start) acc += ds[t];
                    len_sum[t] += acc;
                }
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
            for (int t = 0; t < PT; ++t) len_sum[t] += __shfl_xor_sync(0xffffffffu, len_sum[t], o);      // (the tree of uam_warp_sum)
        }
        double mine = len_sum[0];
#pragma unroll
        for (int t = 1; t < PT; ++t) mine = lane == t ? len_sum[t] : mine;
        if (lane < np) len_path[pb + lane] = mine;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < bg.nbins; i += blockDim.x)
        if (s_hist[i]) atomicAdd(&hist[i], (unsigned)s_hist[i]);
}

// exclusive prefix of hist[0..n) into cursor[0..n) (single CTA, 1024 threads)
__global__ void __launch_bounds__(1024)
uam_k_bin_scan(const unsigned* __restrict__ hist, int n, unsigned* __restrict__ cursor) {
    __shared__ unsigned warp_tot[32];
    const int per = (n + 1023) / 1024;
    const int lo = min((int)threadIdx.x * per, n), hi = min(lo + per, n);
    unsigned local = 0;
    for (int i = lo; i < hi; ++i) local += hist[i];
    unsigned incl = local;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) warp_tot[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        unsigned w = warp_tot[lane], wi = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned t = __shfl_up_sync(0xffffffffu, wi, o);
            if (lane >= o) wi += t;
        }
        warp_tot[lane] = wi - w;
    }
    __syncthreads();
    unsigned run = warp_tot[warp] + incl - local;
    for (int i = lo; i < hi; ++i) {
        const unsigned h = hist[i];
        cursor[i] = run;
        run += h;
    }
}

__global__ void __launch_bounds__(1024)
uam_k_bin_scatter(unsigned long long n_seg, unsigned long long chunk, UamBinGeo bg, const unsigned short* __restrict__ seg_bin,
                  unsigned* __restrict__ cursor, unsigned* __restrict__ sorted_id) {
    extern __shared__ int s_hist[];
    for (int i = threadIdx.x; i < bg.nbins; i += blockDim.x) s_hist[i] = 0;
    __syncthreads();
    const unsigned long long lo = (unsigned long long)blockIdx.x * chunk;
    const unsigned long long hi = lo + chunk < n_seg ? lo + chunk : n_seg;
    // up to KEEP ids per thread stay in registers between the counting and the writing pass (one load of the bin ids)
    constexpr int KEEP = 8;
    const bool keep = chunk <= 1024ull * KEEP;
    unsigned short b[KEEP];
    if (keep) {
#pragma unroll
        for (int t = 0; t < KEEP; ++t) {
            const unsigned long long id = lo + threadIdx.x + 1024u * t;
            b[t] = id < hi ? seg_bin[id] : (unsigned short)0;
        }
#pragma unroll
        for (int t = 0; t < KEEP; ++t)
            if (lo + threadIdx.x + 1024u * t < hi) atomicAdd(&s_hist[b[t]], 1);
    } else {
        for (unsigned long long id = lo + threadIdx.x; id < hi; id += blockDim.x) atomicAdd(&s_hist[seg_bin[id]], 1);
    }
    __syncthreads();
    // reserve this CTA's range in every bin it touches; s_hist becomes the CTA's write cursor (4 independent atomics in flight)
    for (int i0 = threadIdx.x; i0 < bg.nbins; i0 += 4 * 1024) {
        int c[4];
        unsigned r[4];
#pragma unroll
        for (int t = 0; t < 4; ++t) c[t] = i0 + 1024 * t < bg.nbins ? s_hist[i0 + 1024 * t] : 0;
#pragma unroll
        for (int t = 0; t < 4; ++t) r[t] = c[t] ? atomicAdd(&cursor[i0 + 1024 * t], (unsigned)c[t]) : 0u;
#pragma unroll
        for (int t = 0; t < 4; ++t)
            if (c[t]) s_hist[i0 + 1024 * t] = (int)r[t];
    }
    __syncthreads();
    // the sorted order holds 4-byte segment ids only; the scoring kernel rebuilds the segment from its two waypoints
    // (one lane per record, once per group) -- 48-byte records cost 0.33 ms of scattered writes per C3 shard
    if (keep) {
#pragma unroll
        for (int t = 0; t < KEEP; ++t) {
            const unsigned long long id = lo + threadIdx.x + 1024u * t;
            if (id < hi) sorted_id[(unsigned)atomicAdd(&s_hist[b[t]], 1)] = (unsigned)id;
        }
    } else {
        for (unsigned long long id = lo + threadIdx.x; id < hi; id += blockDim.x) {
            const unsigned pos = (unsigned)atomicAdd(&s_hist[seg_bin[id]], 1);
            sorted_id[pos] = (unsigned)id;
        }
    }
}

#define UAM_TS 64                         // variant 3: tile side in cells
#define UAM_TSH (UAM_TS + 1)              // with the halo row / column

// A bilinear tap from the staged tile: (i0, j0) are raster cells, (ti0, tj0) the tile's first cell.  The min() is
// for memory safety only (a correct cut never leaves the tile).
template <int TF>
__device__ __forceinline__ void uam_tap_load_tile(const unsigned char* tile, int ti0, int tj0, const UamRasterParams& rp,
                                                  double u, double v, UamTap<TF>& t) {
    typedef typename UamTexel<TF>::T T;
    int i0, j0;
    uam_cell_frac1(u, rp.W, j0, t.fx);
    uam_cell_frac1(v, rp.H, i0, t.fy);
    const unsigned li = min((unsigned)(i0 - ti0), (unsigned)(UAM_TS - 1)), lj = min((unsigned)(j0 - tj0), (unsigned)(UAM_TS - 1));
    const T* p = reinterpret_cast<const T*>(tile) + (li * UAM_TSH + lj);
    if constexpr (TF == 8) {
        t.q = p[0];
    } else if constexpr (TF == 1) {
        t.q = p[0];
        const unsigned ni = (unsigned)i0 + (t.fy >= 0.5f ? 1u : 0u), nj = (unsigned)j0 + (t.fx >= 0.5f ? 1u : 0u);
        t.ow = __ldg(rp.occ_bits + uam_occ_word(ni, nj, rp.occ_blocks_x));
        t.ob = uam_occ_bit(ni, nj);
    } else {
        t.a = p[0];
        t.b = p[1];
        t.c = p[UAM_TSH];
        t.d = p[UAM_TSH + 1];
    }
}

// x << n with PTX semantics (a shift by 32 or more gives 0; in C++ it would be undefined)
__device__ __forceinline__ unsigned uam_shl_clamp(unsigned x, unsigned n) {
    unsigned r;
    asm("shl.b32 %0, %1, %2;" : "=r"(r) : "r"(x), "r"(n));
    return r;
}

// One warp per group of 32 consecutive sorted records.  The samples of the 32 records are concatenated (record k owns
// the flat indices [P_k, P_{k+1})) and lanes stride the flat index, UAM_TAPS windows of 32 samples per trip, so no
// lane idles on short records.  The record of a flat index is found without branches or dependent shared-memory
// walks: lane l holds P_l; per window one REDUX.OR builds the bitmap of the record starts that fall inside it and
// k(lane) = (#records started before the window) + popc(bitmap & lanes <= lane) - 1.  The record's parameters come
// from a 36-byte-per-record table in shared memory (two LDS.128 + one LDS.32); the loads of all UAM_TAPS taps are
// issued before the first lerp.  Per-lane accumulators are flushed to a 32 x 32 matrix of partials (row = lane,
// column swizzled by lane) when the lane moves on to another record; a fixed-order reduction per record follows.
struct __align__(16) UamGroupRec {
    double U, SU, V, SV;
};
// per-warp shared memory of a group: 33 records (32 + the dummy that owns the flat indices past the end) of 32 B, their
// {P, Q} (8 B), the 32 x 33 partials (row stride 33: conflict-free both ways), the window table and its bit words
#define UAM_GROUP_REC_OFF 0
#define UAM_GROUP_PQ_OFF (33 * 32)
#define UAM_GROUP_PART_OFF (33 * 32 + 33 * 8 + 8)             // 1328: 16-byte aligned
#define UAM_GROUP_TAB_OFF (UAM_GROUP_PART_OFF + 32 * 33 * 4)
#define UAM_GROUP_BITS_OFF (UAM_GROUP_TAB_OFF + 32 * 8)
#define UAM_GROUP_SMEM (UAM_GROUP_BITS_OFF + 32 * 4)          // 5936
#define UAM_GROUP_SEG 1024          // flat samples covered by one fill of the window table (32 windows of 32)

template <int TF> struct UamTapsPerTrip { static const int N = 2; };
template <> struct UamTapsPerTrip<1> { static const int N = 4; };
template <> struct UamTapsPerTrip<8> { static const int N = 4; };

// GRAD: four more 32 x 33 partial matrices behind the group's shared memory, for the per-record sums of dP/du, s dP/du,
// dP/dv and s dP/dv (s = the sample's number in its record); flushed and reduced exactly like the penalty partials.
#define UAM_GROUP_GPART (32 * 33)
#define UAM_GROUP_SMEM_GRAD (UAM_GROUP_SMEM + 4 * UAM_GROUP_GPART * 4)     // 22832

// The sample loop of uam_group_score.  CLAMP = false: the caller guarantees that every sample of the group lies
// strictly inside the raster.
template <int TF, int LAYOUT, int TILE, bool CLAMP, bool GRAD = false>
__device__ __forceinline__ void uam_group_samples(const UamRasterParams& rp, const typename UamTexel<TF>::T* __restrict__ tex,
                                                  const unsigned char* s_tile, int ti0, int tj0, const UamGroupRec* s_rec,
                                                  const int2* s_PQ, float* part, uint2* s_tab, unsigned* s_bits, const int lane,
                                                  const int P, const int S, const int T, float& acc, unsigned& colmask, int& kcur,
                                                  int& pcur, float* gpart, float4& gacc) {
    constexpr int TAPS = UamTapsPerTrip<TF>::N;
    const unsigned le_mask = 0xffffffffu >> (31 - lane);
    // record parameters of this lane's current record (re-read only when the record changes)
    int kc = 0, pc = 0, qc = 0;
    double2 ca, cb;
    {
        const UamGroupRec r0 = s_rec[0];
        const int2 pq0 = s_PQ[0];
        ca = make_double2(r0.U, r0.SU); cb = make_double2(r0.V, r0.SV); pc = pq0.x; qc = pq0.y;
    }
    // The record of a flat index comes from a WINDOW TABLE, filled once per UAM_GROUP_SEG flat samples: entry w =
    // {bitmap of the record starts inside window w, number of records that start before it}; then
    // k(lane) = count + popc(bitmap & lanes <= lane) - 1 -- one LDS.64, a LOP3, a POPC and an add per tap, where a
    // per-window REDUX.OR over freshly built one-hot words cost about ten instructions more.
    // Lanes without a record (S == 0, only past the end of the last group) have P == T and set no bit.  The flat indices
    // past T (the tail of the last trip) belong to a DUMMY record that starts at T (slot = number of records, all-zero
    // parameters: it samples pixel (0, 0)), so the loop needs no "past the end" test anywhere: the dummy's sum and
    // collision bit land in a slot nobody reads (column 32 of the partials / a shift by 32, or the slot of a lane
    // that has no record).
    for (int f0 = 0; f0 < T; f0 += UAM_GROUP_SEG) {
        __syncwarp();
        s_bits[lane] = 0u;
        __syncwarp();
        const unsigned rel0 = (unsigned)(P - f0);
        if (S > 0 && rel0 < (unsigned)UAM_GROUP_SEG) atomicOr(&s_bits[rel0 >> 5], 1u << (rel0 & 31u));
        if (lane == 0 && (unsigned)(T - f0) < (unsigned)UAM_GROUP_SEG) atomicOr(&s_bits[(unsigned)(T - f0) >> 5], 1u << ((unsigned)(T - f0) & 31u));
        __syncwarp();
        {
            const unsigned bits = s_bits[lane];
            const int c = __popc(bits);
            int incl = c;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int t = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += t;
            }
            const int before = __popc(__ballot_sync(0xffffffffu, S > 0 && P < f0));
            s_tab[lane] = make_uint2(bits, (unsigned)(before + incl - c));
        }
        __syncwarp();
        const int t_end = min(T, f0 + UAM_GROUP_SEG);
        for (int t0 = f0; t0 < t_end; t0 += 32 * TAPS) {
            UamTap<TF> tap[TAPS];
            int kk[TAPS], pp[TAPS];
            float ss[TAPS];                 // GRAD: sample number in the record, slopes kept per coordinate
            bool fu[TAPS], fv[TAPS];
            const uint2* tab = s_tab + ((t0 - f0) >> 5);
#pragma unroll
            for (int j = 0; j < TAPS; ++j) {
                const int wb = t0 + 32 * j;
                const uint2 e = tab[j];                 // (a window past the segment's table can only be past T: masked below)
                const int k = (int)e.y + __popc(e.x & le_mask) - 1;
                if (k != kc) {
                    ca = *reinterpret_cast<const double2*>(&s_rec[k].U);
                    cb = *reinterpret_cast<const double2*>(&s_rec[k].V);
                    if constexpr (TILE) {
                        const int2 pq = s_PQ[k];
                        pc = pq.x; qc = pq.y;
                    } else {
                        pc = qc = reinterpret_cast<const int*>(s_PQ)[2 * k];    // whole segments: Q == P (one 4-byte load)
                    }
                    kc = k;
                }
                kk[j] = k;
                pp[j] = pc;
                const double sd = uam_int2double(wb + lane - qc);
                const double u = __dadd_rn(ca.x, __dmul_rn(sd, ca.y)), v = __dadd_rn(cb.x, __dmul_rn(sd, cb.y));
                if constexpr (TILE) uam_tap_load_tile<TF>(s_tile, ti0, tj0, rp, u, v, tap[j]);
                else uam_tap_load<TF, LAYOUT, CLAMP>(tex, rp, u, v, tap[j]);
                if constexpr (GRAD) {
                    ss[j] = (float)(wb + lane - qc);
                    fu[j] = !CLAMP || uam_free_coord(u, rp.W);
                    fv[j] = !CLAMP || uam_free_coord(v, rp.H);
                }
            }
#pragma unroll
            for (int j = 0; j < TAPS; ++j) {
                float pen, du, dv;
                bool occ;
                if constexpr (GRAD) uam_tap_grad<TF>(rp, tap[j], pen, occ, du, dv);
                else uam_tap_eval<TF>(rp, tap[j], pen, occ);
                const int k = kk[j];
                if (k != kcur) {
                    const int row = (lane - pcur) & 31;          // record-local residue class of this lane's samples
                    part[row * 33 + kcur] = acc;
                    acc = 0.0f;
                    if constexpr (GRAD) {
                        gpart[row * 33 + kcur] = gacc.x;
                        gpart[UAM_GROUP_GPART + row * 33 + kcur] = gacc.y;
                        gpart[2 * UAM_GROUP_GPART + row * 33 + kcur] = gacc.z;
                        gpart[3 * UAM_GROUP_GPART + row * 33 + kcur] = gacc.w;
                        gacc = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
                    }
                    kcur = k;
                    pcur = pp[j];
                }
                acc += pen;
                if constexpr (GRAD) {
                    if (!fu[j]) du = 0.0f;
                    if (!fv[j]) dv = 0.0f;
                    gacc.x += du;
                    gacc.y += ss[j] * du;
                    gacc.z += dv;
                    gacc.w += ss[j] * dv;
                }
                colmask |= uam_shl_clamp(occ ? 1u : 0u, (unsigned)k);    // (k = 32, the dummy of a full group: shifted out)
            }
        }
    }
}

// Scores one group.  In: this lane's record (first sample U/V, step SU/SV, S samples starting at sample number s0 of
// its parent segment; S = 0 for a lane without a record).  Out: the record's sample sum (not yet divided by the
// parent's sample count) and its collision bit.  TILE = 0: taps from global memory (tex); TILE = 1: taps from the
// tile staged in shared memory.
// Shared-memory traffic is what the LSU data pipe of this kernel is busiest with (ncu: 256 M shared wavefronts against
// 111 M global ones per C3 launch before the three measures below): (1) the partials are zeroed with conflict-free
// stores (each lane clearing its own row put all 32 lanes on the same 4 banks); (2) a lane re-reads the record
// parameters only when its record changes; (3) a lane's partial for record k goes to the row of its record-local
// residue class (lane - P_k) mod 32, so the final per-record sums are one 32 x 32 transpose-reduce (31 shuffles)
// instead of 32 warp sums (160 shuffles) -- same pairing tree, same bits.
// per-record sums of a 32 x 33 partial matrix: v[s] = this lane's residue class of record s; 32 x 32 transpose-reduce,
// pairing tree (l, l^16), (.., ^8), (.., ^4), (.., ^2), (.., ^1) like uam_warp_sum; lane s ends with the sum of record s
__device__ __forceinline__ float uam_part_reduce(const float* part, const int lane) {
    float v[32];
#pragma unroll
    for (int s = 0; s < 32; ++s) v[s] = part[lane * 33 + s];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const bool hi = (lane & o) != 0;
#pragma unroll
        for (int i = 0; i < o; ++i) {
            const float send = hi ? v[i] : v[i + o];
            const float keep = hi ? v[i + o] : v[i];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, o);
        }
    }
    return v[0];
}

// GRAD: gmine = the record's {sum dP/du, sum s dP/du, sum dP/dv, sum s dP/dv} (slopes of clamped coordinates are 0).
template <int TF, int LAYOUT, int TILE, bool GRAD = false>
__device__ __forceinline__ void uam_group_score(const UamRasterParams& rp, const typename UamTexel<TF>::T* __restrict__ tex,
                                                const unsigned char* s_tile, int ti0, int tj0, unsigned char* warp_smem,
                                                const int lane, const double U, const double V, const double SU,
                                                const double SV, const int S, const int s0, float& mine, bool& collide,
                                                float4* gmine = nullptr) {
    UamGroupRec* s_rec = reinterpret_cast<UamGroupRec*>(warp_smem + UAM_GROUP_REC_OFF);
    int2* s_PQ = reinterpret_cast<int2*>(warp_smem + UAM_GROUP_PQ_OFF);       // {P_k, Q_k = P_k - s0_k}: flat index -> sample number
    float* part = reinterpret_cast<float*>(warp_smem + UAM_GROUP_PART_OFF);
    uint2* s_tab = reinterpret_cast<uint2*>(warp_smem + UAM_GROUP_TAB_OFF);
    unsigned* s_bits = reinterpret_cast<unsigned*>(warp_smem + UAM_GROUP_BITS_OFF);
    int incl = S;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    const int P = incl - S;
    const int T = __shfl_sync(0xffffffffu, incl, 31);
    UamGroupRec mr;
    mr.U = U; mr.SU = SU; mr.V = V; mr.SV = SV;
    s_rec[lane] = mr;
    s_PQ[lane] = make_int2(P, P - s0);
    {
        // the dummy record behind the last real one (the real records are the lanes 0 .. n_rec - 1)
        const int n_rec = __popc(__ballot_sync(0xffffffffu, S > 0));
        if (lane == 0) {
            UamGroupRec z0;
            z0.U = 0.0; z0.SU = 0.0; z0.V = 0.0; z0.SV = 0.0;
            s_rec[n_rec] = z0;
            s_PQ[n_rec] = make_int2(T, T);
        }
    }
#pragma unroll
    for (int q = 0; q < 9; ++q)
        if (q * 32 + lane < 32 * 33 / 4) reinterpret_cast<float4*>(part)[q * 32 + lane] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    float* const gpart = reinterpret_cast<float*>(warp_smem + UAM_GROUP_SMEM);
    if constexpr (GRAD) {
#pragma unroll
        for (int q = 0; q < 33; ++q) reinterpret_cast<float4*>(gpart)[q * 32 + lane] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    }
    __syncwarp();
    // Fast path: when every record of the group lies strictly inside the raster (first and last sample in
    // [0, W-1) x [0, H-1); the samples in between are monotone), the clamps and the saturation of the cell / fraction
    // step cannot act and are left out (same bits).
    bool rec_inside = true;
    if (S > 0 && !TILE) {
        const double ue = __dadd_rn(U, __dmul_rn(uam_int2double(S - 1), SU)), ve = __dadd_rn(V, __dmul_rn(uam_int2double(S - 1), SV));
        const double wl = (double)(rp.W - 1), hl = (double)(rp.H - 1);
        rec_inside = U >= 0.0 && U < wl && ue >= 0.0 && ue < wl && V >= 0.0 && V < hl && ve >= 0.0 && ve < hl;
    }
    const bool all_inside = !TILE && __all_sync(0xffffffffu, rec_inside);
    float acc = 0.0f;
    unsigned colmask = 0;
    int kcur = 0, pcur = 0;     // the record `acc` belongs to and its first flat index
    float4 gacc = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    if (all_inside) uam_group_samples<TF, LAYOUT, TILE, false, GRAD>(rp, tex, s_tile, ti0, tj0, s_rec, s_PQ, part, s_tab, s_bits, lane, P, S, T, acc, colmask, kcur, pcur, gpart, gacc);
    else uam_group_samples<TF, LAYOUT, TILE, true, GRAD>(rp, tex, s_tile, ti0, tj0, s_rec, s_PQ, part, s_tab, s_bits, lane, P, S, T, acc, colmask, kcur, pcur, gpart, gacc);
    {
        const int row = (lane - pcur) & 31;
        part[row * 33 + kcur] = acc;             // (kcur = 32, the dummy of a full group, is the padding column)
        if constexpr (GRAD) {
            gpart[row * 33 + kcur] = gacc.x;
            gpart[UAM_GROUP_GPART + row * 33 + kcur] = gacc.y;
            gpart[2 * UAM_GROUP_GPART + row * 33 + kcur] = gacc.z;
            gpart[3 * UAM_GROUP_GPART + row * 33 + kcur] = gacc.w;
        }
    }
    __syncwarp();
    mine = uam_part_reduce(part, lane);
    if constexpr (GRAD) {
        gmine->x = uam_part_reduce(gpart, lane);
        gmine->y = uam_part_reduce(gpart + UAM_GROUP_GPART, lane);
        gmine->z = uam_part_reduce(gpart + 2 * UAM_GROUP_GPART, lane);
        gmine->w = uam_part_reduce(gpart + 3 * UAM_GROUP_GPART, lane);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) colmask |= __shfl_xor_sync(0xffffffffu, colmask, o);
    collide = ((colmask >> lane) & 1u) != 0u;
    __syncwarp();
}

// GRAD: also part_grad[id] = the segment's share of its two waypoints' penalty gradient (uam_seg_grad); 22.8 KB of shared
// memory per warp, so one CTA of 8 warps per SM.
// Scoring form on quad texels: 3 CTAs (24 warps) per SM, up to 80 registers.  At 4 CTAs the 64-register cap made the sample
// loop spill and re-derive the lane, the shared-memory base and constants inside it (259 instructions per 4 taps against 235);
// on the C3 shard (B200 at 1000 W) the kernel takes 1.455 ms at 3 CTAs, 1.531 ms at 4 and 1.604 ms at 2
// (profiles/r03_ab_group_occupancy.txt).
template <int TF, int LAYOUT, bool GRAD = false>
__global__ void __launch_bounds__(UAM_CTA_THREADS, GRAD ? 1 : (UamIsQuad<TF>::v ? 3 : 4))
uam_k_score_groups(unsigned long long n_seg, int Wp, UamRasterParams rp, const typename UamTexel<TF>::T* __restrict__ tex,
                   const double2* __restrict__ z, const unsigned* __restrict__ sorted_id, float* __restrict__ part_pen,
                   uint8_t* __restrict__ part_col, unsigned* __restrict__ next_group, float4* __restrict__ part_grad) {
    extern __shared__ __align__(128) unsigned char uam_smem[];
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    unsigned char* base = uam_smem + (size_t)warp * (GRAD ? UAM_GROUP_SMEM_GRAD : UAM_GROUP_SMEM);
    const unsigned long long n_groups = (n_seg + 31) >> 5;
    // The groups are handed out through a counter, in sorted order: a warp that finishes early takes the next group instead of
    // idling behind a fixed share (ncu r02 with a fixed round-robin share per warp: the SMs were busy 91 % of the kernel's
    // time on average, 2.84 .. 3.28 M of 3.30 M cycles -- the samples per group vary with the segment lengths), and the groups in
    // flight are always one window of consecutive groups of the sorted order (the L2 working set).  A group's result depends
    // only on its own records: the bits do not depend on which warp takes it.
    for (;;) {
        unsigned gi = 0;
        if (lane == 0) gi = atomicAdd(next_group, 1u);
        const unsigned long long g = __shfl_sync(0xffffffffu, gi, 0);
        if (g >= n_groups) break;
        const unsigned long long ridx = (g << 5) + lane;
        const bool have = ridx < n_seg;
        // this lane's segment, rebuilt from its id (same arithmetic as the binning pass)
        UamSegRec r;
        r.U = 0.0; r.V = 0.0; r.SU = 0.0; r.SV = 0.0; r.S = 0; r.IS = 0.0f; r.id = 0;
        if (have) r = uam_make_segment(z, (unsigned long long)__ldg(sorted_id + ridx), Wp, rp);
        float mine;
        bool col;
        float4 gmine;
        uam_group_score<TF, LAYOUT, 0, GRAD>(rp, tex, nullptr, 0, 0, base, lane, r.U, r.V, r.SU, r.SV, r.S, 0, mine, col, &gmine);
        if constexpr (GRAD) {
            if (have) part_grad[r.id] = uam_seg_grad(gmine, r.IS);
        }
        if (have) {
            if (TF == 8 && rp.w0 >= 0.0f) {
                // sign-packed quads with a weight >= 0: every tap is >= 0, so the partial is >= 0 (or NaN) and its sign bit is
                // free to carry the collision flag (-0.0f = "0, occupied"): one scattered 4-byte store per segment instead of
                // 4 + 1 bytes (uam_k_reduce_paths<., 1> reads it back)
                part_pen[r.id] = __uint_as_float((__float_as_uint(mine * r.IS) & 0x7fffffffu) | (col ? 0x80000000u : 0u));
            } else {
                part_pen[r.id] = mine * r.IS;
                part_col[r.id] = col ? 1 : 0;
            }
        }
    }
}

// one warp per path: fixed-order sum of the per-segment partials + the length term
// BEST: the launch also finds the best candidate (and exchanges it with the peer ranks): uam_best_tail_cta
// PACKED: the collision flag is the sign bit of the partial (uam_k_score_groups<8>), part_col is not read.
// len_path: the paths' length terms from uam_k_bin_hist (the waypoints are then read only when nsamp is asked for).
// GRAD: also grad: waypoint j = segment j's start share + segment j-1's end share (part_grad, fp32, in that order) + the
// fp64 length part.
template <int BEST, int PACKED, bool GRAD = false>
__global__ void __launch_bounds__(UAM_CTA_THREADS)
uam_k_reduce_paths(const double2* __restrict__ z, long long B, int Wp, UamRasterParams rp,
                   const float* __restrict__ part_pen, const uint8_t* __restrict__ part_col,
                   const double* __restrict__ len_path, float* __restrict__ cost,
                   uint8_t* __restrict__ collide, long long* __restrict__ nsamp, UamBestTail tl,
                   const float4* __restrict__ part_grad, double2* __restrict__ grad) {
    const int lane = threadIdx.x & 31;
    const long long warp0 = (long long)blockIdx.x * UAM_WARPS_PER_CTA + (threadIdx.x >> 5);
    const long long nwarps = (long long)gridDim.x * UAM_WARPS_PER_CTA;
    const int N = Wp - 2;
    unsigned long long kbest = UAM_KEY_EMPTY;
    // a warp works on PT consecutive paths at a time (PT independent load streams, interleaved shuffle trees)
    constexpr int PT = 4;
    for (long long pb = warp0 * PT; pb < B; pb += nwarps * PT) {
        float acc[PT];
        long long ns[PT];
        bool col[PT];
#pragma unroll
        for (int t = 0; t < PT; ++t) { acc[t] = 0.0f; ns[t] = 0; col[t] = false; }
        for (int j = lane; j < Wp; j += 32) {
            float pv[PT];
            uint8_t cv[PT];
#pragma unroll
            for (int t = 0; t < PT; ++t) {
                const bool ok = pb + t < B;
                pv[t] = ok ? part_pen[(pb + t) * Wp + j] : 0.0f;
                cv[t] = (!PACKED && ok) ? part_col[(pb + t) * Wp + j] : (uint8_t)0;
            }
#pragma unroll
            for (int t = 0; t < PT; ++t) {
                if (PACKED) {
                    acc[t] += fabsf(pv[t]);
                    col[t] = col[t] || (__float_as_uint(pv[t]) >> 31);
                } else {
                    acc[t] += pv[t];
                    col[t] = col[t] || cv[t];
                }
                if constexpr (GRAD) {
                    if (pb + t < B) {
                        const long long row = (pb + t) * Wp;
                        const float4 a = part_grad[row + j];
                        float pu = a.x, pvv = a.y;
                        if (j >= 1) {
                            const float4 e = part_grad[row + j - 1];
                            pu += e.z;
                            pvv += e.w;
                        }
                        grad[row + j] = uam_grad_point(uam_len_grad(z + row, j, N, z[row + j], rp), pu, pvv, N, rp);
                    }
                }
                if (nsamp && pb + t < B) {
                    long long S = 1;
                    if (j < Wp - 1) {
                        const double2* zp = z + (pb + t) * Wp;
                        const double2 p = zp[j];
                        const double2 q = zp[j + 1];
                        const double dU = __dsub_rn(uam_pix(q.x, rp.x0, rp.dx), uam_pix(p.x, rp.x0, rp.dx));
                        const double dV = __dsub_rn(uam_pix(q.y, rp.y0, rp.dy), uam_pix(p.y, rp.y0, rp.dy));
                        S = (long long)uam_seg_samples(dU, dV, rp.spc);
                    }
                    ns[t] += S;
                }
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
            for (int t = 0; t < PT; ++t) acc[t] += __shfl_xor_sync(0xffffffffu, acc[t], o);              // (the tree of uam_warp_sum)
        }
        float a_mine = acc[0];
        bool c_mine = __any_sync(0xffffffffu, col[0]);
        long long n_mine = 0;
#pragma unroll
        for (int t = 1; t < PT; ++t) {
            const bool ct = __any_sync(0xffffffffu, col[t]);
            a_mine = lane == t ? acc[t] : a_mine;
            c_mine = lane == t ? ct : c_mine;
        }
        if (nsamp) {
#pragma unroll
            for (int t = 0; t < PT; ++t) {
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) ns[t] += __shfl_xor_sync(0xffffffffu, ns[t], o);
                n_mine = lane == t ? ns[t] : n_mine;
            }
        }
        const long long path = pb + lane;
        if (lane < PT && path < B) {
            const double len_sum = len_path[path];
            const float c = (float)((double)(N + 1) * len_sum + (double)a_mine / (double)N);
            if (cost) cost[path] = c;
            if (collide) collide[path] = c_mine ? 1 : 0;
            if (nsamp) nsamp[path] = n_mine;
            if (BEST) {
                const unsigned long long k = uam_best_key(c, tl.offset + (unsigned long long)path);
                kbest = k < kbest ? k : kbest;
            }
        }
    }
    if (BEST) uam_best_tail_cta(tl, uam_cta_min_key(kbest));
}

// ---- integral mode, tile-staged (variant 3) ----------------------------------------------------------------------
// The binned pipeline of variant 2 still gathers every texel through L1 (ncu: l1tex 98 % busy, 25 sectors per load
// request).  Variant 3 removes the gather from the global-memory path altogether: every segment is cut into PIECES
// at the boundaries of 64 x 64-cell raster tiles (a piece = a run of consecutive samples whose bilinear footprint
// lies in one tile + its one-cell halo), the pieces are counting-sorted by tile, and a CTA stages the tile it works
// on -- one contiguous 65 x 65-texel block of the tile-major raster copy -- into shared memory with a single bulk
// async copy (TMA engine, cp.async.bulk + mbarrier) and then samples it with LDS.128 (4 immediate-offset loads per
// sample, no tag lookups, no sector misses).
//   uam_k_piece_count -> uam_k_scan_u32 (paths) + uam_k_tile_scan (tiles, work items) -> [host reads the piece
//   total and sizes the scratch] -> uam_k_piece_scatter -> uam_k_score_tiles -> uam_k_reduce_slots
// Sample positions are computed from the parent segment (U + s * SU, fp64, s counted from the segment start), so
// they are bit-identical to the other variants and to the oracle; the cut points are found with the same
// expression (estimate by division, then corrected until position(c-1) is inside and position(c) outside), so a
// sample can never be assigned to a tile that does not hold its footprint.  Each piece writes its partial sum to a
// slot that depends only on its own path (path-contiguous slot ranges from a prefix sum over per-path piece counts)
// and the last kernel adds a path's slots in a fixed order: results are independent of the rest of the batch.
#define UAM_ITEM_PIECES 2048              // pieces per work item (one tile load per item)

struct __align__(16) UamPieceRec {
    double U, V, SU, SV;   // parent segment: first sample (pixel coordinates) and per-sample step
    int s0;                // first sample of the piece (counted from the segment start)
    int n;                 // samples in the piece
    float IS;              // 1 / S of the parent segment
    unsigned slot;         // index of the piece's partial sum (path-contiguous)
};

struct UamTileGeo {
    int tiles_x, tiles_y, ntiles;
    unsigned tile_stride;  // bytes between tiles in the tile-major copy (multiple of 128)
    unsigned copy_bytes;   // bytes staged per tile (multiple of 16)
};

__device__ __forceinline__ double uam_pos(double U, double SU, int s) { return __dadd_rn(U, __dmul_rn((double)s, SU)); }

// Smallest s' in (s, S] whose sample leaves tile index t along one axis (n cells on that axis), S if none does.
// position(s') is monotone in s', cell(s') = clamp(floor(position), 0, n - 2).
__device__ __forceinline__ int uam_next_cross(double U, double SU, int s, int S, int t, int n) {
    if (SU > 0.0) {
        const int b = (t + 1) << 6;
        if (b > n - 2) return S;                      // the clamp keeps the cell in this tile
        const double bd = (double)b;
        const double e = ceil(__ddiv_rn(__dsub_rn(bd, U), SU));
        int c = s + 1;
        if (e >= (double)S) c = S; else if (e > (double)c) c = (int)e;
        while (c > s + 1 && uam_pos(U, SU, c - 1) >= bd) --c;
        while (c < S && uam_pos(U, SU, c) < bd) ++c;
        return c;
    }
    if (SU < 0.0) {
        if (t == 0) return S;
        const double bd = (double)(t << 6);           // outside once position < bd
        const double e = ceil(__ddiv_rn(__dsub_rn(bd, U), SU));
        int c = s + 1;
        if (e >= (double)S) c = S; else if (e > (double)c) c = (int)e;
        while (c > s + 1 && uam_pos(U, SU, c - 1) < bd) --c;
        while (c < S && uam_pos(U, SU, c) >= bd) ++c;
        return c;
    }
    return S;                                         // zero or NaN step: the cell never changes
}

// Calls emit(tile, s0, n, piece_index) for every piece of the segment, in order; returns the number of pieces.
template <class F>
__device__ __forceinline__ int uam_walk_pieces(const UamSegRec& r, const UamRasterParams& rp, int tiles_x, F&& emit) {
    int s = 0, cnt = 0;
    while (s < r.S) {
        const double u = uam_pos(r.U, r.SU, s), v = uam_pos(r.V, r.SV, s);
        const int tj = min(max(__double2int_rd(u), 0), rp.W - 2) >> 6;
        const int ti = min(max(__double2int_rd(v), 0), rp.H - 2) >> 6;
        const int nxt = min(uam_next_cross(r.U, r.SU, s, r.S, tj, rp.W), uam_next_cross(r.V, r.SV, s, r.S, ti, rp.H));
        emit(ti * tiles_x + tj, s, nxt - s, cnt);
        ++cnt;
        s = nxt;
    }
    return cnt;
}

// warp per path, lanes stride the path's Wp units (Wp - 1 segments + the goal waypoint)
__global__ void __launch_bounds__(UAM_CTA_THREADS)
uam_k_piece_count(const double2* __restrict__ z, long long B, int Wp, UamRasterParams rp, int tiles_x,
                  unsigned* __restrict__ hist, unsigned short* __restrict__ seg_cnt, unsigned* __restrict__ path_cnt) {
    const int lane = threadIdx.x & 31;
    const long long warp0 = (long long)blockIdx.x * UAM_WARPS_PER_CTA + (threadIdx.x >> 5);
    const long long nwarps = (long long)gridDim.x * UAM_WARPS_PER_CTA;
    for (long long path = warp0; path < B; path += nwarps) {
        unsigned tot = 0;
        for (int k = lane; k < Wp; k += 32) {
            const unsigned long long id = (unsigned long long)path * Wp + k;
            const UamSegRec r = uam_make_segment(z, id, Wp, rp);
            const int c = uam_walk_pieces(r, rp, tiles_x, [&](int tile, int, int, int) { atomicAdd(&hist[tile], 1u); });
            seg_cnt[id] = (unsigned short)c;
            tot += (unsigned)c;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) tot += __shfl_xor_sync(0xffffffffu, tot, o);
        if (lane == 0) path_cnt[path] = tot;
    }
}

// exclusive prefix of in[0..n) into out[0..n], out[n] = total (mod 2^32); *total64 = exact total (single CTA)
__global__ void __launch_bounds__(1024)
uam_k_scan_u32(const unsigned* __restrict__ in, long long n, unsigned* __restrict__ out, unsigned long long* __restrict__ total64) {
    __shared__ unsigned long long warp_tot[32];
    const long long per = (n + 1023) / 1024;
    const long long lo = min((long long)threadIdx.x * per, n), hi = min(lo + per, n);
    unsigned long long local = 0;
    for (long long i = lo; i < hi; ++i) local += in[i];
    unsigned long long incl = local;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) warp_tot[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        unsigned long long w = warp_tot[lane], wi = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long t = __shfl_up_sync(0xffffffffu, wi, o);
            if (lane >= o) wi += t;
        }
        warp_tot[lane] = wi - w;
        if (lane == 31) { *total64 = wi; out[n] = (unsigned)wi; }
    }
    __syncthreads();
    unsigned long long run = warp_tot[warp] + incl - local;
    for (long long i = lo; i < hi; ++i) {
        const unsigned h = in[i];
        out[i] = (unsigned)run;
        run += h;
    }
}

// Tiles: exclusive prefix of the piece histogram -> cursor, and the work-item list: tile t with c pieces becomes
// ceil(c / UAM_ITEM_PIECES) items (tile, part).  Single CTA; counters[0] = number of items.
__global__ void __launch_bounds__(1024)
uam_k_tile_scan(const unsigned* __restrict__ hist, int n, unsigned* __restrict__ cursor, uint2* __restrict__ items,
                unsigned* __restrict__ counters) {
    __shared__ unsigned warp_p[32], warp_i[32];
    const int per = (n + 1023) / 1024;
    const int lo = min((int)threadIdx.x * per, n), hi = min(lo + per, n);
    unsigned lp = 0, li = 0;
    for (int i = lo; i < hi; ++i) {
        const unsigned h = hist[i];
        lp += h;
        li += (h + UAM_ITEM_PIECES - 1) / UAM_ITEM_PIECES;
    }
    unsigned ip = lp, ii = li;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned a = __shfl_up_sync(0xffffffffu, ip, o), b = __shfl_up_sync(0xffffffffu, ii, o);
        if (lane >= o) { ip += a; ii += b; }
    }
    if (lane == 31) { warp_p[warp] = ip; warp_i[warp] = ii; }
    __syncthreads();
    if (warp == 0) {
        unsigned a = warp_p[lane], b = warp_i[lane], ai = a, bi = b;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned x = __shfl_up_sync(0xffffffffu, ai, o), y = __shfl_up_sync(0xffffffffu, bi, o);
            if (lane >= o) { ai += x; bi += y; }
        }
        warp_p[lane] = ai - a;
        warp_i[lane] = bi - b;
        if (lane == 31) counters[0] = bi;
    }
    __syncthreads();
    unsigned rp_ = warp_p[warp] + ip - lp, ri = warp_i[warp] + ii - li;
    for (int i = lo; i < hi; ++i) {
        const unsigned h = hist[i];
        cursor[i] = rp_;
        rp_ += h;
        const unsigned ni = (h + UAM_ITEM_PIECES - 1) / UAM_ITEM_PIECES;
        for (unsigned q = 0; q < ni; ++q) items[ri + q] = make_uint2((unsigned)i, q);
        ri += ni;
    }
}

__global__ void __launch_bounds__(UAM_CTA_THREADS)
uam_k_piece_scatter(const double2* __restrict__ z, long long B, int Wp, UamRasterParams rp, int tiles_x,
                    const unsigned short* __restrict__ seg_cnt, const unsigned* __restrict__ path_base,
                    unsigned* __restrict__ cursor, UamPieceRec* __restrict__ recs) {
    const int lane = threadIdx.x & 31;
    const long long warp0 = (long long)blockIdx.x * UAM_WARPS_PER_CTA + (threadIdx.x >> 5);
    const long long nwarps = (long long)gridDim.x * UAM_WARPS_PER_CTA;
    for (long long path = warp0; path < B; path += nwarps) {
        unsigned carry = path_base[path];
        for (int k0 = 0; k0 < Wp; k0 += 32) {
            const int k = k0 + lane;
            const unsigned long long id = (unsigned long long)path * Wp + k;
            const unsigned c = k < Wp ? seg_cnt[id] : 0u;
            unsigned incl = c;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned t = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += t;
            }
            const unsigned base = carry + incl - c;
            carry += __shfl_sync(0xffffffffu, incl, 31);
            if (k < Wp) {
                const UamSegRec r = uam_make_segment(z, id, Wp, rp);
                uam_walk_pieces(r, rp, tiles_x, [&](int tile, int s0, int n, int piece) {
                    const unsigned pos = atomicAdd(&cursor[tile], 1u);
                    UamPieceRec q;
                    q.U = r.U; q.V = r.V; q.SU = r.SU; q.SV = r.SV;
                    q.s0 = s0; q.n = n; q.IS = r.IS; q.slot = base + (unsigned)piece;
                    recs[pos] = q;
                });
            }
        }
    }
}

// ---- bulk async copy (TMA engine, no tensor map: one contiguous block) + mbarrier ------------------------------------
__device__ __forceinline__ unsigned uam_smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void uam_mbar_init(void* bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(uam_smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void uam_bulk_load(void* dst, const void* src, unsigned bytes, void* bar) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(uam_smem_u32(bar)), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(uam_smem_u32(dst)), "l"(src), "r"(bytes), "r"(uam_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void uam_mbar_wait(void* bar, unsigned parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "UAM_WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@!p bra UAM_WAIT_%=;\n\t}"
        ::"r"(uam_smem_u32(bar)), "r"(parity) : "memory");
}

// shared memory of uam_k_score_tiles: [tile (copy_bytes, 128-aligned)] [mbarrier + control, 128 B] [per-warp areas]
#define UAM_TILE_CTL_BYTES 128

template <int TF>
__global__ void __launch_bounds__(UAM_CTA_THREADS, 2)
uam_k_score_tiles(UamRasterParams rp, UamTileGeo tg, const unsigned char* __restrict__ tiles,
                  const unsigned* __restrict__ tile_end, const uint2* __restrict__ items, unsigned* __restrict__ counters,
                  const UamPieceRec* __restrict__ recs, float* __restrict__ part_pen, uint8_t* __restrict__ part_col) {
    extern __shared__ __align__(128) unsigned char uam_smem[];
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    unsigned char* s_tile = uam_smem;
    const unsigned tile_area = (tg.copy_bytes + 127u) & ~127u;
    unsigned long long* s_bar = reinterpret_cast<unsigned long long*>(uam_smem + tile_area);
    volatile unsigned* s_ctl = reinterpret_cast<volatile unsigned*>(uam_smem + tile_area + 16);   // [0] item, [1] next group
    unsigned char* base = uam_smem + tile_area + UAM_TILE_CTL_BYTES + (size_t)warp * UAM_GROUP_SMEM;
    if (threadIdx.x == 0) uam_mbar_init(s_bar, 1);
    __syncthreads();
    const unsigned n_items = counters[0];
    unsigned parity = 0;
    for (;;) {
        // all warps are done with the previous tile and with s_ctl
        __syncthreads();
        if (threadIdx.x == 0) {
            const unsigned it = atomicAdd(&counters[1], 1u);
            s_ctl[0] = it;
            if (it < n_items) {
                const uint2 im = items[it];
                uam_bulk_load(s_tile, tiles + (size_t)im.x * tg.tile_stride, tg.copy_bytes, s_bar);
                s_ctl[1] = (im.x ? tile_end[im.x - 1] : 0u) + im.y * UAM_ITEM_PIECES + UAM_WARPS_PER_CTA * 32;
            }
        }
        __syncthreads();
        const unsigned it = s_ctl[0];
        if (it >= n_items) break;
        const uint2 item = items[it];
        const unsigned t_lo = item.x ? tile_end[item.x - 1] : 0u, t_hi = tile_end[item.x];
        const unsigned lo = t_lo + item.y * UAM_ITEM_PIECES;
        const unsigned hi = min(lo + UAM_ITEM_PIECES, t_hi);
        const int ti0 = (int)(item.x / (unsigned)tg.tiles_x) * UAM_TS, tj0 = (int)(item.x % (unsigned)tg.tiles_x) * UAM_TS;
        uam_mbar_wait(s_bar, parity);
        parity ^= 1u;
        unsigned g = lo + warp * 32;
        while (g < hi) {
            const unsigned ridx = g + lane;
            const bool have = ridx < hi;
            double U = 0.0, V = 0.0, SU = 0.0, SV = 0.0;
            int S = 0, s0 = 0;
            unsigned slot = 0;
            float IS = 0.0f;
            if (have) {
                const double2* rp2 = reinterpret_cast<const double2*>(recs + ridx);
                const double2 a = __ldg(rp2), b = __ldg(rp2 + 1);
                const int4 c = __ldg(reinterpret_cast<const int4*>(rp2 + 2));
                U = a.x; V = a.y; SU = b.x; SV = b.y;
                s0 = c.x;
                S = c.y;
                IS = __int_as_float(c.z);
                slot = (unsigned)c.w;
            }
            float mine;
            bool col;
            uam_group_score<TF, 0, 1>(rp, nullptr, s_tile, ti0, tj0, base, lane, U, V, SU, SV, S, s0, mine, col);
            if (have) {
                part_pen[slot] = mine * IS;
                part_col[slot] = col ? 1 : 0;
            }
            // next group of this item: first come, first served
            unsigned nx = 0;
            if (lane == 0) nx = atomicAdd((unsigned*)&s_ctl[1], 32u);
            g = __shfl_sync(0xffffffffu, nx, 0);
        }
    }
}

// one warp per path: fixed-order sum of the path's piece partials + the length term
__global__ void __launch_bounds__(UAM_CTA_THREADS)
uam_k_reduce_slots(const double2* __restrict__ z, long long B, int Wp, UamRasterParams rp,
                   const unsigned* __restrict__ path_base, const float* __restrict__ part_pen,
                   const uint8_t* __restrict__ part_col, float* __restrict__ cost, uint8_t* __restrict__ collide,
                   long long* __restrict__ nsamp) {
    const int lane = threadIdx.x & 31;
    const long long warp0 = (long long)blockIdx.x * UAM_WARPS_PER_CTA + (threadIdx.x >> 5);
    const long long nwarps = (long long)gridDim.x * UAM_WARPS_PER_CTA;
    const int N = Wp - 2;
    for (long long path = warp0; path < B; path += nwarps) {
        const double2* zp = z + path * Wp;
        float acc = 0.0f;
        double len_sum = 0.0;
        long long ns = 0;
        bool col = false;
        const unsigned s_lo = path_base[path], s_hi = path_base[path + 1];
        for (unsigned s = s_lo + lane; s < s_hi; s += 32) {
            acc += part_pen[s];
            col = col || part_col[s];
        }
        for (int j = lane; j < Wp; j += 32) {
            const double2 p = zp[j];
            len_sum += uam_len_term(zp, j, N, p, rp);
            if (nsamp) {
                long long S = 1;
                if (j < Wp - 1) {
                    const double2 q = zp[j + 1];
                    const double dU = __dsub_rn(uam_pix(q.x, rp.x0, rp.dx), uam_pix(p.x, rp.x0, rp.dx));
                    const double dV = __dsub_rn(uam_pix(q.y, rp.y0, rp.dy), uam_pix(p.y, rp.y0, rp.dy));
                    S = (long long)uam_seg_samples(dU, dV, rp.spc);
                }
                ns += S;
            }
        }
        acc = uam_warp_sum(acc);
        len_sum = uam_warp_sum(len_sum);
        col = __any_sync(0xffffffffu, col);
        if (nsamp) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) ns += __shfl_xor_sync(0xffffffffu, ns, o);
        }
        if (lane == 0) {
            if (cost) cost[path] = (float)((double)(N + 1) * len_sum + (double)acc / (double)N);
            if (collide) collide[path] = col ? 1 : 0;
            if (nsamp) nsamp[path] = ns;
        }
    }
}

// tile-major copy of the texels: tile (ty, tx) = cells [64 ty, 64 ty + 65) x [64 tx, 64 tx + 65), row-major inside
// the tile, zero outside the raster.  One thread per output texel.
template <int TF, int LAYOUT>
__global__ void uam_k_build_tiles(const typename UamTexel<TF>::T* __restrict__ tex, UamRasterParams rp, UamTileGeo tg,
                                  unsigned char* __restrict__ out) {
    typedef typename UamTexel<TF>::T T;
    const unsigned per_tile = UAM_TSH * UAM_TSH;
    const size_t n = (size_t)tg.ntiles * per_tile;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t o = (size_t)blockIdx.x * blockDim.x + threadIdx.x; o < n; o += stride) {
        const unsigned tile = (unsigned)(o / per_tile), w = (unsigned)(o - (size_t)tile * per_tile);
        const unsigned li = w / UAM_TSH, lj = w - li * UAM_TSH;
        const unsigned i = (tile / (unsigned)tg.tiles_x) * UAM_TS + li, j = (tile % (unsigned)tg.tiles_x) * UAM_TS + lj;
        T v;
        if (i < (unsigned)rp.H && j < (unsigned)rp.W) {
            v = tex[uam_tex_row<(UamIsQuad<TF>::v ? 4 : TF), LAYOUT>(i, rp.row_stride) + uam_tex_col<(UamIsQuad<TF>::v ? 4 : TF), LAYOUT>(j)];
        } else {
            if constexpr (TF == 2) v = make_float2(0.0f, 0.0f); else v = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        }
        reinterpret_cast<T*>(out + (size_t)tile * tg.tile_stride)[w] = v;
    }
}

}  // namespace

// ---- host side ---------------------------------------------------------------------------------------------------
int uam_raster_prepare(uam_ctx* ctx, int64_t B, int N, const double* h_p, int n_p, int flags, double spc,
                       UamRasterParams* rp) {
    if (B < 0 || N < 1) return uam_fail(ctx, UAM_ERR_INVALID, "need B >= 0 and N >= 1 (got B=%lld N=%d)", (long long)B, N);
    if (!ctx->has_raster) return uam_fail(ctx, UAM_ERR_STATE, "no raster: call uam_map_set_raster first");
    if (!(spc >= 0.0) || spc > 64.0) return uam_fail(ctx, UAM_ERR_INVALID, "samples_per_cell must be in [0, 64]");
    if (spc > 0.0 && (double)(N + 2) * UAM_MAX_SAMPLES_PER_SEGMENT > 2.0e9)
        return uam_fail(ctx, UAM_ERR_UNSUPPORTED, "N = %d waypoints per path is too many for integral mode", N);
    UamParams prm;
    UAM_TRY(uam_make_params(ctx, h_p, n_p, flags, &prm));
    if (prm.n_regions != ctx->geo.L)
        return uam_fail(ctx, UAM_ERR_INVALID, "p carries %d layer weights, the raster has %d layers", prm.n_regions, ctx->geo.L);
    rp->x0 = ctx->geo.x0; rp->dx = ctx->geo.dx; rp->y0 = ctx->geo.y0; rp->dy = ctx->geo.dy;
    rp->ms_x = prm.ms_x; rp->ms_y = prm.ms_y;
    rp->spc = spc;
    rp->H = ctx->geo.H; rp->W = ctx->geo.W;
    const int tile_texels = ctx->geo.texel_floats == 4 ? 8 : 16;
    rp->row_stride = (unsigned)(ctx->geo.layout ? ctx->geo.tiles_x * tile_texels : ctx->geo.W);
    rp->w0 = (float)prm.w[0];
    rp->w1 = ctx->geo.L > 1 ? (float)prm.w[1] : 0.0f;
    rp->w2 = ctx->geo.L > 2 ? (float)prm.w[2] : 0.0f;
    rp->flags = flags;
    // auto (-1): the binned pipeline pays off once the batch has enough segments to fill the raster bins.  Decided
    // from the whole call (not per pipeline chunk), so host-buffer and device-buffer calls run the same kernels.
    rp->variant = ctx->int_variant >= 0 ? ctx->int_variant : ((unsigned long long)B * (N + 2) >= UAM_LARGE_BATCH_SEGMENTS ? 2 : 0);
    rp->combined = 0;
    return UAM_OK;
}

namespace {

// d_grad != NULL: the gradient forms of the last two kernels (uam_grad_paths_raster; best must be NULL then)
template <int TF, int LAYOUT>
int uam_raster_launch_binned(uam_ctx* ctx, const void* texv, const double2* z, int64_t B, int Wp, const UamRasterParams& rp,
                             float* d_cost, uint8_t* d_collide, long long* d_nsamp, cudaStream_t st, int slot,
                             const UamBestTail* best, bool* best_done, double2* d_grad = nullptr) {
    typedef typename UamTexel<TF>::T T;
    const unsigned long long n_seg = (unsigned long long)B * Wp;
    UamBinGeo bg;
    bg.shift = ctx->bin_shift;
    const int side = std::max(rp.W, rp.H);
    while (((side + (1 << bg.shift) - 1) >> bg.shift) > 128) ++bg.shift;       // at most 128 x 128 bins (64 KiB of smem)
    int p2 = 1;
    while (p2 < ((side + (1 << bg.shift) - 1) >> bg.shift)) p2 <<= 1;
    bg.nbins = p2 * p2;
    bg.hx = (float)(0.5 / rp.dx); bg.hy = (float)(0.5 / rp.dy);
    bg.ox = (float)(-rp.x0 / rp.dx - 0.5); bg.oy = (float)(-rp.y0 / rp.dy - 0.5);
    // scratch: sorted ids (u32) | part_pen (f32) | hist (u32) | cursor (u32) | len_path (f64) | seg_bin (u16) | part_col (u8)
    // (+ gradient: part_grad (float4) behind part_col, 16-byte aligned)
    const size_t need_score = n_seg * (4 + 4 + 2 + 1) + (size_t)bg.nbins * 8 + 16 + (size_t)B * 8 + 256;
    const size_t need = need_score + (d_grad ? n_seg * 16 + 16 : 0);
    UAM_TRY(uam_reserve(ctx, &ctx->d_bin_scratch[slot], &ctx->bin_scratch_bytes[slot], need));
    unsigned* sorted_id = (unsigned*)ctx->d_bin_scratch[slot];
    float* part_pen = (float*)(sorted_id + n_seg);
    unsigned* hist = (unsigned*)(part_pen + n_seg);
    unsigned* next_group = hist + bg.nbins;                   // work counter of uam_k_score_groups (zeroed with the histogram)
    unsigned* cursor = next_group + 4;
    double* len_path = (double*)(cursor + bg.nbins);          // (8-byte aligned: n_seg * 8 + nbins * 8 + 16 bytes in)
    unsigned short* seg_bin = (unsigned short*)(len_path + B);
    uint8_t* part_col = (uint8_t*)(seg_bin + n_seg);
    float4* part_grad = (float4*)(((uintptr_t)(part_col + n_seg) + 15) & ~(uintptr_t)15);
    UAM_NVTX("uam.raster.binned");
    UAM_CUDA(ctx, cudaMemsetAsync(hist, 0, (size_t)(bg.nbins + 4) * 4, st));
    // a CTA of the histogram / scatter kernels owns whole paths: ppc paths = about UAM_BIN_CHUNK segments
    const int ppc = std::max(1, ctx->bin_chunk / Wp);
    const unsigned long long chunk = (unsigned long long)ppc * Wp;
    const unsigned chunks = (unsigned)((B + ppc - 1) / ppc);
    const size_t hsmem = (size_t)bg.nbins * 4;
    if (hsmem > 48 * 1024) {
        UAM_CUDA(ctx, cudaFuncSetAttribute(uam_k_bin_hist<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)hsmem));
        UAM_CUDA(ctx, cudaFuncSetAttribute(uam_k_bin_hist<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)hsmem));
        UAM_CUDA(ctx, cudaFuncSetAttribute(uam_k_bin_hist<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)hsmem));
        UAM_CUDA(ctx, cudaFuncSetAttribute(uam_k_bin_scatter, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)hsmem));
    }
    nvtxRangePushA("uam.raster.bin");
    if (ctx->bin_pt == 1) uam_k_bin_hist<1><<<chunks, 1024, hsmem, st>>>(z, (long long)B, Wp, ppc, rp, bg, seg_bin, hist, len_path);
    else if (ctx->bin_pt == 2) uam_k_bin_hist<2><<<chunks, 1024, hsmem, st>>>(z, (long long)B, Wp, ppc, rp, bg, seg_bin, hist, len_path);
    else uam_k_bin_hist<4><<<chunks, 1024, hsmem, st>>>(z, (long long)B, Wp, ppc, rp, bg, seg_bin, hist, len_path);
    UAM_CHECK_LAUNCH(ctx, "uam_k_bin_hist");
    uam_k_bin_scan<<<1, 1024, 0, st>>>(hist, bg.nbins, cursor);
    UAM_CHECK_LAUNCH(ctx, "uam_k_bin_scan");
    uam_k_bin_scatter<<<chunks, 1024, hsmem, st>>>(n_seg, chunk, bg, seg_bin, cursor, sorted_id);
    UAM_CHECK_LAUNCH(ctx, "uam_k_bin_scatter");
    nvtxRangePop();
    const size_t gsmem = (size_t)UAM_GROUP_SMEM * UAM_WARPS_PER_CTA;
    const unsigned long long n_groups = (n_seg + 31) >> 5;        // (< 2^27: segment ids are 32-bit)
    const long long sctas = std::min<long long>((long long)((n_groups + UAM_WARPS_PER_CTA - 1) / UAM_WARPS_PER_CTA), (long long)ctx->sm_count * 16);
    const bool timed = ctx->time_kernels && slot == 0 && !d_grad;
    if (timed) {
        UAM_TRY(uam_time_begin(ctx, st));
    }
    nvtxRangePushA("uam.raster.score");
    if (d_grad) {
        const size_t gsmem_g = (size_t)UAM_GROUP_SMEM_GRAD * UAM_WARPS_PER_CTA;
        UAM_CUDA(ctx, cudaFuncSetAttribute(uam_k_score_groups<TF, LAYOUT, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gsmem_g));
        uam_k_score_groups<TF, LAYOUT, true><<<(unsigned)sctas, UAM_CTA_THREADS, gsmem_g, st>>>(n_seg, Wp, rp, (const T*)texv, z, sorted_id, part_pen, part_col,
                                                                                             next_group, part_grad);
    } else {
        uam_k_score_groups<TF, LAYOUT><<<(unsigned)sctas, UAM_CTA_THREADS, gsmem, st>>>(n_seg, Wp, rp, (const T*)texv, z, sorted_id, part_pen, part_col, next_group, nullptr);
    }
    nvtxRangePop();
    UAM_CHECK_LAUNCH(ctx, "uam_k_score_groups");
    if (timed) {
        UAM_TRY(uam_time_end(ctx, st));
    }
    const long long rctas = std::min<long long>((B + 4 * UAM_WARPS_PER_CTA - 1) / (4 * UAM_WARPS_PER_CTA), (long long)ctx->sm_count * 16);   // 4 paths per warp and trip
    UAM_NVTX("uam.raster.reduce+best");
    const bool packed = TF == 8 && rp.w0 >= 0.0f;       // the condition uam_k_score_groups tests
    const UamBestTail tl = best ? *best : UamBestTail{};
    const auto reduce = d_grad ? (packed ? uam_k_reduce_paths<0, 1, true> : uam_k_reduce_paths<0, 0, true>)
                      : best   ? (packed ? uam_k_reduce_paths<1, 1> : uam_k_reduce_paths<1, 0>)
                               : (packed ? uam_k_reduce_paths<0, 1> : uam_k_reduce_paths<0, 0>);
    reduce<<<(unsigned)rctas, UAM_CTA_THREADS, 0, st>>>(z, B, Wp, rp, part_pen, part_col, len_path, d_cost, d_collide, d_nsamp, tl,
                                                        d_grad ? part_grad : nullptr, d_grad);
    if (best) *best_done = true;
    UAM_CHECK_LAUNCH(ctx, "uam_k_reduce_paths");
    return UAM_OK;
}

// Tile-major copy of the texels for variant 3, built on first use; `key` names the texel array it was made from
// (raster generation, or generation of the weight-combined texels).
template <int TF, int LAYOUT>
int uam_ensure_tiles(uam_ctx* ctx, const void* texv, uint64_t key, const UamRasterParams& rp, UamTileGeo* tg, cudaStream_t st) {
    typedef typename UamTexel<TF>::T T;
    tg->tiles_x = (rp.W + UAM_TS - 1) / UAM_TS;
    tg->tiles_y = (rp.H + UAM_TS - 1) / UAM_TS;
    tg->ntiles = tg->tiles_x * tg->tiles_y;
    const unsigned raw = (unsigned)(UAM_TSH * UAM_TSH * sizeof(T));
    tg->copy_bytes = (raw + 15u) & ~15u;
    tg->tile_stride = (raw + 127u) & ~127u;
    if (ctx->tiles_valid && ctx->tiles_key == key) return UAM_OK;
    UAM_CUDA(ctx, cudaDeviceSynchronize());      // the old copy may still be read by kernels queued on other streams
    UAM_TRY(uam_reserve(ctx, &ctx->d_tiles, &ctx->tiles_bytes, (size_t)tg->ntiles * tg->tile_stride));
    uam_k_build_tiles<TF, LAYOUT><<<ctx->sm_count * 8, 256, 0, st>>>((const T*)texv, rp, *tg, (unsigned char*)ctx->d_tiles);
    UAM_CHECK_LAUNCH(ctx, "uam_k_build_tiles");
    UAM_CUDA(ctx, cudaStreamSynchronize(st));    // every pipeline stream may use it from now on
    ctx->tiles_valid = true;
    ctx->tiles_key = key;
    return UAM_OK;
}

template <int TF, int LAYOUT>
int uam_raster_launch_tiles(uam_ctx* ctx, const void* texv, uint64_t tex_key, const double2* z, int64_t B, int Wp,
                            const UamRasterParams& rp, float* d_cost, uint8_t* d_collide, long long* d_nsamp, cudaStream_t st,
                            int slot, bool* fell_back) {
    *fell_back = false;
    UamTileGeo tg;
    UAM_TRY((uam_ensure_tiles<TF, LAYOUT>(ctx, texv, tex_key, rp, &tg, st)));
    const unsigned long long n_seg = (unsigned long long)B * Wp;
    // phase 1 scratch: total64 | hist | cursor | counters[4] | path_cnt[B] | path_base[B + 1] | seg_cnt (u16)
    const size_t nt = (size_t)tg.ntiles;
    const size_t need1 = 16 + (2 * nt + 4 + (size_t)B + (size_t)B + 1) * 4 + n_seg * 2 + 256;
    UAM_TRY(uam_reserve(ctx, &ctx->d_bin_scratch[slot], &ctx->bin_scratch_bytes[slot], need1));
    unsigned long long* total64 = (unsigned long long*)ctx->d_bin_scratch[slot];
    unsigned* hist = (unsigned*)(total64 + 2);
    unsigned* cursor = hist + nt;
    unsigned* counters = cursor + nt;
    unsigned* path_cnt = counters + 4;
    unsigned* path_base = path_cnt + B;
    unsigned short* seg_cnt = (unsigned short*)(path_base + B + 1);
    UAM_CUDA(ctx, cudaMemsetAsync(total64, 0, 16 + (2 * nt + 4) * 4, st));
    const long long pctas = std::min<long long>((B + UAM_WARPS_PER_CTA - 1) / UAM_WARPS_PER_CTA, (long long)ctx->sm_count * 16);
    uam_k_piece_count<<<(unsigned)pctas, UAM_CTA_THREADS, 0, st>>>(z, B, Wp, rp, tg.tiles_x, hist, seg_cnt, path_cnt);
    UAM_CHECK_LAUNCH(ctx, "uam_k_piece_count");
    uam_k_scan_u32<<<1, 1024, 0, st>>>(path_cnt, B, path_base, total64);
    UAM_CHECK_LAUNCH(ctx, "uam_k_scan_u32");
    // the scratch for the pieces is sized from their exact number: one 8-byte read-back per call
    unsigned long long total = 0;
    UAM_CUDA(ctx, cudaMemcpyAsync(&total, total64, sizeof total, cudaMemcpyDeviceToHost, st));
    UAM_CUDA(ctx, cudaStreamSynchronize(st));
    if (total >= 0xffffffffull) {              // slots are 32-bit: leave this batch to the binned pipeline
        *fell_back = true;
        return UAM_OK;
    }
    const size_t n_items_max = nt + (size_t)(total / UAM_ITEM_PIECES) + 1;
    const size_t need2 = (size_t)total * (sizeof(UamPieceRec) + 4 + 1) + n_items_max * sizeof(uint2) + 256;
    UAM_TRY(uam_reserve(ctx, &ctx->d_piece_scratch[slot], &ctx->piece_scratch_bytes[slot], need2));
    UamPieceRec* recs = (UamPieceRec*)ctx->d_piece_scratch[slot];
    uint2* items = (uint2*)(recs + total);
    float* part_pen = (float*)(items + n_items_max);
    uint8_t* part_col = (uint8_t*)(part_pen + total);
    uam_k_tile_scan<<<1, 1024, 0, st>>>(hist, tg.ntiles, cursor, items, counters);
    UAM_CHECK_LAUNCH(ctx, "uam_k_tile_scan");
    uam_k_piece_scatter<<<(unsigned)pctas, UAM_CTA_THREADS, 0, st>>>(z, B, Wp, rp, tg.tiles_x, seg_cnt, path_base, cursor, recs);
    UAM_CHECK_LAUNCH(ctx, "uam_k_piece_scatter");
    const size_t smem = (size_t)((tg.copy_bytes + 127u) & ~127u) + UAM_TILE_CTL_BYTES + (size_t)UAM_GROUP_SMEM * UAM_WARPS_PER_CTA;
    UAM_CUDA(ctx, cudaFuncSetAttribute(uam_k_score_tiles<TF>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (ctx->time_kernels && slot == 0) {
        UAM_TRY(uam_time_begin(ctx, st));
    }
    // after the scatter cursor[t] is the END of tile t's pieces
    uam_k_score_tiles<TF><<<(unsigned)(ctx->sm_count * 2), UAM_CTA_THREADS, smem, st>>>(rp, tg, (const unsigned char*)ctx->d_tiles, cursor, items,
                                                                                    counters, recs, part_pen, part_col);
    UAM_CHECK_LAUNCH(ctx, "uam_k_score_tiles");
    if (ctx->time_kernels && slot == 0) {
        UAM_TRY(uam_time_end(ctx, st));
    }
    const long long rctas = std::min<long long>((B + UAM_WARPS_PER_CTA - 1) / UAM_WARPS_PER_CTA, (long long)ctx->sm_count * 16);
    uam_k_reduce_slots<<<(unsigned)rctas, UAM_CTA_THREADS, 0, st>>>(z, B, Wp, rp, path_base, part_pen, part_col, d_cost, d_collide, d_nsamp);
    UAM_CHECK_LAUNCH(ctx, "uam_k_reduce_slots");
    return UAM_OK;
}

// One launch of the scorer (GRAD = false) or of its gradient (GRAD = true, uam_grad_paths_raster) on texels of form TF:
// the waypoint kernel, the warp-per-path integral kernel or the binned pipeline.  Integral variants 1 and 3 have no
// gradient form (uam_raster_grad_supported refuses them first).  The scorer's dominant kernel is timed for slot 0.
template <int TF, int LAYOUT, bool GRAD>
int uam_raster_launch_t(uam_ctx* ctx, const void* texv, uint64_t tex_key, const double2* z, int64_t B, int Wp,
                        const UamRasterParams& rp, float* d_cost, uint8_t* d_collide, long long* d_nsamp, double2* d_grad,
                        cudaStream_t st, int slot, const UamBestTail* best, bool* best_done) {
    typedef typename UamTexel<TF>::T T;
    const T* tex = (const T*)texv;
    const bool timed = !GRAD && ctx->time_kernels && slot == 0;
    if (rp.spc == 0.0) {
        const long long ctas = std::min<long long>((B + UAM_WARPS_PER_CTA - 1) / UAM_WARPS_PER_CTA, (long long)ctx->sm_count * 16);
        if (timed) UAM_TRY(uam_time_begin(ctx, st));
        uam_k_score_raster_wp<TF, LAYOUT, GRAD><<<(unsigned)ctas, UAM_CTA_THREADS, 0, st>>>(z, B, Wp, rp, tex, d_cost, d_collide, d_nsamp, d_grad);
        UAM_CHECK_LAUNCH(ctx, "uam_k_score_raster_wp");
        if (timed) UAM_TRY(uam_time_end(ctx, st));
        return UAM_OK;
    }
    if (rp.variant >= 2 && (unsigned long long)B * Wp < 0xffffffffull) {
        if constexpr (!GRAD) {
            if (rp.variant == 3 && (rp.W + UAM_TS - 1) / UAM_TS + (rp.H + UAM_TS - 1) / UAM_TS < 65535) {
                bool fell_back = false;
                UAM_TRY((uam_raster_launch_tiles<TF, LAYOUT>(ctx, texv, tex_key, z, B, Wp, rp, d_cost, d_collide, d_nsamp, st, slot, &fell_back)));
                if (!fell_back) return UAM_OK;
            }
        }
        return uam_raster_launch_binned<TF, LAYOUT>(ctx, texv, z, B, Wp, rp, d_cost, d_collide, d_nsamp, st, slot, best, best_done, d_grad);
    }
    if constexpr (UamIsQuad<TF>::v) {
        return uam_fail(ctx, UAM_ERR_STATE, "quad texels are not sampled by the warp-per-path integral kernels");
    } else {
        const size_t per_warp = uam_seg_table_bytes(Wp) + (GRAD ? (size_t)Wp * sizeof(float4) : 0);
        const size_t budget = 200 * 1024;
        if (per_warp > budget) return uam_fail(ctx, UAM_ERR_UNSUPPORTED, "N = %d waypoints per path is too many for integral mode", Wp - 2);
        const int wpc = (int)std::max<size_t>(1, std::min<size_t>(UAM_WARPS_PER_CTA, budget / per_warp));
        const size_t smem = per_warp * wpc;
        const long long ctas = std::min<long long>((B + wpc - 1) / wpc, (long long)ctx->sm_count * 16);
        auto kernel = uam_k_score_raster_int<TF, LAYOUT, 0, GRAD>;
        if constexpr (!GRAD) {
            if (rp.variant == 1) kernel = uam_k_score_raster_int<TF, LAYOUT, 1>;
        }
        if (smem > 48 * 1024) UAM_CUDA(ctx, cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        if (timed) UAM_TRY(uam_time_begin(ctx, st));
        kernel<<<(unsigned)ctas, wpc * 32, smem, st>>>(z, B, Wp, rp, tex, d_cost, d_collide, d_nsamp, d_grad);
        UAM_CHECK_LAUNCH(ctx, "uam_k_score_raster_int");
        if (timed) UAM_TRY(uam_time_end(ctx, st));
        return UAM_OK;
    }
}

// Quad texels for the large-batch integral pipelines (variants 2 and 3), whose gather is bound by the number of load
// requests / bytes moved through L1 or shared memory:
//  * the penalty is linear in the layers, sum_l w_l * bilerp(layer_l) = bilerp(sum_l w_l * layer_l), so for a given
//    weight vector an L = 2..3 raster collapses into ONE layer C = sum_l w_l * layer_l (fp32, same rounding class as
//    the per-layer sum it replaces); an L = 1 raster keeps its raw layer and the weight is applied after the lerp;
//  * cell (i, j) then stores its whole bilinear footprint {C(i,j), C(i,j+1), C(i+1,j), C(i+1,j+1)} as one float4, and
//    a bilinear tap is ONE 16-byte load instead of four.  The occupancy flags ride in the sign bits of the four
//    values when every value is >= 0 (checked on the device while building; -0.0 marks an occupied cell of value 0),
//    otherwise they move to a bit-plane (one extra, cache-resident word load per tap).
// Built per (raster, weights) and kept until either changes.
// PACK = 1: store occupied cells' values negated (sign bit = occupancy flag; needs every value >= 0: a negative or NaN
// value raises *bad and the caller rebuilds with PACK = 0 + the bit-plane).
template <int TF, int LAYOUT, int PACK>
__global__ void uam_k_build_quads(const typename UamTexel<TF>::T* __restrict__ tex, int H, int W, unsigned rs_src, unsigned rs_q,
                                  float w0, float w1, float w2, size_t n_out, float4* __restrict__ quad, unsigned* __restrict__ bad) {
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    bool neg = false;
    auto value = [&](int i, int j) -> float {
        if (i >= H || j >= W) return 0.0f;
        const typename UamTexel<TF>::T t = tex[uam_tex_row<TF, LAYOUT>(i, rs_src) + uam_tex_col<TF, LAYOUT>(j)];
        float c, o;
        if constexpr (TF == 2) { c = t.x; o = t.y; } else { c = w0 * t.x + w1 * t.y + w2 * t.z; o = t.w; }
        if constexpr (PACK) {
            neg = neg || !(c >= 0.0f);
            c = fabsf(c);                    // -0.0 -> +0.0
            if (o != 0.0f) c = -c;
        }
        return c;
    };
    for (size_t o = (size_t)blockIdx.x * blockDim.x + threadIdx.x; o < n_out; o += stride) {
        int i, j;                     // o -> cell of the float4 layout (one thread per output texel, coalesced stores)
        if (LAYOUT == 0) {
            i = (int)(o / W);
            j = (int)(o - (size_t)i * W);
        } else {
            const size_t tile = o >> 3;
            const int w = (int)(o & 7), tiles_x = (int)(rs_q >> 3);
            const int ty = (int)(tile / tiles_x), tx = (int)(tile - (size_t)ty * tiles_x);
            i = ty * 2 + ((w >> 1) & 1);
            j = tx * 4 + ((w >> 2) & 1) * 2 + (w & 1);
        }
        quad[o] = make_float4(value(i, j), value(i, j + 1), value(i + 1, j), value(i + 1, j + 1));
    }
    if (PACK && neg) atomicOr(bad, 1u);
}

// one thread per 32-bit word (8 x 4 cells) of the occupancy bit-plane
template <int TF, int LAYOUT>
__global__ void uam_k_build_occ_bits(const typename UamTexel<TF>::T* __restrict__ tex, int H, int W, unsigned rs_src, unsigned blocks_x,
                                     unsigned n_words, unsigned* __restrict__ bits) {
    const unsigned o = blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= n_words) return;
    const unsigned blk = o >> 5, wi = (o >> 2) & 7u, wj = o & 3u;
    const unsigned i0 = (blk / blocks_x) * 32u + wi * 4u, j0 = (blk % blocks_x) * 32u + wj * 8u;
    unsigned word = 0;
    for (unsigned b = 0; b < 32; ++b) {
        const unsigned i = i0 + (b >> 3), j = j0 + (b & 7u);
        if (i < (unsigned)H && j < (unsigned)W) {
            const typename UamTexel<TF>::T t = tex[uam_tex_row<TF, LAYOUT>(i, rs_src) + uam_tex_col<TF, LAYOUT>(j)];
            float occ;
            if constexpr (TF == 2) occ = t.y; else occ = t.w;
            if (occ != 0.0f) word |= 1u << b;
        }
    }
    bits[o] = word;
}

template <int TF, int LAYOUT>
int uam_build_quads_t(uam_ctx* ctx, const UamRasterParams& rp, unsigned rs_q, size_t n_out, cudaStream_t st) {
    typedef typename UamTexel<TF>::T T;
    // first choice: sign-packed quads (no second load per tap); the flag word sits in front of the bit-plane
    unsigned* bad = (unsigned*)ctx->d_occ_bits;
    UAM_CUDA(ctx, cudaMemsetAsync(bad, 0, 4, st));
    uam_k_build_quads<TF, LAYOUT, 1><<<ctx->sm_count * 8, 256, 0, st>>>((const T*)ctx->d_tex, rp.H, rp.W, rp.row_stride, rs_q, rp.w0, rp.w1, rp.w2,
                                                                         n_out, (float4*)ctx->d_tex_comb, bad);
    UAM_CHECK_LAUNCH(ctx, "uam_k_build_quads");
    unsigned h_bad = 0;
    UAM_CUDA(ctx, cudaMemcpyAsync(&h_bad, bad, 4, cudaMemcpyDeviceToHost, st));
    UAM_CUDA(ctx, cudaStreamSynchronize(st));
    ctx->comb_packed = !h_bad && !ctx->no_sign_pack;
    if (ctx->comb_packed) return UAM_OK;
    // negative (or NaN) values somewhere: plain quads + occupancy bit-plane
    UAM_TRY(uam_ensure_occ_bits(ctx, st));
    uam_k_build_quads<TF, LAYOUT, 0><<<ctx->sm_count * 8, 256, 0, st>>>((const T*)ctx->d_tex, rp.H, rp.W, rp.row_stride, rs_q, rp.w0, rp.w1, rp.w2,
                                                                         n_out, (float4*)ctx->d_tex_comb, bad);
    UAM_CHECK_LAUNCH(ctx, "uam_k_build_quads");
    return UAM_OK;
}

// Makes the quad texels of the raster and rp's weights (unless the last ones still fit), then points rp at them: the row
// stride becomes the quads', and the weights of an L = 2..3 raster, now inside the quads, become {1, 0, 0}.
int uam_ensure_quads(uam_ctx* ctx, UamRasterParams* rp, cudaStream_t st) {
    const int W = rp->W, H = rp->H, lay = ctx->geo.layout, tf = ctx->geo.texel_floats;
    const int tiles_x = (W + 3) / 4, tiles_y = (H + 1) / 2;
    const unsigned rs_q = lay ? (unsigned)tiles_x * 8u : (unsigned)W;
    rp->occ_blocks_x = (unsigned)(W + 31) / 32u;
    const bool same_w = tf == 2 || (ctx->comb_w[0] == rp->w0 && ctx->comb_w[1] == rp->w1 && ctx->comb_w[2] == rp->w2);
    if (!(ctx->comb_valid && same_w)) {
        UAM_NVTX("uam.raster.build_quads");
        const size_t n_out = lay ? (size_t)tiles_x * tiles_y * 8 : (size_t)H * W;
        UAM_CUDA(ctx, cudaDeviceSynchronize());      // kernels on other streams may still read the old quads
        UAM_TRY(uam_reserve(ctx, &ctx->d_tex_comb, &ctx->tex_comb_bytes, n_out * sizeof(float4)));
        UAM_TRY(uam_reserve(ctx, &ctx->d_occ_bits, &ctx->occ_bits_bytes, (size_t)(uam_occ_words(H, W) + 4) * 4));
        if (tf == 2) UAM_TRY(lay ? (uam_build_quads_t<2, 1>(ctx, *rp, rs_q, n_out, st)) : (uam_build_quads_t<2, 0>(ctx, *rp, rs_q, n_out, st)));
        else UAM_TRY(lay ? (uam_build_quads_t<4, 1>(ctx, *rp, rs_q, n_out, st)) : (uam_build_quads_t<4, 0>(ctx, *rp, rs_q, n_out, st)));
        UAM_CUDA(ctx, cudaStreamSynchronize(st));    // every pipeline stream may use them from now on
        ctx->comb_valid = true;
        ctx->comb_w[0] = rp->w0; ctx->comb_w[1] = rp->w1; ctx->comb_w[2] = rp->w2;
        ctx->comb_gen += 1;
    }
    rp->occ_bits = (const unsigned*)ctx->d_occ_bits + 4;
    rp->combined = ctx->comb_packed ? 2 : 1;
    rp->row_stride = rs_q;
    if (tf == 4) { rp->w0 = 1.0f; rp->w1 = 0.0f; rp->w2 = 0.0f; }
    return UAM_OK;
}

// One launch of the scorer or of its gradient on the texels the call samples: the quad texels when
// uam_raster_precompute made them for it (rp.combined = 1: + occupancy bit-plane, 2: sign-packed), the raster's own
// otherwise.  slot: which scratch buffer of the ctx the binned pipeline may use (0 = caller-stream calls, 1.. = host
// pipeline stages).  best (nullable, scorer only): also find the best candidate of the launch, which the binned pipeline
// fuses into its last kernel and then reports in *best_done.
template <bool GRAD>
int uam_raster_dispatch(uam_ctx* ctx, const UamRasterParams& rp, const double* d_z, int64_t B, int N, float* d_cost,
                        uint8_t* d_collide, long long* d_nsamp, double* d_grad, cudaStream_t st, int slot,
                        const UamBestTail* best, bool* best_done) {
    const int Wp = N + 2, lay = ctx->geo.layout;
    const double2* z = reinterpret_cast<const double2*>(d_z);
    double2* g = reinterpret_cast<double2*>(d_grad);
    const void* tex = rp.combined ? ctx->d_tex_comb : ctx->d_tex;
    const uint64_t key = rp.combined ? (ctx->comb_gen << 1) | 1u : ctx->raster_gen << 1;
    auto launch = [&](auto form) {
        constexpr int TF = decltype(form)::value;
        return lay ? uam_raster_launch_t<TF, 1, GRAD>(ctx, tex, key, z, B, Wp, rp, d_cost, d_collide, d_nsamp, g, st, slot, best, best_done)
                   : uam_raster_launch_t<TF, 0, GRAD>(ctx, tex, key, z, B, Wp, rp, d_cost, d_collide, d_nsamp, g, st, slot, best, best_done);
    };
    if (rp.combined == 2) return launch(std::integral_constant<int, 8>());
    if (rp.combined) return launch(std::integral_constant<int, 1>());
    if (ctx->geo.texel_floats == 2) return launch(std::integral_constant<int, 2>());
    return launch(std::integral_constant<int, 4>());
}

int uam_raster_launch(uam_ctx* ctx, const double* d_z, int64_t B, int N, const UamRasterParams& rp, float* d_cost,
                      uint8_t* d_collide, long long* d_nsamp, cudaStream_t st, int slot, const UamBestTail* best = nullptr) {
    if (best && !d_cost) return uam_fail(ctx, UAM_ERR_INVALID, "the best-candidate key needs the cost output");
    bool best_done = false;
    UAM_TRY(uam_raster_dispatch<false>(ctx, rp, d_z, B, N, d_cost, d_collide, d_nsamp, nullptr, st, slot, best, &best_done));
    if (best && !best_done) UAM_TRY(uam_best_launch(ctx, d_cost, 0, B, *best, st));
    return UAM_OK;
}

}  // namespace

int uam_ensure_occ_bits(uam_ctx* ctx, cudaStream_t st) {
    if (ctx->occ_bits_valid) return UAM_OK;
    const int H = ctx->geo.H, W = ctx->geo.W, lay = ctx->geo.layout, tf = ctx->geo.texel_floats;
    const unsigned n_words = uam_occ_words(H, W), blocks_x = (unsigned)(W + 31) / 32u;
    const unsigned rs = (unsigned)(lay ? ctx->geo.tiles_x * (tf == 4 ? 8 : 16) : W);    // the raster's own texels
    UAM_TRY(uam_reserve(ctx, &ctx->d_occ_bits, &ctx->occ_bits_bytes, (size_t)(n_words + 4) * 4));
    unsigned* bits = (unsigned*)ctx->d_occ_bits + 4;
    const unsigned grid = (n_words + 255) / 256;
    if (tf == 2 && lay) uam_k_build_occ_bits<2, 1><<<grid, 256, 0, st>>>((const float2*)ctx->d_tex, H, W, rs, blocks_x, n_words, bits);
    else if (tf == 2) uam_k_build_occ_bits<2, 0><<<grid, 256, 0, st>>>((const float2*)ctx->d_tex, H, W, rs, blocks_x, n_words, bits);
    else if (lay) uam_k_build_occ_bits<4, 1><<<grid, 256, 0, st>>>((const float4*)ctx->d_tex, H, W, rs, blocks_x, n_words, bits);
    else uam_k_build_occ_bits<4, 0><<<grid, 256, 0, st>>>((const float4*)ctx->d_tex, H, W, rs, blocks_x, n_words, bits);
    UAM_CHECK_LAUNCH(ctx, "uam_k_build_occ_bits");
    UAM_CUDA(ctx, cudaStreamSynchronize(st));
    ctx->occ_bits_valid = true;
    return UAM_OK;
}

// Once per API call, before any chunk is launched: make the quad texels if this call will use them.
int uam_raster_precompute(uam_ctx* ctx, UamRasterParams* rp, int64_t B, int N, cudaStream_t st) {
    // large batches: integral mode through the binned pipelines, waypoint mode when the batch is worth the one-off build
    const bool big_wp = rp->spc == 0.0 && (unsigned long long)B * (N + 2) >= UAM_LARGE_BATCH_SEGMENTS;
    if (((rp->spc > 0.0 && rp->variant >= 2) || big_wp) && ctx->combine_layers && (unsigned long long)B * (N + 2) < 0xffffffffull) {
        UAM_TRY(uam_ensure_quads(ctx, rp, st));
    }
    return UAM_OK;
}

int uam_raster_grad_supported(uam_ctx* ctx, const UamRasterParams& rp) {
    if (rp.spc > 0.0 && (rp.variant == 1 || rp.variant == 3))
        return uam_fail(ctx, UAM_ERR_UNSUPPORTED, "integral variant %d has no gradient form (use -1, 0 or 2)", rp.variant);
    return UAM_OK;
}

int uam_raster_grad_enqueue(uam_ctx* ctx, const UamRasterParams& rp, const double* d_z, int64_t B, int N, float* d_cost,
                            uint8_t* d_collide, double* d_grad, cudaStream_t st) {
    return uam_raster_dispatch<true>(ctx, rp, d_z, B, N, d_cost, d_collide, nullptr, d_grad, st, 0, nullptr, nullptr);
}

extern "C" int uam_grad_paths_raster(uam_ctx* ctx, const double* d_z, int64_t B, int N, const double* h_p, int n_p, int flags,
                                     double samples_per_cell, float* d_cost, uint8_t* d_collide, double* d_grad, void* stream) {
    if (!ctx) return UAM_ERR_INVALID;
    UamRasterParams rp;
    UAM_TRY(uam_raster_prepare(ctx, B, N, h_p, n_p, flags, samples_per_cell, &rp));
    if (B == 0) return UAM_OK;
    if (!d_z || !d_grad) return uam_fail(ctx, UAM_ERR_INVALID, "paths or gradient pointer is NULL");
    UAM_TRY(uam_raster_grad_supported(ctx, rp));
    UAM_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = uam_pick_stream(ctx, stream);
    UAM_TRY(uam_raster_precompute(ctx, &rp, B, N, st));
    return uam_raster_grad_enqueue(ctx, rp, d_z, B, N, d_cost, d_collide, d_grad, st);
}

static int uam_score_paths_raster_impl(uam_ctx* ctx, const double* d_z, int64_t B, int N, const double* h_p, int n_p, int flags,
                                       double samples_per_cell, float* d_cost, uint8_t* d_collide, int64_t* d_nsamples,
                                       bool want_best, int64_t global_offset, uint64_t* d_key, void* stream) {
    if (!ctx) return UAM_ERR_INVALID;
    UamRasterParams rp;
    UAM_TRY(uam_raster_prepare(ctx, B, N, h_p, n_p, flags, samples_per_cell, &rp));
    if (want_best && (!d_key || global_offset < 0 || global_offset + B > 0x7fffffffll))
        return uam_fail(ctx, UAM_ERR_INVALID, "best key: NULL pointer or global path index beyond 31 bits");
    if (B > 0 && !d_z) return uam_fail(ctx, UAM_ERR_INVALID, "paths pointer is NULL");
    UAM_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = uam_pick_stream(ctx, stream);
    UamBestTail tl;
    if (want_best) UAM_TRY(uam_best_tail(ctx, 0, (unsigned long long)global_offset, (unsigned long long*)d_key, true, false, &tl));
    if (B == 0) {
        // an empty shard still takes part in the exchange (its key is "no candidate")
        if (want_best) UAM_TRY(uam_best_launch(ctx, nullptr, 0, 0, tl, st));
        return UAM_OK;
    }
    UAM_TRY(uam_raster_precompute(ctx, &rp, B, N, st));
    return uam_raster_launch(ctx, d_z, B, N, rp, d_cost, d_collide, (long long*)d_nsamples, st, 0, want_best ? &tl : nullptr);
}

extern "C" int uam_score_paths_raster(uam_ctx* ctx, const double* d_z, int64_t B, int N, const double* h_p, int n_p,
                                      int flags, double samples_per_cell, float* d_cost, uint8_t* d_collide,
                                      int64_t* d_nsamples, void* stream) {
    return uam_score_paths_raster_impl(ctx, d_z, B, N, h_p, n_p, flags, samples_per_cell, d_cost, d_collide, d_nsamples, false, 0,
                                       nullptr, stream);
}

extern "C" int uam_score_paths_raster_best(uam_ctx* ctx, const double* d_z, int64_t B, int N, const double* h_p, int n_p,
                                           int flags, double samples_per_cell, float* d_cost, uint8_t* d_collide,
                                           int64_t global_offset, uint64_t* d_key, void* stream) {
    return uam_score_paths_raster_impl(ctx, d_z, B, N, h_p, n_p, flags, samples_per_cell, d_cost, d_collide, nullptr, true,
                                       global_offset, d_key, stream);
}

// ---- asynchronous host-buffer scoring -------------------------------------------------------------------------------
// A ring of UAM_HOST_PIPE_DEPTH slots, each with its own stream, staging and scratch: submit() queues the upload of the
// caller's (pinned) buffers, the whole-batch scoring pipeline and the download of the results on the slot's stream and
// returns a ticket; wait() blocks until that slot is done.  With two submissions in flight the upload of step s+1 overlaps
// the kernels of step s, so a stream of host-buffer batches runs at max(PCIe time, kernel time) per batch, and every batch
// is binned whole (the chunked synchronous call re-streams the raster through L2 once per chunk).
static int uam_ring_acquire(uam_ctx* ctx, int* slot) {
    const int s = ctx->ring_next;
    if (ctx->ring_busy[s]) {
        UAM_CUDA(ctx, cudaStreamSynchronize(ctx->pipe_stream[s]));      // the oldest ticket: its results are complete now
        ctx->ring_busy[s] = false;
    }
    ctx->ring_next = (s + 1) % UAM_HOST_PIPE_DEPTH;
    if (!ctx->d_ring_key[s]) UAM_CUDA(ctx, cudaMalloc(&ctx->d_ring_key[s], 8));
    *slot = s;
    return UAM_OK;
}

static int uam_raster_submit_impl(uam_ctx* ctx, const double* h_z, const double* h_cand, double jitter_sigma, uint64_t seed,
                                  int64_t B, int N, const double* h_p, int n_p, int flags, double spc, float* h_cost,
                                  uint8_t* h_collide, uint64_t* h_key, int64_t global_offset, int* ticket) {
    if (!ctx) return UAM_ERR_INVALID;
    if (!ticket) return uam_fail(ctx, UAM_ERR_INVALID, "ticket pointer is NULL");
    *ticket = -1;
    UamRasterParams rp;
    UAM_TRY(uam_raster_prepare(ctx, B, N, h_p, n_p, flags, spc, &rp));
    if (B > 0 && !h_z && !h_cand) return uam_fail(ctx, UAM_ERR_INVALID, "paths / candidates pointer is NULL");
    if (h_cand && !(jitter_sigma >= 0.0)) return uam_fail(ctx, UAM_ERR_INVALID, "jitter sigma must be >= 0");
    if (global_offset < 0 || global_offset + B > 0x7fffffffll)
        return uam_fail(ctx, UAM_ERR_UNSUPPORTED, "global path index must fit 31 bits");
    UAM_CUDA(ctx, cudaSetDevice(ctx->device));
    UAM_NVTX("uam.raster.submit (upload -> score -> download)");
    int s;
    UAM_TRY(uam_ring_acquire(ctx, &s));
    cudaStream_t st = ctx->pipe_stream[s];
    *ticket = s;
    ctx->ring_busy[s] = true;
    UamBestTail tl;
    // the exchange with the peer ranks is for caller-stream calls (uam_score_paths_raster_best): here the key is this rank's
    if (h_key) UAM_TRY(uam_best_tail(ctx, 1 + s, (unsigned long long)global_offset, ctx->d_ring_key[s], false, false, &tl));
    if (B == 0) {
        if (h_key) *h_key = UAM_KEY_EMPTY;
        return UAM_OK;
    }
    const size_t row = (size_t)2 * (N + 2) * sizeof(double);
    UAM_TRY(uam_reserve(ctx, &ctx->d_stage_in[s], &ctx->stage_in_bytes[s], (size_t)B * row));
    UAM_TRY(uam_reserve(ctx, &ctx->d_stage_out[s], &ctx->stage_out_bytes[s], (size_t)B * 8));
    float* d_cost = (float*)ctx->d_stage_out[s];
    uint8_t* d_col = (uint8_t*)(d_cost + B);
    // the quad texels are shared by all slots: (re)built here, before anything of this submission is queued
    UAM_TRY(uam_raster_precompute(ctx, &rp, B, N, st));
    if (h_cand) {
        UAM_TRY(uam_reserve(ctx, &ctx->d_ring_cand[s], &ctx->ring_cand_bytes[s], (size_t)B * 5 * sizeof(double)));
        UAM_CUDA(ctx, cudaMemcpyAsync(ctx->d_ring_cand[s], h_cand, (size_t)B * 5 * sizeof(double), cudaMemcpyHostToDevice, st));
        UAM_TRY(uam_make_candidates_launch(ctx, (const double*)ctx->d_ring_cand[s], nullptr, nullptr, N, B, jitter_sigma, seed,
                                           (uint64_t)global_offset, (double*)ctx->d_stage_in[s], st));
    } else {
        UAM_CUDA(ctx, cudaMemcpyAsync(ctx->d_stage_in[s], h_z, (size_t)B * row, cudaMemcpyHostToDevice, st));
    }
    // kernels of consecutive submissions run one after the other (two binned pipelines side by side would halve each
    // other's L2): this slot's kernels wait for the previous submission's, while its upload above and the previous
    // submission's download below overlap them on the copy engines
    if (ctx->ring_last >= 0 && ctx->ring_last != s) UAM_CUDA(ctx, cudaStreamWaitEvent(st, ctx->pipe_event[ctx->ring_last], 0));
    UAM_TRY(uam_raster_launch(ctx, (const double*)ctx->d_stage_in[s], B, N, rp, d_cost, d_col, nullptr, st, 1 + s, h_key ? &tl : nullptr));
    UAM_CUDA(ctx, cudaEventRecord(ctx->pipe_event[s], st));
    ctx->ring_last = s;
    if (h_cost) UAM_CUDA(ctx, cudaMemcpyAsync(h_cost, d_cost, (size_t)B * 4, cudaMemcpyDeviceToHost, st));
    if (h_collide) UAM_CUDA(ctx, cudaMemcpyAsync(h_collide, d_col, (size_t)B, cudaMemcpyDeviceToHost, st));
    if (h_key) UAM_CUDA(ctx, cudaMemcpyAsync(h_key, ctx->d_ring_key[s], 8, cudaMemcpyDeviceToHost, st));
    return UAM_OK;
}

extern "C" int uam_raster_submit_paths_host(uam_ctx* ctx, const double* h_z, int64_t B, int N, const double* h_p, int n_p,
                                            int flags, double samples_per_cell, float* h_cost, uint8_t* h_collide,
                                            uint64_t* h_key, int64_t global_offset, int* ticket) {
    return uam_raster_submit_impl(ctx, h_z, nullptr, 0.0, 0, B, N, h_p, n_p, flags, samples_per_cell, h_cost, h_collide, h_key,
                                  global_offset, ticket);
}

extern "C" int uam_raster_submit_candidates_host(uam_ctx* ctx, const double* h_cand, int64_t B, int N, double jitter_sigma,
                                                 uint64_t seed, const double* h_p, int n_p, int flags, double samples_per_cell,
                                                 float* h_cost, uint8_t* h_collide, uint64_t* h_key, int64_t global_offset,
                                                 int* ticket) {
    return uam_raster_submit_impl(ctx, nullptr, h_cand, jitter_sigma, seed, B, N, h_p, n_p, flags, samples_per_cell, h_cost,
                                  h_collide, h_key, global_offset, ticket);
}

extern "C" int uam_raster_wait(uam_ctx* ctx, int ticket) {
    if (!ctx) return UAM_ERR_INVALID;
    if (ticket < 0 || ticket >= UAM_HOST_PIPE_DEPTH) return uam_fail(ctx, UAM_ERR_INVALID, "bad ticket %d", ticket);
    if (!ctx->ring_busy[ticket]) return UAM_OK;             // already waited for (or reclaimed by a later submission)
    UAM_NVTX("uam.raster.wait");
    UAM_CUDA(ctx, cudaSetDevice(ctx->device));
    UAM_CUDA(ctx, cudaStreamSynchronize(ctx->pipe_stream[ticket]));
    ctx->ring_busy[ticket] = false;
    return UAM_OK;
}

// Host buffers in, host buffers out: the batch is cut into chunks that flow through UAM_HOST_PIPE_DEPTH
// streams (H2D copy of chunk c+1 overlaps the scoring of chunk c and the D2H copy of chunk c-1).
extern "C" int uam_score_paths_raster_host(uam_ctx* ctx, const double* h_z, int64_t B, int N, const double* h_p,
                                           int n_p, int flags, double samples_per_cell, float* h_cost,
                                           uint8_t* h_collide) {
    if (!ctx) return UAM_ERR_INVALID;
    UamRasterParams rp;
    UAM_TRY(uam_raster_prepare(ctx, B, N, h_p, n_p, flags, samples_per_cell, &rp));
    if (B == 0) return UAM_OK;
    if (!h_z) return uam_fail(ctx, UAM_ERR_INVALID, "paths pointer is NULL");
    UAM_CUDA(ctx, cudaSetDevice(ctx->device));
    UAM_CUDA(ctx, cudaDeviceSynchronize());
    UAM_TRY(uam_raster_precompute(ctx, &rp, B, N, ctx->pipe_stream[0]));
    const size_t row = (size_t)2 * (N + 2) * sizeof(double);
    // The pipeline is bound by the kernels (a chunk scores a little slower than it uploads: binning a quarter of the batch
    // streams the raster through L2 once more), so a call lasts about upload(first chunk) + sum of the kernel times.
    // Chunk sizes may change linearly from the first to the last chunk (taper > 0: shrinking, < 0: growing).
    // default: 4 chunks, fewer for small batches (a chunk under ~16 MB of waypoints costs more in launches than its upload hides)
    const int64_t by_bytes = std::max<int64_t>(1, (int64_t)((size_t)B * row / (16u << 20)));
    const int n_chunks = (int)std::min<int64_t>(ctx->host_chunks > 0 ? ctx->host_chunks : std::min<int64_t>(4, by_bytes),
                                                std::max<int64_t>(1, B / 1024));
    const double taper = ctx->host_taper / 100.0;
    auto weight = [&](int c) {
        const double x = n_chunks > 1 ? (double)c / (n_chunks - 1) : 0.0;
        return taper >= 0.0 ? 1.0 - taper * x : 1.0 + taper * (1.0 - x);
    };
    const int64_t max_rows = std::max<int64_t>(1024, (int64_t)((96u << 20) / row));
    std::vector<int64_t> bounds(1, 0);
    {
        double wsum = 0.0, acc = 0.0;
        for (int c = 0; c < n_chunks; ++c) wsum += weight(c);
        for (int c = 0; c < n_chunks; ++c) {
            acc += weight(c) / wsum;
            int64_t e = c + 1 == n_chunks ? B : std::min<int64_t>(B, (int64_t)(acc * (double)B));
            while (e - bounds.back() > max_rows) bounds.push_back(bounds.back() + max_rows);   // staging stays bounded
            if (e > bounds.back()) bounds.push_back(e);
        }
    }
    int64_t chunk = 0;
    for (size_t c = 0; c + 1 < bounds.size(); ++c) chunk = std::max(chunk, bounds[c + 1] - bounds[c]);
    for (size_t c = 0; c + 1 < bounds.size(); ++c) {
        const int s = (int)(c % UAM_HOST_PIPE_DEPTH);
        const int64_t b0 = bounds[c], nb = bounds[c + 1] - bounds[c];
        cudaStream_t st = ctx->pipe_stream[s];
        UAM_TRY(uam_reserve(ctx, &ctx->d_stage_in[s], &ctx->stage_in_bytes[s], (size_t)chunk * row));
        UAM_TRY(uam_reserve(ctx, &ctx->d_stage_out[s], &ctx->stage_out_bytes[s], (size_t)chunk * 8));
        float* d_cost = (float*)ctx->d_stage_out[s];
        uint8_t* d_col = (uint8_t*)(d_cost + chunk);
        UAM_CUDA(ctx, cudaMemcpyAsync(ctx->d_stage_in[s], (const char*)h_z + (size_t)b0 * row, (size_t)nb * row,
                                      cudaMemcpyHostToDevice, st));
        UAM_TRY(uam_raster_launch(ctx, (const double*)ctx->d_stage_in[s], nb, N, rp, d_cost, d_col, nullptr, st, 1 + s));
        if (h_cost) UAM_CUDA(ctx, cudaMemcpyAsync(h_cost + b0, d_cost, (size_t)nb * 4, cudaMemcpyDeviceToHost, st));
        if (h_collide) UAM_CUDA(ctx, cudaMemcpyAsync(h_collide + b0, d_col, (size_t)nb, cudaMemcpyDeviceToHost, st));
    }
    for (int s = 0; s < UAM_HOST_PIPE_DEPTH; ++s) UAM_CUDA(ctx, cudaStreamSynchronize(ctx->pipe_stream[s]));
    return UAM_OK;
}
