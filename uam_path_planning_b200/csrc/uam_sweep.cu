// Swept check of whole path segments against the raster's occupancy, and each path's clearance
// (uam_sweep_paths_raster; include/uam_b200.h has the definition).
//
// Fixed point: a pixel coordinate U becomes Uq = rint(U 2^16) (int64, |Uq| <= 2^47).  The box of cell m dilated by one
// quantum is [m 2^16 - 2^15 - 1, m 2^16 + 2^15 + 1] on either axis.
//
// Kernel: warp per path.  A segment is walked strip by strip along its major axis (u when |dVq| <= |dUq|, else v): strip m
// is the part of the segment inside the dilated slab of column (row) m, and its minor range touches 1 - 3 rows (columns).
// Only strips of raster columns (rows) are listed, so a segment from far outside costs at most max(H, W) strips.  The
// path's strips are flattened (segment k owns the flat indices [P_k, P_{k+1})) and the lanes stride the flat index, as in
// the scorer's variant 0.  A strip's minor range is estimated in fp64 and an exact 128-bit sign test decides a row only
// when the estimate lies within one quantum of that row's box edge (uam_sweep_row_lo / uam_sweep_row_hi).
#include <algorithm>
#include <climits>

#include "uam_internal.cuh"

#define UAM_SWEEP_HALF 32769ll        // half a cell + one quantum, in quanta
#define UAM_SWEEP_D2_CLIP 65535
#define UAM_SWEEP_SMEM_BUDGET (200 * 1024)

namespace {

// Per-warp segment table in shared memory: segment k in its strip frame (major start a, minor start b, major extent
// da >= 0, minor extent db, |db| <= da, slope db / da), its first strip, whether major = v, and the exclusive prefix of the
// strip counts.
__host__ __device__ inline size_t uam_sweep_table_bytes(int n) {
    return ((size_t)n * 56 + 8 + 15) & ~(size_t)15;
}

struct UamSweepSeg {
    long long a, b, da, db;
    double slope;
    int m0, steep;
};

struct UamSweepArgs {
    double x0, dx, y0, dy;
    int H, W;
    const unsigned* occ_bits;     // uam_ensure_occ_bits
    unsigned blocks_x;
    const unsigned short* d2;     // min(EDT d^2, 65535), (H, W) row-major; NULL: no clearance
};

// sign of a b - c d, exact while both products stay below 2^126 in magnitude
__device__ __forceinline__ int uam_sign_det(long long a, long long b, long long c, long long d) {
    const unsigned long long l1 = (unsigned long long)a * (unsigned long long)b, l2 = (unsigned long long)c * (unsigned long long)d;
    const long long hi = __mul64hi(a, b) - __mul64hi(c, d) - (l1 < l2 ? 1ll : 0ll);
    const unsigned long long lo = l1 - l2;
    return hi < 0 ? -1 : ((hi != 0 || lo != 0) ? 1 : 0);
}

// sign of c - w(x), w(x) = b + db (x - a) / da the exact minor coordinate of the segment's line at major coordinate x
// (da = 0 only for a point, where db = 0 and x = a)
__device__ __forceinline__ int uam_sweep_side(const UamSweepSeg& s, long long c, long long x) {
    return uam_sign_det(c - s.b, s.da > 0 ? s.da : 1ll, s.db, x - s.a);
}

// The fp64 estimate of w(x) = b + slope (x - a): x - a <= 2^48 and b are exact doubles and |slope| <= 1 is within 2^-53 of
// db / da, so the slope's error, the product's and the sum's (on magnitudes below 2^49) add up to at most
// 2^-5 + 2^-5 + 2^-4 = 2^-3 quantum.
__device__ __forceinline__ double uam_sweep_minor(const UamSweepSeg& s, long long x) {
    return __dadd_rn((double)s.b, __dmul_rn(s.slope, (double)(x - s.a)));
}

// Lowest row whose dilated box reaches down to w(x): its top edge i 2^16 + HALF >= w(x).  From the estimate we, i satisfies
// e(i - 1) < we <= e(i) (e = the top edge); the true w(x) is within 2^-3 of we, so the answer moves off i only when we is
// within one quantum of e(i - 1) or e(i), and one exact test decides it.
__device__ __forceinline__ long long uam_sweep_row_lo(const UamSweepSeg& s, long long x) {
    const double we = uam_sweep_minor(s, x);
    long long i = (long long)ceil(__dmul_rn(__dsub_rn(we, (double)UAM_SWEEP_HALF), 1.0 / 65536.0));
    const long long below = (i - 1) * 65536 + UAM_SWEEP_HALF, above = i * 65536 + UAM_SWEEP_HALF;
    if (__dsub_rn(we, (double)below) < 1.0) {
        if (uam_sweep_side(s, below, x) >= 0) --i;
    } else if (__dsub_rn((double)above, we) < 1.0) {
        if (uam_sweep_side(s, above, x) < 0) ++i;
    }
    return i;
}

// Highest row whose dilated box reaches up to w(x): its bottom edge i 2^16 - HALF <= w(x); the same correction.
__device__ __forceinline__ long long uam_sweep_row_hi(const UamSweepSeg& s, long long x) {
    const double we = uam_sweep_minor(s, x);
    long long i = (long long)floor(__dmul_rn(__dadd_rn(we, (double)UAM_SWEEP_HALF), 1.0 / 65536.0));
    const long long here = i * 65536 - UAM_SWEEP_HALF, next = (i + 1) * 65536 - UAM_SWEEP_HALF;
    if (__dsub_rn(we, (double)here) < 1.0) {
        if (uam_sweep_side(s, here, x) > 0) --i;
    } else if (__dsub_rn((double)next, we) < 1.0) {
        if (uam_sweep_side(s, next, x) <= 0) ++i;
    }
    return i;
}

__device__ __forceinline__ long long uam_q16(double u) { return __double2ll_rn(__dmul_rn(u, 65536.0)); }

__global__ void __launch_bounds__(UAM_CTA_THREADS)
uam_k_sweep_paths(const double2* __restrict__ z, long long B, int Wp, UamSweepArgs g, uint8_t* __restrict__ flags,
                  int* __restrict__ first_hit, int* __restrict__ d2min) {
    extern __shared__ __align__(16) unsigned char uam_sweep_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wpc = blockDim.x >> 5;
    const int n = Wp - 1;
    long long* const A = reinterpret_cast<long long*>(uam_sweep_smem + (size_t)warp * uam_sweep_table_bytes(n));
    long long* const Bm = A + n;
    long long* const DA = Bm + n;
    long long* const DB = DA + n;
    double* const SL = reinterpret_cast<double*>(DB + n);
    long long* const P = reinterpret_cast<long long*>(SL + n);      // n + 1 entries
    int* const M0 = reinterpret_cast<int*>(P + n + 1);
    int* const ST = M0 + n;
    const long long nwarps = (long long)gridDim.x * wpc;
    for (long long path = (long long)blockIdx.x * wpc + warp; path < B; path += nwarps) {
        const double2* zp = z + path * Wp;
        // A: validity and the outside flag, per waypoint
        bool bad = false, out = false;
        for (int j = lane; j < Wp; j += 32) {
            const double2 p = zp[j];
            const double U = uam_pix(p.x, g.x0, g.dx), V = uam_pix(p.y, g.y0, g.dy);
            bad = bad || !(fabs(U) < 2147483648.0 && fabs(V) < 2147483648.0);
            out = out || !(U >= -0.5 && U <= g.W - 0.5 && V >= -0.5 && V <= g.H - 0.5);
        }
        bad = __any_sync(0xffffffffu, bad);
        out = __any_sync(0xffffffffu, out);
        if (bad) {
            if (lane == 0) {
                flags[path] = UAM_SWEEP_INVALID;
                if (first_hit) first_hit[path] = -1;
                if (d2min) d2min[path] = -1;
            }
            continue;
        }
        // B: every segment in its strip frame, its strips clipped to the raster, the exclusive prefix of the counts
        long long carry = 0;
        for (int k0 = 0; k0 < n; k0 += 32) {
            const int k = k0 + lane;
            long long S = 0;
            if (k < n) {
                const double2 p = zp[k], q = zp[k + 1];
                const long long u0 = uam_q16(uam_pix(p.x, g.x0, g.dx)), v0 = uam_q16(uam_pix(p.y, g.y0, g.dy));
                const long long u1 = uam_q16(uam_pix(q.x, g.x0, g.dx)), v1 = uam_q16(uam_pix(q.y, g.y0, g.dy));
                const long long du = u1 - u0, dv = v1 - v0;
                const bool steep = llabs(dv) > llabs(du);
                long long a = steep ? v0 : u0, b = steep ? u0 : v0, da = steep ? dv : du, db = steep ? du : dv;
                if (da < 0) { a += da; b += db; da = -da; db = -db; }
                const long long m_first = max(-((UAM_SWEEP_HALF - a) >> 16), 0ll);        // ceil((a - HALF) / 2^16)
                const long long m_last = min((a + da + UAM_SWEEP_HALF) >> 16, (long long)(steep ? g.H : g.W) - 1);
                S = m_last >= m_first ? m_last - m_first + 1 : 0;
                A[k] = a; Bm[k] = b; DA[k] = da; DB[k] = db;
                SL[k] = da > 0 ? __ddiv_rn((double)db, (double)da) : 0.0;
                M0[k] = S ? (int)m_first : 0;
                ST[k] = steep ? 1 : 0;
            }
            long long incl = S;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const long long t = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += t;
            }
            if (k < n) P[k] = carry + incl - S;
            carry += __shfl_sync(0xffffffffu, incl, 31);
        }
        if (lane == 0) P[n] = carry;
        __syncwarp();
        // C: flat strip loop
        const long long T = carry;
        int hitk = INT_MAX, dmin = INT_MAX;
        int k = 0;
        long long pk = 0, p1 = P[1];
        UamSweepSeg s = {A[0], Bm[0], DA[0], DB[0], SL[0], M0[0], ST[0]};
        for (long long t0 = 0; t0 < T; t0 += 32) {
            const long long t = t0 + lane;
            if (t < T) {
                if (t >= p1) {
                    do { ++k; p1 = P[k + 1]; } while (t >= p1);
                    pk = P[k];
                    s = {A[k], Bm[k], DA[k], DB[k], SL[k], M0[k], ST[k]};
                }
                const long long m = s.m0 + (t - pk);
                const long long xl = max(m * 65536 - UAM_SWEEP_HALF, s.a), xh = min(m * 65536 + UAM_SWEEP_HALF, s.a + s.da);
                const long long i0 = max(uam_sweep_row_lo(s, s.db >= 0 ? xl : xh), 0ll);
                const long long i1 = min(uam_sweep_row_hi(s, s.db >= 0 ? xh : xl), (long long)(s.steep ? g.W : g.H) - 1);
                for (long long i = i0; i <= i1; ++i) {
                    const unsigned r = (unsigned)(s.steep ? m : i), c = (unsigned)(s.steep ? i : m);
                    const unsigned w = __ldg(g.occ_bits + uam_occ_word(r, c, g.blocks_x));
                    if (((w >> uam_occ_bit(r, c)) & 1u) && hitk == INT_MAX) hitk = k;
                    if (g.d2) dmin = min(dmin, (int)__ldg(g.d2 + (size_t)r * g.W + c));
                }
            }
            // without the clearance the walk ends at the first window with a hit: later windows hold later segments only
            if (!g.d2 && __any_sync(0xffffffffu, hitk != INT_MAX)) break;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            hitk = min(hitk, __shfl_xor_sync(0xffffffffu, hitk, o));
            dmin = min(dmin, __shfl_xor_sync(0xffffffffu, dmin, o));
        }
        if (lane == 0) {
            flags[path] = (uint8_t)((hitk != INT_MAX ? UAM_SWEEP_HIT : 0) | (out ? UAM_SWEEP_OUTSIDE : 0));
            if (first_hit) first_hit[path] = hitk != INT_MAX ? hitk : -1;
            if (d2min) d2min[path] = dmin != INT_MAX ? dmin : -1;
        }
        __syncwarp();                              // the table is rewritten for the next path
    }
}

// occupancy bytes (H, W) from the bit-plane: the input of uam_edt
__global__ void uam_k_occ_bytes(const unsigned* __restrict__ bits, unsigned blocks_x, int H, int W, uint8_t* __restrict__ occ) {
    const size_t n = (size_t)H * W, stride = (size_t)gridDim.x * blockDim.x;
    for (size_t o = (size_t)blockIdx.x * blockDim.x + threadIdx.x; o < n; o += stride) {
        const unsigned i = (unsigned)(o / W), j = (unsigned)(o - (size_t)i * W);
        occ[o] = (uint8_t)((__ldg(bits + uam_occ_word(i, j, blocks_x)) >> uam_occ_bit(i, j)) & 1u);
    }
}

__global__ void uam_k_clip_d2(const int* __restrict__ d2, size_t n, unsigned short* __restrict__ out) {
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t o = (size_t)blockIdx.x * blockDim.x + threadIdx.x; o < n; o += stride)
        out[o] = (unsigned short)min(d2[o], UAM_SWEEP_D2_CLIP);
}

// min(EDT d^2, 65535) of the current raster, built once per upload.  The occupancy bytes and the int32 d^2 (5 B per cell)
// and uam_edt's own scratch (what this build adds to ctx->d_scratch) are freed again; the field itself is 2 B per cell.
int uam_sweep_ensure_d2(uam_ctx* ctx, cudaStream_t st) {
    if (ctx->sweep_d2_gen == ctx->raster_gen) return UAM_OK;
    UAM_NVTX("uam.raster.sweep.build_d2");
    const int H = ctx->geo.H, W = ctx->geo.W;
    const size_t n = (size_t)H * W, occ_bytes = (n + 255) & ~(size_t)255;
    UAM_CUDA(ctx, cudaDeviceSynchronize());        // a sweep on another stream may still read the old field
    UAM_TRY(uam_reserve(ctx, &ctx->d_sweep_d2, &ctx->sweep_d2_bytes, n * 2));
    void* tmp = nullptr;
    UAM_CUDA(ctx, cudaMalloc(&tmp, occ_bytes + n * 4));
    uint8_t* occ = (uint8_t*)tmp;
    int* d2 = (int*)((char*)tmp + occ_bytes);
    const size_t scratch_before = ctx->scratch_bytes;
    auto build = [&]() -> int {
        const unsigned grid = (unsigned)std::min<size_t>((n + 255) / 256, (size_t)ctx->sm_count * 16);
        uam_k_occ_bytes<<<grid, 256, 0, st>>>((const unsigned*)ctx->d_occ_bits + 4, (unsigned)(W + 31) / 32u, H, W, occ);
        UAM_CHECK_LAUNCH(ctx, "uam_k_occ_bytes");
        UAM_TRY(uam_edt(ctx, occ, H, W, 1.0, d2, nullptr, st));
        uam_k_clip_d2<<<grid, 256, 0, st>>>(d2, n, (unsigned short*)ctx->d_sweep_d2);
        UAM_CHECK_LAUNCH(ctx, "uam_k_clip_d2");
        UAM_CUDA(ctx, cudaStreamSynchronize(st));
        return UAM_OK;
    };
    const int rc = build();
    cudaStreamSynchronize(st);
    cudaFree(tmp);
    if (ctx->scratch_bytes > scratch_before) {
        cudaFree(ctx->d_scratch);
        ctx->d_scratch = nullptr;
        ctx->scratch_bytes = 0;
    }
    if (rc == UAM_OK) ctx->sweep_d2_gen = ctx->raster_gen;
    return rc;
}

}  // namespace

extern "C" int uam_sweep_paths_raster(uam_ctx* ctx, const double* d_z, int64_t B, int N, uint8_t* d_flags, int32_t* d_first_hit,
                                      int32_t* d_d2min, void* stream) {
    if (!ctx) return UAM_ERR_INVALID;
    if (B < 0 || N < 0) return uam_fail(ctx, UAM_ERR_INVALID, "need B >= 0 and N >= 0 (got B=%lld N=%d)", (long long)B, N);
    if (B == 0) return UAM_OK;
    if (!d_z || !d_flags) return uam_fail(ctx, UAM_ERR_INVALID, "paths or flags pointer is NULL");
    if (!ctx->has_raster) return uam_fail(ctx, UAM_ERR_STATE, "no raster: call uam_map_set_raster first");
    if (d_d2min && (ctx->geo.H > 23170 || ctx->geo.W > 23170))
        return uam_fail(ctx, UAM_ERR_UNSUPPORTED, "clearance needs a raster of at most 23170 cells per side (uam_edt's limit)");
    const size_t per_warp = uam_sweep_table_bytes((int)std::min<long long>((long long)N + 1, 1 << 24));
    if (per_warp > UAM_SWEEP_SMEM_BUDGET) return uam_fail(ctx, UAM_ERR_UNSUPPORTED, "N = %d waypoints per path is too many", N);
    UAM_NVTX("uam.raster.sweep");
    UAM_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = uam_pick_stream(ctx, stream);
    UAM_TRY(uam_ensure_occ_bits(ctx, st));
    if (d_d2min) UAM_TRY(uam_sweep_ensure_d2(ctx, st));
    UamSweepArgs g;
    g.x0 = ctx->geo.x0; g.dx = ctx->geo.dx; g.y0 = ctx->geo.y0; g.dy = ctx->geo.dy;
    g.H = ctx->geo.H; g.W = ctx->geo.W;
    g.occ_bits = (const unsigned*)ctx->d_occ_bits + 4;
    g.blocks_x = (unsigned)(g.W + 31) / 32u;
    g.d2 = d_d2min ? (const unsigned short*)ctx->d_sweep_d2 : nullptr;
    const int wpc = (int)std::max<size_t>(1, std::min<size_t>(UAM_WARPS_PER_CTA, UAM_SWEEP_SMEM_BUDGET / per_warp));
    const size_t smem = per_warp * wpc;
    const long long ctas = std::min<long long>((B + wpc - 1) / wpc, (long long)ctx->sm_count * 16);
    if (smem > 48 * 1024) UAM_CUDA(ctx, cudaFuncSetAttribute(uam_k_sweep_paths, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    uam_k_sweep_paths<<<(unsigned)ctas, wpc * 32, smem, st>>>(reinterpret_cast<const double2*>(d_z), B, N + 2, g, d_flags,
                                                              d_first_hit, d_d2min);
    UAM_CHECK_LAUNCH(ctx, "uam_k_sweep_paths");
    return UAM_OK;
}
