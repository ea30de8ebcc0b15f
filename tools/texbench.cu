// Microbenchmark: bilinear 2x2 footprint fetch of 3 layers + occupancy along random line segments, L2-resident working
// set: (a) 4 x LDG.128 from the tiled float4 texel array (the product's layout), (b) 4 x tex2Dgather on four R32F
// cudaArrays (texture units).  Prints samples/s for both.  nvcc -arch=sm_100a -O3 tools/texbench.cu -o /tmp/texbench
// Modes 5 and 6 do one load per tap of the weight-folded layer: (5) one LDG.128 of the tiled sign-packed quad (the 2 x 2
// footprint of a cell in one float4, the scorer's TF 8 form), (6) one tex2Dgather<uint4> of the footprint from an R32UI
// cudaArray (4 bytes per cell, block-linear; the TF 16 form).
#include <cstdio>
#include <cstdlib>
#include <vector>
#include <cuda_runtime.h>
#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { printf("%s: %s\n", #x, cudaGetErrorString(e)); exit(1); } } while (0)

__device__ __forceinline__ unsigned tex_index(unsigned i, unsigned j, unsigned row_stride) {
    return (i >> 1) * row_stride + ((i & 1u) << 1) + 2u * j - (j & 1u);
}

// each warp walks `iters` chunks of 32 consecutive samples along its own line inside a window of the raster
// unnormalised texture coordinate c + 1 as a float without the conversion unit (c < 2^23)
__device__ __forceinline__ float fcoord(int c) { return __int_as_float(0x4B000000 | (c + 1)) - 8388608.0f; }

template <int MODE>
__global__ void walk(const float4* __restrict__ tex, cudaTextureObject_t t0, cudaTextureObject_t t1, cudaTextureObject_t t2,
                     cudaTextureObject_t t3, cudaTextureObject_t tu, int n, int win, int iters, float* out) {
    const int lane = threadIdx.x & 31;
    const unsigned warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    unsigned s = warp * 2654435761u + 12345u;
    float acc = 0.f;
    for (int it = 0; it < iters; ++it) {
        s = s * 1664525u + 1013904223u;
        const float ang = (s >> 8) * (6.2831853f / 16777216.f);
        s = s * 1664525u + 1013904223u;
        const float bx = 40.f + (s >> 8) * ((win - 80.f) / 16777216.f);
        s = s * 1664525u + 1013904223u;
        const float by = 40.f + (s >> 8) * ((win - 80.f) / 16777216.f);
        const float u = bx + __cosf(ang) * lane, v = by + __sinf(ang) * lane;
        const int j0 = (int)u, i0 = (int)v;
        const float fx = u - j0, fy = v - i0;
        if (MODE == 5) {
            const unsigned rs = (n / 4) * 8;        // uam_quad_index<1>: (i >> 1) (rs - 4) + 2 (i + j) - (j & 1)
            const float4 q = __ldg(tex + ((unsigned)(i0 >> 1) * (rs - 4u) + ((unsigned)(i0 + j0) << 1) - (j0 & 1u)));
            const float top = fabsf(q.x) + fx * (fabsf(q.y) - fabsf(q.x)), bot = fabsf(q.z) + fx * (fabsf(q.w) - fabsf(q.z));
            acc += top + fy * (bot - top) + (__float_as_int(fy >= 0.5f ? q.z : q.x) < 0 ? 1.0f : 0.0f);
        } else if (MODE == 6) {
            // gather order: (x0,y1) (x1,y1) (x1,y0) (x0,y0)
            const uint4 g = tex2Dgather<uint4>(tu, fcoord(j0), fcoord(i0), 0);
            const float a = fabsf(__uint_as_float(g.w)), b = fabsf(__uint_as_float(g.z));
            const float c = fabsf(__uint_as_float(g.x)), d = fabsf(__uint_as_float(g.y));
            const float top = a + fx * (b - a), bot = c + fx * (d - c);
            acc += top + fy * (bot - top) + ((int)(fy >= 0.5f ? g.x : g.w) < 0 ? 1.0f : 0.0f);
        } else if (MODE == 0) {
            const unsigned rs = (n / 4) * 8;
            const float4 a = __ldg(tex + tex_index(i0, j0, rs)), b = __ldg(tex + tex_index(i0, j0 + 1, rs));
            const float4 c = __ldg(tex + tex_index(i0 + 1, j0, rs)), d = __ldg(tex + tex_index(i0 + 1, j0 + 1, rs));
            const float wa = (1 - fx) * (1 - fy), wb = fx * (1 - fy), wc = (1 - fx) * fy, wd = fx * fy;
            acc += wa * (a.x + a.y + a.z + a.w) + wb * (b.x + b.y + b.z + b.w) + wc * (c.x + c.y + c.z + c.w) + wd * (d.x + d.y + d.z + d.w);
        } else if (MODE >= 2) {
            const float wa = (1 - fx) * (1 - fy), wb = fx * (1 - fy), wc = (1 - fx) * fy, wd = fx * fy;
            if (MODE == 2 || MODE == 4) {       // float2 texels, 4 x 4 tiles
                const float2* t2 = reinterpret_cast<const float2*>(tex);
                const unsigned rs = (n / 4) * 16;
                auto idx = [rs](unsigned i, unsigned j) { return (i >> 2) * rs + ((i & 2u) << 2) + ((i & 1u) << 1) + ((j >> 2) << 4) + ((j & 2u) << 1) + (j & 1u); };
                const float2 a = __ldg(t2 + idx(i0, j0)), b = __ldg(t2 + idx(i0, j0 + 1)), c = __ldg(t2 + idx(i0 + 1, j0)), d = __ldg(t2 + idx(i0 + 1, j0 + 1));
                acc += wa * (a.x + a.y) + wb * (b.x + b.y) + wc * (c.x + c.y) + wd * (d.x + d.y);
            }
            if (MODE == 3 || MODE == 4) {
                const float x = j0 + 1.0f, y = i0 + 1.0f;
                const float4 g0 = tex2Dgather<float4>(t0, x, y, 0), g1 = tex2Dgather<float4>(t1, x, y, 0);
                acc += wa * (g0.w + g1.w) + wb * (g0.z + g1.z) + wc * (g0.x + g1.x) + wd * (g0.y + g1.y);
            }
        } else {
            const float x = j0 + 1.0f, y = i0 + 1.0f;
            const float4 g0 = tex2Dgather<float4>(t0, x, y, 0), g1 = tex2Dgather<float4>(t1, x, y, 0);
            const float4 g2 = tex2Dgather<float4>(t2, x, y, 0), g3 = tex2Dgather<float4>(t3, x, y, 0);
            // gather order: (x0,y1) (x1,y1) (x1,y0) (x0,y0)
            const float wa = (1 - fx) * (1 - fy), wb = fx * (1 - fy), wc = (1 - fx) * fy, wd = fx * fy;
            acc += wa * (g0.w + g1.w + g2.w + g3.w) + wb * (g0.z + g1.z + g2.z + g3.z) + wc * (g0.x + g1.x + g2.x + g3.x) +
                   wd * (g0.y + g1.y + g2.y + g3.y);
        }
    }
    if (acc == 123.456f) out[0] = acc;
}

int main(int argc, char** argv) {
    const int n = 8192, win = argc > 1 ? atoi(argv[1]) : 2048;      // window side: working set = win^2 * 16 B
    const size_t cells = (size_t)n * n;
    float4* tex;
    CK(cudaMalloc(&tex, cells * sizeof(float4)));
    CK(cudaMemset(tex, 0, cells * sizeof(float4)));
    cudaTextureObject_t to[4];
    cudaChannelFormatDesc desc = cudaCreateChannelDesc<float>();
    for (int k = 0; k < 4; ++k) {
        cudaArray_t arr;
        CK(cudaMallocArray(&arr, &desc, n, n, cudaArrayTextureGather));
        cudaResourceDesc rd = {};
        rd.resType = cudaResourceTypeArray;
        rd.res.array.array = arr;
        cudaTextureDesc td = {};
        td.addressMode[0] = td.addressMode[1] = cudaAddressModeClamp;
        td.filterMode = cudaFilterModePoint;
        td.readMode = cudaReadModeElementType;
        td.normalizedCoords = 0;
        CK(cudaCreateTextureObject(&to[k], &rd, &td, nullptr));
    }
    cudaTextureObject_t tu;
    {
        cudaChannelFormatDesc du = cudaCreateChannelDesc<unsigned>();
        cudaArray_t arr;
        CK(cudaMallocArray(&arr, &du, n, n, cudaArrayTextureGather));
        cudaResourceDesc rd = {};
        rd.resType = cudaResourceTypeArray;
        rd.res.array.array = arr;
        cudaTextureDesc td = {};
        td.addressMode[0] = td.addressMode[1] = cudaAddressModeClamp;
        td.filterMode = cudaFilterModePoint;
        td.readMode = cudaReadModeElementType;
        td.normalizedCoords = 0;
        CK(cudaCreateTextureObject(&tu, &rd, &td, nullptr));
    }
    float* out;
    CK(cudaMalloc(&out, 4));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, 0));
    printf("device %s, %d SMs, maxTexture2DGather %d x %d\n", prop.name, prop.multiProcessorCount, prop.maxTexture2DGather[0],
           prop.maxTexture2DGather[1]);
    const int blocks = 148 * 16, threads = 256, iters = 4000;
    const double samples = (double)blocks * threads * iters;
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    const char* names[7] = {"LDG.128 x4 (tiled float4)", "tex2Dgather x4 (R32F planes)", "LDG.64 x4 (tiled float2)", "tex2Dgather x2",
                            "LDG.64 x4 + tex2Dgather x2", "LDG.128 x1 (sign-packed quad)", "tex2Dgather<uint4> x1 (R32UI folded)"};
    const int mode0 = argc > 2 ? atoi(argv[2]) : 0;     // first mode to run (5: only the one-load-per-tap pair)
    for (int mode = mode0; mode < 7; ++mode) {
        for (int rep = 0; rep < 3; ++rep) {
            cudaEventRecord(e0);
            if (mode == 0) walk<0><<<blocks, threads>>>(tex, to[0], to[1], to[2], to[3], tu, n, win, iters, out);
            else if (mode == 1) walk<1><<<blocks, threads>>>(tex, to[0], to[1], to[2], to[3], tu, n, win, iters, out);
            else if (mode == 2) walk<2><<<blocks, threads>>>(tex, to[0], to[1], to[2], to[3], tu, n, win, iters, out);
            else if (mode == 3) walk<3><<<blocks, threads>>>(tex, to[0], to[1], to[2], to[3], tu, n, win, iters, out);
            else if (mode == 4) walk<4><<<blocks, threads>>>(tex, to[0], to[1], to[2], to[3], tu, n, win, iters, out);
            else if (mode == 5) walk<5><<<blocks, threads>>>(tex, to[0], to[1], to[2], to[3], tu, n, win, iters, out);
            else walk<6><<<blocks, threads>>>(tex, to[0], to[1], to[2], to[3], tu, n, win, iters, out);
            cudaEventRecord(e1);
            CK(cudaDeviceSynchronize());
            float ms;
            cudaEventElapsedTime(&ms, e0, e1);
            if (rep == 2) printf("win=%d mode=%s: %.3f ms, %.3e samples/s\n", win, names[mode], ms, samples / (ms * 1e-3));
        }
    }
    return 0;
}
