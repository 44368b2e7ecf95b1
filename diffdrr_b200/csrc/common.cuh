// common.cuh -- shared helpers for the sm_100a DRR kernels.
//
// The per-ray math (ray_math.cuh) is written as host+device functions so that tests/hostemu can compile the very
// same source with g++ and check it against the oracle in the CPU-only container.  That emulation is test
// infrastructure; the product library contains device code only and has no CPU path.
#pragma once

#include <math.h>
#include <stdint.h>

#if defined(__CUDACC__)
#include <cuda_runtime.h>
#define B200_HD __host__ __device__ __forceinline__
#else
#define B200_HD inline
struct float4 {  // host emulation only (tests/hostemu): the CUDA headers provide it for device builds
    float x, y, z, w;
};
#endif

namespace b200drr {

constexpr int kWarp = 32;

struct VolDims {
    int d[3];
};

B200_HD float ldg(const float* p)
{
#if defined(__CUDA_ARCH__)
    return __ldg(p);  // (an L2::256B prefetch hint was measured: no effect, L2 already hits 80 %)
#else
    return *p;
#endif
}

// single-rounding multiply / add that the compiler may not contract into an fma
B200_HD float mul_rn(float a, float b)
{
#if defined(__CUDA_ARCH__)
    return __fmul_rn(a, b);
#else
    volatile float r = a * b;
    return r;
#endif
}
B200_HD float add_rn(float a, float b)
{
#if defined(__CUDA_ARCH__)
    return __fadd_rn(a, b);
#else
    volatile float r = a + b;
    return r;
#endif
}

// A pair of floats updated by one packed f32x2 instruction on sm_100a (FADD2 / FMUL2 / FFMA2: both lanes rounded exactly
// as the scalar add.rn / mul.rn / fma.rn); two scalar operations in the host emulation, which is compiled without contraction.
#if defined(__CUDACC__)
using Pair = float2;
#else
struct Pair {
    float x, y;
};
#endif
B200_HD Pair add2_rn(Pair a, Pair b)
{
#if defined(__CUDA_ARCH__)
    return __fadd2_rn(a, b);
#else
    return Pair{a.x + b.x, a.y + b.y};
#endif
}
B200_HD Pair sub2_rn(Pair a, Pair b)
{
#if defined(__CUDA_ARCH__)
    return __fadd2_rn(a, make_float2(-b.x, -b.y));
#else
    return Pair{a.x - b.x, a.y - b.y};
#endif
}
B200_HD Pair mul2_rn(Pair a, Pair b)
{
#if defined(__CUDA_ARCH__)
    return __fmul2_rn(a, b);
#else
    return Pair{a.x * b.x, a.y * b.y};
#endif
}
B200_HD Pair fma2_rn(Pair a, Pair b, Pair c)
{
#if defined(__CUDA_ARCH__)
    return __ffma2_rn(a, b, c);
#else
    return Pair{fmaf(a.x, b.x, c.x), fmaf(a.y, b.y, c.y)};
#endif
}

// accumulate into the volume gradient: red.global.add.f32 on the device, plain add in the host emulation
B200_HD void red_add(float* addr, float v)
{
#if defined(__CUDA_ARCH__)
    asm volatile("red.global.add.f32 [%0], %1;" ::"l"(addr), "f"(v) : "memory");
#else
    *addr += v;
#endif
}

// One ray: d = (target - source) + eps (renderers.py:104-106), inv = 1/d.
struct Ray {
    float s[3];
    float d[3];
    float inv[3];
};

B200_HD Ray load_ray(const float* src, const float* tgt, int b, int64_t r, float eps)
{
    Ray ray;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        ray.s[a] = ldg(src + b * 3 + a);
        ray.d[a] = (ldg(tgt + r * 3 + a) - ray.s[a]) + eps;
        ray.inv[a] = 1.0f / ray.d[a];
    }
    return ray;
}

// alpha of plane i on axis a with the reference's own rounding sequence ((i - shift) - s) / d
B200_HD float plane_alpha(const Ray& ray, int a, float i, float shift) { return ((i - shift) - ray.s[a]) / ray.d[a]; }

#if defined(__CUDACC__)
__device__ __forceinline__ float warp_sum(float v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Block-wide sum of `v` (blockDim.x multiple of 32, <= 1024); result valid in thread 0.
__device__ __forceinline__ float block_sum(float v, float* smem /* >= 32 floats */)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    v = warp_sum(v);
    __syncthreads();  // protect smem reuse between consecutive calls
    if (lane == 0) smem[warp] = v;
    __syncthreads();
    const int nwarp = (blockDim.x + 31) >> 5;
    v = (threadIdx.x < nwarp) ? smem[threadIdx.x] : 0.0f;
    if (warp == 0) v = warp_sum(v);
    return v;
}

// Ray handled by this thread of a 128-thread CTA: row order (W == 0, any ray set) or, for a full detector grid of width W,
// a 16 x 8 pixel tile made of four 8 x 4 warp bundles (neighbouring rays gather neighbouring voxels).  -1 = no ray.
__device__ __forceinline__ int64_t tiled_ray_index(int64_t N, int W)
{
    if (W <= 0) {
        const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
        return n < N ? n : -1;
    }
    const int H = (int)(N / W), tiles_x = (W + 15) / 16;
    const int tile_x = blockIdx.x % tiles_x, tile_y = blockIdx.x / tiles_x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int px = tile_x * 16 + (warp & 1) * 8 + (lane & 7), py = tile_y * 8 + (warp >> 1) * 4 + (lane >> 3);
    return (px < W && py < H) ? (int64_t)py * W + px : -1;
}
inline dim3 tiled_ray_grid(int B, int64_t N, int W)
{
    if (W <= 0) return dim3((unsigned)((N + 127) / 128), (unsigned)B, 1);
    const int64_t H = N / W;
    return dim3((unsigned)(((W + 15) / 16) * ((H + 7) / 8)), (unsigned)B, 1);
}

// Optional in-kernel ray generation ("pose-in" entry points): when G != nullptr the rays of pose b are made from
//   target_voxel(h, w) = G[b] . (cols[w], rows[h], 1, 1),   raylen(h, w) = | Wd[b] . (cols[w], rows[h], 1, 1) |
// (G = affine_inverse . extrinsic . reorient . calibration, Wd = the same without affine_inverse and with the source
// subtracted; reference detector.py:144-154 + drr.py:201-205 collapsed into two 3x4 matrices per pose), so the
// (B, N, 3) target tensor and the ray-length image never exist in HBM.
struct PoseRays {
    const float* G;     // [B][3][4]
    const float* Wd;    // [B][3][4]
    const float* rows;  // [H]  canonical detector y of image row h   (detector.py:114-126)
    const float* cols;  // [W]  canonical detector x of image column w
};

__device__ __forceinline__ Ray make_ray(const PoseRays& pr, const float* __restrict__ src, const float* __restrict__ tgt,
                                        const float* __restrict__ raylen, int b, int64_t r, int px, int py, float eps,
                                        float& L)
{
    if (pr.G == nullptr) {
        L = __ldg(raylen + r);
        return load_ray(src, tgt, b, r, eps);
    }
    const float c = __ldg(pr.cols + px), rr = __ldg(pr.rows + py);
    const float* g = pr.G + b * 12;
    const float* wd = pr.Wd + b * 12;
    Ray ray;
    float l2 = 0.0f;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const float t = fmaf(__ldg(g + a * 4), c, fmaf(__ldg(g + a * 4 + 1), rr, __ldg(g + a * 4 + 2) + __ldg(g + a * 4 + 3)));
        const float dw = fmaf(__ldg(wd + a * 4), c, fmaf(__ldg(wd + a * 4 + 1), rr, __ldg(wd + a * 4 + 2) + __ldg(wd + a * 4 + 3)));
        l2 = fmaf(dw, dw, l2);
        ray.s[a] = __ldg(src + b * 3 + a);
        ray.d[a] = (t - ray.s[a]) + eps;
        ray.inv[a] = 1.0f / ray.d[a];
    }
    L = sqrtf(l2);
    return ray;
}
#endif

}  // namespace b200drr
