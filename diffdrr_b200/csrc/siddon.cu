// siddon.cu -- Siddon exact-path DRR kernels for sm_100a (forward, backward, visit counter).
// One thread walks one ray (ray_math.cuh); blockIdx.y is the pose, blockIdx.x tiles the rays of that pose.
#include <stdlib.h>

#include "kernels.h"
#ifdef B200DRR_EXPERIMENTS
#include "psync.cuh"  // rejected experiments live only in the opt-in experimental build (build.py)
#endif
#include "ray_math.cuh"

namespace b200drr {

constexpr int kThreads = 128;

__global__ void __launch_bounds__(kThreads) siddon_fwd_general_kernel(const float* __restrict__ vol, VolDims dims,
                                                                      const float* __restrict__ src,
                                                                      const float* __restrict__ tgt,
                                                                      const float* __restrict__ raylen,
                                                                      float* __restrict__ out, int64_t N, float shift,
                                                                      float eps, int reduce, int align_corners)
{
    const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    const int b = blockIdx.y;
    const int64_t r = (int64_t)b * N + n;
    const Ray ray = load_ray(src, tgt, b, r, eps);
    out[r] = siddon_ray_general(vol, dims, ray, __ldg(raylen + r), shift, reduce, align_corners);
}

__global__ void __launch_bounds__(kThreads) siddon_fwd_fast_kernel(const float* __restrict__ vol, VolDims dims,
                                                                   const float* __restrict__ src,
                                                                   const float* __restrict__ tgt,
                                                                   const float* __restrict__ raylen,
                                                                   float* __restrict__ out, int64_t N, float shift,
                                                                   float eps)
{
    const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    const int b = blockIdx.y;
    const int64_t r = (int64_t)b * N + n;
    const Ray ray = load_ray(src, tgt, b, r, eps);
    // arbitrary ray sets (sub-sampled / patched / user rays): no tiling is possible, the kernel is bound by DRAM/L2
    // locality (measured: the lean walk is 10 % SLOWER here because it thrashes the caches faster), so keep the plain walk
    out[r] = __ldg(raylen + r) * siddon_ray_fast<false>(vol, dims, ray, shift, nullptr);
}

__global__ void __launch_bounds__(kThreads) siddon_visits_kernel(VolDims dims, const float* __restrict__ src,
                                                                 const float* __restrict__ tgt,
                                                                 int32_t* __restrict__ visits, int64_t N, float shift,
                                                                 float eps)
{
    const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    const int b = blockIdx.y;
    const int64_t r = (int64_t)b * N + n;
    const Ray ray = load_ray(src, tgt, b, r, eps);
    int count = 0;
    siddon_ray_fast<true>(nullptr, dims, ray, shift, &count);
    visits[r] = count;
}

__global__ void __launch_bounds__(kThreads) siddon_bwd_kernel(const float* __restrict__ vol, VolDims dims,
                                                              const float* __restrict__ src,
                                                              const float* __restrict__ tgt,
                                                              const float* __restrict__ raylen,
                                                              const float* __restrict__ gout,
                                                              float* __restrict__ g_src, float* __restrict__ g_tgt,
                                                              float* __restrict__ g_raylen, float* __restrict__ g_vol,
                                                              int64_t N, float shift, float eps, int stop_grad)
{
    __shared__ float red[32];
    const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int b = blockIdx.y;
    const bool active = n < N;
    float gs[3] = {0.0f, 0.0f, 0.0f};
    if (active) {
        const int64_t r = (int64_t)b * N + n;
        const Ray ray = load_ray(src, tgt, b, r, eps);
        const float L = __ldg(raylen + r), g = __ldg(gout + r);
        float gt[3];
        float acc;
        if ((int64_t)dims.d[0] * dims.d[1] * dims.d[2] < (int64_t)INT32_MAX) {
            const int lo_v[3] = {0, 0, 0};
            float A[3] = {0.0f, 0.0f, 0.0f}, C[3] = {0.0f, 0.0f, 0.0f};
            const float gL = g * L;
            const bool want_vol = g_vol != nullptr && !stop_grad;
            acc = want_vol ? siddon_ray_bwd_lean_box<4, true>(vol, dims, lo_v, dims.d, dims.d[1] * dims.d[2], dims.d[2], 1, ray,
                                                              shift, gL, g_vol, A, C)
                           : siddon_ray_bwd_lean_box<4, false>(vol, dims, lo_v, dims.d, dims.d[1] * dims.d[2], dims.d[2], 1, ray,
                                                               shift, gL, nullptr, A, C);
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                gt[a] = -gL * A[a] * ray.inv[a];
                gs[a] = gL * (A[a] - C[a]) * ray.inv[a];
            }
        } else {
            acc = siddon_ray_bwd(vol, dims, ray, shift, g * L, stop_grad ? nullptr : g_vol, gs, gt);
        }
        if (g_tgt) {
#pragma unroll
            for (int a = 0; a < 3; ++a) g_tgt[r * 3 + a] = gt[a];
        }
        if (g_raylen) g_raylen[r] = stop_grad ? 0.0f : g * acc;
    }
    if (g_src) {
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            const float tot = block_sum(gs[a], red);
            if (threadIdx.x == 0) atomicAdd(g_src + b * 3 + a, tot);
        }
    }
}

// ---------------------------------------------------------------------------------------------------
// Detector-grid kernel: the rays of a pose are the full H x W detector (n = h*W + w).  A CTA owns a
// TW x TH pixel tile and every warp an 8 x 4 sub-tile, so the 32 lanes of a warp walk a compact ray
// bundle (~16 x 8 voxels across) and their gathers share 128-byte lines / 32-byte sectors in L1.
// U = voxel loads kept in flight per thread.
// ---------------------------------------------------------------------------------------------------
template <int TW, int TH, int U, int LEAN>
__global__ void __launch_bounds__(TW* TH) siddon_fwd_grid_kernel(const float* __restrict__ vol, VolDims dims,
                                                                 const float* __restrict__ src,
                                                                 const float* __restrict__ tgt,
                                                                 const float* __restrict__ raylen,
                                                                 float* __restrict__ out, int H, int W, float shift,
                                                                 float eps)
{
    constexpr int WX = TW / 8;  // warps per tile row
    const int tiles_x = (W + TW - 1) / TW;
    const int tile_x = blockIdx.x % tiles_x, tile_y = blockIdx.x / tiles_x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int px = tile_x * TW + (warp % WX) * 8 + (lane & 7);
    const int py = tile_y * TH + (warp / WX) * 4 + (lane >> 3);
    if (px >= W || py >= H) return;
    const int b = blockIdx.y;
    const int64_t r = ((int64_t)b * H + py) * W + px;
    const Ray ray = load_ray(src, tgt, b, r, eps);
    out[r] = __ldg(raylen + r) *
             (LEAN ? siddon_ray_lean<U>(vol, dims, ray, shift) : siddon_ray_fast_ilp<U>(vol, dims, ray, shift));
}

// ---------------------------------------------------------------------------------------------------
// Slab-major detector-grid kernel.  The volume is cut into slabs of `slab` planes along axis 0 (the
// slowest axis: a slab is one contiguous chunk of memory sized to stay resident in the 126 MB L2).
// blockIdx.x enumerates (slab, pose, tile) with the slab SLOWEST, so the CTAs in flight at any time --
// across all poses of the batch -- gather from the same few slabs and the volume streams from HBM about
// once per BATCH instead of once per pose.  Each CTA integrates its rays over its slab only (splitting a
// ray at voxel planes is exact) and adds the partial line integral to out with red.global.add.f32
// (out is zero-filled by the launcher).
// ---------------------------------------------------------------------------------------------------
// MAJ = true: `slab` is a piece COUNT along each ray's own major axis (major_axis_piece; batches of one or two poses).
template <int TW, int TH, int U, bool MAJ = false>
__global__ void __launch_bounds__(TW* TH) siddon_fwd_slab_kernel(const float* __restrict__ vol, VolDims dims,
                                                                 const float* __restrict__ src,
                                                                 const float* __restrict__ tgt,
                                                                 const float* __restrict__ raylen,
                                                                 float* __restrict__ out, int B, int H, int W, int slab,
                                                                 float shift, float eps, PoseRays pr)
{
    constexpr int WX = TW / 8;
    const int tiles_x = (W + TW - 1) / TW, tiles_y = (H + TH - 1) / TH;
    const int tiles = tiles_x * tiles_y;
    int id = blockIdx.x;
    const int tile = id % tiles;
    id /= tiles;
    const int b = id % B;
    const int sl = id / B;
    const int tile_x = tile % tiles_x, tile_y = tile / tiles_x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int px = tile_x * TW + (warp % WX) * 8 + (lane & 7);
    const int py = tile_y * TH + (warp / WX) * 4 + (lane >> 3);
    if (px >= W || py >= H) return;
    const int64_t r = ((int64_t)b * H + py) * W + px;
    float L;
    const Ray ray = make_ray(pr, src, tgt, raylen, b, r, px, py, eps, L);
    int lo_v[3] = {sl * slab, 0, 0};
    int hi_v[3] = {min(dims.d[0], (sl + 1) * slab), dims.d[1], dims.d[2]};
    if (MAJ && !major_axis_piece(ray, dims, sl, slab, lo_v, hi_v)) return;
    if (box_surely_missed(ray, lo_v, hi_v, shift)) return;  // most (ray, slab) pairs: skip the walk set-up
    const float part = siddon_ray_lean_box<U>(vol, lo_v, hi_v, dims.d[1] * dims.d[2], dims.d[2], 1, ray, shift);
    if (part != 0.0f) red_add(out + r, L * part);
}

template <int TW, int TH, int U, bool MAJ = false>
static cudaError_t launch_slab_variant(const float* vol, VolDims dims, const float* src, const float* tgt,
                                       const float* raylen, float* out, int B, int H, int W, int slab, float shift,
                                       float eps, cudaStream_t stream, PoseRays pr = PoseRays{nullptr, nullptr, nullptr, nullptr})
{
    const int n_slabs = MAJ ? slab : (dims.d[0] + slab - 1) / slab;
    const int64_t blocks = (int64_t)((W + TW - 1) / TW) * ((H + TH - 1) / TH) * B * n_slabs;
    if (blocks > INT32_MAX) return cudaErrorInvalidValue;
    cudaError_t e = cudaMemsetAsync(out, 0, sizeof(float) * (size_t)B * H * W, stream);
    if (e != cudaSuccess) return e;
    siddon_fwd_slab_kernel<TW, TH, U, MAJ><<<(unsigned)blocks, TW * TH, 0, stream>>>(vol, dims, src, tgt, raylen, out, B, H, W,
                                                                                   slab, shift, eps, pr);
    return cudaGetLastError();
}

#ifdef B200DRR_EXPERIMENTS
// ---------------------------------------------------------------------------------------------------
// EXPERIMENT (opt-in, b200drr_x_*): slab-major forward over a major-axis-fastest copy with per-lane chunk reuse
// (ray_math.cuh: siddon_ray_lean_box_chunk).  Not on any default path; kept compiled so the next tuning round can time it.
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) transpose_volume_kernel(const float* __restrict__ vol, VolDims dims, int axis,
                                                               float* __restrict__ out)
{
    // out[i_p][i_q][i_axis], (p, q) = the other two axes in ascending order; one thread per OUTPUT element
    const int64_t total = (int64_t)dims.d[0] * dims.d[1] * dims.d[2];
    const int p = axis == 0 ? 1 : 0, q = axis == 2 ? 1 : 2;
    for (int64_t o = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; o < total; o += (int64_t)gridDim.x * blockDim.x) {
        int idx[3];
        idx[axis] = (int)(o % dims.d[axis]);
        const int64_t t = o / dims.d[axis];
        idx[q] = (int)(t % dims.d[q]);
        idx[p] = (int)(t / dims.d[q]);
        out[o] = __ldg(vol + ((int64_t)idx[0] * dims.d[1] + idx[1]) * dims.d[2] + idx[2]);
    }
}

cudaError_t launch_x_transpose_volume(const float* vol, VolDims dims, int axis, float* out, cudaStream_t stream)
{
    const int64_t total = (int64_t)dims.d[0] * dims.d[1] * dims.d[2];
    cudaError_t e = cudaMemsetAsync(out + total, 0, sizeof(float) * 4, stream);  // the padding chunk
    if (e != cudaSuccess) return e;
    transpose_volume_kernel<<<148 * 8, 256, 0, stream>>>(vol, dims, axis, out);
    return cudaGetLastError();
}

template <int TW, int TH, int U, int CW>
__global__ void __launch_bounds__(TW* TH) siddon_fwd_slab_chunk_kernel(const float* __restrict__ volT, VolDims dims, int axis,
                                                                       const float* __restrict__ src,
                                                                       const float* __restrict__ tgt,
                                                                       const float* __restrict__ raylen,
                                                                       float* __restrict__ out, int B, int H, int W, int slab,
                                                                       float shift, float eps)
{
    constexpr int WX = TW / 8;
    const int tiles_x = (W + TW - 1) / TW, tiles_y = (H + TH - 1) / TH;
    const int tiles = tiles_x * tiles_y;
    int id = blockIdx.x;
    const int tile = id % tiles;
    id /= tiles;
    const int b = id % B;
    const int sl = id / B;
    const int tile_x = tile % tiles_x, tile_y = tile / tiles_x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int px = tile_x * TW + (warp % WX) * 8 + (lane & 7);
    const int py = tile_y * TH + (warp / WX) * 4 + (lane >> 3);
    if (px >= W || py >= H) return;
    const int64_t r = ((int64_t)b * H + py) * W + px;
    const Ray ray = load_ray(src, tgt, b, r, eps);
    const int lo_v[3] = {sl * slab, 0, 0};
    const int hi_v[3] = {min(dims.d[0], (sl + 1) * slab), dims.d[1], dims.d[2]};
    if (box_surely_missed(ray, lo_v, hi_v, shift)) return;
    // element strides of the copy whose fastest axis is `axis` (the other two keep their order)
    const int d0 = dims.d[0], d1 = dims.d[1], d2 = dims.d[2];
    const int st0 = axis == 0 ? 1 : (axis == 1 ? d1 * d2 : d2 * d1);  // out[i_p][i_q][i_axis], p < q
    const int st1 = axis == 1 ? 1 : (axis == 0 ? d0 * d2 : d2);
    const int st2 = axis == 2 ? 1 : (axis == 0 ? d0 : d1);
    const float part = siddon_ray_lean_box_chunk<U, CW>(volT, lo_v, hi_v, st0, st1, st2, ray, shift);
    if (part != 0.0f) red_add(out + r, __ldg(raylen + r) * part);
}

cudaError_t launch_x_siddon_fwd_chunk(const float* volT, VolDims dims, int axis, const float* src, const float* tgt,
                                      const float* raylen, float* out, int B, int H, int W, float shift, float eps,
                                      int variant, cudaStream_t stream)
{
    if ((int64_t)dims.d[0] * dims.d[1] * dims.d[2] >= (int64_t)INT32_MAX) return cudaErrorInvalidValue;
    cudaError_t e = cudaMemsetAsync(out, 0, sizeof(float) * (size_t)B * H * W, stream);
    if (e != cudaSuccess) return e;
#define XC(id, TW, TH, U, CW, SLAB)                                                                                      \
    case id: {                                                                                                           \
        const int n_slabs = (dims.d[0] + SLAB - 1) / SLAB;                                                               \
        const int64_t blocks = (int64_t)((W + TW - 1) / TW) * ((H + TH - 1) / TH) * B * n_slabs;                         \
        if (blocks > INT32_MAX) return cudaErrorInvalidValue;                                                            \
        siddon_fwd_slab_chunk_kernel<TW, TH, U, CW><<<(unsigned)blocks, TW * TH, 0, stream>>>(                           \
            volT, dims, axis, src, tgt, raylen, out, B, H, W, SLAB, shift, eps);                                         \
        return cudaGetLastError();                                                                                       \
    }
    switch (variant) {
        XC(0, 16, 16, 4, 4, 32)
        XC(1, 16, 16, 4, 2, 32)
        XC(2, 16, 8, 4, 4, 32)
        XC(3, 8, 16, 4, 4, 32)
        XC(4, 16, 16, 2, 4, 32)
        XC(5, 16, 16, 8, 4, 32)
        XC(6, 16, 16, 4, 4, 48)
        XC(7, 8, 16, 8, 2, 48)
        default: return cudaErrorInvalidValue;
    }
#undef XC
}

// ---------------------------------------------------------------------------------------------------
// Plane-synchronous slab-major kernel (psync.cuh): same decomposition as siddon_fwd_slab_kernel, but every
// lane advances one MAJOR-axis plane per iteration and the lanes of a warp are aligned onto the same plane
// (WarpAlign), so the 8x4 ray bundle gathers from one voxel plane at a time and shares sectors.
// ---------------------------------------------------------------------------------------------------
struct WarpAlign {
    __device__ __forceinline__ int operator()(int m, bool pos, int p_start, bool active) const
    {
        const unsigned full = 0xffffffffu;
        const unsigned act = __ballot_sync(full, active);
        if (act == 0u) return 0;
        const int key = m * 2 + (pos ? 1 : 0);
        const int lkey = __shfl_sync(full, key, __ffs(act) - 1);
        const bool uniform = __all_sync(full, !active || key == lkey);
        const int t = pos ? p_start : -p_start;  // position along the direction of travel
        const int tmin = __reduce_min_sync(full, active ? t : 0x7fffffff);
        return (uniform && active) ? t - tmin : 0;
    }
};

template <int TW, int TH, int U, int ALIGN>
__global__ void __launch_bounds__(TW* TH) siddon_fwd_psync_kernel(const float* __restrict__ vol, VolDims dims,
                                                                  const float* __restrict__ src,
                                                                  const float* __restrict__ tgt,
                                                                  const float* __restrict__ raylen,
                                                                  float* __restrict__ out, int B, int H, int W, int slab,
                                                                  float shift, float eps)
{
    constexpr int WX = TW / 8;
    const int tiles_x = (W + TW - 1) / TW, tiles_y = (H + TH - 1) / TH;
    const int tiles = tiles_x * tiles_y;
    int id = blockIdx.x;
    const int tile = id % tiles;
    id /= tiles;
    const int b = id % B;
    const int sl = id / B;
    const int tile_x = tile % tiles_x, tile_y = tile / tiles_x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int px = tile_x * TW + (warp % WX) * 8 + (lane & 7);
    const int py = tile_y * TH + (warp / WX) * 4 + (lane >> 3);
    const bool valid = px < W && py < H;  // out-of-image lanes shadow the last pixel: the warp stays convergent
    const int64_t r = ((int64_t)b * H + min(py, H - 1)) * W + min(px, W - 1);
    const Ray ray = load_ray(src, tgt, b, r, eps);
    const int lo_v[3] = {sl * slab, 0, 0};
    const int hi_v[3] = {min(dims.d[0], (sl + 1) * slab), dims.d[1], dims.d[2]};
    const unsigned nvox = (unsigned)(dims.d[0] * dims.d[1] * dims.d[2]);
    float part;
    if (ALIGN)
        part = siddon_ray_psync<U>(vol, nvox, lo_v, hi_v, dims.d[1] * dims.d[2], dims.d[2], 1, ray, shift, WarpAlign());
    else
        part = siddon_ray_psync<U>(vol, nvox, lo_v, hi_v, dims.d[1] * dims.d[2], dims.d[2], 1, ray, shift, NoAlign());
    if (valid && part != 0.0f) red_add(out + r, __ldg(raylen + r) * part);
}

template <int TW, int TH, int U, int ALIGN>
static cudaError_t launch_psync_variant(const float* vol, VolDims dims, const float* src, const float* tgt,
                                        const float* raylen, float* out, int B, int H, int W, int slab, float shift,
                                        float eps, cudaStream_t stream)
{
    const int n_slabs = (dims.d[0] + slab - 1) / slab;
    const int64_t blocks = (int64_t)((W + TW - 1) / TW) * ((H + TH - 1) / TH) * B * n_slabs;
    if (blocks > INT32_MAX || (int64_t)dims.d[0] * dims.d[1] * dims.d[2] >= (int64_t)INT32_MAX) return cudaErrorInvalidValue;
    cudaError_t e = cudaMemsetAsync(out, 0, sizeof(float) * (size_t)B * H * W, stream);
    if (e != cudaSuccess) return e;
    siddon_fwd_psync_kernel<TW, TH, U, ALIGN><<<(unsigned)blocks, TW * TH, 0, stream>>>(vol, dims, src, tgt, raylen, out, B,
                                                                                      H, W, slab, shift, eps);
    return cudaGetLastError();
}

#endif  // B200DRR_EXPERIMENTS

// ---------------------------------------------------------------------------------------------------
// Slab-major detector-grid BACKWARD kernel: same decomposition as siddon_fwd_slab_kernel.  Every CTA adds its
// slab's share of g_tgt / g_raylen / g_src (and optionally g_vol) with red.global.add; the launcher zero-fills.
// ---------------------------------------------------------------------------------------------------
template <int TW, int TH, int U, int MINB>
__global__ void __launch_bounds__(TW* TH, MINB) siddon_bwd_slab_kernel(const float* __restrict__ vol, VolDims dims,
                                                                 const float* __restrict__ src,
                                                                 const float* __restrict__ tgt,
                                                                 const float* __restrict__ raylen,
                                                                 const float* __restrict__ gout, float* __restrict__ g_src,
                                                                 float* __restrict__ g_tgt, float* __restrict__ g_raylen,
                                                                 float* __restrict__ g_vol, int B, int H, int W, int slab,
                                                                 float shift, float eps, int stop_grad, PoseRays pr)
{
    constexpr int WX = TW / 8;
    const int tiles_x = (W + TW - 1) / TW, tiles_y = (H + TH - 1) / TH;
    const int tiles = tiles_x * tiles_y;
    int id = blockIdx.x;
    const int tile = id % tiles;
    id /= tiles;
    const int b = id % B;
    const int sl = id / B;
    const int tile_x = tile % tiles_x, tile_y = tile / tiles_x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int px = tile_x * TW + (warp % WX) * 8 + (lane & 7);
    const int py = tile_y * TH + (warp / WX) * 4 + (lane >> 3);
    float gs[3] = {0.0f, 0.0f, 0.0f};
    if (px < W && py < H) {
        const int64_t r = ((int64_t)b * H + py) * W + px;
        float L;
        const Ray ray = make_ray(pr, src, tgt, raylen, b, r, px, py, eps, L);
        const int lo_v[3] = {sl * slab, 0, 0};
        const int hi_v[3] = {min(dims.d[0], (sl + 1) * slab), dims.d[1], dims.d[2]};
        const float g = __ldg(gout + r);
        const float gL = g * L;
        float A[3] = {0.0f, 0.0f, 0.0f}, C[3] = {0.0f, 0.0f, 0.0f};
        const bool want_vol = g_vol != nullptr && !stop_grad;
        float acc = 0.0f;
        if (!box_surely_missed(ray, lo_v, hi_v, shift))  // most (ray, slab) pairs are misses: skip the walk set-up
            acc = want_vol ? siddon_ray_bwd_lean_box<U, true>(vol, dims, lo_v, hi_v, dims.d[1] * dims.d[2], dims.d[2], 1, ray,
                                                              shift, gL, g_vol, A, C)
                           : siddon_ray_bwd_lean_box<U, false>(vol, dims, lo_v, hi_v, dims.d[1] * dims.d[2], dims.d[2], 1, ray,
                                                               shift, gL, nullptr, A, C);
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            const float gt = -gL * A[a] * ray.inv[a];
            gs[a] = gL * (A[a] - C[a]) * ray.inv[a];
            if (g_tgt && gt != 0.0f) red_add(g_tgt + r * 3 + a, gt);
        }
        if (g_raylen && !stop_grad && acc != 0.0f) red_add(g_raylen + r, g * acc);
    }
    if (g_src) {
        // warp-level reduction + one atomic per warp: no block barrier, so warps whose rays finish early retire
        // instead of waiting for the slowest warp of the CTA (ncu: 19 % of stalls were on that barrier)
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            const float tot = warp_sum(gs[a]);
            if ((threadIdx.x & 31) == 0 && tot != 0.0f) atomicAdd(g_src + b * 3 + a, tot);
        }
    }
}

template <int TW, int TH, int U, int MINB>
static cudaError_t launch_bwd_slab_variant(const float* vol, VolDims dims, const float* src, const float* tgt,
                                           const float* raylen, const float* gout, float* g_src, float* g_tgt,
                                           float* g_raylen, float* g_vol, int B, int H, int W, int slab, float shift,
                                           float eps, int stop_grad, cudaStream_t stream,
                                           PoseRays pr = PoseRays{nullptr, nullptr, nullptr, nullptr})
{
    const int n_slabs = (dims.d[0] + slab - 1) / slab;
    const int64_t blocks = (int64_t)((W + TW - 1) / TW) * ((H + TH - 1) / TH) * B * n_slabs;
    if (blocks > INT32_MAX || (int64_t)dims.d[0] * dims.d[1] * dims.d[2] >= (int64_t)INT32_MAX) return cudaErrorInvalidValue;
    const size_t n = (size_t)B * H * W;
    cudaError_t e = cudaSuccess;
    if (g_src) e = cudaMemsetAsync(g_src, 0, sizeof(float) * 3 * (size_t)B, stream);
    if (e == cudaSuccess && g_tgt) e = cudaMemsetAsync(g_tgt, 0, sizeof(float) * 3 * n, stream);
    if (e == cudaSuccess && g_raylen) e = cudaMemsetAsync(g_raylen, 0, sizeof(float) * n, stream);
    if (e != cudaSuccess) return e;
    siddon_bwd_slab_kernel<TW, TH, U, MINB><<<(unsigned)blocks, TW * TH, 0, stream>>>(
        vol, dims, src, tgt, raylen, gout, g_src, g_tgt, g_raylen, g_vol, B, H, W, slab, shift, eps, stop_grad, pr);
    return cudaGetLastError();
}

cudaError_t launch_siddon_bwd_grid(const float* vol, VolDims dims, const float* src, const float* tgt,
                                   const float* raylen, const float* gout, float* g_src, float* g_tgt, float* g_raylen,
                                   float* g_vol, int B, int H, int W, float shift, float eps, int stop_grad, int variant,
                                   cudaStream_t stream)
{
#define BV(id, TW, TH, U, SLAB, MINB)                                                                                    \
    case id:                                                                                                             \
        return launch_bwd_slab_variant<TW, TH, U, MINB>(vol, dims, src, tgt, raylen, gout, g_src, g_tgt, g_raylen, g_vol, B, \
                                                        H, W, SLAB, shift, eps, stop_grad, stream);
    switch (variant) {
        BV(0, 16, 8, 4, 64, 8)
        BV(10, 16, 16, 4, 32, 1)
        BV(1, 16, 8, 4, 32, 1)
        BV(2, 16, 16, 2, 32, 1)
        BV(3, 16, 16, 4, 64, 1)
        BV(4, 16, 16, 4, 64, 4)
        BV(5, 16, 16, 2, 64, 4)
        BV(6, 16, 8, 4, 64, 8)
        BV(7, 16, 8, 2, 64, 8)
        BV(8, 16, 16, 4, 128, 4)
        BV(9, 16, 8, 4, 64, 6)
        default: return cudaErrorInvalidValue;
    }
#undef BV
}

template <int TW, int TH, int U, int LEAN>
static cudaError_t launch_grid_variant(const float* vol, VolDims dims, const float* src, const float* tgt,
                                       const float* raylen, float* out, int B, int H, int W, float shift, float eps,
                                       cudaStream_t stream)
{
    const dim3 grid((unsigned)(((W + TW - 1) / TW) * ((H + TH - 1) / TH)), (unsigned)B, 1);
    if (LEAN && (int64_t)dims.d[0] * dims.d[1] * dims.d[2] >= (int64_t)INT32_MAX)  // 32-bit offsets would overflow
        siddon_fwd_grid_kernel<TW, TH, U, 0><<<grid, TW * TH, 0, stream>>>(vol, dims, src, tgt, raylen, out, H, W, shift, eps);
    else
        siddon_fwd_grid_kernel<TW, TH, U, LEAN><<<grid, TW * TH, 0, stream>>>(vol, dims, src, tgt, raylen, out, H, W, shift,
                                                                              eps);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------------
// Pose-in entry points: rays generated in-kernel (PoseRays), gradients reduced to the 3x4 matrices.
// ---------------------------------------------------------------------------------------------------
int small_batch_pieces(const VolDims& dims, int B, int H, int W, bool sens);  // defined next to the sensitivities launchers below

cudaError_t launch_siddon_fwd_pose(const float* vol, VolDims dims, const float* src, const float* G, const float* Wd,
                                   const float* rows, const float* cols, float* out, int B, int H, int W, float shift,
                                   float eps, cudaStream_t stream)
{
    const int pieces = small_batch_pieces(dims, B, H, W, false);
    if (pieces > 0 && (int64_t)dims.d[0] * dims.d[1] * dims.d[2] < (int64_t)INT32_MAX)
        return launch_slab_variant<16, 16, 4, true>(vol, dims, src, nullptr, nullptr, out, B, H, W, pieces, shift, eps, stream,
                                                    PoseRays{G, Wd, rows, cols});
    return launch_slab_variant<16, 16, 4>(vol, dims, src, nullptr, nullptr, out, B, H, W, 32, shift, eps, stream,
                                          PoseRays{G, Wd, rows, cols});
}

// g_G[b][a][k] = sum_n g_tgt[b][n][a] * p_k(n),  g_Wd[b][a][k] = sum_n g_raylen[b][n] * delta_a(n)/L(n) * p_k(n),
// p(n) = (cols[w], rows[h], 1, 1): the chain rule through the in-kernel ray generation of make_ray().
__global__ void __launch_bounds__(256) pose_grad_reduce_kernel(const float* __restrict__ g_tgt,
                                                                const float* __restrict__ g_raylen,
                                                                const float* __restrict__ Wd,
                                                                const float* __restrict__ rows,
                                                                const float* __restrict__ cols, float* __restrict__ g_G,
                                                                float* __restrict__ g_Wd, int H, int W)
{
    __shared__ float red[32];
    const int b = blockIdx.y;
    const int64_t N = (int64_t)H * W;
    float acc[18];
#pragma unroll
    for (int i = 0; i < 18; ++i) acc[i] = 0.0f;
    const float* wd = Wd + b * 12;
    for (int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; n < N; n += (int64_t)gridDim.x * blockDim.x) {
        const int h = (int)(n / W), w = (int)(n % W);
        const float c = __ldg(cols + w), r = __ldg(rows + h);
        const int64_t ray = (int64_t)b * N + n;
        float dl[3], l2 = 0.0f;
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            dl[a] = fmaf(__ldg(wd + a * 4), c, fmaf(__ldg(wd + a * 4 + 1), r, __ldg(wd + a * 4 + 2) + __ldg(wd + a * 4 + 3)));
            l2 = fmaf(dl[a], dl[a], l2);
        }
        const float gl = g_raylen ? __ldg(g_raylen + ray) * rsqrtf(fmaxf(l2, 1e-30f)) : 0.0f;
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            const float gt = __ldg(g_tgt + ray * 3 + a), u = gl * dl[a];
            acc[a * 3 + 0] = fmaf(gt, c, acc[a * 3 + 0]);
            acc[a * 3 + 1] = fmaf(gt, r, acc[a * 3 + 1]);
            acc[a * 3 + 2] += gt;
            acc[9 + a * 3 + 0] = fmaf(u, c, acc[9 + a * 3 + 0]);
            acc[9 + a * 3 + 1] = fmaf(u, r, acc[9 + a * 3 + 1]);
            acc[9 + a * 3 + 2] += u;
        }
    }
#pragma unroll
    for (int i = 0; i < 18; ++i) {
        const float tot = block_sum(acc[i], red);
        if (threadIdx.x == 0) {
            float* dst = (i < 9 ? g_G : g_Wd) + b * 12;
            const int a = (i % 9) / 3, k = i % 3;
            atomicAdd(dst + a * 4 + k, tot);
            if (k == 2) atomicAdd(dst + a * 4 + 3, tot);  // the homogeneous 1 multiplies column 3 as well
        }
    }
}

cudaError_t launch_siddon_bwd_pose(const float* vol, VolDims dims, const float* src, const float* G, const float* Wd,
                                   const float* rows, const float* cols, const float* gout, float* g_src, float* g_G,
                                   float* g_Wd, float* g_vol, float* ws_tgt, float* ws_len, int B, int H, int W, float shift,
                                   float eps, int stop_grad, cudaStream_t stream)
{
    cudaError_t e = launch_bwd_slab_variant<16, 8, 4, 8>(vol, dims, src, nullptr, nullptr, gout, g_src, ws_tgt,
                                                        stop_grad ? nullptr : ws_len, g_vol, B, H, W, 64, shift, eps,
                                                        stop_grad, stream, PoseRays{G, Wd, rows, cols});
    if (e != cudaSuccess) return e;
    e = cudaMemsetAsync(g_G, 0, sizeof(float) * 12 * (size_t)B, stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(g_Wd, 0, sizeof(float) * 12 * (size_t)B, stream);
    if (e != cudaSuccess) return e;
    const int chunks = (int)min((int64_t)64, ((int64_t)H * W + 255) / 256);
    pose_grad_reduce_kernel<<<dim3((unsigned)chunks, (unsigned)B), 256, 0, stream>>>(ws_tgt, stop_grad ? nullptr : ws_len, Wd,
                                                                                   rows, cols, g_G, g_Wd, H, W);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------------
// Forward WITH per-ray sensitivities: one walk produces the line integral AND its derivative with respect to the
// ray's own end points (forward-mode; each pixel depends on one ray only, so the whole Jacobian is 6 numbers per
// ray).  The crossing coefficients A_a, C_a of the closed-form backward (SURVEY.md 8a-G) do not depend on the
// incoming gradient, so they are accumulated here and the backward pass shrinks to an elementwise product with g:
//   sens[r] = { dI/dt0, dI/dt1, dI/dt2, S = sum v*dalpha,  dI/ds0, dI/ds1, dI/ds2, 0 },   out[r] = L * S.
// Same slab-major decomposition as siddon_bwd_slab_kernel; partial sums via red.global.add (zero-filled by the launcher).
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ void red_add4(float* addr, float a, float b, float c, float d)
{
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

// MAJ = true: `slab` is a piece COUNT and the volume is cut along each ray's own major axis (major_axis_piece; small batches).
template <int TW, int TH, int U, int MINB, bool MAJ = false>
__global__ void __launch_bounds__(TW* TH, MINB) siddon_sens_slab_kernel(const float* __restrict__ vol, VolDims dims,
                                                                  const float* __restrict__ src,
                                                                  const float* __restrict__ tgt,
                                                                  const float* __restrict__ raylen, float* __restrict__ out,
                                                                  float* __restrict__ sens, int B, int H, int W, int slab,
                                                                  float shift, float eps, PoseRays pr)
{
    constexpr int WX = TW / 8;
    const int tiles_x = (W + TW - 1) / TW, tiles_y = (H + TH - 1) / TH;
    const int tiles = tiles_x * tiles_y;
    int id = blockIdx.x;
    const int tile = id % tiles;
    id /= tiles;
    const int b = id % B;
    const int sl = id / B;
    const int tile_x = tile % tiles_x, tile_y = tile / tiles_x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int px = tile_x * TW + (warp % WX) * 8 + (lane & 7);
    const int py = tile_y * TH + (warp / WX) * 4 + (lane >> 3);
    if (px >= W || py >= H) return;
    const int64_t r = ((int64_t)b * H + py) * W + px;
    float L;
    const Ray ray = make_ray(pr, src, tgt, raylen, b, r, px, py, eps, L);
    int lo_v[3] = {sl * slab, 0, 0};
    int hi_v[3] = {min(dims.d[0], (sl + 1) * slab), dims.d[1], dims.d[2]};
    if (MAJ && !major_axis_piece(ray, dims, sl, slab, lo_v, hi_v)) return;
    if (box_surely_missed(ray, lo_v, hi_v, shift)) return;  // most (ray, slab) pairs: skip the walk set-up
    float A[3] = {0.0f, 0.0f, 0.0f}, C[3] = {0.0f, 0.0f, 0.0f};
    const float S = siddon_ray_sens_box<U, LoadPlain, MAJ>(vol, dims, lo_v, hi_v, dims.d[1] * dims.d[2], dims.d[2], 1, ray, shift, A, C);
    float jt[3], js[3];
    bool any = S != 0.0f;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const float k = L * ray.inv[a];
        jt[a] = -k * A[a];
        js[a] = k * (A[a] - C[a]);
        any = any || jt[a] != 0.0f || js[a] != 0.0f;
    }
    if (any) {  // rays that miss this slab (or see only zeros) add nothing
        red_add4(sens + r * 8, jt[0], jt[1], jt[2], S);
        red_add4(sens + r * 8 + 4, js[0], js[1], js[2], 0.0f);
        red_add(out + r, L * S);
    }
}

template <int TW, int TH, int U, int MINB, bool MAJ = false>
static cudaError_t launch_sens_slab_variant(const float* vol, VolDims dims, const float* src, const float* tgt,
                                            const float* raylen, float* out, float* sens, int B, int H, int W, int slab,
                                            float shift, float eps, cudaStream_t stream,
                                            PoseRays pr = PoseRays{nullptr, nullptr, nullptr, nullptr})
{
    const int n_slabs = MAJ ? slab : (dims.d[0] + slab - 1) / slab;
    const int64_t blocks = (int64_t)((W + TW - 1) / TW) * ((H + TH - 1) / TH) * B * n_slabs;
    if (blocks > INT32_MAX || (int64_t)dims.d[0] * dims.d[1] * dims.d[2] >= (int64_t)INT32_MAX) return cudaErrorInvalidValue;
    const size_t n = (size_t)B * H * W;
    cudaError_t e = cudaMemsetAsync(out, 0, sizeof(float) * n, stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(sens, 0, sizeof(float) * 8 * n, stream);
    if (e != cudaSuccess) return e;
    siddon_sens_slab_kernel<TW, TH, U, MINB, MAJ><<<(unsigned)blocks, TW * TH, 0, stream>>>(vol, dims, src, tgt, raylen, out, sens,
                                                                                         B, H, W, slab, shift, eps, pr);
    return cudaGetLastError();
}

#ifdef B200DRR_EXPERIMENTS
// EXPERIMENT: the sensitivities walk (training step) with the same chunk reuse.  Same outputs as siddon_sens_slab_kernel.
template <int TW, int TH, int U, int CW, int MINB>
__global__ void __launch_bounds__(TW* TH, MINB) siddon_sens_slab_chunk_kernel(const float* __restrict__ volT, VolDims dims,
                                                                        int axis, const float* __restrict__ src,
                                                                        const float* __restrict__ tgt,
                                                                        const float* __restrict__ raylen,
                                                                        float* __restrict__ out, float* __restrict__ sens,
                                                                        int B, int H, int W, int slab, float shift, float eps)
{
    constexpr int WX = TW / 8;
    const int tiles_x = (W + TW - 1) / TW, tiles_y = (H + TH - 1) / TH;
    const int tiles = tiles_x * tiles_y;
    int id = blockIdx.x;
    const int tile = id % tiles;
    id /= tiles;
    const int b = id % B;
    const int sl = id / B;
    const int tile_x = tile % tiles_x, tile_y = tile / tiles_x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int px = tile_x * TW + (warp % WX) * 8 + (lane & 7);
    const int py = tile_y * TH + (warp / WX) * 4 + (lane >> 3);
    if (px >= W || py >= H) return;
    const int64_t r = ((int64_t)b * H + py) * W + px;
    const Ray ray = load_ray(src, tgt, b, r, eps);
    const float L = __ldg(raylen + r);
    const int lo_v[3] = {sl * slab, 0, 0};
    const int hi_v[3] = {min(dims.d[0], (sl + 1) * slab), dims.d[1], dims.d[2]};
    if (box_surely_missed(ray, lo_v, hi_v, shift)) return;
    const int d0 = dims.d[0], d1 = dims.d[1], d2 = dims.d[2];
    const int st0 = axis == 0 ? 1 : (axis == 1 ? d1 * d2 : d2 * d1);
    const int st1 = axis == 1 ? 1 : (axis == 0 ? d0 * d2 : d2);
    const int st2 = axis == 2 ? 1 : (axis == 0 ? d0 : d1);
    float A[3] = {0.0f, 0.0f, 0.0f}, C[3] = {0.0f, 0.0f, 0.0f};
    const float S = siddon_ray_sens_box<U, LoadChunk<CW>>(volT, dims, lo_v, hi_v, st0, st1, st2, ray, shift, A, C);
    float jt[3], js[3];
    bool any = S != 0.0f;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const float k = L * ray.inv[a];
        jt[a] = -k * A[a];
        js[a] = k * (A[a] - C[a]);
        any = any || jt[a] != 0.0f || js[a] != 0.0f;
    }
    if (any) {
        red_add4(sens + r * 8, jt[0], jt[1], jt[2], S);
        red_add4(sens + r * 8 + 4, js[0], js[1], js[2], 0.0f);
        red_add(out + r, L * S);
    }
}

cudaError_t launch_x_siddon_sens_chunk(const float* volT, VolDims dims, int axis, const float* src, const float* tgt,
                                       const float* raylen, float* out, float* sens, int B, int H, int W, float shift,
                                       float eps, int variant, cudaStream_t stream)
{
    if ((int64_t)dims.d[0] * dims.d[1] * dims.d[2] >= (int64_t)INT32_MAX) return cudaErrorInvalidValue;
    const size_t n = (size_t)B * H * W;
    cudaError_t e = cudaMemsetAsync(out, 0, sizeof(float) * n, stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(sens, 0, sizeof(float) * 8 * n, stream);
    if (e != cudaSuccess) return e;
#define XS(id, TW, TH, U, CW, SLAB, MINB)                                                                                \
    case id: {                                                                                                           \
        const int n_slabs = (dims.d[0] + SLAB - 1) / SLAB;                                                               \
        const int64_t blocks = (int64_t)((W + TW - 1) / TW) * ((H + TH - 1) / TH) * B * n_slabs;                         \
        if (blocks > INT32_MAX) return cudaErrorInvalidValue;                                                            \
        siddon_sens_slab_chunk_kernel<TW, TH, U, CW, MINB><<<(unsigned)blocks, TW * TH, 0, stream>>>(                    \
            volT, dims, axis, src, tgt, raylen, out, sens, B, H, W, SLAB, shift, eps);                                   \
        return cudaGetLastError();                                                                                       \
    }
    switch (variant) {
        XS(0, 8, 16, 4, 4, 48, 8)
        XS(1, 8, 16, 4, 2, 48, 8)
        XS(2, 8, 16, 8, 4, 48, 6)
        XS(3, 8, 16, 8, 2, 48, 8)
        XS(4, 16, 8, 4, 4, 48, 8)
        XS(5, 8, 16, 4, 4, 32, 8)
        default: return cudaErrorInvalidValue;
    }
#undef XS
}

#endif  // B200DRR_EXPERIMENTS

// Major-axis pieces (MAJ kernels): every ray is cut into K pieces along its OWN major axis, a thread per (ray, piece).
// Why: (1) the registration loop renders ONE pose per step -- 256^2 rays are 21 % of a B200's thread slots, each walking ~670
// voxels in series; (2) slabs along a FIXED axis give a ray that runs across them one to three pieces of very different length,
// so the lanes of a warp finish at different times, while the major-axis pieces of a warp's rays carry equal shares of the visits.
// Measured on B200, 512^3 -> 256^2 (profiles/r02_tune_small_batch.log; us per launch):
//   forward   B = 1: 187 (32-plane slabs) -> 95 (K = 12);  2: 250 -> 152;  4: 365 -> 248;  8: 601 (brick 591) -> 504;
//             16: 1142 (brick 1099) -> 1032 (K = 16)  -- the fastest forward kernel at every batch size measured (41 % of HBM roofline)
//   sens      B = 1: 193 (thread per ray) -> 115 (K = 8..16);  2: 281 -> 192;  4: 394 (96-plane slabs) -> 312;  8: 637 (48-plane
//             slabs) -> 639;  16: 1243 -> 1273  -- the slab-major kernel keeps batches >= 8 (its volume re-use through L2 pays there).
//             Re-measured at 16 poses with the packed-pair sensitivities step (profiles/r03_tune_sens_routing.log, 3 runs): 48-plane
//             slabs 1182-1191, pieces K = 8 / 12 / 16: 1260-1309 / 1254-1311 / 1288-1321 -- the slabs still win
// `load` = B * H * W in units of 256^2 rays.  Pieces thinner than ~24 planes only add set-up; volumes below 384^3 were not measured
// at batch sizes > 4 (the slab-major tuning of BASELINE config 2 stands there), volumes below 96 voxels keep one thread per ray.
// Returns K, 0 = not used.
// B200DRR_MAJOR_PIECES / B200DRR_MAJOR_MAXB override it for kernel A/B runs (K for every batch up to MAXB poses).
int small_batch_pieces(const VolDims& dims, int B, int H, int W, bool sens)
{
    static const int env_k = [] { const char* e = getenv("B200DRR_MAJOR_PIECES"); return e ? atoi(e) : -1; }();
    static const int env_b = [] { const char* e = getenv("B200DRR_MAJOR_MAXB"); return e ? atoi(e) : -1; }();
    if (env_k >= 0 || env_b >= 0) {
        if (B > (env_b >= 0 ? env_b : 2)) return 0;
        if (env_k >= 0) return env_k > 64 ? 64 : env_k;
    }
    const int dmax = dims.d[0] > dims.d[1] ? (dims.d[0] > dims.d[2] ? dims.d[0] : dims.d[2]) : (dims.d[1] > dims.d[2] ? dims.d[1] : dims.d[2]);
    if (dmax < 96) return 0;  // tiny volumes: a launch is latency-bound whatever the decomposition
    const double load = (double)B * H * W / 65536.0;
    const double max_load = dmax < 384 ? 4.0 : (sens ? 6.0 : 16.0);
    if (load > max_load) return 0;
    int k = (!sens && load > 4.0) ? 16 : 12;
    if (k > dmax / 24) k = dmax / 24;
    return k < 2 ? 0 : k;
}

cudaError_t launch_siddon_fwd_sens_grid(const float* vol, VolDims dims, const float* src, const float* tgt,
                                        const float* raylen, float* out, float* sens, int B, int H, int W, float shift,
                                        float eps, int variant, cudaStream_t stream)
{
#define SV(id, TW, TH, U, SLAB, MINB)                                                                                   \
    case id:                                                                                                             \
        return launch_sens_slab_variant<TW, TH, U, MINB>(vol, dims, src, tgt, raylen, out, sens, B, H, W, SLAB, shift, eps, \
                                                         stream);
    if (variant > 100 && variant <= 164)  // tuning: 101..164 = that many major-axis pieces, whatever the batch size
        return launch_sens_slab_variant<8, 16, 8, 8, true>(vol, dims, src, tgt, raylen, out, sens, B, H, W, variant - 100, shift, eps,
                                                           stream);
    if (variant > 300 && variant <= 364)
        return launch_sens_slab_variant<16, 8, 8, 8, true>(vol, dims, src, tgt, raylen, out, sens, B, H, W, variant - 300, shift, eps,
                                                           stream);
    if (variant > 400 && variant <= 464)
        return launch_sens_slab_variant<8, 16, 4, 8, true>(vol, dims, src, tgt, raylen, out, sens, B, H, W, variant - 400, shift, eps,
                                                           stream);
    if (variant == 0) {
        const int pieces = small_batch_pieces(dims, B, H, W, true);
        if (pieces > 0)
            return launch_sens_slab_variant<8, 16, 8, 8, true>(vol, dims, src, tgt, raylen, out, sens, B, H, W, pieces, shift, eps,
                                                               stream);
    }
    if (variant == 0 && B <= 2)  // few poses: no cross-pose L2 sharing to win, skip the slab decomposition
        return launch_sens_slab_variant<8, 16, 8, 8>(vol, dims, src, tgt, raylen, out, sens, B, H, W, dims.d[0], shift, eps,
                                                     stream);
    switch (variant) {
        SV(0, 8, 16, 8, 48, 8)  // tuned default (profiles/r01_tune_sens.log)
        SV(38, 8, 16, 8, 48, 8)  // the same kernel by an explicit id, for batches whose default is the major-axis-pieces kernel
        SV(32, 16, 8, 8, 48, 8)
        SV(33, 8, 16, 8, 128, 8)
        SV(34, 8, 16, 8, 512, 8)
        SV(35, 8, 16, 8, 96, 8)
        SV(36, 8, 16, 8, 256, 8)
        SV(37, 8, 16, 8, 64, 8)
        SV(22, 16, 8, 4, 64, 8)
        SV(1, 16, 8, 4, 32, 8)
        SV(2, 16, 16, 4, 64, 4)
        SV(3, 16, 16, 4, 32, 4)
        SV(4, 16, 8, 2, 64, 8)
        SV(5, 16, 8, 4, 64, 6)
        SV(6, 16, 16, 4, 128, 4)
        SV(7, 16, 8, 4, 128, 8)
        SV(8, 16, 8, 6, 64, 6)
        SV(9, 16, 8, 8, 64, 4)
        SV(10, 8, 8, 4, 64, 16)
        SV(11, 16, 16, 2, 64, 4)
        SV(12, 16, 8, 4, 64, 10)
        SV(13, 16, 8, 8, 32, 4)
        SV(14, 16, 8, 8, 32, 8)
        SV(15, 16, 8, 6, 32, 8)
        SV(16, 16, 8, 8, 16, 8)
        SV(17, 16, 16, 8, 32, 4)
        SV(18, 16, 8, 12, 32, 4)
        SV(20, 16, 16, 8, 32, 3)
        SV(24, 32, 4, 8, 48, 8)
        SV(25, 16, 8, 8, 40, 8)
        SV(26, 16, 8, 8, 56, 8)
        SV(27, 16, 4, 8, 48, 16)
        SV(28, 8, 8, 8, 48, 16)
        SV(29, 16, 8, 6, 48, 8)
        SV(30, 16, 8, 10, 48, 6)
        SV(31, 32, 8, 8, 48, 4)
        SV(21, 8, 8, 8, 32, 16)
        default: return cudaErrorInvalidValue;
    }
#undef SV
}

cudaError_t launch_siddon_fwd_sens_pose(const float* vol, VolDims dims, const float* src, const float* G, const float* Wd,
                                        const float* rows, const float* cols, float* out, float* sens, int B, int H, int W,
                                        float shift, float eps, cudaStream_t stream)
{
    const int pieces = small_batch_pieces(dims, B, H, W, true);
    if (pieces > 0)
        return launch_sens_slab_variant<8, 16, 8, 8, true>(vol, dims, src, nullptr, nullptr, out, sens, B, H, W, pieces, shift, eps,
                                                           stream, PoseRays{G, Wd, rows, cols});
    // slabs exist to share the volume through L2 across the poses of a batch; with one or two poses they only repeat the
    // per-ray set-up (measured at B = 1: 0.147 ms with 48-plane slabs, 0.136 ms unslabbed)
    return launch_sens_slab_variant<8, 16, 8, 8>(vol, dims, src, nullptr, nullptr, out, sens, B, H, W,
                                                 B <= 2 ? dims.d[0] : 48, shift, eps, stream,
                                                 PoseRays{G, Wd, rows, cols});
}

// Backward from the saved sensitivities, arbitrary-ray layout: g_tgt = g * dI/dt, g_raylen = g * S, g_src = sum_n g * dI/ds.
__global__ void __launch_bounds__(256) sens_bwd_kernel(const float4* __restrict__ sens, const float* __restrict__ gout,
                                                       float* __restrict__ g_src, float* __restrict__ g_tgt,
                                                       float* __restrict__ g_raylen, int64_t N, int stop_grad)
{
    __shared__ float red[32];
    const int b = blockIdx.y;
    float gs[3] = {0.0f, 0.0f, 0.0f};
    for (int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; n < N; n += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = (int64_t)b * N + n;
        const float g = __ldg(gout + r);
        const float4 t = __ldg(sens + r * 2), s = __ldg(sens + r * 2 + 1);
        if (g_tgt) {
            g_tgt[r * 3 + 0] = g * t.x;
            g_tgt[r * 3 + 1] = g * t.y;
            g_tgt[r * 3 + 2] = g * t.z;
        }
        if (g_raylen) g_raylen[r] = stop_grad ? 0.0f : g * t.w;
        gs[0] = fmaf(g, s.x, gs[0]);
        gs[1] = fmaf(g, s.y, gs[1]);
        gs[2] = fmaf(g, s.z, gs[2]);
    }
    if (g_src) {
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            const float tot = block_sum(gs[a], red);
            if (threadIdx.x == 0) atomicAdd(g_src + b * 3 + a, tot);
        }
    }
}

cudaError_t launch_siddon_bwd_sens(const float* sens, const float* gout, float* g_src, float* g_tgt, float* g_raylen,
                                   int B, int64_t N, int stop_grad, cudaStream_t stream)
{
    if (g_src) {
        const cudaError_t e = cudaMemsetAsync(g_src, 0, sizeof(float) * 3 * (size_t)B, stream);
        if (e != cudaSuccess) return e;
    }
    const int chunks = (int)min((int64_t)64, (N + 255) / 256);
    sens_bwd_kernel<<<dim3((unsigned)chunks, (unsigned)B), 256, 0, stream>>>((const float4*)sens, gout, g_src, g_tgt, g_raylen,
                                                                           N, stop_grad);
    return cudaGetLastError();
}

// Backward from the saved sensitivities, pose-in layout: the chain rule through make_ray() as in
// pose_grad_reduce_kernel, with g_tgt = g * dI/dt and g_raylen = g * S formed on the fly.
__global__ void __launch_bounds__(256) sens_bwd_pose_kernel(const float4* __restrict__ sens, const float* __restrict__ gout,
                                                            const float* __restrict__ Wd, const float* __restrict__ rows,
                                                            const float* __restrict__ cols, float* __restrict__ g_src,
                                                            float* __restrict__ g_G, float* __restrict__ g_Wd, int H, int W,
                                                            int stop_grad)
{
    __shared__ float red[32];
    const int b = blockIdx.y;
    const int64_t N = (int64_t)H * W;
    float acc[21];
#pragma unroll
    for (int i = 0; i < 21; ++i) acc[i] = 0.0f;
    const float* wd = Wd + b * 12;
    for (int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; n < N; n += (int64_t)gridDim.x * blockDim.x) {
        const int h = (int)(n / W), w = (int)(n % W);
        const float c = __ldg(cols + w), r = __ldg(rows + h);
        const int64_t ray = (int64_t)b * N + n;
        const float g = __ldg(gout + ray);
        const float4 t = __ldg(sens + ray * 2), s = __ldg(sens + ray * 2 + 1);
        float dl[3], l2 = 0.0f;
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            dl[a] = fmaf(__ldg(wd + a * 4), c, fmaf(__ldg(wd + a * 4 + 1), r, __ldg(wd + a * 4 + 2) + __ldg(wd + a * 4 + 3)));
            l2 = fmaf(dl[a], dl[a], l2);
        }
        const float gl = stop_grad ? 0.0f : g * t.w * rsqrtf(fmaxf(l2, 1e-30f));
        const float gt[3] = {g * t.x, g * t.y, g * t.z};
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            const float u = gl * dl[a];
            acc[a * 3 + 0] = fmaf(gt[a], c, acc[a * 3 + 0]);
            acc[a * 3 + 1] = fmaf(gt[a], r, acc[a * 3 + 1]);
            acc[a * 3 + 2] += gt[a];
            acc[9 + a * 3 + 0] = fmaf(u, c, acc[9 + a * 3 + 0]);
            acc[9 + a * 3 + 1] = fmaf(u, r, acc[9 + a * 3 + 1]);
            acc[9 + a * 3 + 2] += u;
        }
        acc[18] = fmaf(g, s.x, acc[18]);
        acc[19] = fmaf(g, s.y, acc[19]);
        acc[20] = fmaf(g, s.z, acc[20]);
    }
#pragma unroll
    for (int i = 0; i < 21; ++i) {
        const float tot = block_sum(acc[i], red);
        if (threadIdx.x == 0) {
            if (i >= 18) {
                atomicAdd(g_src + b * 3 + (i - 18), tot);
            } else {
                float* dst = (i < 9 ? g_G : g_Wd) + b * 12;
                const int a = (i % 9) / 3, k = i % 3;
                atomicAdd(dst + a * 4 + k, tot);
                if (k == 2) atomicAdd(dst + a * 4 + 3, tot);  // the homogeneous 1 multiplies column 3 as well
            }
        }
    }
}

cudaError_t launch_siddon_bwd_sens_pose(const float* sens, const float* gout, const float* Wd, const float* rows,
                                        const float* cols, float* g_src, float* g_G, float* g_Wd, int B, int H, int W,
                                        int stop_grad, cudaStream_t stream)
{
    cudaError_t e = cudaMemsetAsync(g_src, 0, sizeof(float) * 3 * (size_t)B, stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(g_G, 0, sizeof(float) * 12 * (size_t)B, stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(g_Wd, 0, sizeof(float) * 12 * (size_t)B, stream);
    if (e != cudaSuccess) return e;
    const int chunks = (int)min((int64_t)64, ((int64_t)H * W + 255) / 256);
    sens_bwd_pose_kernel<<<dim3((unsigned)chunks, (unsigned)B), 256, 0, stream>>>((const float4*)sens, gout, Wd, rows, cols,
                                                                                g_src, g_G, g_Wd, H, W, stop_grad);
    return cudaGetLastError();
}

cudaError_t launch_siddon_fwd_grid(const float* vol, VolDims dims, const float* src, const float* tgt,
                                   const float* raylen, float* out, int B, int H, int W, float shift, float eps,
                                   int variant, cudaStream_t stream)
{
#define V(id, TW, TH, U, LEAN) \
    case id: return launch_grid_variant<TW, TH, U, LEAN>(vol, dims, src, tgt, raylen, out, B, H, W, shift, eps, stream);
#define S0(id, TW, TH, U, SLAB) \
    case id: return launch_slab_variant<TW, TH, U>(vol, dims, src, tgt, raylen, out, B, H, W, SLAB, shift, eps, stream);
    if (variant > 100 && variant <= 164)  // tuning: 101..164 = that many major-axis pieces, whatever the batch size
        return launch_slab_variant<16, 16, 4, true>(vol, dims, src, tgt, raylen, out, B, H, W, variant - 100, shift, eps, stream);
    if (variant > 200 && variant <= 264)
        return launch_slab_variant<8, 16, 8, true>(vol, dims, src, tgt, raylen, out, B, H, W, variant - 200, shift, eps, stream);
    if (variant > 300 && variant <= 364)
        return launch_slab_variant<16, 8, 4, true>(vol, dims, src, tgt, raylen, out, B, H, W, variant - 300, shift, eps, stream);
    if (variant > 400 && variant <= 464)
        return launch_slab_variant<8, 16, 4, true>(vol, dims, src, tgt, raylen, out, B, H, W, variant - 400, shift, eps, stream);
    if (variant == 0) {
        const int pieces = small_batch_pieces(dims, B, H, W, false);
        if (pieces > 0) return launch_slab_variant<16, 16, 4, true>(vol, dims, src, tgt, raylen, out, B, H, W, pieces, shift, eps, stream);
    }
    switch (variant) {
        S0(0, 16, 16, 4, 32)
        V(30, 16, 8, 4, 1)
        V(1, 16, 8, 8, 0)
        V(2, 16, 8, 2, 1)
        V(3, 16, 8, 8, 1)
        V(4, 16, 16, 4, 1)
        V(5, 32, 8, 4, 1)
        V(6, 8, 8, 4, 1)
        V(7, 8, 16, 4, 1)
        V(8, 16, 8, 6, 1)
        V(9, 8, 8, 8, 1)
#define S(id, TW, TH, U, SLAB) \
    case id: return launch_slab_variant<TW, TH, U>(vol, dims, src, tgt, raylen, out, B, H, W, SLAB, shift, eps, stream);
        S(10, 16, 8, 4, 32)
        S(11, 16, 8, 4, 16)
        S(12, 16, 8, 4, 64)
        S(13, 16, 8, 2, 32)
        S(14, 16, 8, 8, 32)
        S(15, 16, 16, 4, 32)
        S(16, 8, 8, 4, 32)
        S(17, 16, 8, 4, 8)
        S(18, 16, 8, 4, 128)
        S(19, 32, 8, 4, 32)
        S(40, 8, 16, 4, 32)
        S(41, 8, 16, 8, 32)
        S(42, 8, 16, 4, 48)
        S(43, 16, 8, 8, 48)
        S(44, 16, 16, 8, 32)
        S(45, 8, 16, 6, 32)
#undef S
#ifdef B200DRR_EXPERIMENTS
#define P(id, TW, TH, U, SLAB, ALIGN) \
    case id: return launch_psync_variant<TW, TH, U, ALIGN>(vol, dims, src, tgt, raylen, out, B, H, W, SLAB, shift, eps, stream);
        P(20, 16, 8, 2, 32, 1)
        P(21, 16, 8, 2, 32, 0)
        P(22, 16, 8, 1, 32, 1)
        P(23, 16, 8, 2, 64, 1)
        P(24, 16, 16, 2, 32, 1)
        P(25, 16, 16, 2, 64, 1)
        P(26, 16, 8, 3, 32, 1)
        P(27, 16, 8, 2, 512, 1)
        P(28, 8, 8, 2, 32, 1)
        P(29, 16, 16, 1, 32, 1)
#undef P
#endif

        default: return cudaErrorInvalidValue;
    }
#undef V
}

// mask_to_channels forward: out [B][C][N], zero-filled by the launcher; one thread per ray owns out[b][:][n].
__global__ void __launch_bounds__(kThreads) siddon_fwd_mask_kernel(const float* __restrict__ vol,
                                                                   const float* __restrict__ mask, VolDims dims,
                                                                   const float* __restrict__ src,
                                                                   const float* __restrict__ tgt,
                                                                   const float* __restrict__ raylen, float* out, int64_t N,
                                                                   int C, float shift, float eps, int W)
{
    const int64_t n = tiled_ray_index(N, W);
    if (n < 0) return;
    const int b = blockIdx.y;
    const int64_t r = (int64_t)b * N + n;
    const Ray ray = load_ray(src, tgt, b, r, eps);
    siddon_ray_lean_mask<4>(vol, mask, dims, ray, shift, __ldg(raylen + r), out + (int64_t)b * C * N + n, N, C);
}

// Full detector grid: the slab-major decomposition of siddon_fwd_slab_kernel (the poses of a batch share each 32-plane slab of
// BOTH the density and the label volume through L2), label runs flushed per (ray, slab) with red.global.add.
__global__ void __launch_bounds__(256) siddon_fwd_mask_slab_kernel(const float* __restrict__ vol, const float* __restrict__ mask,
                                                                   VolDims dims, const float* __restrict__ src,
                                                                   const float* __restrict__ tgt, const float* __restrict__ raylen,
                                                                   float* __restrict__ out, int B, int H, int W, int C, int slab,
                                                                   float shift, float eps)
{
    const int tiles_x = (W + 15) / 16, tiles = tiles_x * ((H + 15) / 16);
    int id = blockIdx.x;
    const int tile = id % tiles;
    id /= tiles;
    const int b = id % B, sl = id / B;
    const int tile_x = tile % tiles_x, tile_y = tile / tiles_x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int px = tile_x * 16 + (warp % 2) * 8 + (lane & 7), py = tile_y * 16 + (warp / 2) * 4 + (lane >> 3);
    if (px >= W || py >= H) return;
    const int64_t N = (int64_t)H * W, n = (int64_t)py * W + px, r = (int64_t)b * N + n;
    const Ray ray = load_ray(src, tgt, b, r, eps);
    const int lo_v[3] = {sl * slab, 0, 0};
    const int hi_v[3] = {min(dims.d[0], (sl + 1) * slab), dims.d[1], dims.d[2]};
    if (box_surely_missed(ray, lo_v, hi_v, shift)) return;
    siddon_ray_lean_mask_box<4, true>(vol, mask, lo_v, hi_v, dims.d[1] * dims.d[2], dims.d[2], 1, ray, shift, __ldg(raylen + r),
                                      out + (int64_t)b * C * N + n, N, C);
}

cudaError_t launch_siddon_fwd_mask(const float* vol, const float* mask, VolDims dims, const float* src, const float* tgt,
                                   const float* raylen, float* out, int B, int64_t N, int C, float shift, float eps,
                                   cudaStream_t stream, int W)
{
    static_assert(kThreads == 128, "tiled_ray_index assumes 128-thread CTAs");
    cudaError_t e = cudaMemsetAsync(out, 0, sizeof(float) * (size_t)B * C * N, stream);
    if (e != cudaSuccess) return e;
    if (W > 0) {
        const int H = (int)(N / W), slab = 32, n_slabs = (dims.d[0] + slab - 1) / slab;
        const int64_t blocks = (int64_t)((W + 15) / 16) * ((H + 15) / 16) * B * n_slabs;
        if (blocks <= INT32_MAX) {
            siddon_fwd_mask_slab_kernel<<<(unsigned)blocks, 256, 0, stream>>>(vol, mask, dims, src, tgt, raylen, out, B, H, W, C, slab,
                                                                            shift, eps);
            return cudaGetLastError();
        }
    }
    siddon_fwd_mask_kernel<<<tiled_ray_grid(B, N, W), kThreads, 0, stream>>>(
        vol, mask, dims, src, tgt, raylen, out, N, C, shift, eps, W);
    return cudaGetLastError();
}

// Backward for the options the fast kernels do not cover: reducefn="max" and/or align_corners=True (general walk).
__global__ void __launch_bounds__(kThreads) siddon_bwd_general_kernel(
    const float* __restrict__ vol, VolDims dims, const float* __restrict__ src, const float* __restrict__ tgt,
    const float* __restrict__ raylen, const float* __restrict__ gout, float* __restrict__ g_src, float* __restrict__ g_tgt,
    float* __restrict__ g_raylen, float* __restrict__ g_vol, int64_t N, float shift, float eps, int stop_grad, int reduce,
    int align_corners, int mode)
{
    __shared__ float red[32];
    const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int b = blockIdx.y;
    float gs[3] = {0.0f, 0.0f, 0.0f};
    if (n < N) {
        const int64_t r = (int64_t)b * N + n;
        const Ray ray = load_ray(src, tgt, b, r, eps);
        const float L = __ldg(raylen + r), g = __ldg(gout + r);
        float gt[3];
        float acc;
        if (mode == 0)
            acc = siddon_ray_general_bwd(vol, dims, ray, L, g * L, shift, reduce, align_corners, stop_grad ? nullptr : g_vol,
                                         gs, gt);
        else  // mode="bilinear" (reduce "sum"): trilinear sampling at the segment midpoints
            siddon_ray_bilinear<true>(vol, dims, ray, L, shift, 0, align_corners, g, stop_grad != 0,
                                      stop_grad ? nullptr : g_vol, gs, gt, acc);
        if (g_tgt) {
#pragma unroll
            for (int a = 0; a < 3; ++a) g_tgt[r * 3 + a] = gt[a];
        }
        if (g_raylen) g_raylen[r] = stop_grad ? 0.0f : g * acc;
    }
    if (g_src) {
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            const float tot = block_sum(gs[a], red);
            if (threadIdx.x == 0) atomicAdd(g_src + b * 3 + a, tot);
        }
    }
}

cudaError_t launch_siddon_bwd_general(const float* vol, VolDims dims, const float* src, const float* tgt, const float* raylen,
                                      const float* gout, float* g_src, float* g_tgt, float* g_raylen, float* g_vol, int B,
                                      int64_t N, float shift, float eps, int stop_grad, int reduce, int align_corners,
                                      int mode, cudaStream_t stream)
{
    if (mode != 0 && reduce != 0) return cudaErrorNotSupported;
    if (g_src) {
        const cudaError_t e = cudaMemsetAsync(g_src, 0, sizeof(float) * 3 * (size_t)B, stream);
        if (e != cudaSuccess) return e;
    }
    siddon_bwd_general_kernel<<<dim3((unsigned)((N + kThreads - 1) / kThreads), (unsigned)B, 1), kThreads, 0, stream>>>(
        vol, dims, src, tgt, raylen, gout, g_src, g_tgt, g_raylen, g_vol, N, shift, eps, stop_grad, reduce, align_corners,
        mode);
    return cudaGetLastError();
}

// Forward of the general walk with the sampling mode selectable (0 = nearest: the reference default, 1 = bilinear).
__global__ void __launch_bounds__(kThreads) siddon_fwd_bilinear_kernel(const float* __restrict__ vol, VolDims dims,
                                                                       const float* __restrict__ src,
                                                                       const float* __restrict__ tgt,
                                                                       const float* __restrict__ raylen,
                                                                       float* __restrict__ out, int64_t N, float shift,
                                                                       float eps, int reduce, int align_corners)
{
    const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    const int b = blockIdx.y;
    const int64_t r = (int64_t)b * N + n;
    const Ray ray = load_ray(src, tgt, b, r, eps);
    float gs[3], gt[3], sum_tl;
    out[r] = siddon_ray_bilinear<false>(vol, dims, ray, __ldg(raylen + r), shift, reduce, align_corners, 0.0f, true, nullptr,
                                        gs, gt, sum_tl);
}

cudaError_t launch_siddon_fwd_general(const float* vol, VolDims dims, const float* src, const float* tgt, const float* raylen,
                                      float* out, int B, int64_t N, float shift, float eps, int reduce, int align_corners,
                                      int mode, cudaStream_t stream)
{
    const dim3 grid((unsigned)((N + kThreads - 1) / kThreads), (unsigned)B, 1);
    if (mode == 0)
        siddon_fwd_general_kernel<<<grid, kThreads, 0, stream>>>(vol, dims, src, tgt, raylen, out, N, shift, eps, reduce,
                                                                 align_corners);
    else
        siddon_fwd_bilinear_kernel<<<grid, kThreads, 0, stream>>>(vol, dims, src, tgt, raylen, out, N, shift, eps, reduce,
                                                                  align_corners);
    return cudaGetLastError();
}

// mask_to_channels backward (autograd of renderers.py:77-89): gout [B][C][N]; the segment in voxel j receives the
// gradient of the channel it was scattered to, g_j = gout[b][label_j][n], i.e. the closed-form walk with v_j -> g_j v_j.
__global__ void __launch_bounds__(kThreads) siddon_bwd_mask_kernel(
    const float* __restrict__ vol, const float* __restrict__ mask, VolDims dims, const float* __restrict__ src,
    const float* __restrict__ tgt, const float* __restrict__ raylen, const float* __restrict__ gout,
    float* __restrict__ g_src, float* __restrict__ g_tgt, float* __restrict__ g_raylen, float* __restrict__ g_vol, int64_t N,
    int C, float shift, float eps, int stop_grad, int W)
{
    __shared__ float red[32];
    const int64_t n = tiled_ray_index(N, W);  // W > 0: full detector grid, threads in pixel tiles
    const int b = blockIdx.y;
    float gs[3] = {0.0f, 0.0f, 0.0f};
    if (n >= 0) {
        const int64_t r = (int64_t)b * N + n;
        const Ray ray = load_ray(src, tgt, b, r, eps);
        const float L = __ldg(raylen + r);
        float gt[3];
        const FetchMasked fetch{vol, mask, gout + (int64_t)b * C * N + n, N, C};
        const float acc = siddon_ray_bwd_f(fetch, dims, ray, shift, L, stop_grad ? nullptr : g_vol, gs, gt);
        if (g_tgt) {
#pragma unroll
            for (int a = 0; a < 3; ++a) g_tgt[r * 3 + a] = gt[a];
        }
        if (g_raylen) g_raylen[r] = stop_grad ? 0.0f : acc;
    }
    if (g_src) {
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            const float tot = block_sum(gs[a], red);
            if (threadIdx.x == 0) atomicAdd(g_src + b * 3 + a, tot);
        }
    }
}

cudaError_t launch_siddon_bwd_mask(const float* vol, const float* mask, VolDims dims, const float* src, const float* tgt,
                                   const float* raylen, const float* gout, float* g_src, float* g_tgt, float* g_raylen,
                                   float* g_vol, int B, int64_t N, int C, float shift, float eps, int stop_grad,
                                   cudaStream_t stream, int W)
{
    if (g_src) {
        const cudaError_t e = cudaMemsetAsync(g_src, 0, sizeof(float) * 3 * (size_t)B, stream);
        if (e != cudaSuccess) return e;
    }
    siddon_bwd_mask_kernel<<<tiled_ray_grid(B, N, W), kThreads, 0, stream>>>(
        vol, mask, dims, src, tgt, raylen, gout, g_src, g_tgt, g_raylen, g_vol, N, C, shift, eps, stop_grad, W);
    return cudaGetLastError();
}

static inline dim3 ray_grid(int B, int64_t N) { return dim3((unsigned)((N + kThreads - 1) / kThreads), (unsigned)B, 1); }

cudaError_t launch_siddon_fwd(const float* vol, VolDims dims, const float* src, const float* tgt,
                              const float* raylen, float* out, int B, int64_t N, float shift, float eps, int reduce,
                              int align_corners, cudaStream_t stream)
{
    if (reduce == 0 && !align_corners)
        siddon_fwd_fast_kernel<<<ray_grid(B, N), kThreads, 0, stream>>>(vol, dims, src, tgt, raylen, out, N, shift, eps);
    else
        siddon_fwd_general_kernel<<<ray_grid(B, N), kThreads, 0, stream>>>(vol, dims, src, tgt, raylen, out, N, shift,
                                                                          eps, reduce, align_corners);
    return cudaGetLastError();
}

cudaError_t launch_siddon_visits(VolDims dims, const float* src, const float* tgt, int32_t* visits, int B, int64_t N,
                                 float shift, float eps, cudaStream_t stream)
{
    siddon_visits_kernel<<<ray_grid(B, N), kThreads, 0, stream>>>(dims, src, tgt, visits, N, shift, eps);
    return cudaGetLastError();
}

// Forward with sensitivities for ARBITRARY ray sets (sub-sampled / patched / user rays): one thread per ray over the
// whole volume, plain stores (no slabs, so no partial sums).  Volumes too large for 32-bit offsets are refused.
__global__ void __launch_bounds__(kThreads) siddon_sens_kernel(const float* __restrict__ vol, VolDims dims,
                                                               const float* __restrict__ src, const float* __restrict__ tgt,
                                                               const float* __restrict__ raylen, float* __restrict__ out,
                                                               float* __restrict__ sens, int64_t N, float shift, float eps)
{
    const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    const int b = blockIdx.y;
    const int64_t r = (int64_t)b * N + n;
    const Ray ray = load_ray(src, tgt, b, r, eps);
    const float L = __ldg(raylen + r);
    const int lo_v[3] = {0, 0, 0};
    float A[3] = {0.0f, 0.0f, 0.0f}, C[3] = {0.0f, 0.0f, 0.0f};
    const float S = siddon_ray_sens_box<4>(vol, dims, lo_v, dims.d, dims.d[1] * dims.d[2], dims.d[2], 1, ray, shift, A, C);
    float4 t, s4;
    t.x = -L * ray.inv[0] * A[0];
    t.y = -L * ray.inv[1] * A[1];
    t.z = -L * ray.inv[2] * A[2];
    t.w = S;
    s4.x = L * ray.inv[0] * (A[0] - C[0]);
    s4.y = L * ray.inv[1] * (A[1] - C[1]);
    s4.z = L * ray.inv[2] * (A[2] - C[2]);
    s4.w = 0.0f;
    reinterpret_cast<float4*>(sens)[r * 2] = t;
    reinterpret_cast<float4*>(sens)[r * 2 + 1] = s4;
    out[r] = L * S;
}

// ---------------------------------------------------------------------------------------------------
// Slab-major kernels for ARBITRARY ray sets that the caller has put in a locality order (sub-sampled detectors, patches,
// user rays: the module sorts them by the Morton code of their target points, renderers._locality_order): ray i of a
// pose is simply thread i, so the 32 lanes of a warp walk 32 spatial neighbours and share 128-byte lines exactly like
// the 8 x 4 pixel bundles of the detector-grid kernels.  Same slab decomposition, same per-ray math, same atomics.
// ---------------------------------------------------------------------------------------------------
template <int THREADS, int U>
__global__ void __launch_bounds__(THREADS) siddon_fwd_slab_linear_kernel(const float* __restrict__ vol, VolDims dims,
                                                                         const float* __restrict__ src,
                                                                         const float* __restrict__ tgt,
                                                                         const float* __restrict__ raylen,
                                                                         float* __restrict__ out, int B, int64_t N, int slab,
                                                                         float shift, float eps)
{
    const int64_t tiles = (N + THREADS - 1) / THREADS;
    int64_t id = blockIdx.x;
    const int64_t tile = id % tiles;
    id /= tiles;
    const int b = (int)(id % B);
    const int sl = (int)(id / B);
    const int64_t n = tile * THREADS + threadIdx.x;
    if (n >= N) return;
    const int64_t r = (int64_t)b * N + n;
    const Ray ray = load_ray(src, tgt, b, r, eps);
    const int lo_v[3] = {sl * slab, 0, 0};
    const int hi_v[3] = {min(dims.d[0], (sl + 1) * slab), dims.d[1], dims.d[2]};
    if (box_surely_missed(ray, lo_v, hi_v, shift)) return;
    const float part = siddon_ray_lean_box<U>(vol, lo_v, hi_v, dims.d[1] * dims.d[2], dims.d[2], 1, ray, shift);
    if (part != 0.0f) red_add(out + r, __ldg(raylen + r) * part);
}

template <int THREADS, int U>
__global__ void __launch_bounds__(THREADS, 2048 / THREADS / 4) siddon_sens_slab_linear_kernel(
    const float* __restrict__ vol, VolDims dims, const float* __restrict__ src, const float* __restrict__ tgt,
    const float* __restrict__ raylen, float* __restrict__ out, float* __restrict__ sens, int B, int64_t N, int slab, float shift,
    float eps)
{
    const int64_t tiles = (N + THREADS - 1) / THREADS;
    int64_t id = blockIdx.x;
    const int64_t tile = id % tiles;
    id /= tiles;
    const int b = (int)(id % B);
    const int sl = (int)(id / B);
    const int64_t n = tile * THREADS + threadIdx.x;
    if (n >= N) return;
    const int64_t r = (int64_t)b * N + n;
    const Ray ray = load_ray(src, tgt, b, r, eps);
    const float L = __ldg(raylen + r);
    const int lo_v[3] = {sl * slab, 0, 0};
    const int hi_v[3] = {min(dims.d[0], (sl + 1) * slab), dims.d[1], dims.d[2]};
    if (box_surely_missed(ray, lo_v, hi_v, shift)) return;
    float A[3] = {0.0f, 0.0f, 0.0f}, C[3] = {0.0f, 0.0f, 0.0f};
    const float S = siddon_ray_sens_box<U>(vol, dims, lo_v, hi_v, dims.d[1] * dims.d[2], dims.d[2], 1, ray, shift, A, C);
    float jt[3], js[3];
    bool any = S != 0.0f;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const float k = L * ray.inv[a];
        jt[a] = -k * A[a];
        js[a] = k * (A[a] - C[a]);
        any = any || jt[a] != 0.0f || js[a] != 0.0f;
    }
    if (any) {
        red_add4(sens + r * 8, jt[0], jt[1], jt[2], S);
        red_add4(sens + r * 8 + 4, js[0], js[1], js[2], 0.0f);
        red_add(out + r, L * S);
    }
}

cudaError_t launch_siddon_fwd_sorted(const float* vol, VolDims dims, const float* src, const float* tgt, const float* raylen,
                                     float* out, int B, int64_t N, float shift, float eps, cudaStream_t stream)
{
    constexpr int T = 128, SLAB = 32;
    if ((int64_t)dims.d[0] * dims.d[1] * dims.d[2] >= (int64_t)INT32_MAX) return cudaErrorInvalidValue;
    const int n_slabs = B >= 3 ? (dims.d[0] + SLAB - 1) / SLAB : 1;  // one or two poses: no batch to share a slab with
    const int slab = B >= 3 ? SLAB : dims.d[0];
    const int64_t blocks = ((N + T - 1) / T) * B * n_slabs;
    if (blocks > INT32_MAX) return cudaErrorInvalidValue;
    cudaError_t e = cudaMemsetAsync(out, 0, sizeof(float) * (size_t)B * N, stream);
    if (e != cudaSuccess) return e;
    siddon_fwd_slab_linear_kernel<T, 4><<<(unsigned)blocks, T, 0, stream>>>(vol, dims, src, tgt, raylen, out, B, N, slab, shift, eps);
    return cudaGetLastError();
}

cudaError_t launch_siddon_fwd_sens_sorted(const float* vol, VolDims dims, const float* src, const float* tgt, const float* raylen,
                                          float* out, float* sens, int B, int64_t N, float shift, float eps, cudaStream_t stream)
{
    constexpr int T = 128, SLAB = 48;
    if ((int64_t)dims.d[0] * dims.d[1] * dims.d[2] >= (int64_t)INT32_MAX) return cudaErrorInvalidValue;
    const int n_slabs = B >= 3 ? (dims.d[0] + SLAB - 1) / SLAB : 1;
    const int slab = B >= 3 ? SLAB : dims.d[0];
    const int64_t blocks = ((N + T - 1) / T) * B * n_slabs;
    if (blocks > INT32_MAX) return cudaErrorInvalidValue;
    cudaError_t e = cudaMemsetAsync(out, 0, sizeof(float) * (size_t)B * N, stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(sens, 0, sizeof(float) * 8 * (size_t)B * N, stream);
    if (e != cudaSuccess) return e;
    siddon_sens_slab_linear_kernel<T, 8><<<(unsigned)blocks, T, 0, stream>>>(vol, dims, src, tgt, raylen, out, sens, B, N, slab, shift,
                                                                            eps);
    return cudaGetLastError();
}

cudaError_t launch_siddon_fwd_sens(const float* vol, VolDims dims, const float* src, const float* tgt, const float* raylen,
                                   float* out, float* sens, int B, int64_t N, float shift, float eps, cudaStream_t stream)
{
    if ((int64_t)dims.d[0] * dims.d[1] * dims.d[2] >= (int64_t)INT32_MAX) return cudaErrorInvalidValue;
    siddon_sens_kernel<<<ray_grid(B, N), kThreads, 0, stream>>>(vol, dims, src, tgt, raylen, out, sens, N, shift, eps);
    return cudaGetLastError();
}

cudaError_t launch_siddon_bwd(const float* vol, VolDims dims, const float* src, const float* tgt,
                              const float* raylen, const float* gout, float* g_src, float* g_tgt, float* g_raylen,
                              float* g_vol, int B, int64_t N, float shift, float eps, int stop_grad,
                              cudaStream_t stream)
{
    if (g_src) {
        cudaError_t e = cudaMemsetAsync(g_src, 0, sizeof(float) * 3 * (size_t)B, stream);
        if (e != cudaSuccess) return e;
    }
    siddon_bwd_kernel<<<ray_grid(B, N), kThreads, 0, stream>>>(vol, dims, src, tgt, raylen, gout, g_src, g_tgt,
                                                               g_raylen, g_vol, N, shift, eps, stop_grad);
    return cudaGetLastError();
}

}  // namespace b200drr
