// Launch plumbing shared by the kernels: error channel, argument checks,
// block reductions.  The library never allocates: every buffer is caller-owned.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "dmh_math.cuh"

namespace dmh {

void set_error(const char* fmt, ...);
void count_launches(int n);   // bookkeeping for dmh_launch_count()
// true iff div_const(a, c, *rc_out) == a / c bit for bit for every float a (verified exhaustively on the current
// device the first time a constant is seen: one small launch + a synchronous 4-byte read-back; cached).  While
// `caller` (the stream the kernel will be launched on) is being captured, an unseen constant reports false.
bool const_div_exact(int c, float* rc_out, cudaStream_t caller);

#define DMH_REQUIRE(cond, ...)                    \
    do {                                          \
        if (!(cond)) {                            \
            dmh::set_error(__VA_ARGS__);          \
            return DMH_ERR_INVALID;               \
        }                                         \
    } while (0)

#define DMH_CHECK_LAUNCH(name)                                                           \
    do {                                                                                 \
        cudaError_t e__ = cudaGetLastError();                                            \
        if (e__ != cudaSuccess) {                                                        \
            dmh::set_error("%s: CUDA launch failed: %s", name, cudaGetErrorString(e__)); \
            return DMH_ERR_CUDA;                                                         \
        }                                                                                \
    } while (0)

// <<<>>> with launch accounting: DMH_LAUNCH(kernel, grid, block, smem, stream)(args...)
#define DMH_LAUNCH(kernel, grid, block, smem, st) dmh::count_launches(1), kernel<<<grid, block, smem, st>>>

static inline int ceil_div(long long a, long long b) { return (int)((a + b - 1) / b); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Sum over the block; result valid in thread 0.  `red` needs >= 32 floats.
__device__ __forceinline__ float block_sum(float v, float* red) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int nthreads = blockDim.x * blockDim.y * blockDim.z;
    v = warp_sum(v);
    __syncthreads();
    if (lane == 0) red[wid] = v;
    __syncthreads();
    if (wid == 0) {
        v = (lane < (nthreads + 31) / 32) ? red[lane] : 0.0f;
        v = warp_sum(v);
    }
    return v;
}

// ATen upsample_bilinear2d (align_corners=False) source taps: src = max(scale*(dst+0.5)-0.5, 0)
struct UpTap { int i0, i1; float l0, l1; };
__device__ __forceinline__ UpTap up_tap(int dst, float scale, int in_size) {
    UpTap t;
    const float src = fmaxf(scale * ((float)dst + 0.5f) - 0.5f, 0.0f);
    t.i0 = min((int)src, in_size - 1);
    t.i1 = t.i0 + ((t.i0 < in_size - 1) ? 1 : 0);
    t.l1 = src - (float)t.i0;
    t.l0 = 1.0f - t.l1;
    return t;
}

// A (h,w) disparity map read as if F.interpolate'd to (H,W) (trainer.py:481-482);
// direct read when the sizes match.
struct DispSrc {
    const float* ptr;
    int h, w;
    float sh, sw;      // h/H, w/W
};
__device__ __forceinline__ float load_disp(const DispSrc& d, int b, int iy, int ix, int H, int W) {
    const float* p = d.ptr + (size_t)b * d.h * d.w;
    if (d.h == H && d.w == W) return __ldg(p + (size_t)iy * W + ix);
    const UpTap ty = up_tap(iy, d.sh, d.h), tx = up_tap(ix, d.sw, d.w);
    return ty.l0 * (tx.l0 * __ldg(p + ty.i0 * d.w + tx.i0) + tx.l1 * __ldg(p + ty.i0 * d.w + tx.i1)) +
           ty.l1 * (tx.l0 * __ldg(p + ty.i1 * d.w + tx.i0) + tx.l1 * __ldg(p + ty.i1 * d.w + tx.i1));
}

// depth-hints arguments of dmh_photo_scale_dh, for the single-source fast kernel (photo_fast.cu) and the general one
struct FastDhArgs {
    const float* hint_reproj;
    const float* hint_depth;
    const float* hint_valid;
    float* grad_hint;
    int nblk;              // stride between the four partial-sum arrays (set by the launcher of the fast kernel)
};

}  // namespace dmh
