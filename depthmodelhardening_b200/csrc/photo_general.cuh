// The general photometric tile: 32 x 16 target pixels with a 2-px reflect halo, 256 threads -- photo_scale_kernel
// (photo_objective.cu: the objective, any number of sources) and reproj_grad_kernel (photo_image_grad.cu: its
// colour-frame gradients).  The backward is only correct if it recomputes the forward's sample points and window
// statistics bit for bit, so both kernels take the tile geometry, the staging of the target and depth tile and the
// window statistics from here.
#pragma once
#include "photo_launch.cuh"

namespace {

#define PH_TW 32
#define PH_TH 16
#define PH_R2W (PH_TW + 4)
#define PH_R2H (PH_TH + 4)
#define PH_R1W (PH_TW + 2)
#define PH_R1H (PH_TH + 2)
#define PH_R2 (PH_R2W * PH_R2H)
#define PH_R1 (PH_R1W * PH_R1H)
#define PH_THREADS 256

// 3x3 window statistics for one channel plane pair [R2] in shared memory around R2 position (r+1, c+1).
// Same arithmetic as the single-source fast kernel and the identity-loss kernel (row sums of 3, then 3 rows,
// mean = sum * (1/9)) so that the automask compares like with like.
__device__ __forceinline__ SsimStatsRows window_stats(const float* __restrict__ xs, const float* __restrict__ ys, int r,
                                                      int c) {
    Row5 rows[3];
#pragma unroll
    for (int dy = 0; dy < 3; ++dy) {
        const float* x = xs + (r + dy) * PH_R2W + c;
        const float* y = ys + (r + dy) * PH_R2W + c;
        rows[dy] = row5(x[0], x[1], x[2], y[0], y[1], y[2]);
    }
    return ssim_stats_rows(rows[0], rows[1], rows[2]);
}

// The target tile tgt [3][R2] and the depth dep [R2] of the tile at (x0, y0) of batch item b, 2-px reflect halo;
// the disparity is up-sampled in the read.  is_depth: the network output is a depth map, used as it is.
__device__ __forceinline__ void load_target_depth(const float* target, const DispSrc& disp, const DepthScale& ds,
                                                  bool is_depth, int b, int x0, int y0, int H, int W, size_t N,
                                                  float* tgt, float* dep) {
    for (int i = threadIdx.x; i < PH_R2; i += PH_THREADS) {
        const int r = i / PH_R2W, c = i % PH_R2W;
        const int iy = ext_to_img(y0 - 2 + r, H), ix = ext_to_img(x0 - 2 + c, W);
        const size_t o = (size_t)iy * W + ix;
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) tgt[ch * PH_R2 + i] = __ldg(target + ((size_t)b * 3 + ch) * N + o);
        const float dv = load_disp(disp, b, iy, ix, H, W);
        dep[i] = is_depth ? dv : disp_to_depth(dv, ds);
    }
}

}  // namespace
