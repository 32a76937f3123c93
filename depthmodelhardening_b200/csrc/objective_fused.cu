// Glue kernels of the fused multi-scale objective (M2/trainer.py:589-674):
//
//   dmh_smooth_fused      A16 forward AND the gradient w.r.t. the normalised
//                         disparity in one pass per scale (per-block partials)
//   dmh_objective_finish  one launch for ALL scales: per-image mean / correction
//                         scalars of the normalisation backward, the per-scale
//                         losses and the total (deterministic, fp64 accumulate)
//   dmh_disp_grad         backward: one launch per scale turns the speculative
//                         gradients into d(total)/d(disp_s) =
//                           u_s * [ F.interpolate^T(grad wrt up-sampled disp)
//                                   + w_s * (gN / (mean+eps) - corr) ]
//                         where u_s is the incoming autograd scalar(s), read on
//                         the device (no host sync, no extra elementwise pass).
//
// With these the whole objective is 4 x (photo + 2 smooth launches) + ident +
// finish forward and 4 launches backward, instead of ~250 ATen kernels per
// (scale, frame) round trip in the reference.
#include <string.h>

#include "../../include/dmh_b200.h"
#include "dmh_common.cuh"

using namespace dmh;

namespace {

#define SF_NB1 64
#define SF_THREADS 256
// CTA tile of sf_main_kernel: 128 x 32 pixels (8 warps x 4 rows, 4 pixels per lane)
#define SF_TW 128
#define SF_TH 32
#define SF_RPW 4
#define SF_BLOCKS(h, w) ((((w) + SF_TW - 1) / SF_TW) * (((h) + SF_TH - 1) / SF_TH))

// bx < SF_NB1 = block of this image
__device__ __forceinline__ void sf_mean_body(const float* __restrict__ disp, int hw, float* __restrict__ part, int b,
                                             int bx, float* red) {
    const float* d = disp + (size_t)b * hw;
    float s = 0.f;
    const int stride = SF_NB1 * SF_THREADS, t = bx * SF_THREADS + threadIdx.x;
    if (((uintptr_t)d & 15) == 0) {
        // 128-bit loads, four of them in flight per thread (the kernel is pure latency otherwise)
        const float4* d4 = reinterpret_cast<const float4*>(d);
        const int n4 = hw >> 2;
        int i = t;
        for (; i + 3 * stride < n4; i += 4 * stride) {
            const float4 a = __ldg(d4 + i), b4 = __ldg(d4 + i + stride), c = __ldg(d4 + i + 2 * stride),
                         e = __ldg(d4 + i + 3 * stride);
            s += ((a.x + a.y) + (a.z + a.w)) + ((b4.x + b4.y) + (b4.z + b4.w)) + ((c.x + c.y) + (c.z + c.w)) +
                 ((e.x + e.y) + (e.z + e.w));
        }
        for (; i < n4; i += stride) {
            const float4 a = __ldg(d4 + i);
            s += (a.x + a.y) + (a.z + a.w);
        }
        for (int j = (n4 << 2) + t; j < hw; j += stride) s += d[j];
    } else {
        for (int i = t; i < hw; i += stride) s += d[i];
    }
    s = block_sum(s, red);
    if (threadIdx.x == 0) part[b * SF_NB1 + bx] = s;
}

__global__ void __launch_bounds__(SF_THREADS)
sf_mean_kernel(const float* __restrict__ disp, int hw, float* __restrict__ part) {
    __shared__ float red[32];
    sf_mean_body(disp, hw, part, blockIdx.y, blockIdx.x, red);
}

// mean(disp_b) + 1e-7 from the 64 partials; called by the 32 lanes of one warp, same
// summation order wherever it is used (forward normalisation and its backward)
__device__ __forceinline__ float mean_eps_warp(const float* __restrict__ mean_part, int b, int hw) {
    const int l = threadIdx.x & 31;
    float s = mean_part[b * SF_NB1 + l] + mean_part[b * SF_NB1 + 32 + l];
    s = warp_sum(s);
    return s / (float)hw + 1e-7f;
}

__device__ __forceinline__ float sgn(float v) { return v > 0.f ? 1.f : (v < 0.f ? -1.f : 0.f); }
// exp(-s / C) for s >= 0 as one multiply + MUFU.EX2 (relative error 2^-22, far inside the 1e-5 tolerance of the
// smoothness term; expf's range reduction costs ~8 more issue slots per edge)
__device__ __forceinline__ float edge_weight(float sabs, float neg_inv_c_log2e) {
    float r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(sabs * neg_inv_c_log2e));
    return r;
}

// four consecutive pixels of one row (x .. x+3); zeros beyond the row end
__device__ __forceinline__ void load_px4(const float* __restrict__ row, int x, int w, bool vec, float v[4]) {
    if (vec && x + 3 < w) {
        const float4 t = __ldg(reinterpret_cast<const float4*>(row + x));
        v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
    } else {
#pragma unroll
        for (int j = 0; j < 4; ++j) v[j] = (x + j < w) ? __ldg(row + x + j) : 0.f;
    }
}

// (Every product-sum below is written with an explicit rounding sequence -- mul_rn / fmaf -- so that the result does
// not depend on the compiler's FMA contraction choices.)
// A16 forward + gradient w.r.t. the normalised disparity.  A lane owns 4 consecutive pixels of a row and
// walks down SF_RPW rows keeping the previous row in registers, so every disparity / colour value is loaded
// once per warp (128-bit loads) plus one row of overlap above and below; the edge weight exp(-mean_c|dI|)
// of every edge is evaluated once by the pixel on its left / top ("owner") and reaches the right / bottom
// neighbour through a register or a warp shuffle.
template <int C>
__device__ __forceinline__ void sf_main_body(const float* __restrict__ disp, const float* __restrict__ img, int h, int w,
                                             const float* __restrict__ mean_part, float inv_nx, float inv_ny, int vec,
                                             float* __restrict__ gN, float* __restrict__ part, int bx, int by, int b,
                                             int gx, int gy) {
    __shared__ float s_m;
    __shared__ float s_red[3][SF_THREADS / 32];
    const int hw = h * w;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (threadIdx.x < 32) {
        const float m0 = mean_eps_warp(mean_part, b, hw);
        if (threadIdx.x == 0) s_m = 1.0f / m0;
    }
    __syncthreads();
    const float inv_m = s_m;
    const float nicl = -1.4426950408889634f / (float)C;
    const float* d = disp + (size_t)b * hw;
    const float* im = img + (size_t)b * C * hw;
    const int x = bx * SF_TW + 4 * lane;
    const int xr = bx * SF_TW + SF_TW;                      // first pixel right of the tile
    const int xl = bx * SF_TW - 1;                          // last pixel left of the tile
    const int yb = by * SF_TH + SF_RPW * wid;               // first output row of this warp
    const bool vok = vec != 0;

    float dc[4], ic[C][4];                                  // owner row y: normalised disparity, colour
    float dn_[4], in_[C][4];                                // row y + 1
    float gy_up[4] = {0.f, 0.f, 0.f, 0.f};                  // y-edge terms owned by row y - 1
    float sum_x = 0.f, sum_y = 0.f, sum_g = 0.f;

    int y = yb - 1;
    if (y >= 0 && y < h) {
        load_px4(d + (size_t)y * w, x, w, vok, dc);
#pragma unroll
        for (int c = 0; c < C; ++c) load_px4(im + (size_t)c * hw + (size_t)y * w, x, w, vok, ic[c]);
    } else {
#pragma unroll
        for (int j = 0; j < 4; ++j) { dc[j] = 0.f; for (int c = 0; c < C; ++c) ic[c][j] = 0.f; }
    }
#pragma unroll
    for (int r = -1; r < SF_RPW; ++r, ++y) {
        const bool row_ok = y >= 0 && y < h;
        const bool below_ok = y + 1 < h && y + 1 >= 0;
        if (below_ok) {
            load_px4(d + (size_t)(y + 1) * w, x, w, vok, dn_);
#pragma unroll
            for (int c = 0; c < C; ++c) load_px4(im + (size_t)c * hw + (size_t)(y + 1) * w, x, w, vok, in_[c]);
        } else {
#pragma unroll
            for (int j = 0; j < 4; ++j) { dn_[j] = 0.f; for (int c = 0; c < C; ++c) in_[c][j] = 0.f; }
        }
        // y-edge owned by (y, x+j): valid iff y and y+1 are rows of the image
        float gy[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            float sabs = 0.f;
#pragma unroll
            for (int c = 0; c < C; ++c) sabs += fabsf(ic[c][j] - in_[c][j]);
            const float e = edge_weight(sabs, nicl);
            const float diff = sub_rn(mul_rn(dc[j], inv_m), mul_rn(dn_[j], inv_m));
            const bool ok = row_ok && below_ok && x + j < w;
            gy[j] = ok ? sgn(diff) * e : 0.f;
            if (r >= 0 && ok) sum_y = fmaf(fabsf(diff), e, sum_y);
        }
        if (r >= 0) {
            // right neighbour of pixel 3: lane+1's pixel 0, or (lane 31) the first pixel of the next tile
            float dr = __shfl_down_sync(0xffffffffu, dc[0], 1);
            float ir[C];
#pragma unroll
            for (int c = 0; c < C; ++c) ir[c] = __shfl_down_sync(0xffffffffu, ic[c][0], 1);
            if (lane == 31 && row_ok && xr < w) {
                dr = __ldg(d + (size_t)y * w + xr);
#pragma unroll
                for (int c = 0; c < C; ++c) ir[c] = __ldg(im + (size_t)c * hw + (size_t)y * w + xr);
            }
            float gx[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                float sabs = 0.f;
#pragma unroll
                for (int c = 0; c < C; ++c) sabs += fabsf(ic[c][j] - (j < 3 ? ic[c][j + 1] : ir[c]));
                const float e = edge_weight(sabs, nicl);
                const float diff = sub_rn(mul_rn(dc[j], inv_m), mul_rn(j < 3 ? dc[j + 1] : dr, inv_m));
                const bool ok = row_ok && x + j < w - 1;
                gx[j] = ok ? sgn(diff) * e : 0.f;
                if (ok) sum_x = fmaf(fabsf(diff), e, sum_x);
            }
            // x-edge owned by the pixel left of pixel 0: lane-1's gx[3], or (lane 0) recomputed across the tile border
            float gl = __shfl_up_sync(0xffffffffu, gx[3], 1);
            if (lane == 0) {
                gl = 0.f;
                if (row_ok && xl >= 0 && x < w) {
                    float sabs = 0.f;
#pragma unroll
                    for (int c = 0; c < C; ++c) sabs += fabsf(__ldg(im + (size_t)c * hw + (size_t)y * w + xl) - ic[c][0]);
                    const float diff = sub_rn(mul_rn(__ldg(d + (size_t)y * w + xl), inv_m), mul_rn(dc[0], inv_m));
                    gl = sgn(diff) * edge_weight(sabs, nicl);
                }
            }
            if (row_ok) {
                float g[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    g[j] = fmaf(gx[j] - (j > 0 ? gx[j - 1] : gl), inv_nx, mul_rn(gy[j] - gy_up[j], inv_ny));
                    if (x + j < w) sum_g = fmaf(g[j], dc[j], sum_g);
                }
                float* go = gN + (size_t)b * hw + (size_t)y * w + x;
                if (vok && x + 3 < w) {
                    *reinterpret_cast<float4*>(go) = make_float4(g[0], g[1], g[2], g[3]);
                } else {
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        if (x + j < w) go[j] = g[j];
                }
            }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            gy_up[j] = gy[j];
            dc[j] = dn_[j];
#pragma unroll
            for (int c = 0; c < C; ++c) ic[c][j] = in_[c][j];
        }
    }
    // one combined reduction of the three partial sums (warp shuffles, then 3 x 8 values in shared memory)
    const float r0 = warp_sum(sum_x), r1 = warp_sum(sum_y), r2 = warp_sum(sum_g);
    if (lane == 0) { s_red[0][wid] = r0; s_red[1][wid] = r1; s_red[2][wid] = r2; }
    __syncthreads();
    if (threadIdx.x < 3) {
        float t = 0.f;
#pragma unroll
        for (int i = 0; i < SF_THREADS / 32; ++i) t += s_red[threadIdx.x][i];
        part[((size_t)b * gx * gy + by * gx + bx) * 3 + threadIdx.x] = t;
    }
}

template <int C>
__global__ void __launch_bounds__(SF_THREADS, 4)
sf_main_kernel(const float* __restrict__ disp, const float* __restrict__ img, int h, int w,
               const float* __restrict__ mean_part, float inv_nx, float inv_ny, int vec, float* __restrict__ gN,
               float* __restrict__ part) {
    sf_main_body<C>(disp, img, h, w, mean_part, inv_nx, inv_ny, vec, gN, part, blockIdx.x, blockIdx.y, blockIdx.z,
                    gridDim.x, gridDim.y);
}

#define FIN_MAXS 8
struct FinishParams {
    const float* smooth_ws[FIN_MAXS];     // [B*64 mean partials][B*nb*3 partials]
    const float* photo_part[FIN_MAXS];
    int photo_n[FIN_MAXS];
    int h[FIN_MAXS], w[FIN_MAXS];
    float smooth_weight[FIN_MAXS];
    int S, B;
    double inv_photo_den;
    float* img_scalars;                   // (S,B,2): 1/(mean+eps), corr
    float* losses;                        // (S+1): per-scale, total
    double* img_sums;                     // workspace (S,B,3): photo, smooth-x, smooth-y numerators
    unsigned* ticket;                     // workspace: arrival counter (zeroed by the launcher)
};

__device__ __forceinline__ double block_sum_d(double v, double* red) {
    v = warp_sum_d(v);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    __syncthreads();
    if (lane == 0) red[wid] = v;
    __syncthreads();
    double t = 0.0;
    if (threadIdx.x == 0)
        for (int i = 0; i < (int)(blockDim.x >> 5); ++i) t += red[i];
    return t;
}

// One CTA per (scale, image): reduces that image's partial sums in a fixed order; the CTA that
// arrives last (atomic ticket) adds the S*B results up, again in a fixed order -> deterministic.
__global__ void __launch_bounds__(256)
finish_kernel(const FinishParams p) {
    __shared__ double red4[4][8];
    __shared__ bool s_last;
    const int blk = blockIdx.x;
    const int s = blk / p.B, b = blk % p.B;
    const int hw = p.h[s] * p.w[s];
    const int nb = SF_BLOCKS(p.h[s], p.w[s]);
    const float* mean_part = p.smooth_ws[s];
    const float* part = p.smooth_ws[s] + (size_t)p.B * SF_NB1 + (size_t)b * nb * 3;
    double sx = 0.0, sy = 0.0, sg = 0.0, ph = 0.0;
    for (int i = threadIdx.x; i < nb; i += blockDim.x) {
        sx += (double)part[(size_t)i * 3 + 0];
        sy += (double)part[(size_t)i * 3 + 1];
        sg += (double)part[(size_t)i * 3 + 2];
    }
    // this CTA's share of the photo partial sums (any fixed partition is fine)
    const long long n = p.photo_n[s];
    const long long lo = n * b / p.B, hi = n * (b + 1) / p.B;
    for (long long i = lo + threadIdx.x; i < hi; i += blockDim.x) ph += (double)p.photo_part[s][i];
    // the four block sums share one pair of barriers (fixed order: lanes by shuffle tree, then warps 0..7)
    sx = warp_sum_d(sx); sy = warp_sum_d(sy); sg = warp_sum_d(sg); ph = warp_sum_d(ph);
    if ((threadIdx.x & 31) == 0) {
        const int wid = threadIdx.x >> 5;
        red4[0][wid] = sx; red4[1][wid] = sy; red4[2][wid] = sg; red4[3][wid] = ph;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        sx = sy = sg = ph = 0.0;
        for (int i = 0; i < 8; ++i) { sx += red4[0][i]; sy += red4[1][i]; sg += red4[2][i]; ph += red4[3][i]; }
    }
    float m = 0.f;
    if (threadIdx.x < 32) m = mean_eps_warp(mean_part, b, hw);
    if (threadIdx.x == 0) {
        const float inv_m = 1.0f / m;
        p.img_scalars[((size_t)s * p.B + b) * 2 + 0] = inv_m;
        p.img_scalars[((size_t)s * p.B + b) * 2 + 1] = (float)(sg / (double)hw) * inv_m * inv_m;
        double* o = p.img_sums + ((size_t)s * p.B + b) * 3;
        o[0] = ph; o[1] = sx; o[2] = sy;
        __threadfence();
        s_last = atomicAdd(p.ticket, 1u) == (unsigned)(p.S * p.B - 1);
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    // last CTA: warp ss adds up scale ss (lane bb takes images bb, bb+32, ... in order; fixed shuffle tree)
    const int lane = threadIdx.x & 31, ss = threadIdx.x >> 5;
    __shared__ double s_loss[8];
    if (ss < p.S) {
        double a = 0.0, bx = 0.0, by = 0.0;
        for (int bb = lane; bb < p.B; bb += 32) {
            const volatile double* o = p.img_sums + ((size_t)ss * p.B + bb) * 3;
            a += o[0]; bx += o[1]; by += o[2];
        }
        a = warp_sum_d(a); bx = warp_sum_d(bx); by = warp_sum_d(by);
        if (lane == 0) {
            const double inv_nx = 1.0 / ((double)p.B * p.h[ss] * (p.w[ss] - 1));
            const double inv_ny = 1.0 / ((double)p.B * (p.h[ss] - 1) * p.w[ss]);
            const double loss = a * p.inv_photo_den + (double)p.smooth_weight[ss] * (bx * inv_nx + by * inv_ny);
            p.losses[ss] = (float)loss;
            s_loss[ss] = loss;
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double total = 0.0;
        for (int i = 0; i < p.S; ++i) total += s_loss[i];
        p.losses[p.S] = (float)(total / (double)p.S);
        *p.ticket = 0u;
    }
}

// Transposed bilinear up-sampling (F.interpolate backward) + normalisation backward + upstream scaling.
// Integer up-scale factor R (2, 4, 8): full-res pixel X = R*c - R/2 + j (chunk c, j < R) reads low-res
// pixels c-1 (weight 1-l_j) and c (weight l_j), so low-res pixel x gathers chunk x and chunk x+1.
// CTA = 32 x 8 low-res pixels.  Stage 1: a warp takes one full-res row, lane c loads chunk c with one or
// two 128/64-bit loads (coalesced; every full-res value is read once) and reduces it against both weight
// sets; the contribution to the left neighbour travels by shuffle; row results go to shared memory.
// Stage 2: one thread per low-res pixel sums its 2R rows.  Deterministic (no atomics; ATen's CUDA
// backward of upsample_bilinear2d scatters with atomicAdd).  R == 1: plain copy; other factors: generic
// conservative window (one thread per low-res pixel).
template <int R>
__device__ __forceinline__ void load_chunk(const float* __restrict__ grow, int X, int W, float v[R]) {
    if (X >= 0 && X + R <= W) {
        if (R == 8) {
            const float4 a = __ldg(reinterpret_cast<const float4*>(grow + X));
            const float4 b = __ldg(reinterpret_cast<const float4*>(grow + X + 4));
            v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4 % R] = b.x; v[5 % R] = b.y; v[6 % R] = b.z; v[7 % R] = b.w;
        } else if (R == 4) {
            const float2 a = __ldg(reinterpret_cast<const float2*>(grow + X));
            const float2 b = __ldg(reinterpret_cast<const float2*>(grow + X + 2));
            v[0] = a.x; v[1] = a.y; v[2 % R] = b.x; v[3 % R] = b.y;
        } else {
#pragma unroll
            for (int j = 0; j < R; ++j) v[j] = __ldg(grow + X + j);
        }
    } else {
#pragma unroll
        for (int j = 0; j < R; ++j) v[j] = (X + j >= 0 && X + j < W) ? __ldg(grow + X + j) : 0.f;
    }
}

// Integer factors 2 / 4 / 8 with a TALL tile: 32 x (64/R) low-res pixels per CTA, i.e. ~66-72 full-res rows of
// 32*R columns (16-64 KB of gradient per CTA, 9 row loads per thread in flight in batches) -- the 32 x 8 tile of
// the general kernel below spends its time in per-CTA latency (weights, two barriers) for 2-3 loads per thread.
template <int R>
__device__ __forceinline__ void load_chunk(const float* __restrict__ grow, int X, int W, float v[R]);

// shared memory of one tall-tile CTA (floats): weights 64/R x 2R + 32 x 2R, row results (64 + R) x 32
#define DG_UP_SMEM(R) (128 + 64 * (R) + (64 + (R)) * 32)
template <int R>
__device__ __forceinline__ void disp_grad_up_body(const float* __restrict__ G_full, const float* __restrict__ gN,
                                                  const float* __restrict__ img_scalars, float smooth_weight,
                                                  const float* __restrict__ g_total, const float* __restrict__ g_scale,
                                                  const float* __restrict__ g_smooth, float inv_S, int h, int w, int H,
                                                  int W, float sh, float sw, float* __restrict__ grad, int bx, int by,
                                                  int b, int lane, int wid, float* smem) {
    constexpr int RW = 2 * R, LR = 64 / R, NR = R * LR + R, NPW = (NR + 7) / 8, BS = R >= 8 ? 3 : (R >= 4 ? 5 : NPW);
    float (*s_wy)[RW] = reinterpret_cast<float (*)[RW]>(smem);                       // [LR][RW]
    float (*s_wx)[RW] = reinterpret_cast<float (*)[RW]>(smem + LR * RW);             // [32][RW]
    float (*s_h)[32] = reinterpret_cast<float (*)[32]>(smem + LR * RW + 32 * RW);    // [NR][32]
    const int x = bx * 32 + lane;
    const float* g = G_full + (size_t)b * H * W;
    const int t = wid * 32 + lane;
    // weights depend only on (y, offset) / (x, offset): tabulated once per CTA with the forward's up_tap
    for (int i = t; i < LR * RW + 32 * RW; i += 256) {
        if (i < LR * RW) {
            const int ly = i / RW, j = i % RW;
            const int yy = by * LR + ly, Y = R * yy - R / 2 + j;
            float wv = 0.f;
            if (yy < h && Y >= 0 && Y < H) { const UpTap tp = up_tap(Y, sh, h); wv = (tp.i0 == yy ? tp.l0 : 0.f) + (tp.i1 == yy ? tp.l1 : 0.f); }
            s_wy[ly][j] = wv;
        } else {
            const int k = i - LR * RW;
            const int lx = k / RW, j = k % RW;
            const int xx = bx * 32 + lx, X = R * xx - R / 2 + j;
            float wv = 0.f;
            if (xx < w && X >= 0 && X < W) { const UpTap tp = up_tap(X, sw, w); wv = (tp.i0 == xx ? tp.l0 : 0.f) + (tp.i1 == xx ? tp.l1 : 0.f); }
            s_wx[lx][j] = wv;
        }
    }
    __syncthreads();
    float wA[R], wB[R], wE[R];                              // chunk c -> low-res c, chunk c -> low-res c-1, chunk 32 -> 31
#pragma unroll
    for (int j = 0; j < R; ++j) {
        wA[j] = s_wx[lane][j];
        wB[j] = lane > 0 ? s_wx[lane - 1][R + j] : 0.f;
        wE[j] = s_wx[31][R + j];
    }
    const int Xc = R * x - R / 2;                            // first full-res column of this lane's chunk
    const int Xe = R * (bx * 32 + 32) - R / 2;      // chunk 32 (lane 0 takes it)
    const int Yt = R * (by * LR) - R / 2;           // first full-res row of the tile's window
#pragma unroll
    for (int i0 = 0; i0 < NPW; i0 += BS) {
        float v[BS][R], ve[BS][R];
#pragma unroll
        for (int i = 0; i < BS; ++i) {
            const int ry = wid + 8 * (i0 + i), Y = Yt + ry;
            const bool ok = i0 + i < NPW && ry < NR && Y >= 0 && Y < H;          // warp-uniform
            const float* grow = g + (size_t)(ok ? Y : 0) * W;
            if (ok) load_chunk<R>(grow, Xc, W, v[i]);
            else {
#pragma unroll
                for (int j = 0; j < R; ++j) v[i][j] = 0.f;
            }
            if (ok && lane == 0) load_chunk<R>(grow, Xe, W, ve[i]);
            else {
#pragma unroll
                for (int j = 0; j < R; ++j) ve[i][j] = 0.f;
            }
        }
#pragma unroll
        for (int i = 0; i < BS; ++i) {
            const int ry = wid + 8 * (i0 + i);
            float a = 0.f, bm = 0.f, e = 0.f;
#pragma unroll
            for (int j = 0; j < R; ++j) {
                a = fmaf(wA[j], v[i][j], a); bm = fmaf(wB[j], v[i][j], bm); e = fmaf(wE[j], ve[i][j], e);
            }
            float nb = __shfl_down_sync(0xffffffffu, bm, 1);
            const float ee = __shfl_sync(0xffffffffu, e, 0);
            if (lane == 31) nb = ee;
            if (i0 + i < NPW && ry < NR) s_h[ry][lane] = a + nb;
        }
    }
    __syncthreads();
    if (x >= w) return;
    const float up = add_rn(g_total ? mul_rn(g_total[0], inv_S) : 0.0f, g_scale ? g_scale[0] : 0.0f);
    float inv_m = 0.f, corr = 0.f;
    if (gN) { inv_m = img_scalars[b * 2]; corr = img_scalars[b * 2 + 1]; }
#pragma unroll
    for (int m = 0; m < LR / 8; ++m) {
        const int ly = wid + 8 * m, y = by * LR + ly;
        if (y >= h) continue;
        float acc = 0.0f;
#pragma unroll
        for (int j = 0; j < RW; ++j) acc = fmaf(s_wy[ly][j], s_h[R * ly + j][lane], acc);
        const size_t o = (size_t)b * h * w + (size_t)y * w + x;
        const float sm = gN ? mul_rn(smooth_weight, fmaf(gN[o], inv_m, -corr)) : 0.0f;
        grad[o] = g_smooth ? fmaf(g_smooth[0], sm, mul_rn(up, acc)) : mul_rn(up, add_rn(acc, sm));
    }
}

template <int R>
__global__ void __launch_bounds__(256)
disp_grad_up_kernel(const float* __restrict__ G_full, const float* __restrict__ gN,
                    const float* __restrict__ img_scalars, float smooth_weight, const float* __restrict__ g_total,
                    const float* __restrict__ g_scale, const float* __restrict__ g_smooth, float inv_S, int h, int w,
                    int H, int W, float sh, float sw, float* __restrict__ grad) {
    __shared__ float smem[DG_UP_SMEM(R)];
    disp_grad_up_body<R>(G_full, gN, img_scalars, smooth_weight, g_total, g_scale, g_smooth, inv_S, h, w, H, W, sh, sw,
                         grad, blockIdx.x, blockIdx.y, blockIdx.z, threadIdx.x, threadIdx.y, smem);
}

// Same-size case (scale 0) of dmh_disp_grad: pure elementwise, 4 pixels per thread (128-bit loads / stores).
__device__ __forceinline__ void disp_grad_same_body(const float4* __restrict__ G4, const float4* __restrict__ gN4,
                                                    const float* __restrict__ img_scalars, float smooth_weight,
                                                    const float* __restrict__ g_total, const float* __restrict__ g_scale,
                                                    const float* __restrict__ g_smooth, float inv_S, int n4,
                                                    float4* __restrict__ grad4, int i, int b) {
    if (i >= n4) return;
    const float up = add_rn(g_total ? mul_rn(g_total[0], inv_S) : 0.0f, g_scale ? g_scale[0] : 0.0f);
    const size_t o = (size_t)b * n4 + i;
    const float4 a = __ldg(G4 + o);
    float acc[4] = {a.x, a.y, a.z, a.w}, sm[4] = {0.f, 0.f, 0.f, 0.f}, out[4];
    if (gN4) {
        const float inv_m = img_scalars[b * 2], corr = img_scalars[b * 2 + 1];
        const float4 n = __ldg(gN4 + o);
        const float nv[4] = {n.x, n.y, n.z, n.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) sm[j] = mul_rn(smooth_weight, fmaf(nv[j], inv_m, -corr));
    }
    const float gsm = g_smooth ? g_smooth[0] : 0.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) out[j] = g_smooth ? fmaf(gsm, sm[j], mul_rn(up, acc[j])) : mul_rn(up, add_rn(acc[j], sm[j]));
    grad4[o] = make_float4(out[0], out[1], out[2], out[3]);
}

__global__ void __launch_bounds__(256)
disp_grad_same_kernel(const float4* __restrict__ G4, const float4* __restrict__ gN4, const float* __restrict__ img_scalars,
                      float smooth_weight, const float* __restrict__ g_total, const float* __restrict__ g_scale,
                      const float* __restrict__ g_smooth, float inv_S, int n4, float4* __restrict__ grad4) {
    disp_grad_same_body(G4, gN4, img_scalars, smooth_weight, g_total, g_scale, g_smooth, inv_S, n4, grad4,
                        blockIdx.x * blockDim.x + threadIdx.x, blockIdx.y);
}

template <int R>
__global__ void __launch_bounds__(256)
disp_grad_kernel(const float* __restrict__ G_full, const float* __restrict__ gN,
                 const float* __restrict__ img_scalars, float smooth_weight, const float* __restrict__ g_total,
                 const float* __restrict__ g_scale, const float* __restrict__ g_smooth, float inv_S, int h, int w,
                 int H, int W, float sh, float sw, float* __restrict__ grad) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    const bool in = x < w && y < h;
    if (R <= 1 && !in) return;                            // (R > 1: every thread works on the tile)
    const int b = blockIdx.z;
    const float up = add_rn(g_total ? mul_rn(g_total[0], inv_S) : 0.0f, g_scale ? g_scale[0] : 0.0f);
    const float* g = G_full + (size_t)b * H * W;
    float acc;
    if (R == 1) {
        acc = __ldg(g + (size_t)y * W + x);
    } else if (R > 1) {
        constexpr int RW = R > 0 ? 2 * R : 1, RR = R > 0 ? R : 1, NR = 9 * RR;
        __shared__ float s_wy[8][RW], s_wx[32][RW];
        __shared__ float s_h[NR][32];
        const int lane = threadIdx.x, wid = threadIdx.y;
        const int t = wid * 32 + lane;
        // weights depend only on (y, offset) / (x, offset): tabulated once per CTA with the forward's up_tap
        for (int i = t; i < 8 * RW + 32 * RW; i += 256) {
            if (i < 8 * RW) {
                const int ly = i / RW, j = i % RW;
                const int yy = blockIdx.y * 8 + ly, Y = R * yy - R / 2 + j;
                float wv = 0.f;
                if (yy < h && Y >= 0 && Y < H) { const UpTap tp = up_tap(Y, sh, h); wv = (tp.i0 == yy ? tp.l0 : 0.f) + (tp.i1 == yy ? tp.l1 : 0.f); }
                s_wy[ly][j] = wv;
            } else {
                const int k = i - 8 * RW;
                const int lx = k / RW, j = k % RW;
                const int xx = blockIdx.x * 32 + lx, X = R * xx - R / 2 + j;
                float wv = 0.f;
                if (xx < w && X >= 0 && X < W) { const UpTap tp = up_tap(X, sw, w); wv = (tp.i0 == xx ? tp.l0 : 0.f) + (tp.i1 == xx ? tp.l1 : 0.f); }
                s_wx[lx][j] = wv;
            }
        }
        __syncthreads();
        float wA[RR], wB[RR], wE[RR];                       // chunk c -> low-res c, chunk c -> low-res c-1, chunk 32 -> 31
#pragma unroll
        for (int j = 0; j < RR; ++j) {
            wA[j] = s_wx[lane][j];
            wB[j] = lane > 0 ? s_wx[lane - 1][RR + j] : 0.f;
            wE[j] = s_wx[31][RR + j];
        }
        const int Xc = R * x - R / 2;                        // first full-res column of this lane's chunk
        const int Xe = R * (blockIdx.x * 32 + 32) - R / 2;  // chunk 32 (lane 0 takes it)
        const int Yt = R * (blockIdx.y * 8) - R / 2;        // first full-res row of the tile's window
        // rows of this warp: wid, wid + 8, ...; the loads of a batch of rows are issued before any is consumed
        constexpr int NPW = (NR + 7) / 8, BS = RR >= 8 ? 3 : NPW;
#pragma unroll
        for (int i0 = 0; i0 < NPW; i0 += BS) {
            float v[BS][RR], ve[BS][RR];
#pragma unroll
            for (int i = 0; i < BS; ++i) {
                const int ry = wid + 8 * (i0 + i), Y = Yt + ry;
                const bool ok = i0 + i < NPW && ry < NR && Y >= 0 && Y < H;      // warp-uniform
                const float* grow = g + (size_t)(ok ? Y : 0) * W;
                if (ok) load_chunk<RR>(grow, Xc, W, v[i]);
                else {
#pragma unroll
                    for (int j = 0; j < RR; ++j) v[i][j] = 0.f;
                }
                if (ok && lane == 0) load_chunk<RR>(grow, Xe, W, ve[i]);
                else {
#pragma unroll
                    for (int j = 0; j < RR; ++j) ve[i][j] = 0.f;
                }
            }
#pragma unroll
            for (int i = 0; i < BS; ++i) {
                const int ry = wid + 8 * (i0 + i);
                float a = 0.f, bm = 0.f, e = 0.f;
#pragma unroll
                for (int j = 0; j < RR; ++j) {
                    a = fmaf(wA[j], v[i][j], a); bm = fmaf(wB[j], v[i][j], bm); e = fmaf(wE[j], ve[i][j], e);
                }
                float nb = __shfl_down_sync(0xffffffffu, bm, 1);
                const float ee = __shfl_sync(0xffffffffu, e, 0);
                if (lane == 31) nb = ee;
                if (i0 + i < NPW && ry < NR) s_h[ry][lane] = a + nb;
            }
        }
        __syncthreads();
        if (!in) return;
        acc = 0.0f;
#pragma unroll
        for (int j = 0; j < RW; ++j) acc = fmaf(s_wy[wid][j], s_h[R * wid + j][lane], acc);
    } else {
        const float rh = 1.0f / sh, rw = 1.0f / sw;
        const int Y0 = max(0, (int)floorf(((float)y - 0.5f) * rh - 0.5f) - 1);
        const int Y1 = min(H - 1, (int)ceilf(((float)y + 1.5f) * rh - 0.5f) + 1);
        const int X0 = max(0, (int)floorf(((float)x - 0.5f) * rw - 0.5f) - 1);
        const int X1 = min(W - 1, (int)ceilf(((float)x + 1.5f) * rw - 0.5f) + 1);
        acc = 0.0f;
        for (int Y = Y0; Y <= Y1; ++Y) {
            const UpTap ty = up_tap(Y, sh, h);
            const float wy = (ty.i0 == y ? ty.l0 : 0.0f) + (ty.i1 == y ? ty.l1 : 0.0f);
            if (wy == 0.0f) continue;
            float row = 0.0f;
            for (int X = X0; X <= X1; ++X) {
                const UpTap tx = up_tap(X, sw, w);
                const float wx = (tx.i0 == x ? tx.l0 : 0.0f) + (tx.i1 == x ? tx.l1 : 0.0f);
                if (wx != 0.0f) row = fmaf(wx, __ldg(g + (size_t)Y * W + X), row);
            }
            acc = fmaf(wy, row, acc);
        }
    }
    float sm = 0.0f;
    if (gN) {
        const float inv_m = img_scalars[b * 2], corr = img_scalars[b * 2 + 1];
        sm = mul_rn(smooth_weight, fmaf(gN[(size_t)b * h * w + (size_t)y * w + x], inv_m, -corr));
    }
    // g_smooth: separate upstream weight of the smoothness term (depth-hints objective: the photometric
    // gradients arrive already weighted by their masked-mean denominators)
    grad[(size_t)b * h * w + (size_t)y * w + x] = g_smooth ? fmaf(g_smooth[0], sm, mul_rn(up, acc)) : mul_rn(up, add_rn(acc, sm));
}

}  // namespace

extern "C" {

long long dmh_smooth_fused_workspace_floats(int B, int h, int w) {
    return (long long)B * SF_NB1 + 3LL * B * SF_BLOCKS(h, w);
}

int dmh_smooth_fused(const float* disp, const float* img, int B, int C, int h, int w, float* ws, float* gN,
                     dmh_stream_t stream) {
    DMH_REQUIRE(disp && img && ws && gN, "dmh_smooth_fused: null pointer");
    DMH_REQUIRE(B > 0 && B <= 65535 && (C == 3 || C == 1) && h >= 2 && w >= 2,
                "dmh_smooth_fused: bad shape (the image must have 3 channels or 1)");
    cudaStream_t st = (cudaStream_t)stream;
    DMH_LAUNCH(sf_mean_kernel, dim3(SF_NB1, B), 256, 0, st)(disp, h * w, ws);
    const float inv_nx = (float)(1.0 / ((double)B * h * (w - 1))), inv_ny = (float)(1.0 / ((double)B * (h - 1) * w));
    const int vec = (w % 4 == 0) && (((uintptr_t)disp | (uintptr_t)img | (uintptr_t)gN) % 16 == 0);
    const dim3 grid(ceil_div(w, SF_TW), ceil_div(h, SF_TH), B);
    float* part = ws + (size_t)B * SF_NB1;
    if (C == 3)
        DMH_LAUNCH(sf_main_kernel<3>, grid, SF_THREADS, 0, st)(disp, img, h, w, ws, inv_nx, inv_ny, vec, gN, part);
    else
        DMH_LAUNCH(sf_main_kernel<1>, grid, SF_THREADS, 0, st)(disp, img, h, w, ws, inv_nx, inv_ny, vec, gN, part);
    DMH_CHECK_LAUNCH("dmh_smooth_fused");
    return DMH_OK;
}

long long dmh_objective_finish_workspace_bytes(int S, int B) { return 16 + 24LL * S * B; }

int dmh_objective_finish(int S, int B, const float* const* smooth_ws_host, const int* h_host, const int* w_host,
                         const float* const* photo_part_host, const int* photo_n_host,
                         const float* smooth_weight_host, double photo_den, void* workspace, float* img_scalars,
                         float* losses, dmh_stream_t stream) {
    DMH_REQUIRE(S >= 1 && S <= FIN_MAXS && B > 0, "dmh_objective_finish: S=%d outside [1,%d] or B <= 0", S, FIN_MAXS);
    DMH_REQUIRE(smooth_ws_host && h_host && w_host && photo_part_host && photo_n_host && smooth_weight_host &&
                    workspace && img_scalars && losses && photo_den > 0.0,
                "dmh_objective_finish: null pointer");
    DMH_REQUIRE(((uintptr_t)workspace & 15) == 0, "dmh_objective_finish: workspace must be 16-byte aligned");
    FinishParams p;
    for (int s = 0; s < S; ++s) {
        DMH_REQUIRE(smooth_ws_host[s] && photo_part_host[s], "dmh_objective_finish: null buffer for scale %d", s);
        p.smooth_ws[s] = smooth_ws_host[s];
        p.photo_part[s] = photo_part_host[s];
        p.photo_n[s] = photo_n_host[s];
        p.h[s] = h_host[s];
        p.w[s] = w_host[s];
        p.smooth_weight[s] = smooth_weight_host[s];
    }
    p.S = S; p.B = B; p.inv_photo_den = 1.0 / photo_den; p.img_scalars = img_scalars; p.losses = losses;
    p.ticket = reinterpret_cast<unsigned*>(workspace);
    p.img_sums = reinterpret_cast<double*>(reinterpret_cast<char*>(workspace) + 16);
    cudaError_t e = cudaMemsetAsync(workspace, 0, 16, (cudaStream_t)stream);
    if (e != cudaSuccess) { set_error("dmh_objective_finish: memset failed: %s", cudaGetErrorString(e)); return DMH_ERR_CUDA; }
    DMH_LAUNCH(finish_kernel, S * B, 256, 0, (cudaStream_t)stream)(p);
    DMH_CHECK_LAUNCH("dmh_objective_finish");
    return DMH_OK;
}

int dmh_disp_grad(const float* G_full, const float* gN, const float* img_scalars, float smooth_weight,
                  const float* g_total, const float* g_scale, const float* g_smooth, float inv_S, int B, int h, int w,
                  int H, int W, float* grad_disp, dmh_stream_t stream) {
    DMH_REQUIRE(G_full && grad_disp && (g_total || g_scale), "dmh_disp_grad: null pointer");
    DMH_REQUIRE(!gN || img_scalars, "dmh_disp_grad: gN given without img_scalars");
    DMH_REQUIRE(B > 0 && B <= 65535 && h >= 1 && w >= 1 && H >= h && W >= w, "dmh_disp_grad: bad shape");
    dim3 block(32, 8), grid(ceil_div(w, 32), ceil_div(h, 8), B);
    const float sh = (float)h / (float)H, sw = (float)w / (float)W;
    cudaStream_t st = (cudaStream_t)stream;
    int R = 0;                                   // integer up-scale factor shared by both axes, else generic
    if (H % h == 0 && W % w == 0 && H / h == W / w) R = H / h;
    if (R > 1 && ((uintptr_t)G_full % 16 != 0 || W % 4 != 0)) R = 0;   // vector loads need aligned rows
#define DMH_DG(RR) DMH_LAUNCH(disp_grad_kernel<RR>, grid, block, 0, st)(G_full, gN, img_scalars, smooth_weight, g_total, \
                                                                       g_scale, g_smooth, inv_S, h, w, H, W, sh, sw, grad_disp)
    if (R == 1 && ((size_t)h * w) % 4 == 0 && (uintptr_t)G_full % 16 == 0 && (uintptr_t)grad_disp % 16 == 0 &&
        (!gN || (uintptr_t)gN % 16 == 0)) {
        const int n4 = (int)(((size_t)h * w) / 4);
        DMH_LAUNCH(disp_grad_same_kernel, dim3(ceil_div(n4, 256), B), 256, 0, st)(
            reinterpret_cast<const float4*>(G_full), reinterpret_cast<const float4*>(gN), img_scalars, smooth_weight,
            g_total, g_scale, g_smooth, inv_S, n4, reinterpret_cast<float4*>(grad_disp));
    } else if (R == 1) DMH_DG(1);
    else if (R == 2 || R == 4 || R == 8) {
        const dim3 gtall(ceil_div(w, 32), ceil_div(h, 64 / R), B);
#define DMH_DGU(RR) DMH_LAUNCH(disp_grad_up_kernel<RR>, gtall, block, 0, st)(G_full, gN, img_scalars, smooth_weight, g_total, \
                                                                           g_scale, g_smooth, inv_S, h, w, H, W, sh, sw, grad_disp)
        if (R == 2) DMH_DGU(2);
        else if (R == 4) DMH_DGU(4);
        else DMH_DGU(8);
#undef DMH_DGU
    }
    else DMH_DG(0);
#undef DMH_DG
    DMH_CHECK_LAUNCH("dmh_disp_grad");
    return DMH_OK;
}

}  // extern "C"
