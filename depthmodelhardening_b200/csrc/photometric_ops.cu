// Op-level kernels behind the drop-in classes BackprojectDepth, Project3D, SSIM,
// compute_reprojection_loss, F.grid_sample (bilinear) and disp_to_depth.
// These keep the reference's tensor boundaries (one op = one materialised
// tensor); the fused fast path lives in photometric_fused.cu.
//
// All kernels are HBM-streaming: one thread per pixel (or 4 pixels), coalesced
// along W, grids sized by the problem (>= several waves of 148 SMs at the
// benchmark sizes).  No tensor cores: the largest contraction on this path has
// inner dimension 4 (SURVEY.md section 2, "ATen call sites").
#include "../../include/dmh_b200.h"
#include "dmh_common.cuh"

using namespace dmh;

namespace {

// ------------------------------------------------------------------ A9
__global__ void disp_to_depth_kernel(const float* __restrict__ disp, long long n, DepthScale ds,
                                     float* __restrict__ scaled, float* __restrict__ depth) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (; i < n; i += stride) {
        const float s = add_rn(ds.min_disp, mul_rn(ds.range, disp[i]));
        if (scaled) scaled[i] = s;
        if (depth) depth[i] = div_rn(1.0f, s);
    }
}

// ------------------------------------------------------------------ A10
__global__ void backproject_fwd_kernel(const float* __restrict__ depth, const float* __restrict__ inv_K, int H,
                                       int W, float* __restrict__ points) {
    const int b = blockIdx.y;
    const int N = H * W;
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    Camera cam;
    const float* iK = inv_K + b * 16;
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) cam.iK[i * 3 + j] = __ldg(iK + i * 4 + j);
    const float x = (float)(n % W), y = (float)(n / W);
    float ray[3];
    pixel_ray(cam, x, y, ray);
    const float d = depth[(size_t)b * N + n];
    float* out = points + (size_t)b * 4 * N + n;
    out[0] = mul_rn(d, ray[0]);
    out[(size_t)N] = mul_rn(d, ray[1]);
    out[(size_t)2 * N] = mul_rn(d, ray[2]);
    out[(size_t)3 * N] = 1.0f;
}

#define BP_BWD_THREADS 256
// grad_depth (nullable) and, when giK_partial != nullptr, the per-block partials of
// d/d(inv_K[:3,:3])_ij = sum_n g_i(n) * depth(n) * pix_j(n), pix = (x, y, 1)
__global__ void __launch_bounds__(BP_BWD_THREADS)
backproject_bwd_kernel(const float* __restrict__ gpts, const float* __restrict__ depth,
                       const float* __restrict__ inv_K, int H, int W, float* __restrict__ gdepth,
                       float* __restrict__ giK_partial) {
    __shared__ float red[32];
    const int b = blockIdx.y;
    const int N = H * W;
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    float gd[3] = {0.f, 0.f, 0.f};
    float pix[3] = {0.f, 0.f, 0.f};
    if (n < N) {
        const float* g = gpts + (size_t)b * 4 * N + n;
        gd[0] = g[0]; gd[1] = g[(size_t)N]; gd[2] = g[(size_t)2 * N];
        pix[0] = (float)(n % W); pix[1] = (float)(n / W); pix[2] = 1.0f;
        if (gdepth) {
            Camera cam;
            const float* iK = inv_K + b * 16;
#pragma unroll
            for (int i = 0; i < 3; ++i)
#pragma unroll
                for (int j = 0; j < 3; ++j) cam.iK[i * 3 + j] = __ldg(iK + i * 4 + j);
            float ray[3];
            pixel_ray(cam, pix[0], pix[1], ray);
            gdepth[(size_t)b * N + n] = gd[0] * ray[0] + gd[1] * ray[1] + gd[2] * ray[2];
        }
        if (giK_partial) {
            const float d = depth[(size_t)b * N + n];
            gd[0] *= d; gd[1] *= d; gd[2] *= d;
        }
    }
    if (giK_partial) {
        float* out = giK_partial + ((size_t)b * gridDim.x + blockIdx.x) * 9;
#pragma unroll
        for (int i = 0; i < 3; ++i)
#pragma unroll
            for (int j = 0; j < 3; ++j) {
                const float s = block_sum(gd[i] * pix[j], red);
                if (threadIdx.x == 0) out[i * 3 + j] = s;
            }
    }
}

// ------------------------------------------------------------------ A11
__device__ __forceinline__ void load_P(const float* K, const float* T, int b, float P[12]) {
    const float* k = K + b * 16;
    const float* t = T + b * 16;
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            float acc = __ldg(k + i * 4) * __ldg(t + j);
            acc = fmaf(__ldg(k + i * 4 + 1), __ldg(t + 4 + j), acc);
            acc = fmaf(__ldg(k + i * 4 + 2), __ldg(t + 8 + j), acc);
            acc = fmaf(__ldg(k + i * 4 + 3), __ldg(t + 12 + j), acc);
            P[i * 4 + j] = acc;
        }
}

__global__ void project3d_fwd_kernel(const float* __restrict__ points, const float* __restrict__ K,
                                     const float* __restrict__ T, int H, int W, float eps,
                                     float* __restrict__ grid) {
    const int b = blockIdx.y;
    const int N = H * W;
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    float P[12];
    load_P(K, T, b, P);
    const float* pt = points + (size_t)b * 4 * N + n;
    const float X = pt[0], Y = pt[(size_t)N], Z = pt[(size_t)2 * N], Wh = pt[(size_t)3 * N];
    float p[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        float acc = P[i * 4] * X;
        acc = fmaf(P[i * 4 + 1], Y, acc);
        acc = fmaf(P[i * 4 + 2], Z, acc);
        acc = fmaf(P[i * 4 + 3], Wh, acc);
        p[i] = acc;
    }
    const float z = add_rn(p[2], eps);
    float2 g;
    g.x = normalise_coord(p[0], z, W);
    g.y = normalise_coord(p[1], z, H);
    reinterpret_cast<float2*>(grid)[(size_t)b * N + n] = g;
}

#define P3D_BWD_THREADS 256
__global__ void project3d_bwd_kernel(const float* __restrict__ ggrid, const float* __restrict__ points,
                                     const float* __restrict__ K, const float* __restrict__ T, int H, int W,
                                     float eps, float* __restrict__ gpoints, float* __restrict__ gP_partial) {
    __shared__ float red[32];
    const int b = blockIdx.y;
    const int N = H * W;
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    float P[12];
    load_P(K, T, b, P);
    float dp[3] = {0.f, 0.f, 0.f};
    float pt4[4] = {0.f, 0.f, 0.f, 0.f};
    if (n < N) {
        const float* pt = points + (size_t)b * 4 * N + n;
        pt4[0] = pt[0]; pt4[1] = pt[(size_t)N]; pt4[2] = pt[(size_t)2 * N]; pt4[3] = pt[(size_t)3 * N];
        float p[3];
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            float acc = P[i * 4] * pt4[0];
            acc = fmaf(P[i * 4 + 1], pt4[1], acc);
            acc = fmaf(P[i * 4 + 2], pt4[2], acc);
            acc = fmaf(P[i * 4 + 3], pt4[3], acc);
            p[i] = acc;
        }
        const float z = add_rn(p[2], eps);
        const float inv_z = 1.0f / z;
        const float u = div_rn(p[0], z), v = div_rn(p[1], z);
        const float2 g = reinterpret_cast<const float2*>(ggrid)[(size_t)b * N + n];
        const float gu = g.x * (2.0f / (float)(W - 1));
        const float gv = g.y * (2.0f / (float)(H - 1));
        dp[0] = gu * inv_z;
        dp[1] = gv * inv_z;
        dp[2] = -(gu * u + gv * v) * inv_z;
        if (gpoints) {
            float* go = gpoints + (size_t)b * 4 * N + n;
#pragma unroll
            for (int j = 0; j < 4; ++j) go[(size_t)j * N] = P[j] * dp[0] + P[4 + j] * dp[1] + P[8 + j] * dp[2];
        }
    }
    if (gP_partial) {
        float* out = gP_partial + ((size_t)b * gridDim.x + blockIdx.x) * 12;
#pragma unroll
        for (int i = 0; i < 3; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float s = block_sum(dp[i] * pt4[j], red);
                if (threadIdx.x == 0) out[i * 4 + j] = s;
            }
    }
}

// ------------------------------------------------------------------ A12
struct SampleCoord { float ix, iy, mx, my; };

// A NaN coordinate under border padding: ATen's CUDA forward clips with fmin/fmax (NaN -> 0, the sample reads
// column / row 0), while its backward clips with comparisons (clip_coordinates_set_grad lets NaN through) and then
// safe_downgrade_to_int_range sends it to -100, so the gradient pass scatters nothing.  `for_grad` picks the latter.
__device__ __forceinline__ SampleCoord sample_coord(float gx, float gy, int Ws, int Hs, int padding_mode,
                                                    bool align_corners, bool for_grad) {
    SampleCoord s;
    float ux = unnormalise_coord(gx, Ws, align_corners);
    float uy = unnormalise_coord(gy, Hs, align_corners);
    float cx = 1.0f, cy = 1.0f;
    if (padding_mode == DMH_PAD_BORDER) {
        ux = (ux == ux || for_grad) ? clip_coord(ux, Ws, cx) : (cx = 0.0f, 0.0f);
        uy = (uy == uy || for_grad) ? clip_coord(uy, Hs, cy) : (cy = 0.0f, 0.0f);
    }
    s.ix = safe_coord(ux);
    s.iy = safe_coord(uy);
    s.mx = cx * unnormalise_mult(Ws, align_corners);
    s.my = cy * unnormalise_mult(Hs, align_corners);
    return s;
}

__global__ void grid_sample_fwd_kernel(const float* __restrict__ src, const float* __restrict__ grid, int C, int Hs,
                                       int Ws, int Ho, int Wo, int padding_mode, int align_corners,
                                       float* __restrict__ out) {
    const int b = blockIdx.y;
    const int No = Ho * Wo;
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= No) return;
    const float2 g = reinterpret_cast<const float2*>(grid)[(size_t)b * No + n];
    const SampleCoord sc = sample_coord(g.x, g.y, Ws, Hs, padding_mode, align_corners != 0, false);
    const Bilinear bl = bilinear_setup(sc.ix, sc.iy);
    const bool x0in = bl.x0 >= 0 && bl.x0 < Ws, x1in = bl.x0 + 1 >= 0 && bl.x0 + 1 < Ws;
    const bool y0in = bl.y0 >= 0 && bl.y0 < Hs, y1in = bl.y0 + 1 >= 0 && bl.y0 + 1 < Hs;
    const size_t plane = (size_t)Hs * Ws;
    const float* s = src + (size_t)b * C * plane;
    const long long o00 = (long long)bl.y0 * Ws + bl.x0;
    for (int c = 0; c < C; ++c) {
        const float* sp = s + c * plane;
        float acc = 0.0f;
        if (y0in && x0in) acc = fmaf(__ldg(sp + o00), bl.wnw, acc);
        if (y0in && x1in) acc = fmaf(__ldg(sp + o00 + 1), bl.wne, acc);
        if (y1in && x0in) acc = fmaf(__ldg(sp + o00 + Ws), bl.wsw, acc);
        if (y1in && x1in) acc = fmaf(__ldg(sp + o00 + Ws + 1), bl.wse, acc);
        out[((size_t)b * C + c) * No + n] = acc;
    }
}

__global__ void grid_sample_bwd_kernel(const float* __restrict__ gout, const float* __restrict__ src,
                                       const float* __restrict__ grid, int C, int Hs, int Ws, int Ho, int Wo,
                                       int padding_mode, int align_corners, float* __restrict__ gsrc,
                                       float* __restrict__ ggrid) {
    const int b = blockIdx.y;
    const int No = Ho * Wo;
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= No) return;
    const float2 g = reinterpret_cast<const float2*>(grid)[(size_t)b * No + n];
    const SampleCoord sc = sample_coord(g.x, g.y, Ws, Hs, padding_mode, align_corners != 0, true);
    const Bilinear bl = bilinear_setup(sc.ix, sc.iy);
    const bool x0in = bl.x0 >= 0 && bl.x0 < Ws, x1in = bl.x0 + 1 >= 0 && bl.x0 + 1 < Ws;
    const bool y0in = bl.y0 >= 0 && bl.y0 < Hs, y1in = bl.y0 + 1 >= 0 && bl.y0 + 1 < Hs;
    const size_t plane = (size_t)Hs * Ws;
    const long long o00 = (long long)bl.y0 * Ws + bl.x0;
    float gix = 0.0f, giy = 0.0f;
    for (int c = 0; c < C; ++c) {
        const float go = gout[((size_t)b * C + c) * No + n];
        const float* sp = src + ((size_t)b * C + c) * plane;
        float* gp = gsrc ? gsrc + ((size_t)b * C + c) * plane : nullptr;
        if (y0in && x0in) {
            const float v = __ldg(sp + o00);
            gix -= v * bl.ty1 * go; giy -= v * bl.tx1 * go;
            if (gp) atomicAdd(gp + o00, bl.wnw * go);
        }
        if (y0in && x1in) {
            const float v = __ldg(sp + o00 + 1);
            gix += v * bl.ty1 * go; giy -= v * bl.tx0 * go;
            if (gp) atomicAdd(gp + o00 + 1, bl.wne * go);
        }
        if (y1in && x0in) {
            const float v = __ldg(sp + o00 + Ws);
            gix -= v * bl.ty0 * go; giy += v * bl.tx1 * go;
            if (gp) atomicAdd(gp + o00 + Ws, bl.wsw * go);
        }
        if (y1in && x1in) {
            const float v = __ldg(sp + o00 + Ws + 1);
            gix += v * bl.ty0 * go; giy += v * bl.tx0 * go;
            if (gp) atomicAdd(gp + o00 + Ws + 1, bl.wse * go);
        }
    }
    if (ggrid) {
        float2 r;
        r.x = sc.mx * gix;
        r.y = sc.my * giy;
        reinterpret_cast<float2*>(ggrid)[(size_t)b * No + n] = r;
    }
}

// ------------------------------------------------------------------ A13 / A14 forward
// One thread per output pixel; the 3x3 windows are read straight from global
// through the read-only path (L1 holds the row reuse).  Row-major 9-term sums
// then /9, the order ATen's avg_pool2d uses.
__device__ __forceinline__ float ssim_at(const float* __restrict__ xp, const float* __restrict__ yp, int px, int py,
                                         int H, int W) {
    float sx = 0.f, sy = 0.f, sxx = 0.f, syy = 0.f, sxy = 0.f;
#pragma unroll
    for (int dy = -1; dy <= 1; ++dy) {
        const int ry = reflect1(py + dy, H);
#pragma unroll
        for (int dx = -1; dx <= 1; ++dx) {
            const int rx = reflect1(px + dx, W);
            const float a = __ldg(xp + (size_t)ry * W + rx);
            const float c = __ldg(yp + (size_t)ry * W + rx);
            sx = add_rn(sx, a);
            sy = add_rn(sy, c);
            sxx = add_rn(sxx, mul_rn(a, a));
            syy = add_rn(syy, mul_rn(c, c));
            sxy = add_rn(sxy, mul_rn(a, c));
        }
    }
    float pass;
    return ssim_value(ssim_stats(sx, sy, sxx, syy, sxy), pass);
}

__global__ void ssim_fwd_kernel(const float* __restrict__ x, const float* __restrict__ y, int H, int W,
                                float* __restrict__ out) {
    const int px = blockIdx.x * blockDim.x + threadIdx.x;
    const int py = blockIdx.y * blockDim.y + threadIdx.y;
    if (px >= W || py >= H) return;
    const size_t plane = (size_t)H * W;
    const size_t base = (size_t)blockIdx.z * plane;
    out[base + (size_t)py * W + px] = ssim_at(x + base, y + base, px, py, H, W);
}

__global__ void reproj_loss_fwd_kernel(const float* __restrict__ pred, const float* __restrict__ target, int C,
                                       int H, int W, int no_ssim, float* __restrict__ out) {
    const int px = blockIdx.x * blockDim.x + threadIdx.x;
    const int py = blockIdx.y * blockDim.y + threadIdx.y;
    if (px >= W || py >= H) return;
    const int b = blockIdx.z;
    const size_t plane = (size_t)H * W;
    const size_t pix = (size_t)py * W + px;
    float l1 = 0.f, ss = 0.f;
    for (int c = 0; c < C; ++c) {
        const size_t base = ((size_t)b * C + c) * plane;
        l1 = add_rn(l1, fabsf(sub_rn(__ldg(target + base + pix), __ldg(pred + base + pix))));
        if (!no_ssim) ss = add_rn(ss, ssim_at(pred + base, target + base, px, py, H, W));
    }
    l1 = div_rn(l1, (float)C);
    float r = l1;
    if (!no_ssim) r = add_rn(mul_rn(0.85f, div_rn(ss, (float)C)), mul_rn(0.15f, l1));
    out[(size_t)b * plane + pix] = r;
}

// ------------------------------------------------------------------ A13 / A14 backward
// Tile kernel: x/y tiles with a 2-px (reflect) halo in shared memory; phase 1
// turns every valid window centre q of the 1-px ring into the gated linear
// coefficients of dS/d(tap) (dmh_math.cuh: ssim_coef); phase 2 is a weighted
// 3x3 box sum of those coefficient planes.  The box weights carry the
// reflection multiplicity: the pad row -1 is pixel row 1 again, so window centre
// 0 reaches pixel 1 twice.
#define ST_TW 32
#define ST_TH 16
#define ST_R2W (ST_TW + 4)
#define ST_R2H (ST_TH + 4)
#define ST_R1W (ST_TW + 2)
#define ST_R1H (ST_TH + 2)
#define ST_THREADS 256

// mode 0: SSIM op   (grad_out is (B,C,H,W), weight 1)
// mode 1: reprojection loss (grad_out is (B,1,H,W); SSIM weight 0.85/C, L1 weight 0.15/C; no_ssim: L1 weight 1/C)
__global__ void __launch_bounds__(ST_THREADS)
ssim_bwd_kernel(const float* __restrict__ gout, const float* __restrict__ x, const float* __restrict__ y, int C,
                int H, int W, int mode, int no_ssim, float* __restrict__ gx, float* __restrict__ gy) {
    __shared__ float sx[ST_R2H][ST_R2W];
    __shared__ float sy[ST_R2H][ST_R2W];
    __shared__ float cax[ST_R1H][ST_R1W];
    __shared__ float cay[ST_R1H][ST_R1W];
    __shared__ float cb[ST_R1H][ST_R1W];
    __shared__ float cc[ST_R1H][ST_R1W];
    const int tid = threadIdx.x;
    const int x0 = blockIdx.x * ST_TW, y0 = blockIdx.y * ST_TH;
    const int bc = blockIdx.z;
    const int b = bc / C;
    const size_t plane = (size_t)H * W;
    const float* xp = x + (size_t)bc * plane;
    const float* yp = y + (size_t)bc * plane;
    const float* gp = mode == 0 ? gout + (size_t)bc * plane : gout + (size_t)b * plane;
    const float w_ssim = mode == 0 ? 1.0f : (no_ssim ? 0.0f : 0.85f / (float)C);
    const float w_l1 = mode == 0 ? 0.0f : (no_ssim ? 1.0f / (float)C : 0.15f / (float)C);

    for (int i = tid; i < ST_R2H * ST_R2W; i += ST_THREADS) {
        const int r = i / ST_R2W, c = i % ST_R2W;
        const int iy = ext_to_img(y0 - 2 + r, H), ix = ext_to_img(x0 - 2 + c, W);
        sx[r][c] = __ldg(xp + (size_t)iy * W + ix);
        sy[r][c] = __ldg(yp + (size_t)iy * W + ix);
    }
    __syncthreads();
    for (int i = tid; i < ST_R1H * ST_R1W; i += ST_THREADS) {
        const int r = i / ST_R1W, c = i % ST_R1W;
        const int qy = y0 - 1 + r, qx = x0 - 1 + c;
        float k_ax = 0.f, k_ay = 0.f, k_b = 0.f, k_c = 0.f;
        if (w_ssim != 0.0f && qy >= 0 && qy < H && qx >= 0 && qx < W) {
            float s1 = 0.f, s2 = 0.f, s11 = 0.f, s22 = 0.f, s12 = 0.f;
#pragma unroll
            for (int dy = 0; dy < 3; ++dy)
#pragma unroll
                for (int dx = 0; dx < 3; ++dx) {
                    const float a = sx[r + dy][c + dx], d = sy[r + dy][c + dx];
                    s1 = add_rn(s1, a);
                    s2 = add_rn(s2, d);
                    s11 = add_rn(s11, mul_rn(a, a));
                    s22 = add_rn(s22, mul_rn(d, d));
                    s12 = add_rn(s12, mul_rn(a, d));
                }
            const SsimStats st = ssim_stats(s1, s2, s11, s22, s12);
            float pass;
            ssim_value(st, pass);
            const float g = __ldg(gp + (size_t)qy * W + qx) * w_ssim * pass;
            if (g != 0.0f) {
                const SsimCoef k = ssim_coef(st);
                k_ax = g * k.ax; k_ay = g * k.ay; k_b = g * k.b; k_c = g * k.c;
            }
        }
        cax[r][c] = k_ax; cay[r][c] = k_ay; cb[r][c] = k_b; cc[r][c] = k_c;
    }
    __syncthreads();
    for (int i = tid; i < ST_TH * ST_TW; i += ST_THREADS) {
        const int r = i / ST_TW, c = i % ST_TW;
        const int py = y0 + r, px = x0 + c;
        if (py >= H || px >= W) continue;
        float a_x = 0.f, a_y = 0.f, sb = 0.f, sc = 0.f;
#pragma unroll
        for (int dy = 0; dy < 3; ++dy) {
            const float wy = reflect_mult(py, py - 1 + dy, H);
#pragma unroll
            for (int dx = 0; dx < 3; ++dx) {
                const float w = wy * reflect_mult(px, px - 1 + dx, W);
                a_x = fmaf(w, cax[r + dy][c + dx], a_x);
                a_y = fmaf(w, cay[r + dy][c + dx], a_y);
                sb = fmaf(w, cb[r + dy][c + dx], sb);
                sc = fmaf(w, cc[r + dy][c + dx], sc);
            }
        }
        const float xv = sx[r + 2][c + 2], yv = sy[r + 2][c + 2];
        float l1 = 0.0f;
        if (w_l1 != 0.0f) {
            const float d = xv - yv;
            const float sg = d > 0.f ? 1.f : (d < 0.f ? -1.f : 0.f);
            l1 = __ldg(gp + (size_t)py * W + px) * w_l1 * sg;   // d|y-x|/dx
        }
        const size_t o = (size_t)bc * plane + (size_t)py * W + px;
        if (gx) gx[o] = a_x + sb * xv + sc * yv + l1;
        if (gy) gy[o] = a_y + sb * yv + sc * xv - l1;
    }
}

}  // namespace

// ============================================================================ C ABI
extern "C" {

int dmh_disp_to_depth(const float* disp, long long n, float min_depth, float max_depth, float* scaled_disp,
                      float* depth, dmh_stream_t stream) {
    DMH_REQUIRE(disp && n > 0, "dmh_disp_to_depth: null input or n <= 0");
    DepthScale ds;
    ds.min_disp = (float)(1.0 / (double)max_depth);
    ds.range = (float)(1.0 / (double)min_depth - 1.0 / (double)max_depth);
    const int blocks = (int)((n + 255) / 256 < 148 * 16 ? (n + 255) / 256 : 148 * 16);
    DMH_LAUNCH(disp_to_depth_kernel, blocks, 256, 0, (cudaStream_t)stream)(disp, n, ds, scaled_disp, depth);
    DMH_CHECK_LAUNCH("dmh_disp_to_depth");
    return DMH_OK;
}

int dmh_backproject_fwd(const float* depth, const float* inv_K, int B, int H, int W, float* points,
                        dmh_stream_t stream) {
    DMH_REQUIRE(depth && inv_K && points, "dmh_backproject_fwd: null pointer");
    DMH_REQUIRE(B > 0 && H > 0 && W > 0 && B <= 65535, "dmh_backproject_fwd: bad shape B=%d H=%d W=%d", B, H, W);
    dim3 grid(ceil_div((long long)H * W, 256), B);
    DMH_LAUNCH(backproject_fwd_kernel, grid, 256, 0, (cudaStream_t)stream)(depth, inv_K, H, W, points);
    DMH_CHECK_LAUNCH("dmh_backproject_fwd");
    return DMH_OK;
}

int dmh_backproject_bwd_blocks(int H, int W) { return ceil_div((long long)H * W, BP_BWD_THREADS); }

int dmh_backproject_bwd(const float* grad_points, const float* depth, const float* inv_K, int B, int H, int W,
                        float* grad_depth, float* grad_inv_K_partial, dmh_stream_t stream) {
    DMH_REQUIRE(grad_points && inv_K && (grad_depth || grad_inv_K_partial), "dmh_backproject_bwd: null pointer");
    DMH_REQUIRE(depth || !grad_inv_K_partial, "dmh_backproject_bwd: null pointer (depth is needed for grad_inv_K)");
    DMH_REQUIRE(B > 0 && H > 0 && W > 0 && B <= 65535, "dmh_backproject_bwd: bad shape");
    dim3 grid(dmh_backproject_bwd_blocks(H, W), B);
    DMH_LAUNCH(backproject_bwd_kernel, grid, BP_BWD_THREADS, 0, (cudaStream_t)stream)(grad_points, depth, inv_K, H, W,
                                                                                  grad_depth, grad_inv_K_partial);
    DMH_CHECK_LAUNCH("dmh_backproject_bwd");
    return DMH_OK;
}

int dmh_project3d_fwd(const float* points, const float* K, const float* T, int B, int H, int W, float eps,
                      float* grid_out, dmh_stream_t stream) {
    DMH_REQUIRE(points && K && T && grid_out, "dmh_project3d_fwd: null pointer");
    DMH_REQUIRE(B > 0 && H > 1 && W > 1 && B <= 65535, "dmh_project3d_fwd: bad shape");
    dim3 grid(ceil_div((long long)H * W, 256), B);
    DMH_LAUNCH(project3d_fwd_kernel, grid, 256, 0, (cudaStream_t)stream)(points, K, T, H, W, eps, grid_out);
    DMH_CHECK_LAUNCH("dmh_project3d_fwd");
    return DMH_OK;
}

int dmh_project3d_bwd_blocks(int H, int W) { return ceil_div((long long)H * W, P3D_BWD_THREADS); }

int dmh_project3d_bwd(const float* grad_grid, const float* points, const float* K, const float* T, int B, int H,
                      int W, float eps, float* grad_points, float* grad_P_partial, dmh_stream_t stream) {
    DMH_REQUIRE(grad_grid && points && K && T, "dmh_project3d_bwd: null pointer");
    DMH_REQUIRE(B > 0 && H > 1 && W > 1 && B <= 65535, "dmh_project3d_bwd: bad shape");
    dim3 grid(dmh_project3d_bwd_blocks(H, W), B);
    DMH_LAUNCH(project3d_bwd_kernel, grid, P3D_BWD_THREADS, 0, (cudaStream_t)stream)(grad_grid, points, K, T, H, W, eps,
                                                                            grad_points, grad_P_partial);
    DMH_CHECK_LAUNCH("dmh_project3d_bwd");
    return DMH_OK;
}

int dmh_grid_sample_fwd(const float* src, const float* grid, int B, int C, int Hs, int Ws, int Ho, int Wo,
                        int padding_mode, int align_corners, float* out, dmh_stream_t stream) {
    DMH_REQUIRE(src && grid && out, "dmh_grid_sample_fwd: null pointer");
    DMH_REQUIRE(B > 0 && C > 0 && Hs > 0 && Ws > 0 && Ho > 0 && Wo > 0 && B <= 65535, "dmh_grid_sample_fwd: bad shape");
    if (padding_mode != DMH_PAD_ZEROS && padding_mode != DMH_PAD_BORDER) {
        set_error("dmh_grid_sample_fwd: padding_mode %d unsupported (zeros|border only)", padding_mode);
        return DMH_ERR_UNSUPPORTED;
    }
    dim3 g(ceil_div((long long)Ho * Wo, 256), B);
    DMH_LAUNCH(grid_sample_fwd_kernel, g, 256, 0, (cudaStream_t)stream)(src, grid, C, Hs, Ws, Ho, Wo, padding_mode,
                                                               align_corners, out);
    DMH_CHECK_LAUNCH("dmh_grid_sample_fwd");
    return DMH_OK;
}

int dmh_grid_sample_bwd(const float* grad_out, const float* src, const float* grid, int B, int C, int Hs, int Ws,
                        int Ho, int Wo, int padding_mode, int align_corners, float* grad_src, float* grad_grid,
                        dmh_stream_t stream) {
    DMH_REQUIRE(grad_out && src && grid, "dmh_grid_sample_bwd: null pointer");
    DMH_REQUIRE(B > 0 && C > 0 && Hs > 0 && Ws > 0 && Ho > 0 && Wo > 0 && B <= 65535, "dmh_grid_sample_bwd: bad shape");
    if (padding_mode != DMH_PAD_ZEROS && padding_mode != DMH_PAD_BORDER) {
        set_error("dmh_grid_sample_bwd: padding_mode %d unsupported (zeros|border only)", padding_mode);
        return DMH_ERR_UNSUPPORTED;
    }
    dim3 g(ceil_div((long long)Ho * Wo, 256), B);
    DMH_LAUNCH(grid_sample_bwd_kernel, g, 256, 0, (cudaStream_t)stream)(grad_out, src, grid, C, Hs, Ws, Ho, Wo, padding_mode,
                                                               align_corners, grad_src, grad_grid);
    DMH_CHECK_LAUNCH("dmh_grid_sample_bwd");
    return DMH_OK;
}

int dmh_ssim_fwd(const float* x, const float* y, int B, int C, int H, int W, float* out, dmh_stream_t stream) {
    DMH_REQUIRE(x && y && out, "dmh_ssim_fwd: null pointer");
    DMH_REQUIRE(B > 0 && C > 0 && H >= 2 && W >= 2 && (long long)B * C <= 65535, "dmh_ssim_fwd: bad shape");
    dim3 block(32, 8), grid(ceil_div(W, 32), ceil_div(H, 8), B * C);
    DMH_LAUNCH(ssim_fwd_kernel, grid, block, 0, (cudaStream_t)stream)(x, y, H, W, out);
    DMH_CHECK_LAUNCH("dmh_ssim_fwd");
    return DMH_OK;
}

static int launch_ssim_bwd(const char* name, const float* grad_out, const float* x, const float* y, int B, int C,
                           int H, int W, int mode, int no_ssim, float* gx, float* gy, dmh_stream_t stream) {
    DMH_REQUIRE(grad_out && x && y, "%s: null pointer", name);
    DMH_REQUIRE(B > 0 && C > 0 && H >= 2 && W >= 2 && (long long)B * C <= 65535, "%s: bad shape", name);
    dim3 grid(ceil_div(W, ST_TW), ceil_div(H, ST_TH), B * C);
    DMH_LAUNCH(ssim_bwd_kernel, grid, ST_THREADS, 0, (cudaStream_t)stream)(grad_out, x, y, C, H, W, mode, no_ssim, gx, gy);
    DMH_CHECK_LAUNCH(name);
    return DMH_OK;
}

int dmh_ssim_bwd(const float* grad_out, const float* x, const float* y, int B, int C, int H, int W, float* grad_x,
                 float* grad_y, dmh_stream_t stream) {
    return launch_ssim_bwd("dmh_ssim_bwd", grad_out, x, y, B, C, H, W, 0, 0, grad_x, grad_y, stream);
}

int dmh_reproj_loss_fwd(const float* pred, const float* target, int B, int C, int H, int W, int no_ssim,
                        float* out, dmh_stream_t stream) {
    DMH_REQUIRE(pred && target && out, "dmh_reproj_loss_fwd: null pointer");
    DMH_REQUIRE(B > 0 && C > 0 && H >= 2 && W >= 2 && B <= 65535, "dmh_reproj_loss_fwd: bad shape");
    dim3 block(32, 8), grid(ceil_div(W, 32), ceil_div(H, 8), B);
    DMH_LAUNCH(reproj_loss_fwd_kernel, grid, block, 0, (cudaStream_t)stream)(pred, target, C, H, W, no_ssim, out);
    DMH_CHECK_LAUNCH("dmh_reproj_loss_fwd");
    return DMH_OK;
}

int dmh_reproj_loss_bwd(const float* grad_out, const float* pred, const float* target, int B, int C, int H, int W,
                        int no_ssim, float* grad_pred, float* grad_target, dmh_stream_t stream) {
    return launch_ssim_bwd("dmh_reproj_loss_bwd", grad_out, pred, target, B, C, H, W, 1, no_ssim, grad_pred,
                           grad_target, stream);
}

}  // extern "C"
