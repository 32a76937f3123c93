// A9-A12 fused gather (disp -> depth -> backproject -> project -> bilinear border
// warp) forward/backward, the smoothness term A16, and the deterministic sum.
//
// Roofline: HBM.  Algorithmic bytes per target pixel (fp32, C=3):
//   warp fwd  : 4 (disp) + 12 (src, gathered through L2) + 12 (warped out) = 28 B
//   warp bwd  : 12 (grad_warped) + 12 (src) + 4 (disp) + 4 (grad_disp)      = 32 B
//   smooth fwd: 4 (disp) + 12 (img) = 16 B ; bwd: 16 + 4 (grad_disp)       = 20 B
#include "../../include/dmh_b200.h"
#include "dmh_common.cuh"

using namespace dmh;

namespace {

#define WARP_THREADS 256

__device__ __forceinline__ void load_camera(const float* K, const float* inv_K, const float* T, int b,
                                            Camera& cam, float* smem /* >= 21 floats */) {
    // first 21 threads compose P and inv_K[:3,:3] once per CTA
    const int t = threadIdx.x;
    if (t < 12) {
        const int i = t / 4, j = t % 4;
        const float* k = K + b * 16 + i * 4;
        const float* tt = T + b * 16 + j;
        float acc = __ldg(k) * __ldg(tt);
        acc = fmaf(__ldg(k + 1), __ldg(tt + 4), acc);
        acc = fmaf(__ldg(k + 2), __ldg(tt + 8), acc);
        acc = fmaf(__ldg(k + 3), __ldg(tt + 12), acc);
        smem[t] = acc;
    } else if (t < 21) {
        const int i = (t - 12) / 3, j = (t - 12) % 3;
        smem[t] = __ldg(inv_K + b * 16 + i * 4 + j);
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 12; ++i) cam.P[i] = smem[i];
#pragma unroll
    for (int i = 0; i < 9; ++i) cam.iK[i] = smem[12 + i];
}

template <int C>
__global__ void __launch_bounds__(WARP_THREADS)
warp_fwd_kernel(const float* __restrict__ disp, int input_is_depth, DepthScale ds, const float* __restrict__ src,
                const float* __restrict__ K, const float* __restrict__ inv_K, const float* __restrict__ T, int Cdyn,
                int H, int W, float* __restrict__ warped, float* __restrict__ grid_out,
                float* __restrict__ depth_out) {
    __shared__ float cam_s[24];
    const int b = blockIdx.y;
    Camera cam;
    load_camera(K, inv_K, T, b, cam, cam_s);
    const int N = H * W;
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    const int px = n % W, py = n / W;
    const float dv = disp[(size_t)b * N + n];
    const bool is_depth = (input_is_depth & 1) != 0;
    const bool half_pixel = (input_is_depth & 2) != 0;      // grid_sample(align_corners=False): the depth-hints warp
    const float depth = is_depth ? dv : disp_to_depth(dv, ds);
    if (depth_out) depth_out[(size_t)b * N + n] = depth;
    const WarpCoord wc = warp_coord(cam, (float)px, (float)py, depth, W, H, 1e-7f);
    const float gxn = normalise_coord(wc.u_raw, 1.0f, W);   // u_raw already divided by z
    const float gyn = normalise_coord(wc.v_raw, 1.0f, H);
    if (grid_out) reinterpret_cast<float2*>(grid_out)[(size_t)b * N + n] = make_float2(gxn, gyn);
    float six = wc.ix, siy = wc.iy;
    if (half_pixel) {       // same op sequence as Project3D -> grid_sample(border, align_corners=False)
        six = clip_coord_fwd(unnormalise_coord(gxn, W, false), W);
        siy = clip_coord_fwd(unnormalise_coord(gyn, H, false), H);
    }
    const Bilinear bl = bilinear_setup(six, siy);
    const bool x0in = bl.x0 >= 0 && bl.x0 < W, x1in = bl.x0 + 1 >= 0 && bl.x0 + 1 < W;
    const bool y0in = bl.y0 >= 0 && bl.y0 < H, y1in = bl.y0 + 1 >= 0 && bl.y0 + 1 < H;
    const long long o00 = (long long)bl.y0 * W + bl.x0;
    const int Cn = C > 0 ? C : Cdyn;
#pragma unroll
    for (int c = 0; c < Cn; ++c) {
        const float* sp = src + ((size_t)b * Cn + c) * N;
        float acc = 0.0f;
        if (y0in && x0in) acc = fmaf(__ldg(sp + o00), bl.wnw, acc);
        if (y0in && x1in) acc = fmaf(__ldg(sp + o00 + 1), bl.wne, acc);
        if (y1in && x0in) acc = fmaf(__ldg(sp + o00 + W), bl.wsw, acc);
        if (y1in && x1in) acc = fmaf(__ldg(sp + o00 + W + 1), bl.wse, acc);
        warped[((size_t)b * Cn + c) * N + n] = acc;
    }
}

template <int C>
__global__ void __launch_bounds__(WARP_THREADS)
warp_bwd_kernel(const float* __restrict__ gwarped, const float* __restrict__ disp, int input_is_depth, DepthScale ds,
                const float* __restrict__ src, const float* __restrict__ K, const float* __restrict__ inv_K,
                const float* __restrict__ T, int Cdyn, int H, int W, float* __restrict__ gdisp,
                float* __restrict__ gsrc, float* __restrict__ gP_partial) {
    __shared__ float cam_s[24];
    __shared__ float red[32];
    const int b = blockIdx.y;
    Camera cam;
    load_camera(K, inv_K, T, b, cam, cam_s);
    const int N = H * W;
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    const bool active = n < N;
    const int nn = active ? n : N - 1;
    const int px = nn % W, py = nn / W;
    const float dv = disp[(size_t)b * N + nn];
    const float depth = input_is_depth ? dv : disp_to_depth(dv, ds);
    const WarpCoord wc = warp_coord(cam, (float)px, (float)py, depth, W, H, 1e-7f);
    const Bilinear bl = bilinear_setup(wc.ix, wc.iy);
    const bool x0in = bl.x0 >= 0 && bl.x0 < W, x1in = bl.x0 + 1 >= 0 && bl.x0 + 1 < W;
    const bool y0in = bl.y0 >= 0 && bl.y0 < H, y1in = bl.y0 + 1 >= 0 && bl.y0 + 1 < H;
    const long long o00 = (long long)bl.y0 * W + bl.x0;
    const int Cn = C > 0 ? C : Cdyn;
    const unsigned lane = threadIdx.x & 31;
    // east tap of this lane == west tap of lane+1 ?
    bool merge_e = false, recv_w = false;
    if (gsrc) {
        const int nx0 = __shfl_down_sync(0xffffffffu, bl.x0, 1);
        const int ny0 = __shfl_down_sync(0xffffffffu, bl.y0, 1);
        const int nact = __shfl_down_sync(0xffffffffu, (int)active, 1);
        merge_e = active && lane < 31 && nact && nx0 == bl.x0 + 1 && ny0 == bl.y0;
        recv_w = __shfl_up_sync(0xffffffffu, (int)merge_e, 1) != 0;
    }
    float gix = 0.0f, giy = 0.0f;
#pragma unroll
    for (int c = 0; c < Cn; ++c) {
        const float go = active ? gwarped[((size_t)b * Cn + c) * N + nn] : 0.0f;
        const float* sp = src + ((size_t)b * Cn + c) * N;
        if (y0in && x0in) { const float v = __ldg(sp + o00);         gix -= v * bl.ty1 * go; giy -= v * bl.tx1 * go; }
        if (y0in && x1in) { const float v = __ldg(sp + o00 + 1);     gix += v * bl.ty1 * go; giy -= v * bl.tx0 * go; }
        if (y1in && x0in) { const float v = __ldg(sp + o00 + W);     gix -= v * bl.ty0 * go; giy += v * bl.tx1 * go; }
        if (y1in && x1in) { const float v = __ldg(sp + o00 + W + 1); gix += v * bl.ty0 * go; giy += v * bl.tx0 * go; }
        if (gsrc) {
            float* gp = gsrc + ((size_t)b * Cn + c) * N;
            scatter_row(gp, o00, active && y0in && x0in, active && y0in && x1in, bl.wnw * go, bl.wne * go,
                        merge_e && y0in, recv_w, lane);
            scatter_row(gp, o00 + W, active && y1in && x0in, active && y1in && x1in, bl.wsw * go, bl.wse * go,
                        merge_e && y1in, recv_w, lane);
        }
    }
    float dp[3];
    float g_depth = warp_coord_bwd(cam, wc, gix, giy, W, H, dp);
    if (!active) { g_depth = 0.f; dp[0] = dp[1] = dp[2] = 0.f; }
    if (active && gdisp) gdisp[(size_t)b * N + n] = input_is_depth ? g_depth : g_depth * ddepth_ddisp(depth, ds);
    if (gP_partial) {
        const float pt[4] = {depth * wc.ray[0], depth * wc.ray[1], depth * wc.ray[2], 1.0f};
        float* out = gP_partial + ((size_t)b * gridDim.x + blockIdx.x) * 12;
#pragma unroll
        for (int i = 0; i < 3; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float s = block_sum(dp[i] * pt[j], red);
                if (threadIdx.x == 0) out[i * 4 + j] = s;
            }
    }
}

// ---------------------------------------------------------------------------- A16
#define SM_NB1 64          // partial blocks per image for the mean
#define SM_THREADS 256

__global__ void smooth_mean_kernel(const float* __restrict__ disp, int hw, float* __restrict__ part) {
    __shared__ float red[32];
    const int b = blockIdx.y;
    const float* d = disp + (size_t)b * hw;
    float s = 0.f;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < hw; i += gridDim.x * blockDim.x) s += d[i];
    s = block_sum(s, red);
    if (threadIdx.x == 0) part[b * SM_NB1 + blockIdx.x] = s;
}

// per-image denominator of trainer.py:663: mean(disp) + 1e-7 (1 when not normalising)
__device__ __forceinline__ float image_mean_eps(const float* part, int b, int hw, int normalise) {
    if (!normalise) return 1.0f;
    float s = 0.f;
    for (int i = 0; i < SM_NB1; ++i) s += part[b * SM_NB1 + i];
    return s / (float)hw + 1e-7f;
}

__device__ __forceinline__ float edge_weight(const float* __restrict__ img, int C, size_t plane, size_t a, size_t b2) {
    float s = 0.f;
    for (int c = 0; c < C; ++c) s += fabsf(img[c * plane + a] - img[c * plane + b2]);
    return expf(-(s / (float)C));
}
__device__ __forceinline__ float sgn(float v) { return v > 0.f ? 1.f : (v < 0.f ? -1.f : 0.f); }

__global__ void __launch_bounds__(SM_THREADS)
smooth_fwd_kernel(const float* __restrict__ disp, const float* __restrict__ img, int C, int h, int w, int normalise,
                  const float* __restrict__ mean_part, float* __restrict__ loss_part) {
    __shared__ float red[32];
    const int b = blockIdx.y;
    const int hw = h * w;
    const float m = image_mean_eps(mean_part, b, hw, normalise);
    const float* d = disp + (size_t)b * hw;
    const float* im = img + (size_t)b * C * hw;
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    float sx = 0.f, sy = 0.f;
    if (n < hw) {
        const int x = n % w, y = n / w;
        const float dn = div_rn(d[n], m);
        if (x < w - 1) sx = fabsf(dn - div_rn(d[n + 1], m)) * edge_weight(im, C, hw, n, n + 1);
        if (y < h - 1) sy = fabsf(dn - div_rn(d[n + w], m)) * edge_weight(im, C, hw, n, n + w);
    }
    sx = block_sum(sx, red);
    sy = block_sum(sy, red);
    if (threadIdx.x == 0) {
        float* o = loss_part + ((size_t)b * gridDim.x + blockIdx.x) * 2;
        o[0] = sx;
        o[1] = sy;
    }
}

__global__ void smooth_loss_reduce_kernel(const float* __restrict__ loss_part, int nblk, double inv_nx, double inv_ny,
                                          float* __restrict__ loss_out) {
    __shared__ double rx[32], ry[32];
    double sx = 0.0, sy = 0.0;
    for (int i = threadIdx.x; i < nblk; i += blockDim.x) {
        sx += (double)loss_part[2 * i];
        sy += (double)loss_part[2 * i + 1];
    }
    sx = warp_sum_d(sx);
    sy = warp_sum_d(sy);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (lane == 0) { rx[wid] = sx; ry[wid] = sy; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double tx = 0.0, ty = 0.0;
        for (int i = 0; i < (int)(blockDim.x >> 5); ++i) { tx += rx[i]; ty += ry[i]; }
        loss_out[0] = (float)(tx * inv_nx + ty * inv_ny);
    }
}

// gN = d loss / d norm_disp ; also per-block sum of gN * disp for the mean term
__global__ void __launch_bounds__(SM_THREADS)
smooth_bwd_kernel(const float* __restrict__ disp, const float* __restrict__ img, int C, int h, int w, int normalise,
                  const float* __restrict__ mean_part, float inv_nx, float inv_ny, const float* __restrict__ grad_loss,
                  float weight, float* __restrict__ gn_out, float* __restrict__ gd_part,
                  float* __restrict__ grad_img) {
    __shared__ float red[32];
    const int b = blockIdx.y;
    const int hw = h * w;
    const float m = image_mean_eps(mean_part, b, hw, normalise);
    const float up = weight * (grad_loss ? grad_loss[0] : 1.0f);
    const float* d = disp + (size_t)b * hw;
    const float* im = img + (size_t)b * C * hw;
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    float g = 0.f, dv = 0.f;
    if (n < hw) {
        const int x = n % w, y = n / w;
        dv = d[n];
        const float dn = div_rn(dv, m);
        float gi[8];
        const bool want_img = grad_img != nullptr && C <= 8;
        if (want_img)
            for (int c = 0; c < C; ++c) gi[c] = 0.f;
        if (x < w - 1) {
            const float diff = dn - div_rn(d[n + 1], m);
            const float e = edge_weight(im, C, hw, n, n + 1);
            g += sgn(diff) * e * inv_nx;
            if (want_img)
                for (int c = 0; c < C; ++c)
                    gi[c] -= fabsf(diff) * e * inv_nx / (float)C * sgn(im[c * hw + n] - im[c * hw + n + 1]);
        }
        if (x > 0) {
            const float diff = div_rn(d[n - 1], m) - dn;
            const float e = edge_weight(im, C, hw, n - 1, n);
            g -= sgn(diff) * e * inv_nx;
            if (want_img)
                for (int c = 0; c < C; ++c)
                    gi[c] += fabsf(diff) * e * inv_nx / (float)C * sgn(im[c * hw + n - 1] - im[c * hw + n]);
        }
        if (y < h - 1) {
            const float diff = dn - div_rn(d[n + w], m);
            const float e = edge_weight(im, C, hw, n, n + w);
            g += sgn(diff) * e * inv_ny;
            if (want_img)
                for (int c = 0; c < C; ++c)
                    gi[c] -= fabsf(diff) * e * inv_ny / (float)C * sgn(im[c * hw + n] - im[c * hw + n + w]);
        }
        if (y > 0) {
            const float diff = div_rn(d[n - w], m) - dn;
            const float e = edge_weight(im, C, hw, n - w, n);
            g -= sgn(diff) * e * inv_ny;
            if (want_img)
                for (int c = 0; c < C; ++c)
                    gi[c] += fabsf(diff) * e * inv_ny / (float)C * sgn(im[c * hw + n - w] - im[c * hw + n]);
        }
        g *= up;
        gn_out[(size_t)b * hw + n] = g;
        if (want_img)
            for (int c = 0; c < C; ++c) grad_img[((size_t)b * C + c) * hw + n] = gi[c] * up;
    }
    if (normalise) {
        const float s = block_sum(g * dv, red);
        if (threadIdx.x == 0) gd_part[(size_t)b * gridDim.x + blockIdx.x] = s;
    }
}

// grad_disp = gN/(m+eps) - (sum_i gN_i d_i) / (N (m+eps)^2)
__global__ void __launch_bounds__(SM_THREADS)
smooth_bwd_finalize_kernel(int hw, int nblk, const float* __restrict__ mean_part, const float* __restrict__ gd_part,
                           float* __restrict__ grad_disp) {
    __shared__ float s_corr, s_invm;
    const int b = blockIdx.y;
    if (threadIdx.x == 0) {
        const float inv_m = 1.0f / image_mean_eps(mean_part, b, hw, 1);
        double s = 0.0;
        for (int i = 0; i < nblk; ++i) s += (double)gd_part[(size_t)b * nblk + i];
        s_invm = inv_m;
        s_corr = (float)(s / (double)hw) * inv_m * inv_m;
    }
    __syncthreads();
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n < hw) {
        float* g = grad_disp + (size_t)b * hw + n;
        *g = *g * s_invm - s_corr;
    }
}


// ---------------------------------------------------------------------------- bilinear up-sample
// F.interpolate(disp, [H,W], mode="bilinear", align_corners=False) of trainer.py:481-482
// (ATen upsample_bilinear2d: src = max(scale*(dst+0.5)-0.5, 0)), forward and a
// DETERMINISTIC gather backward (ATen's CUDA backward scatters with atomics).
__global__ void upsample_fwd_kernel(const float* __restrict__ in, int h, int w, int H, int W, float sh, float sw,
                                    float* __restrict__ out) {
    const int X = blockIdx.x * blockDim.x + threadIdx.x;
    const int Y = blockIdx.y * blockDim.y + threadIdx.y;
    if (X >= W || Y >= H) return;
    const float* p = in + (size_t)blockIdx.z * h * w;
    const UpTap ty = up_tap(Y, sh, h), tx = up_tap(X, sw, w);
    const float v = ty.l0 * (tx.l0 * __ldg(p + ty.i0 * w + tx.i0) + tx.l1 * __ldg(p + ty.i0 * w + tx.i1)) +
                    ty.l1 * (tx.l0 * __ldg(p + ty.i1 * w + tx.i0) + tx.l1 * __ldg(p + ty.i1 * w + tx.i1));
    out[(size_t)blockIdx.z * H * W + (size_t)Y * W + X] = v;
}

// one thread per LOW-res pixel gathers every high-res pixel that read it
__global__ void upsample_bwd_kernel(const float* __restrict__ gout, int h, int w, int H, int W, float sh, float sw,
                                    const float* __restrict__ gscale, float* __restrict__ gin) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= w || y >= h) return;
    const float* g = gout + (size_t)blockIdx.z * H * W;
    const float rh = 1.0f / sh, rw = 1.0f / sw;
    const int Y0 = max(0, (int)floorf(((float)y - 0.5f) * rh - 0.5f) - 1);
    const int Y1 = min(H - 1, (int)ceilf(((float)y + 1.5f) * rh - 0.5f) + 1);
    const int X0 = max(0, (int)floorf(((float)x - 0.5f) * rw - 0.5f) - 1);
    const int X1 = min(W - 1, (int)ceilf(((float)x + 1.5f) * rw - 0.5f) + 1);
    float acc = 0.0f;
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
    if (gscale) acc *= gscale[0];
    gin[(size_t)blockIdx.z * h * w + (size_t)y * w + x] = acc;
}

// ---------------------------------------------------------------------------- reduce
// (one block per row: blockIdx.x selects the row of a (rows, n) array; rows == 1 for dmh_reduce_sum)
__global__ void reduce_sum_kernel(const float* __restrict__ in, long long n, float scale, int accumulate,
                                  float* __restrict__ out) {
    __shared__ double red[32];
    double s = 0.0;
    in += (size_t)blockIdx.x * n;
    out += blockIdx.x;
    for (long long i = threadIdx.x; i < n; i += blockDim.x) s += (double)in[i];
    s = warp_sum_d(s);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (lane == 0) red[wid] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int i = 0; i < (int)(blockDim.x >> 5); ++i) t += red[i];
        const float r = (float)(t * (double)scale);
        out[0] = accumulate ? out[0] + r : r;
    }
}

DepthScale make_depth_scale(float min_depth, float max_depth) {
    DepthScale ds;
    ds.min_disp = (float)(1.0 / (double)max_depth);
    ds.range = (float)(1.0 / (double)min_depth - 1.0 / (double)max_depth);
    return ds;
}

}  // namespace

extern "C" {

int dmh_warp_fwd(const float* disp, int input_is_depth, float min_depth, float max_depth, const float* src,
                 const float* K, const float* inv_K, const float* T, int B, int C, int H, int W, float* warped,
                 float* grid_out, float* depth_out, dmh_stream_t stream) {
    DMH_REQUIRE(disp && src && K && inv_K && T && warped, "dmh_warp_fwd: null pointer");
    DMH_REQUIRE(B > 0 && C > 0 && H > 1 && W > 1 && B <= 65535, "dmh_warp_fwd: bad shape B=%d C=%d H=%d W=%d", B, C, H, W);
    DMH_REQUIRE((input_is_depth & 1) || (min_depth > 0.f && max_depth > min_depth), "dmh_warp_fwd: bad depth range");
    const DepthScale ds = (input_is_depth & 1) ? DepthScale{0.f, 0.f} : make_depth_scale(min_depth, max_depth);
    dim3 grid(ceil_div((long long)H * W, WARP_THREADS), B);
    if (C == 3)
        DMH_LAUNCH(warp_fwd_kernel<3>, grid, WARP_THREADS, 0, (cudaStream_t)stream)(disp, input_is_depth, ds, src, K, inv_K, T,
                                                                           C, H, W, warped, grid_out, depth_out);
    else
        DMH_LAUNCH(warp_fwd_kernel<0>, grid, WARP_THREADS, 0, (cudaStream_t)stream)(disp, input_is_depth, ds, src, K, inv_K, T,
                                                                           C, H, W, warped, grid_out, depth_out);
    DMH_CHECK_LAUNCH("dmh_warp_fwd");
    return DMH_OK;
}

int dmh_warp_bwd_blocks(int H, int W) { return ceil_div((long long)H * W, WARP_THREADS); }

int dmh_warp_bwd(const float* grad_warped, const float* disp, int input_is_depth, float min_depth, float max_depth,
                 const float* src, const float* K, const float* inv_K, const float* T, int B, int C, int H, int W,
                 float* grad_disp, float* grad_src, float* grad_P_partial, dmh_stream_t stream) {
    DMH_REQUIRE(grad_warped && disp && src && K && inv_K && T, "dmh_warp_bwd: null pointer");
    DMH_REQUIRE(B > 0 && C > 0 && H > 1 && W > 1 && B <= 65535, "dmh_warp_bwd: bad shape");
    DMH_REQUIRE(input_is_depth || (min_depth > 0.f && max_depth > min_depth), "dmh_warp_bwd: bad depth range");
    const DepthScale ds = input_is_depth ? DepthScale{0.f, 0.f} : make_depth_scale(min_depth, max_depth);
    dim3 grid(dmh_warp_bwd_blocks(H, W), B);
    if (C == 3)
        DMH_LAUNCH(warp_bwd_kernel<3>, grid, WARP_THREADS, 0, (cudaStream_t)stream)(
            grad_warped, disp, input_is_depth, ds, src, K, inv_K, T, C, H, W, grad_disp, grad_src, grad_P_partial);
    else
        DMH_LAUNCH(warp_bwd_kernel<0>, grid, WARP_THREADS, 0, (cudaStream_t)stream)(
            grad_warped, disp, input_is_depth, ds, src, K, inv_K, T, C, H, W, grad_disp, grad_src, grad_P_partial);
    DMH_CHECK_LAUNCH("dmh_warp_bwd");
    return DMH_OK;
}

static inline int smooth_blocks(int h, int w) { return ceil_div((long long)h * w, SM_THREADS); }

long long dmh_smooth_workspace_floats(int B, int h, int w) {
    return (long long)B * SM_NB1 + 3LL * B * smooth_blocks(h, w);
}

int dmh_smooth_fwd(const float* disp, const float* img, int B, int C, int h, int w, int normalise, float* ws,
                   float* loss_out, dmh_stream_t stream) {
    DMH_REQUIRE(disp && img && ws && loss_out, "dmh_smooth_fwd: null pointer");
    DMH_REQUIRE(B > 0 && C > 0 && h >= 2 && w >= 2 && B <= 65535, "dmh_smooth_fwd: bad shape");
    const int nb = smooth_blocks(h, w);
    float* mean_part = ws;
    float* loss_part = ws + (size_t)B * SM_NB1;
    cudaStream_t st = (cudaStream_t)stream;
    if (normalise) DMH_LAUNCH(smooth_mean_kernel, dim3(SM_NB1, B), 256, 0, st)(disp, h * w, mean_part);
    DMH_LAUNCH(smooth_fwd_kernel, dim3(nb, B), SM_THREADS, 0, st)(disp, img, C, h, w, normalise, mean_part, loss_part);
    const double inv_nx = 1.0 / ((double)B * h * (w - 1)), inv_ny = 1.0 / ((double)B * (h - 1) * w);
    DMH_LAUNCH(smooth_loss_reduce_kernel, 1, 256, 0, st)(loss_part, B * nb, inv_nx, inv_ny, loss_out);
    DMH_CHECK_LAUNCH("dmh_smooth_fwd");
    return DMH_OK;
}

int dmh_smooth_bwd(const float* disp, const float* img, int B, int C, int h, int w, int normalise,
                   const float* grad_loss, float weight, float* ws, float* grad_disp, float* grad_img,
                   dmh_stream_t stream) {
    DMH_REQUIRE(disp && img && ws && grad_disp, "dmh_smooth_bwd: null pointer");
    DMH_REQUIRE(B > 0 && C > 0 && h >= 2 && w >= 2 && B <= 65535, "dmh_smooth_bwd: bad shape");
    DMH_REQUIRE(!grad_img || C <= 8, "dmh_smooth_bwd: grad_img needs C <= 8");
    const int nb = smooth_blocks(h, w);
    float* mean_part = ws;
    float* gd_part = ws + (size_t)B * SM_NB1 + 2 * (size_t)B * nb;
    cudaStream_t st = (cudaStream_t)stream;
    if (normalise) DMH_LAUNCH(smooth_mean_kernel, dim3(SM_NB1, B), 256, 0, st)(disp, h * w, mean_part);
    const float inv_nx = (float)(1.0 / ((double)B * h * (w - 1))), inv_ny = (float)(1.0 / ((double)B * (h - 1) * w));
    DMH_LAUNCH(smooth_bwd_kernel, dim3(nb, B), SM_THREADS, 0, st)(disp, img, C, h, w, normalise, mean_part, inv_nx, inv_ny,
                                                          grad_loss, weight, grad_disp, gd_part, grad_img);
    if (normalise)
        DMH_LAUNCH(smooth_bwd_finalize_kernel, dim3(nb, B), SM_THREADS, 0, st)(h * w, nb, mean_part, gd_part, grad_disp);
    DMH_CHECK_LAUNCH("dmh_smooth_bwd");
    return DMH_OK;
}

int dmh_upsample_bilinear_fwd(const float* in, int planes, int h, int w, int H, int W, float* out,
                              dmh_stream_t stream) {
    DMH_REQUIRE(in && out, "dmh_upsample_bilinear_fwd: null pointer");
    DMH_REQUIRE(planes > 0 && planes <= 65535 && h > 0 && w > 0 && H > 0 && W > 0, "dmh_upsample_bilinear_fwd: bad shape");
    dim3 block(32, 8), grid(ceil_div(W, 32), ceil_div(H, 8), planes);
    DMH_LAUNCH(upsample_fwd_kernel, grid, block, 0, (cudaStream_t)stream)(in, h, w, H, W, (float)h / (float)H,
                                                                 (float)w / (float)W, out);
    DMH_CHECK_LAUNCH("dmh_upsample_bilinear_fwd");
    return DMH_OK;
}

int dmh_upsample_bilinear_bwd(const float* grad_out, int planes, int h, int w, int H, int W, const float* grad_scale,
                              float* grad_in, dmh_stream_t stream) {
    DMH_REQUIRE(grad_out && grad_in, "dmh_upsample_bilinear_bwd: null pointer");
    DMH_REQUIRE(planes > 0 && planes <= 65535 && h > 0 && w > 0 && H > 0 && W > 0, "dmh_upsample_bilinear_bwd: bad shape");
    dim3 block(32, 8), grid(ceil_div(w, 32), ceil_div(h, 8), planes);
    DMH_LAUNCH(upsample_bwd_kernel, grid, block, 0, (cudaStream_t)stream)(grad_out, h, w, H, W, (float)h / (float)H,
                                                                 (float)w / (float)W, grad_scale, grad_in);
    DMH_CHECK_LAUNCH("dmh_upsample_bilinear_bwd");
    return DMH_OK;
}

int dmh_reduce_sum(const float* in, long long n, float scale, int accumulate, float* out, dmh_stream_t stream) {
    DMH_REQUIRE(in && out && n > 0, "dmh_reduce_sum: null pointer or n <= 0");
    DMH_LAUNCH(reduce_sum_kernel, 1, 1024, 0, (cudaStream_t)stream)(in, n, scale, accumulate, out);
    DMH_CHECK_LAUNCH("dmh_reduce_sum");
    return DMH_OK;
}

int dmh_reduce_rows(const float* in, int rows, long long n, float scale, float* out, dmh_stream_t stream) {
    DMH_REQUIRE(in && out && n > 0 && rows > 0 && rows <= 65535, "dmh_reduce_rows: null pointer or bad shape");
    DMH_LAUNCH(reduce_sum_kernel, rows, 1024, 0, (cudaStream_t)stream)(in, n, scale, 0, out);
    DMH_CHECK_LAUNCH("dmh_reduce_rows");
    return DMH_OK;
}

}  // extern "C"
