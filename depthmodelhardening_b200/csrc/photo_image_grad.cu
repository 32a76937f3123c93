// Colour-frame gradients of the fused photometric objective (backward of ops.objective w.r.t. the target, the
// source frames and the colour pyramid), recomputed from the saved frames, the disparities and the per-scale
// selections `sel` of the forward -- no warped image, SSIM map or autograd intermediate is kept.
//
//   dmh_identity_image_grad  one launch for all scales (the identity losses do not depend on the scale): the
//                            identity candidates' terms on the un-warped pair (src_f, target), gated per pixel by
//                            sum_s u_s [sel_s == identity of f].  INITIALISES grad_target and every grad_src[f].
//   dmh_photo_image_grad     one launch per scale, the tile machinery of photo_scale_kernel (photo_objective.cu):
//                            disparity up-sampling fused into the read, the same coordinate chain (and the same
//                            verified division rule), the warped tile with its 2-px reflect halo, gated SSIM
//                            coefficient planes and their box sums.  The reprojection terms are added into
//                            grad_target in place (each pixel is owned by one thread; launches run in stream order:
//                            deterministic) and scattered into grad_src[f] through the bilinear taps by RED
//                            (warp-aggregated, as dmh_warp_bwd).
//                            With DMH_PHOTO_INPUT_IS_DEPTH the network output is a depth map, used as it is (the
//                            forward's chain); with DMH_PHOTO_PIXEL_SUM the loss is the sum over the pixels, not
//                            their mean (ops.photo_scale_sum).
//   dmh_photo_image_grad_dh  the same kernel for the depth-hints objective (depth_hints.py): the reprojection term
//                            counts wherever the identity did not win the argmin over [reprojection, identity,
//                            hint] and goes to the forward's first-minimum source frame (or 1/F to each under
//                            avg_reprojection); the identity and hint candidates carry no gradient there.
//   dmh_smooth_image_grad    u_s * w_s * d(edge-aware smoothness)/d(colour(0, s)); scale 0 adds into grad_target.
//
// u_s = g_total / S + g_scale[s] (depth hints: the masked mean's u_r[s]) is read on the device: no host
// synchronisation, CUDA-graph capturable.
//
// Algorithmic bytes per target pixel (fp32, F source frames, S scales):
//   dmh_photo_image_grad     read 12 (target) + 12 F (gathered sources) + <= 4 (disparity) + 1 (sel);
//                            write 24 (target read-modify-write) + 12 F (source RED)
//   dmh_identity_image_grad  read 12 + 12 F + S (sel); write 12 + 12 F
#include "photo_general.cuh"

namespace {

#define IG_MAXF DMH_PHOTO_MAX_FRAMES
#define IG_MAXS 8

__device__ __forceinline__ float upstream(const float* g_total, const float* g_scale, float inv_S) {
    return add_rn(g_total ? mul_rn(g_total[0], inv_S) : 0.0f, g_scale ? g_scale[0] : 0.0f);
}

// Gated SSIM coefficient planes k[4][3][R1] (ax, b, c, ay) of R(x, y) at every ring position whose gate is non-zero
// (zero elsewhere).  xs / ys: [3][R2] tiles of the prediction / the target.
__device__ __forceinline__ void coef_planes(const float* __restrict__ xs, const float* __restrict__ ys,
                                            const float* __restrict__ gate, float w_ssim, float* __restrict__ k) {
    for (int i = threadIdx.x; i < PH_R1; i += PH_THREADS) {
        const int r = i / PH_R1W, c = i % PH_R1W;
        const float g = gate[i];
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) {
            float a = 0.f, bq = 0.f, cq = 0.f, d = 0.f;
            if (g != 0.f) {
                float pass;
                SsimCoef kk;
                ssim_value_coef(window_stats(xs + ch * PH_R2, ys + ch * PH_R2, r, c), pass, kk);
                const float gg = g * w_ssim * pass;
                a = gg * kk.ax; bq = gg * kk.b; cq = gg * kk.c; d = gg * kk.ay;
            }
            k[(0 * 3 + ch) * PH_R1 + i] = a;
            k[(1 * 3 + ch) * PH_R1 + i] = bq;
            k[(2 * 3 + ch) * PH_R1 + i] = cq;
            k[(3 * 3 + ch) * PH_R1 + i] = d;
        }
    }
}

// d/d(x) and d/d(y) at interior tile pixel (r, c) = image (py, px): box sums of the coefficient planes over the
// window centres reaching it (reflection multiplicities), plus the L1 term of its own window
__device__ __forceinline__ void pixel_grads(const float* __restrict__ xs, const float* __restrict__ ys,
                                            const float* __restrict__ k, const float* __restrict__ gate, int r, int c,
                                            int py, int px, int H, int W, bool ssim, float w_l1, float gx[3],
                                            float gy[3]) {
    const int ci2 = (r + 2) * PH_R2W + (c + 2);
    const float gl1 = gate[(r + 1) * PH_R1W + (c + 1)] * w_l1;
    float wy[3], wx[3];
#pragma unroll
    for (int d = 0; d < 3; ++d) {
        wy[d] = reflect_mult(py, py - 1 + d, H);
        wx[d] = reflect_mult(px, px - 1 + d, W);
    }
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) {
        float sa = 0.f, sb = 0.f, sc = 0.f, sd = 0.f;
        if (ssim) {
#pragma unroll
            for (int dy = 0; dy < 3; ++dy)
#pragma unroll
                for (int dx = 0; dx < 3; ++dx) {
                    const float w = wy[dy] * wx[dx];
                    const int o = ch * PH_R1 + (r + dy) * PH_R1W + c + dx;
                    sa = fmaf(w, k[o], sa);
                    sb = fmaf(w, k[3 * PH_R1 + o], sb);
                    sc = fmaf(w, k[6 * PH_R1 + o], sc);
                    sd = fmaf(w, k[9 * PH_R1 + o], sd);
                }
        }
        reproj_pixel_grad(sa, sb, sc, sd, xs[ch * PH_R2 + ci2], ys[ch * PH_R2 + ci2], gl1, gx[ch], gy[ch]);
    }
}

// the [3][R2] tile of frame `img` (B,3,H,W) at batch b with its 2-px reflect halo
__device__ __forceinline__ void load_tile(const float* __restrict__ img, int b, int x0, int y0, int H, int W,
                                          float* __restrict__ out) {
    const size_t N = (size_t)H * W;
    for (int i = threadIdx.x; i < PH_R2; i += PH_THREADS) {
        const int r = i / PH_R2W, c = i % PH_R2W;
        const size_t o = (size_t)ext_to_img(y0 - 2 + r, H) * W + ext_to_img(x0 - 2 + c, W);
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) out[ch * PH_R2 + i] = __ldg(img + ((size_t)b * 3 + ch) * N + o);
    }
}

// ---------------------------------------------------------------------------------------------- identity terms
struct IdentGradParams {
    const float* target;
    const float* src[IG_MAXF];
    const uint8_t* sel[IG_MAXS];
    const float* g_total;
    const float* g_scales;
    float inv_S, inv_den;
    float* grad_target;
    float* grad_src[IG_MAXF];
    int B, H, W, F, S, n_ident, flags;
};

size_t ident_smem_bytes() { return sizeof(float) * ((size_t)6 * PH_R2 + 13 * PH_R1); }

__global__ void __launch_bounds__(PH_THREADS)
identity_grad_kernel(const IdentGradParams p) {
    extern __shared__ float smem[];
    float* tgt = smem;                          // [3][R2]
    float* xs = tgt + 3 * PH_R2;                // [3][R2] source frame f
    float* k = xs + 3 * PH_R2;                  // [4][3][R1]
    float* gate = k + 12 * PH_R1;               // [R1]
    __shared__ float us[IG_MAXS];

    const int H = p.H, W = p.W, b = blockIdx.z;
    const int x0 = blockIdx.x * PH_TW, y0 = blockIdx.y * PH_TH;
    const size_t N = (size_t)H * W;
    const bool no_ssim = (p.flags & DMH_PHOTO_NO_SSIM) != 0;
    const bool avg = (p.flags & DMH_PHOTO_AVG_REPROJECTION) != 0;
    const float w_ssim = no_ssim ? 0.0f : 0.85f / 3.0f;
    const float w_l1 = no_ssim ? 1.0f / 3.0f : 0.15f / 3.0f;

    if (threadIdx.x < p.S)
        us[threadIdx.x] = upstream(p.g_total, p.g_scales ? p.g_scales + threadIdx.x : nullptr, p.inv_S) * p.inv_den;
    load_tile(p.target, b, x0, y0, H, W, tgt);
    __syncthreads();

    float g_tgt[2][3] = {{0.f, 0.f, 0.f}, {0.f, 0.f, 0.f}};
    for (int f = 0; f < p.F; ++f) {
        bool any = false;
        for (int i = threadIdx.x; i < PH_R1; i += PH_THREADS) {
            const int qy = y0 - 1 + i / PH_R1W, qx = x0 - 1 + i % PH_R1W;
            float g = 0.f;
            if (p.n_ident > 0 && qy >= 0 && qy < H && qx >= 0 && qx < W) {
                const size_t qo = (size_t)b * N + (size_t)qy * W + qx;
                for (int s = 0; s < p.S; ++s) g = fmaf(us[s], ident_gate(p.sel[s][qo], f, p.n_ident, p.F, avg), g);
            }
            gate[i] = g;
            any |= g != 0.f;
        }
        float* gs = p.grad_src[f] ? p.grad_src[f] + (size_t)b * 3 * N : nullptr;
        if (!__syncthreads_or(any)) {
            // no pixel of the tile picked this identity at any scale: the tile's source gradient starts at zero
            for (int slot = 0; slot < 2 && gs; ++slot) {
                const int i = threadIdx.x + slot * PH_THREADS;
                const int py = y0 + i / PH_TW, px = x0 + i % PH_TW;
                if (py < H && px < W)
                    for (int ch = 0; ch < 3; ++ch) gs[ch * N + (size_t)py * W + px] = 0.f;
            }
            continue;
        }
        load_tile(p.src[f], b, x0, y0, H, W, xs);
        __syncthreads();
        if (!no_ssim) {
            coef_planes(xs, tgt, gate, w_ssim, k);
            __syncthreads();
        }
#pragma unroll
        for (int slot = 0; slot < 2; ++slot) {
            const int i = threadIdx.x + slot * PH_THREADS;
            const int r = i / PH_TW, c = i % PH_TW;
            const int py = y0 + r, px = x0 + c;
            if (py >= H || px >= W) continue;
            float gx[3], gy[3];
            pixel_grads(xs, tgt, k, gate, r, c, py, px, H, W, !no_ssim, w_l1, gx, gy);
#pragma unroll
            for (int ch = 0; ch < 3; ++ch) {
                if (gs) gs[ch * N + (size_t)py * W + px] = gx[ch];
                g_tgt[slot][ch] += gy[ch];
            }
        }
        __syncthreads();
    }
    if (p.grad_target) {
#pragma unroll
        for (int slot = 0; slot < 2; ++slot) {
            const int i = threadIdx.x + slot * PH_THREADS;
            const int py = y0 + i / PH_TW, px = x0 + i % PH_TW;
            if (py >= H || px >= W) continue;
#pragma unroll
            for (int ch = 0; ch < 3; ++ch)
                p.grad_target[((size_t)b * 3 + ch) * N + (size_t)py * W + px] = g_tgt[slot][ch];
        }
    }
}

// ---------------------------------------------------------------------------------------- reprojection terms
struct ReprojGradParams {
    const float* target;
    const float* src[IG_MAXF];
    const float* T[IG_MAXF];
    DispSrc disp;
    const float* K;
    const float* inv_K;
    const uint8_t* sel;
    const float* g_total;
    const float* g_scale;
    float inv_S, inv_den;
    float* grad_target;
    float* grad_src[IG_MAXF];
    int B, H, W, F, n_ident, flags;
    DepthScale ds;
    float rcw, rch;              // 1/(W-1), 1/(H-1) for the verified 3-instruction division
    const float* u_dh;           // depth-hints mode: device scalar, the reprojection term's upstream weight of this scale
};

size_t reproj_smem_bytes() { return sizeof(float) * ((size_t)7 * PH_R2 + 13 * PH_R1 + IG_MAXF * 24); }

// DH: the depth-hints objective (sel from dmh_photo_scale_dh with DMH_PHOTO_SEL_SOURCE, gate reproj_gate_dh, upstream
// weight *u_dh); otherwise monodepth2's (reproj_gate, upstream(...) * inv_den).  DEPTH_IN: the network output is a
// depth map (DMH_PHOTO_INPUT_IS_DEPTH), not a disparity.
template <bool FASTDIV, bool DH, bool DEPTH_IN>
__global__ void __launch_bounds__(PH_THREADS)
reproj_grad_kernel(const ReprojGradParams p) {
    extern __shared__ float smem[];
    float* tgt = smem;                          // [3][R2]
    float* dep = tgt + 3 * PH_R2;               // [R2]
    float* pred = dep + PH_R2;                  // [3][R2] source f warped into the target view
    float* k = pred + 3 * PH_R2;                // [4][3][R1]
    float* gate = k + 12 * PH_R1;               // [R1]
    float* cams = gate + PH_R1;                 // [F][24]
    __shared__ float s_u;

    const int tid = threadIdx.x;
    const int H = p.H, W = p.W, b = blockIdx.z;
    const int x0 = blockIdx.x * PH_TW, y0 = blockIdx.y * PH_TH;
    const size_t N = (size_t)H * W;
    const bool no_ssim = (p.flags & DMH_PHOTO_NO_SSIM) != 0;
    const bool avg = (p.flags & DMH_PHOTO_AVG_REPROJECTION) != 0;
    const float w_ssim = no_ssim ? 0.0f : 0.85f / 3.0f;
    const float w_l1 = no_ssim ? 1.0f / 3.0f : 0.15f / 3.0f;
    const unsigned lane = tid & 31;

    // ---- cameras, target tile and depth: the forward's operations (photo_scale_kernel)
    load_cameras(cams, p, p.F, b, tid);
    if (tid == 0) s_u = DH ? __ldg(p.u_dh) : upstream(p.g_total, p.g_scale, p.inv_S) * p.inv_den;
    load_target_depth(p.target, p.disp, p.ds, DEPTH_IN, b, x0, y0, H, W, N, tgt, dep);
    __syncthreads();
    const float u = s_u;

    float g_tgt[2][3] = {{0.f, 0.f, 0.f}, {0.f, 0.f, 0.f}};
    for (int f = 0; f < p.F; ++f) {
        bool any = false;
        for (int i = tid; i < PH_R1; i += PH_THREADS) {
            const int qy = y0 - 1 + i / PH_R1W, qx = x0 - 1 + i % PH_R1W;
            float g = 0.f;
            if (qy >= 0 && qy < H && qx >= 0 && qx < W) {
                const int sel = p.sel[(size_t)b * N + (size_t)qy * W + qx];
                g = u * (DH ? reproj_gate_dh(sel, f, p.F, avg) : reproj_gate(sel, f, p.n_ident, p.F, avg));
            }
            gate[i] = g;
            any |= g != 0.f;
        }
        if (!__syncthreads_or(any)) continue;       // no pixel of the tile picked this reprojection
        Camera cam;
#pragma unroll
        for (int i = 0; i < 12; ++i) cam.P[i] = cams[f * 24 + i];
#pragma unroll
        for (int i = 0; i < 9; ++i) cam.iK[i] = cams[f * 24 + 12 + i];
        const float* sp = p.src[f] + (size_t)b * 3 * N;
        for (int i = tid; i < PH_R2; i += PH_THREADS) {
            const int r = i / PH_R2W, c = i % PH_R2W;
            const int iy = ext_to_img(y0 - 2 + r, H), ix = ext_to_img(x0 - 2 + c, W);
            const WarpCoord wc = warp_coord<FASTDIV>(cam, (float)ix, (float)iy, dep[i], W, H, 1e-7f, p.rcw, p.rch);
            const Bilinear bl = bilinear_setup(wc.ix, wc.iy);
            const Taps t = make_taps(bl, H, W);
#pragma unroll
            for (int ch = 0; ch < 3; ++ch) {
                const float* s = sp + ch * N;
                float acc = 0.0f;
                if (t.nw) acc = fmaf(__ldg(s + t.o00), bl.wnw, acc);
                if (t.ne) acc = fmaf(__ldg(s + t.o00 + 1), bl.wne, acc);
                if (t.sw) acc = fmaf(__ldg(s + t.o00 + W), bl.wsw, acc);
                if (t.se) acc = fmaf(__ldg(s + t.o00 + W + 1), bl.wse, acc);
                pred[ch * PH_R2 + i] = acc;
            }
        }
        __syncthreads();
        if (!no_ssim) {
            coef_planes(pred, tgt, gate, w_ssim, k);
            __syncthreads();
        }
        float* gs = p.grad_src[f] ? p.grad_src[f] + (size_t)b * 3 * N : nullptr;
#pragma unroll
        for (int slot = 0; slot < 2; ++slot) {
            // a warp holds 32 consecutive pixels of one tile row: every lane takes part in the aggregated scatter
            const int i = tid + slot * PH_THREADS;
            const int r = i / PH_TW, c = i % PH_TW;
            const int py = y0 + r, px = x0 + c;
            const bool active = py < H && px < W;
            float gx[3] = {0.f, 0.f, 0.f}, gy[3];
            if (active) {
                pixel_grads(pred, tgt, k, gate, r, c, py, px, H, W, !no_ssim, w_l1, gx, gy);
#pragma unroll
                for (int ch = 0; ch < 3; ++ch) g_tgt[slot][ch] += gy[ch];
            }
            if (!gs) continue;
            Bilinear bl = {};
            Taps t = {};
            if (active) {
                const WarpCoord wc = warp_coord<FASTDIV>(cam, (float)px, (float)py, dep[(r + 2) * PH_R2W + (c + 2)], W,
                                                         H, 1e-7f, p.rcw, p.rch);
                bl = bilinear_setup(wc.ix, wc.iy);
                t = make_taps(bl, H, W);
            }
            // east tap of this lane == west tap of lane+1 ?
            const int nx0 = __shfl_down_sync(0xffffffffu, bl.x0, 1);
            const int ny0 = __shfl_down_sync(0xffffffffu, bl.y0, 1);
            const int nact = __shfl_down_sync(0xffffffffu, (int)active, 1);
            const bool merge_e = active && lane < 31 && nact && nx0 == bl.x0 + 1 && ny0 == bl.y0;
            const bool recv_w = __shfl_up_sync(0xffffffffu, (int)merge_e, 1) != 0;
#pragma unroll
            for (int ch = 0; ch < 3; ++ch) {
                const float go = gx[ch];
                float* gp = gs + ch * N;
                scatter_row(gp, t.o00, active && t.nw, active && t.ne, bl.wnw * go, bl.wne * go, merge_e && t.nw && t.ne,
                            recv_w, lane);
                scatter_row(gp, t.o00 + W, active && t.sw, active && t.se, bl.wsw * go, bl.wse * go,
                            merge_e && t.sw && t.se, recv_w, lane);
            }
        }
        __syncthreads();
    }
    if (p.grad_target) {
#pragma unroll
        for (int slot = 0; slot < 2; ++slot) {
            const int i = tid + slot * PH_THREADS;
            const int py = y0 + i / PH_TW, px = x0 + i % PH_TW;
            if (py >= H || px >= W) continue;
#pragma unroll
            for (int ch = 0; ch < 3; ++ch) p.grad_target[((size_t)b * 3 + ch) * N + (size_t)py * W + px] += g_tgt[slot][ch];
        }
    }
}

// ------------------------------------------------------------------------------------------------ smoothness
// d/d(img) of w_s * [inv_nx * sum |dn_x| exp(-mean_c |d_x I|) + inv_ny * sum |dn_y| exp(-mean_c |d_y I|)],
// dn = disp / (mean + 1e-7) with the forward's 1/(mean + 1e-7) (img_scalars), one thread per pixel gathering its
// (up to) four edges
__global__ void __launch_bounds__(256)
smooth_img_grad_kernel(const float* __restrict__ disp, const float* __restrict__ img, int h, int w,
                       const float* __restrict__ img_scalars, float weight, const float* __restrict__ g_total,
                       const float* __restrict__ g_scale, float inv_S, float inv_nx, float inv_ny, int accumulate,
                       float* __restrict__ grad_img) {
    const int b = blockIdx.y;
    const int hw = h * w;
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= hw) return;
    const float inv_m = img_scalars[b * 2];
    const float up = upstream(g_total, g_scale, inv_S) * weight;
    const float* d = disp + (size_t)b * hw;
    const float* im = img + (size_t)b * 3 * hw;
    const int x = n % w, y = n / w;
    float gi[3] = {0.f, 0.f, 0.f};
    // edge (a, a + step) with this pixel at a (sign +1) or at a + step (sign -1)
    auto edge = [&](int a, int step, float inv_cnt, float sign) {
        float ia[3], ib[3], sabs = 0.f;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            ia[c] = __ldg(im + (size_t)c * hw + a);
            ib[c] = __ldg(im + (size_t)c * hw + a + step);
            sabs += fabsf(ia[c] - ib[c]);
        }
        const float diff = sub_rn(mul_rn(__ldg(d + a), inv_m), mul_rn(__ldg(d + a + step), inv_m));
        const float de = fabsf(diff) * expf(-sabs / 3.0f) * inv_cnt;
#pragma unroll
        for (int c = 0; c < 3; ++c) gi[c] += sign * smooth_edge_img_grad(de, ia[c], ib[c], 3);
    };
    if (x < w - 1) edge(n, 1, inv_nx, 1.f);
    if (x > 0) edge(n - 1, 1, inv_nx, -1.f);
    if (y < h - 1) edge(n, w, inv_ny, 1.f);
    if (y > 0) edge(n - w, w, inv_ny, -1.f);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        float* o = grad_img + ((size_t)b * 3 + c) * hw + n;
        const float v = gi[c] * up;
        *o = accumulate ? *o + v : v;
    }
}

// dmh_photo_image_grad (DH = false) and dmh_photo_image_grad_dh: the argument checks and the launch shared by both.
// p arrives with the upstream weight of its mode filled in; `name` is the public entry point, for the errors.  A depth
// input is a mode of dmh_photo_image_grad only.
template <bool DH>
int reproj_grad_launch(const char* name, ReprojGradParams& p, const float* target, const float* const* src_host,
                       const float* const* T_host, int F, const float* disp, int disp_h, int disp_w, const float* K,
                       const float* inv_K, const uint8_t* sel, int B, int H, int W, float min_depth, float max_depth,
                       int flags, float* grad_target, float* const* grad_src_host, cudaStream_t st) {
    DMH_REQUIRE(target && src_host && T_host && disp && K && inv_K && sel && grad_src_host, "%s: null pointer", name);
    DMH_REQUIRE(F >= 1 && F <= IG_MAXF, "%s: F=%d outside [1,%d]", name, F, IG_MAXF);
    DMH_REQUIRE(B > 0 && B <= 65535 && H >= 2 && W >= 2, "%s: bad shape B=%d H=%d W=%d", name, B, H, W);
    DMH_REQUIRE(disp_h >= 1 && disp_w >= 1 && disp_h <= H && disp_w <= W, "%s: bad disparity size %dx%d", name, disp_h,
                disp_w);
    const bool depth_in = (flags & DMH_PHOTO_INPUT_IS_DEPTH) != 0;
    DMH_REQUIRE(!(DH && depth_in), "%s: no depth-input mode", name);
    DMH_REQUIRE(depth_in || (min_depth > 0.f && max_depth > min_depth), "%s: bad depth range", name);
    p.target = target;
    for (int f = 0; f < F; ++f) {
        DMH_REQUIRE(src_host[f] && T_host[f], "%s: null src/T for frame %d", name, f);
        p.src[f] = src_host[f];
        p.T[f] = T_host[f];
        p.grad_src[f] = grad_src_host[f];
    }
    p.disp.ptr = disp; p.disp.h = disp_h; p.disp.w = disp_w;
    p.disp.sh = (float)disp_h / (float)H; p.disp.sw = (float)disp_w / (float)W;
    p.K = K; p.inv_K = inv_K; p.sel = sel;
    p.grad_target = grad_target;
    p.B = B; p.H = H; p.W = W; p.F = F; p.flags = flags;
    p.ds = depth_scale(min_depth, max_depth, depth_in);
    // the division rule of the forward kernels: bit-identical either way, the verified one is shorter
    const bool fastdiv = const_div_exact(W - 1, &p.rcw, st) && const_div_exact(H - 1, &p.rch, st);
    const size_t smem = reproj_smem_bytes();
    static KernelSetup setup;
    // the depth-input instantiations exist for DH = false only (for DH = true the last two repeat the first two)
    const void* kernels[4] = {(const void*)reproj_grad_kernel<false, DH, false>,
                              (const void*)reproj_grad_kernel<true, DH, false>,
                              (const void*)reproj_grad_kernel<false, DH, !DH>,
                              (const void*)reproj_grad_kernel<true, DH, !DH>};
    if (setup.sms(name, kernels, DH ? 2 : 4, smem) == 0) return DMH_ERR_CUDA;
    const dim3 grid(ceil_div(W, PH_TW), ceil_div(H, PH_TH), B);
    void (*kernel)(const ReprojGradParams) =
        depth_in ? (fastdiv ? reproj_grad_kernel<true, DH, !DH> : reproj_grad_kernel<false, DH, !DH>)
                 : (fastdiv ? reproj_grad_kernel<true, DH, false> : reproj_grad_kernel<false, DH, false>);
    DMH_LAUNCH(kernel, grid, PH_THREADS, smem, st)(p);
    DMH_CHECK_LAUNCH(name);
    return DMH_OK;
}

}  // namespace

extern "C" {

int dmh_identity_image_grad(const float* target, const float* const* src_host, int F, const uint8_t* const* sel_host,
                            int S, const float* g_total, const float* g_scales, int B, int H, int W, int flags,
                            int automask, float* grad_target, float* const* grad_src_host, dmh_stream_t stream) {
    DMH_REQUIRE(target && src_host && sel_host && grad_src_host && (g_total || g_scales),
                "dmh_identity_image_grad: null pointer");
    DMH_REQUIRE(F >= 1 && F <= IG_MAXF, "dmh_identity_image_grad: F=%d outside [1,%d]", F, IG_MAXF);
    DMH_REQUIRE(S >= 1 && S <= IG_MAXS, "dmh_identity_image_grad: S=%d outside [1,%d]", S, IG_MAXS);
    DMH_REQUIRE(B > 0 && B <= 65535 && H >= 2 && W >= 2, "dmh_identity_image_grad: bad shape B=%d H=%d W=%d", B, H, W);
    IdentGradParams p = {};
    p.target = target;
    for (int f = 0; f < F; ++f) {
        DMH_REQUIRE(src_host[f], "dmh_identity_image_grad: null src for frame %d", f);
        p.src[f] = src_host[f];
        p.grad_src[f] = grad_src_host[f];
    }
    for (int s = 0; s < S; ++s) {
        DMH_REQUIRE(sel_host[s], "dmh_identity_image_grad: null sel for scale %d", s);
        p.sel[s] = sel_host[s];
    }
    p.g_total = g_total; p.g_scales = g_scales;
    p.inv_S = 1.0f / (float)S;
    p.inv_den = (float)(1.0 / ((double)B * H * W));
    p.grad_target = grad_target;
    p.B = B; p.H = H; p.W = W; p.F = F; p.S = S; p.flags = flags;
    p.n_ident = automask ? ((flags & DMH_PHOTO_AVG_REPROJECTION) ? 1 : F) : 0;
    const size_t smem = ident_smem_bytes();
    static KernelSetup setup;
    const void* kernel = (const void*)identity_grad_kernel;
    if (setup.sms("dmh_identity_image_grad", &kernel, 1, smem) == 0) return DMH_ERR_CUDA;
    const dim3 grid(ceil_div(W, PH_TW), ceil_div(H, PH_TH), B);
    DMH_LAUNCH(identity_grad_kernel, grid, PH_THREADS, smem, (cudaStream_t)stream)(p);
    DMH_CHECK_LAUNCH("dmh_identity_image_grad");
    return DMH_OK;
}

int dmh_photo_image_grad(const float* target, const float* const* src_host, const float* const* T_host, int F,
                         const float* disp, int disp_h, int disp_w, const float* K, const float* inv_K,
                         const uint8_t* sel, int scale, int S, const float* g_total, const float* g_scales, int B,
                         int H, int W, float min_depth, float max_depth, int flags, int automask, float* grad_target,
                         float* const* grad_src_host, dmh_stream_t stream) {
    DMH_REQUIRE(g_total || g_scales, "dmh_photo_image_grad: null pointer");
    DMH_REQUIRE(S >= 1 && scale >= 0 && scale < S, "dmh_photo_image_grad: scale %d of %d", scale, S);
    ReprojGradParams p = {};
    p.g_total = g_total; p.g_scale = g_scales ? g_scales + scale : nullptr;
    p.inv_S = 1.0f / (float)S;
    p.inv_den = (flags & DMH_PHOTO_PIXEL_SUM) ? 1.0f : (float)(1.0 / ((double)B * H * W));
    p.n_ident = automask ? ((flags & DMH_PHOTO_AVG_REPROJECTION) ? 1 : F) : 0;
    return reproj_grad_launch<false>("dmh_photo_image_grad", p, target, src_host, T_host, F, disp, disp_h, disp_w, K,
                                     inv_K, sel, B, H, W, min_depth, max_depth, flags, grad_target, grad_src_host,
                                     (cudaStream_t)stream);
}

int dmh_photo_image_grad_dh(const float* target, const float* const* src_host, const float* const* T_host, int F,
                            const float* disp, int disp_h, int disp_w, const float* K, const float* inv_K,
                            const uint8_t* sel, const float* u, int B, int H, int W, float min_depth, float max_depth,
                            int flags, float* grad_target, float* const* grad_src_host, dmh_stream_t stream) {
    DMH_REQUIRE(u, "dmh_photo_image_grad_dh: null pointer");
    ReprojGradParams p = {};
    p.u_dh = u;
    return reproj_grad_launch<true>("dmh_photo_image_grad_dh", p, target, src_host, T_host, F, disp, disp_h, disp_w, K,
                                    inv_K, sel, B, H, W, min_depth, max_depth, flags, grad_target, grad_src_host,
                                    (cudaStream_t)stream);
}

int dmh_smooth_image_grad(const float* disp, const float* img, int B, int h, int w, const float* img_scalars,
                          float smooth_weight, int scale, int S, const float* g_total, const float* g_scales,
                          int accumulate, float* grad_img, dmh_stream_t stream) {
    DMH_REQUIRE(disp && img && img_scalars && grad_img && (g_total || g_scales), "dmh_smooth_image_grad: null pointer");
    DMH_REQUIRE(S >= 1 && scale >= 0 && scale < S, "dmh_smooth_image_grad: scale %d of %d", scale, S);
    DMH_REQUIRE(B > 0 && B <= 65535 && h >= 2 && w >= 2, "dmh_smooth_image_grad: bad shape");
    const float inv_nx = (float)(1.0 / ((double)B * h * (w - 1))), inv_ny = (float)(1.0 / ((double)B * (h - 1) * w));
    const dim3 grid(ceil_div((long long)h * w, 256), B);
    DMH_LAUNCH(smooth_img_grad_kernel, grid, 256, 0, (cudaStream_t)stream)(
        disp, img, h, w, img_scalars, smooth_weight, g_total, g_scales ? g_scales + scale : nullptr, 1.0f / (float)S,
        inv_nx, inv_ny, accumulate, grad_img);
    DMH_CHECK_LAUNCH("dmh_smooth_image_grad");
    return DMH_OK;
}

}  // extern "C"
