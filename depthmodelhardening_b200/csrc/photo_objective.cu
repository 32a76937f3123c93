// A9-A15 fused: ONE kernel per scale does, for a 32x16 tile of target pixels,
//   disp -> depth -> backproject -> project -> bilinear border warp of every
//   source frame (with a 2-px reflect halo), 3x3 SSIM + L1 reprojection loss,
//   per-pixel min over [identity+noise, reprojection] (automask), the partial
//   sum of to_optimise, AND the backward pass down to d(loss)/d(disp)
//   (+ optional pose-gradient partials), without ever materialising the warped
//   images, the SSIM maps or any autograd intermediate in HBM.
//
// Restates M2/trainer.py:485-519 (generate_images_pred) and :589-660
// (compute_losses) for one scale.  The backward is emitted speculatively in the
// forward call (the loss is a mean with a static upstream weight); the autograd
// wrapper multiplies by the incoming scalar gradient.
//
// Algorithmic bytes per target pixel and scale (fp32, F source frames):
//   read  12 (target) + 12 F (sources, gathered via L2) + 4 (disp) + 4 Fi (ident)
//         + 4 Fi (noise);  write 4 (grad_disp)  [+1 sel]
// Shared memory per CTA: (3 + 1 + 3F) * 720 + 9 * 612 + 612 floats (~43 KB, F=1).
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
#define PH_MAXF DMH_PHOTO_MAX_FRAMES

struct PhotoParams {
    const float* target;
    const float* src[PH_MAXF];
    const float* T[PH_MAXF];
    DispSrc disp;
    const float* K;
    const float* inv_K;
    const float* ident;
    const float* noise;
    float* loss_partial;
    float* grad_disp;
    float* grad_P_partial;
    uint8_t* sel;
    float* warped[PH_MAXF];
    int B, H, W, F, flags;
    DepthScale ds;
    float grad_scale;
    // depth-hints mode (DMH_PHOTO_DEPTH_HINTS; DH/trainer.py:541-590, 666-713)
    int dh;                        // 1: min over frames first, argmin [reprojection, identity, hint], masked sums
    const float* hint_reproj;      // (B,1,H,W) hint reprojection loss + 1000*(1-valid); NULL: no hints
    const float* hint_depth;       // (B,1,H,W)
    const float* hint_valid;       // (B,1,H,W)
    float* grad_hint;              // (B,1,H,W) d(sum proxy*mask_h)/d(up-sampled disp)
};

__device__ __forceinline__ int ext_to_img(int e, int n) {
    e = e < -1 ? -1 : (e > n ? n : e);
    return reflect1(e, n);
}
__device__ __forceinline__ float reflect_mult(int p, int q, int n) {
    float m = 1.0f;
    if (p == 1 && q == 0) m += 1.0f;
    if (p == n - 2 && q == n - 1) m += 1.0f;
    return m;
}

struct Taps {
    long long o00;
    bool nw, ne, sw, se;
};
__device__ __forceinline__ Taps make_taps(const Bilinear& bl, int H, int W) {
    Taps t;
    const bool x0in = bl.x0 >= 0 && bl.x0 < W, x1in = bl.x0 + 1 >= 0 && bl.x0 + 1 < W;
    const bool y0in = bl.y0 >= 0 && bl.y0 < H, y1in = bl.y0 + 1 >= 0 && bl.y0 + 1 < H;
    t.o00 = (long long)bl.y0 * W + bl.x0;
    t.nw = y0in && x0in; t.ne = y0in && x1in; t.sw = y1in && x0in; t.se = y1in && x1in;
    return t;
}

// 3x3 window statistics for one channel plane in shared memory around R2 position (r+1, c+1).
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

template <int F>
__global__ void __launch_bounds__(PH_THREADS)
photo_scale_kernel(const PhotoParams p) {
    extern __shared__ float smem[];
    float* tgt = smem;                          // [3][R2]
    float* dep = tgt + 3 * PH_R2;               // [R2]
    float* pred = dep + PH_R2;                  // [F][3][R2]
    float* ka = pred + F * 3 * PH_R2;           // [3][R1]  gated SSIM coefficient planes
    float* kb = ka + 3 * PH_R1;
    float* kc = kb + 3 * PH_R1;
    float* gl1 = kc + 3 * PH_R1;                // [R1] gate of the winning frame for the L1 term / win index
    float* cams = gl1 + PH_R1;                  // [F][24]
    float* red = cams + F * 24;                 // [32]

    const int tid = threadIdx.x;
    const int H = p.H, W = p.W;
    const int b = blockIdx.z;
    const int x0 = blockIdx.x * PH_TW, y0 = blockIdx.y * PH_TH;
    const size_t N = (size_t)H * W;
    const bool no_ssim = (p.flags & DMH_PHOTO_NO_SSIM) != 0;
    const bool avg = (p.flags & DMH_PHOTO_AVG_REPROJECTION) != 0;
    const bool is_depth = (p.flags & DMH_PHOTO_INPUT_IS_DEPTH) != 0;
    const float w_ssim = no_ssim ? 0.0f : 0.85f / 3.0f;
    const float w_l1 = no_ssim ? 1.0f / 3.0f : 0.15f / 3.0f;

    // ---- cameras
    if (tid < F * 21) {
        const int f = tid / 21, t = tid % 21;
        if (t < 12) {
            const int i = t / 4, j = t % 4;
            const float* k = p.K + b * 16 + i * 4;
            const float* tt = p.T[f] + b * 16 + j;
            float acc = __ldg(k) * __ldg(tt);
            acc = fmaf(__ldg(k + 1), __ldg(tt + 4), acc);
            acc = fmaf(__ldg(k + 2), __ldg(tt + 8), acc);
            acc = fmaf(__ldg(k + 3), __ldg(tt + 12), acc);
            cams[f * 24 + t] = acc;
        } else {
            const int i = (t - 12) / 3, j = (t - 12) % 3;
            cams[f * 24 + t] = __ldg(p.inv_K + b * 16 + i * 4 + j);
        }
    }
    // ---- target tile + depth, 2-px reflect halo
    for (int i = tid; i < PH_R2; i += PH_THREADS) {
        const int r = i / PH_R2W, c = i % PH_R2W;
        const int iy = ext_to_img(y0 - 2 + r, H), ix = ext_to_img(x0 - 2 + c, W);
        const size_t o = (size_t)iy * W + ix;
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) tgt[ch * PH_R2 + i] = __ldg(p.target + ((size_t)b * 3 + ch) * N + o);
        const float dv = load_disp(p.disp, b, iy, ix, H, W);
        dep[i] = is_depth ? dv : disp_to_depth(dv, p.ds);
    }
    __syncthreads();

    // ---- warp every source frame into shared memory
#pragma unroll
    for (int f = 0; f < F; ++f) {
        Camera cam;
#pragma unroll
        for (int i = 0; i < 12; ++i) cam.P[i] = cams[f * 24 + i];
#pragma unroll
        for (int i = 0; i < 9; ++i) cam.iK[i] = cams[f * 24 + 12 + i];
        const float* sp = p.src[f] + (size_t)b * 3 * N;
        for (int i = tid; i < PH_R2; i += PH_THREADS) {
            const int r = i / PH_R2W, c = i % PH_R2W;
            const int iy = ext_to_img(y0 - 2 + r, H), ix = ext_to_img(x0 - 2 + c, W);
            const WarpCoord wc = warp_coord(cam, (float)ix, (float)iy, dep[i], W, H, 1e-7f);
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
                pred[(f * 3 + ch) * PH_R2 + i] = acc;
            }
            if (p.warped[f]) {
                const int ey = y0 - 2 + r, ex = x0 - 2 + c;
                if (r >= 2 && r < PH_TH + 2 && c >= 2 && c < PH_TW + 2 && ey < H && ex < W) {
#pragma unroll
                    for (int ch = 0; ch < 3; ++ch)
                        p.warped[f][((size_t)b * 3 + ch) * N + (size_t)ey * W + ex] = pred[(f * 3 + ch) * PH_R2 + i];
                }
            }
        }
    }
    __syncthreads();

    // ---- forward loss at every valid window centre q of the 1-px ring; argmin; loss sum
    const int Fi = p.ident ? (avg ? 1 : F) : 0;      // identity candidates
    float loss_local = 0.0f;
    float dh_r = 0.f, dh_rm = 0.f, dh_h = 0.f, dh_hm = 0.f;      // depth-hints mode: the four masked sums
    for (int i = tid; i < PH_R1; i += PH_THREADS) {
        const int r = i / PH_R1W, c = i % PH_R1W;
        const int qy = y0 - 1 + r, qx = x0 - 1 + c;
        float win = -1.0f;                           // winning source frame (or -1: identity / invalid)
        if (qy >= 0 && qy < H && qx >= 0 && qx < W) {
            const size_t qo = (size_t)qy * W + qx;
            const int ci = (r + 1) * PH_R2W + (c + 1);
            float rp[F];
            float rp_avg = 0.f;
#pragma unroll
            for (int f = 0; f < F; ++f) {
                float l1 = 0.f, ss = 0.f;
#pragma unroll
                for (int ch = 0; ch < 3; ++ch) {
                    const float* xs = pred + (f * 3 + ch) * PH_R2;
                    const float* ys = tgt + ch * PH_R2;
                    l1 += fabsf(ys[ci] - xs[ci]);
                    if (!no_ssim) {
                        float pass;
                        SsimCoef kk;
                        ss += ssim_value_coef(window_stats(xs, ys, r, c), pass, kk);
                    }
                }
                l1 *= (1.0f / 3.0f);
                rp[f] = no_ssim ? l1 : fmaf(0.85f, ss * (1.0f / 3.0f), 0.15f * l1);
                rp_avg = add_rn(rp_avg, rp[f]);
            }
            rp_avg = div_rn(rp_avg, (float)F);
            const bool interior = r >= 1 && r <= PH_TH && c >= 1 && c <= PH_TW;
            if (p.dh) {
                // depth-hints objective: reduce over the frames FIRST (DH/trainer.py:670-672, 683-685), one
                // tie-break noise plane, argmin over [reprojection, identity, hint] (:541-590)
                float rpm = avg ? rp_avg : rp[0];
                int fb = 0;
                if (!avg) {
#pragma unroll
                    for (int f = 1; f < F; ++f)
                        if (rp[f] < rpm) { rpm = rp[f]; fb = f; }
                }
                int idx = 0;
                float best = rpm;
                if (Fi > 0) {
                    float idv = __ldg(p.ident + ((size_t)b * F) * N + qo);
                    if (avg) {
                        for (int f = 1; f < F; ++f) idv = add_rn(idv, __ldg(p.ident + ((size_t)b * F + f) * N + qo));
                        idv = div_rn(idv, (float)F);
                    } else {
                        for (int f = 1; f < F; ++f) idv = fminf(idv, __ldg(p.ident + ((size_t)b * F + f) * N + qo));
                    }
                    if (p.noise) idv = add_rn(idv, __ldg(p.noise + (size_t)b * N + qo));
                    if (idv < best) { best = idv; idx = 1; }
                }
                if (p.hint_reproj) {
                    const float hv = __ldg(p.hint_reproj + (size_t)b * N + qo);
                    if (hv < best) { best = hv; idx = 2; }
                }
                win = (idx != 1) ? (float)fb : -1.0f;       // reprojection mask = argmin != identity
                if (interior) {
                    if (idx != 1) { dh_r += rpm; dh_rm += 1.0f; }
                    if (p.hint_reproj) {
                        const float m_h = (idx == 2) ? 1.0f : 0.0f;
                        const float depth = dep[ci];
                        const float hd = __ldg(p.hint_depth + (size_t)b * N + qo);
                        const float va = __ldg(p.hint_valid + (size_t)b * N + qo);
                        const float diff = sub_rn(hd, depth);
                        const float a1 = add_rn(fabsf(diff), 1.0f);
                        dh_h += mul_rn(mul_rn(logf(a1), va), m_h);
                        dh_hm += m_h;
                        const float sg = diff > 0.f ? -1.f : (diff < 0.f ? 1.f : 0.f);
                        const float gd = m_h * va * sg / a1;
                        p.grad_hint[(size_t)b * N + qo] = is_depth ? gd : gd * ddepth_ddisp(depth, p.ds);
                    }
                    if (p.sel) p.sel[(size_t)b * N + qo] = (uint8_t)idx;
                }
            } else {
            // candidates in the reference's cat order: identity first, then reprojection
            float best = 3.4e38f;
            int best_idx = 0, idx = 0;
            if (Fi > 0) {
                if (avg) {
                    float s = 0.f;
                    for (int f = 0; f < F; ++f) s = add_rn(s, __ldg(p.ident + ((size_t)b * F + f) * N + qo));
                    float v = div_rn(s, (float)F);
                    if (p.noise) v = add_rn(v, __ldg(p.noise + (size_t)b * N + qo));
                    best = v; best_idx = 0; idx = 1;
                } else {
                    for (int f = 0; f < F; ++f) {
                        float v = __ldg(p.ident + ((size_t)b * F + f) * N + qo);
                        if (p.noise) v = add_rn(v, __ldg(p.noise + ((size_t)b * F + f) * N + qo));
                        if (idx == 0 || v < best) { best = v; best_idx = idx; }
                        ++idx;
                    }
                }
            }
            if (avg) {
                if (idx == 0 || rp_avg < best) { best = rp_avg; best_idx = idx; win = 0.0f; }
            } else {
#pragma unroll
                for (int f = 0; f < F; ++f) {
                    if (idx == 0 || rp[f] < best) { best = rp[f]; best_idx = idx; win = (float)f; }
                    ++idx;
                }
            }
            if (interior) {
                loss_local += best;
                if (p.sel) p.sel[(size_t)b * N + qo] = (uint8_t)best_idx;
            }
            }
        }
        gl1[i] = win;
    }
    __syncthreads();

    // ---- backward, one source frame at a time
    float g_depth_acc[2] = {0.f, 0.f};             // this thread owns interior pixels tid and tid+256
    float gP[F][12];
#pragma unroll
    for (int f = 0; f < F; ++f)
#pragma unroll
        for (int k = 0; k < 12; ++k) gP[f][k] = 0.f;

#pragma unroll
    for (int f = 0; f < F; ++f) {
        // phase A: gated SSIM coefficients of frame f at every ring position
        for (int i = tid; i < PH_R1; i += PH_THREADS) {
            const int r = i / PH_R1W, c = i % PH_R1W;
            const float win = gl1[i];
            const float gate = avg ? (win >= 0.f ? 1.0f / (float)F : 0.f) : (win == (float)f ? 1.0f : 0.f);
#pragma unroll
            for (int ch = 0; ch < 3; ++ch) {
                float a = 0.f, bq = 0.f, cq = 0.f;
                if (gate != 0.f && !no_ssim) {
                    const SsimStatsRows st = window_stats(pred + (f * 3 + ch) * PH_R2, tgt + ch * PH_R2, r, c);
                    float pass;
                    SsimCoef k;
                    ssim_value_coef(st, pass, k);
                    const float g = gate * w_ssim * pass;
                    a = g * k.ax; bq = g * k.b; cq = g * k.c;
                }
                ka[ch * PH_R1 + i] = a; kb[ch * PH_R1 + i] = bq; kc[ch * PH_R1 + i] = cq;
            }
        }
        __syncthreads();
        // phase B: box-sum the coefficient planes -> d/d(pred), chain through the warp
        Camera cam;
#pragma unroll
        for (int i = 0; i < 12; ++i) cam.P[i] = cams[f * 24 + i];
#pragma unroll
        for (int i = 0; i < 9; ++i) cam.iK[i] = cams[f * 24 + 12 + i];
        const float* sp = p.src[f] + (size_t)b * 3 * N;
#pragma unroll
        for (int slot = 0; slot < 2; ++slot) {
            const int i = tid + slot * PH_THREADS;
            const int r = i / PH_TW, c = i % PH_TW;
            const int py = y0 + r, px = x0 + c;
            if (py >= H || px >= W) continue;
            const int ci2 = (r + 2) * PH_R2W + (c + 2);
            const int ci1 = (r + 1) * PH_R1W + (c + 1);
            const float win = gl1[ci1];
            const float gate = avg ? (win >= 0.f ? 1.0f / (float)F : 0.f) : (win == (float)f ? 1.0f : 0.f);
            float wy[3], wx[3];
#pragma unroll
            for (int d = 0; d < 3; ++d) {
                wy[d] = reflect_mult(py, py - 1 + d, H);
                wx[d] = reflect_mult(px, px - 1 + d, W);
            }
            float g_pred[3];
#pragma unroll
            for (int ch = 0; ch < 3; ++ch) {
                float sa = 0.f, sb = 0.f, sc = 0.f;
                if (!no_ssim) {
#pragma unroll
                    for (int dy = 0; dy < 3; ++dy)
#pragma unroll
                        for (int dx = 0; dx < 3; ++dx) {
                            const float w = wy[dy] * wx[dx];
                            const int o = ch * PH_R1 + (r + dy) * PH_R1W + c + dx;
                            sa = fmaf(w, ka[o], sa);
                            sb = fmaf(w, kb[o], sb);
                            sc = fmaf(w, kc[o], sc);
                        }
                }
                const float xv = pred[(f * 3 + ch) * PH_R2 + ci2], yv = tgt[ch * PH_R2 + ci2];
                const float d = xv - yv;
                const float sg = d > 0.f ? 1.f : (d < 0.f ? -1.f : 0.f);
                g_pred[ch] = sa + sb * xv + sc * yv + gate * w_l1 * sg;
            }
            // chain through the bilinear gather (recomputed: taps are L1/L2 hits)
            const WarpCoord wc = warp_coord(cam, (float)px, (float)py, dep[ci2], W, H, 1e-7f);
            const Bilinear bl = bilinear_setup(wc.ix, wc.iy);
            const Taps t = make_taps(bl, H, W);
            float gix = 0.f, giy = 0.f;
#pragma unroll
            for (int ch = 0; ch < 3; ++ch) {
                const float* s = sp + ch * N;
                const float go = g_pred[ch];
                if (t.nw) { const float v = __ldg(s + t.o00);         gix -= v * bl.ty1 * go; giy -= v * bl.tx1 * go; }
                if (t.ne) { const float v = __ldg(s + t.o00 + 1);     gix += v * bl.ty1 * go; giy -= v * bl.tx0 * go; }
                if (t.sw) { const float v = __ldg(s + t.o00 + W);     gix -= v * bl.ty0 * go; giy += v * bl.tx1 * go; }
                if (t.se) { const float v = __ldg(s + t.o00 + W + 1); gix += v * bl.ty0 * go; giy += v * bl.tx0 * go; }
            }
            float dp[3];
            g_depth_acc[slot] += warp_coord_bwd(cam, wc, gix, giy, W, H, dp);
            if (p.grad_P_partial) {
                const float depth = dep[ci2];
                const float pt[4] = {depth * wc.ray[0], depth * wc.ray[1], depth * wc.ray[2], 1.0f};
#pragma unroll
                for (int a = 0; a < 3; ++a)
#pragma unroll
                    for (int k = 0; k < 4; ++k) gP[f][a * 4 + k] = fmaf(dp[a], pt[k], gP[f][a * 4 + k]);
            }
        }
        __syncthreads();
    }

    // ---- outputs
#pragma unroll
    for (int slot = 0; slot < 2; ++slot) {
        const int i = tid + slot * PH_THREADS;
        const int r = i / PH_TW, c = i % PH_TW;
        const int py = y0 + r, px = x0 + c;
        if (py >= H || px >= W) continue;
        const float depth = dep[(r + 2) * PH_R2W + (c + 2)];
        const float g = g_depth_acc[slot] * p.grad_scale;
        p.grad_disp[(size_t)b * N + (size_t)py * W + px] = is_depth ? g : g * ddepth_ddisp(depth, p.ds);
    }
    const int blk = (b * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x;
    if (p.dh) {
        // [4][B * tiles]: sum reproj*mask_r, sum mask_r, sum proxy*mask_h, sum mask_h
        const int nblk = p.B * gridDim.x * gridDim.y;
        float s = block_sum(dh_r, red);
        if (tid == 0) p.loss_partial[blk] = s;
        s = block_sum(dh_rm, red);
        if (tid == 0) p.loss_partial[nblk + blk] = s;
        s = block_sum(dh_h, red);
        if (tid == 0) p.loss_partial[2 * nblk + blk] = s;
        s = block_sum(dh_hm, red);
        if (tid == 0) p.loss_partial[3 * nblk + blk] = s;
    } else {
        const float s = block_sum(loss_local, red);
        if (tid == 0) p.loss_partial[blk] = s;
    }
    if (p.grad_P_partial) {
        const int tiles = gridDim.x * gridDim.y;
        const int tile = blockIdx.y * gridDim.x + blockIdx.x;
#pragma unroll
        for (int f = 0; f < F; ++f) {
            float* out = p.grad_P_partial + (((size_t)f * p.B + b) * tiles + tile) * 12;
#pragma unroll
            for (int k = 0; k < 12; ++k) {
                const float s = block_sum(gP[f][k] * p.grad_scale, red);
                if (tid == 0) out[k] = s;
            }
        }
    }
}

size_t photo_smem_bytes(int F) {
    return sizeof(float) * ((size_t)(3 + 1 + 3 * F) * PH_R2 + 9 * PH_R1 + PH_R1 + (size_t)F * 24 + 32);
}

template <int F>
int launch_photo(const PhotoParams& p, dim3 grid, cudaStream_t st) {
    const size_t smem = photo_smem_bytes(F);
    static KernelSetup setup;
    const void* kernel = (const void*)photo_scale_kernel<F>;
    if (setup.sms("dmh_photo_scale", &kernel, 1, smem) == 0) return DMH_ERR_CUDA;
    DMH_LAUNCH(photo_scale_kernel<F>, grid, PH_THREADS, smem, st)(p);
    return DMH_OK;
}

}  // namespace

namespace dmh {
int photo_fast_tiles(int H, int W);
int launch_photo_fast(const float* target, const float* src, const float* T, const float* disp, int disp_h,
                      int disp_w, const float* K, const float* inv_K, const float* ident, const float* noise, int B, int H, int W, float min_depth,
                      float max_depth, int flags, float grad_scale, float* loss_partial, float* grad_disp,
                      uint8_t* sel, float* warped, const FastDhArgs* dh, cudaStream_t st);
int launch_ident_bf16(const uint16_t* target, const uint16_t* src, int B, int H, int W, int no_ssim, float* out,
                      float* packed, float* tgt_f32, cudaStream_t st);
int launch_ident_fast(const float* target, const float* const* src_host, int F, int B, int H, int W, int no_ssim,
                      float* out, float* packed, cudaStream_t st);
}  // namespace dmh

namespace {

// dmh_photo_scale (dh == nullptr) and dmh_photo_scale_dh: argument checks, then the single-source fast kernel or the
// general one.  With depth hints, loss_partial holds the four [B * dmh_photo_tiles] arrays of the depth-hints sums
// and the fast path also excludes DMH_PHOTO_AVG_REPROJECTION.  `name` is the public entry point, for the errors.
int photo_scale_launch(const char* name, const float* target, const float* const* src_host, const float* const* T_host,
                       int F, const float* disp, int disp_h, int disp_w, const float* K, const float* inv_K,
                       const float* ident, const float* noise, int B, int H, int W, float min_depth, float max_depth,
                       int flags, float grad_scale, float* loss_partial, float* grad_disp, float* grad_P_partial,
                       uint8_t* sel, float* const* warped_host, const FastDhArgs* dh, cudaStream_t st) {
    DMH_REQUIRE(target && src_host && T_host && disp && K && inv_K && loss_partial && grad_disp, "%s: null pointer", name);
    DMH_REQUIRE(F >= 1 && F <= PH_MAXF, "%s: F=%d outside [1,%d]", name, F, PH_MAXF);
    DMH_REQUIRE(B > 0 && B <= 65535 && H >= 2 && W >= 2, "%s: bad shape B=%d H=%d W=%d", name, B, H, W);
    DMH_REQUIRE(disp_h >= 1 && disp_w >= 1 && disp_h <= H && disp_w <= W, "%s: bad disparity size %dx%d", name, disp_h,
                disp_w);
    const bool is_depth = (flags & DMH_PHOTO_INPUT_IS_DEPTH) != 0;
    DMH_REQUIRE(is_depth || (min_depth > 0.f && max_depth > min_depth), "%s: bad depth range", name);
    DMH_REQUIRE(!(flags & DMH_PHOTO_SRC_PACKED) || (uintptr_t)src_host[0] % 16 == 0,
                "%s: DMH_PHOTO_SRC_PACKED needs a 16-byte aligned source", name);
    const int fast_excl = DMH_PHOTO_NO_SSIM | DMH_PHOTO_INPUT_IS_DEPTH | (dh ? DMH_PHOTO_AVG_REPROJECTION : 0);
    const bool fast_ok = F == 1 && !grad_P_partial && !(warped_host && warped_host[0]) && !(flags & fast_excl) &&
                         H * (long long)W < (1ll << 28);
    DMH_REQUIRE(!(flags & DMH_PHOTO_SRC_PACKED) || fast_ok,
                "%s: DMH_PHOTO_SRC_PACKED needs the single-source fast path (F == 1, SSIM on, disparity input, no pose "
                "gradient, no warped output)", name);
    const int nblk = B * dmh_photo_tiles(H, W);
    if (fast_ok) {
        // single source frame, no pose gradient: the 32x32-tile fast kernel (photo_fast.cu).  It writes fewer partial
        // sums than dmh_photo_tiles() promises (at the head of each array); zero the rest so the caller's reduction is
        // exact.
        DMH_REQUIRE(src_host[0] && T_host[0], "%s: null src/T for frame 0", name);
        const int used = B * photo_fast_tiles(H, W);
        cudaError_t e = cudaSuccess;
        if (dh) e = cudaMemsetAsync(loss_partial, 0, sizeof(float) * 4 * (size_t)nblk, st);
        else if (nblk > used) e = cudaMemsetAsync(loss_partial + used, 0, sizeof(float) * (size_t)(nblk - used), st);
        if (e != cudaSuccess) { set_error("%s: memset failed: %s", name, cudaGetErrorString(e)); return DMH_ERR_CUDA; }
        FastDhArgs a = {};
        if (dh) { a = *dh; a.nblk = nblk; }
        const int rc = launch_photo_fast(target, src_host[0], T_host[0], disp, disp_h, disp_w, K, inv_K, ident, noise, B, H,
                                         W, min_depth, max_depth, flags, grad_scale, loss_partial, grad_disp, sel,
                                         warped_host ? warped_host[0] : nullptr, dh ? &a : nullptr, st);
        if (rc != DMH_OK) return rc;
        DMH_CHECK_LAUNCH(name);
        return DMH_OK;
    }
    PhotoParams p;
    p.target = target;
    for (int f = 0; f < PH_MAXF; ++f) {
        p.src[f] = f < F ? src_host[f] : nullptr;
        p.T[f] = f < F ? T_host[f] : nullptr;
        p.warped[f] = (warped_host && f < F) ? warped_host[f] : nullptr;
        DMH_REQUIRE(f >= F || (p.src[f] && p.T[f]), "%s: null src/T for frame %d", name, f);
    }
    p.disp.ptr = disp; p.disp.h = disp_h; p.disp.w = disp_w;
    p.disp.sh = (float)disp_h / (float)H; p.disp.sw = (float)disp_w / (float)W;
    p.K = K; p.inv_K = inv_K; p.ident = ident; p.noise = noise;
    p.loss_partial = loss_partial; p.grad_disp = grad_disp; p.grad_P_partial = grad_P_partial; p.sel = sel;
    p.B = B; p.H = H; p.W = W; p.F = F; p.flags = flags;
    p.ds = depth_scale(min_depth, max_depth, is_depth);
    p.grad_scale = grad_scale;
    p.dh = dh != nullptr;
    p.hint_reproj = dh ? dh->hint_reproj : nullptr; p.hint_depth = dh ? dh->hint_depth : nullptr;
    p.hint_valid = dh ? dh->hint_valid : nullptr; p.grad_hint = dh ? dh->grad_hint : nullptr;
    dim3 grid(ceil_div(W, PH_TW), ceil_div(H, PH_TH), B);
    int rc = DMH_OK;
    switch (F) {
        case 1: rc = launch_photo<1>(p, grid, st); break;
        case 2: rc = launch_photo<2>(p, grid, st); break;
        case 3: rc = launch_photo<3>(p, grid, st); break;
        default: rc = launch_photo<4>(p, grid, st); break;
    }
    if (rc != DMH_OK) return rc;
    DMH_CHECK_LAUNCH(name);
    return DMH_OK;
}

}  // namespace

extern "C" {

int dmh_identity_loss(const float* target, const float* const* src_host, int F, int B, int H, int W, int no_ssim,
                      float* ident, dmh_stream_t stream) {
    DMH_REQUIRE(target && src_host && ident, "dmh_identity_loss: null pointer");
    DMH_REQUIRE(F >= 1 && F <= PH_MAXF, "dmh_identity_loss: F=%d outside [1,%d]", F, PH_MAXF);
    DMH_REQUIRE(B > 0 && (long long)B * F <= 65535 && H >= 2 && W >= 2, "dmh_identity_loss: bad shape");
    for (int f = 0; f < F; ++f) DMH_REQUIRE(src_host[f], "dmh_identity_loss: null src for frame %d", f);
    const int rc = launch_ident_fast(target, src_host, F, B, H, W, no_ssim, ident, nullptr, (cudaStream_t)stream);
    if (rc != DMH_OK) return rc;
    DMH_CHECK_LAUNCH("dmh_identity_loss");
    return DMH_OK;
}

int dmh_identity_loss_pack(const float* target, const float* src, int B, int H, int W, int no_ssim, float* ident,
                           float* src_packed, dmh_stream_t stream) {
    DMH_REQUIRE(target && src && src_packed, "dmh_identity_loss_pack: null pointer");
    DMH_REQUIRE(B > 0 && B <= 65535 && H >= 2 && W >= 2, "dmh_identity_loss_pack: bad shape");
    DMH_REQUIRE((uintptr_t)src_packed % 16 == 0, "dmh_identity_loss_pack: src_packed must be 16-byte aligned");
    const float* srcs[1] = {src};
    const int rc = launch_ident_fast(target, srcs, 1, B, H, W, no_ssim, ident, src_packed, (cudaStream_t)stream);
    if (rc != DMH_OK) return rc;
    DMH_CHECK_LAUNCH("dmh_identity_loss_pack");
    return DMH_OK;
}

int dmh_identity_loss_pack_bf16(const uint16_t* target_bf16, const uint16_t* src_bf16, int B, int H, int W, int no_ssim,
                                float* ident, float* src_packed, float* target_f32, dmh_stream_t stream) {
    DMH_REQUIRE(target_bf16 && src_bf16 && src_packed && target_f32, "dmh_identity_loss_pack_bf16: null pointer");
    DMH_REQUIRE(B > 0 && B <= 65535 && H >= 2 && W >= 2, "dmh_identity_loss_pack_bf16: bad shape");
    DMH_REQUIRE(W % 8 == 0 && (uintptr_t)target_bf16 % 16 == 0 && (uintptr_t)src_bf16 % 16 == 0,
                "dmh_identity_loss_pack_bf16: needs W %% 8 == 0 and 16-byte aligned frames (128-bit loads of 8 bf16)");
    DMH_REQUIRE((uintptr_t)src_packed % 16 == 0, "dmh_identity_loss_pack_bf16: src_packed must be 16-byte aligned");
    const int rc = launch_ident_bf16(target_bf16, src_bf16, B, H, W, no_ssim, ident, src_packed, target_f32,
                                     (cudaStream_t)stream);
    if (rc != DMH_OK) return rc;
    DMH_CHECK_LAUNCH("dmh_identity_loss_pack_bf16");
    return DMH_OK;
}

int dmh_photo_tiles(int H, int W) { return ceil_div(W, PH_TW) * ceil_div(H, PH_TH); }

int dmh_photo_scale(const float* target, const float* const* src_host, const float* const* T_host, int F,
                    const float* disp, int disp_h, int disp_w, const float* K, const float* inv_K, const float* ident,
                    const float* noise, int B, int H, int W, float min_depth, float max_depth, int flags, float grad_scale,
                    float* loss_partial, float* grad_disp, float* grad_P_partial, uint8_t* sel,
                    float* const* warped_host, dmh_stream_t stream) {
    return photo_scale_launch("dmh_photo_scale", target, src_host, T_host, F, disp, disp_h, disp_w, K, inv_K, ident,
                              noise, B, H, W, min_depth, max_depth, flags, grad_scale, loss_partial, grad_disp,
                              grad_P_partial, sel, warped_host, nullptr, (cudaStream_t)stream);
}

int dmh_photo_scale_dh(const float* target, const float* const* src_host, const float* const* T_host, int F,
                       const float* disp, int disp_h, int disp_w, const float* K, const float* inv_K,
                       const float* ident, const float* noise, const float* hint_reproj, const float* hint_depth,
                       const float* hint_valid, int B, int H, int W, float min_depth, float max_depth, int flags,
                       float* sums_partial, float* grad_disp, float* grad_disp_hint, float* grad_P_partial,
                       uint8_t* sel, dmh_stream_t stream) {
    DMH_REQUIRE(!hint_reproj || (hint_depth && hint_valid && grad_disp_hint),
                "dmh_photo_scale_dh: depth hints need hint_depth, hint_valid and grad_disp_hint");
    DMH_REQUIRE(!noise || ident, "dmh_photo_scale_dh: noise without identity losses");
    const FastDhArgs dh = {hint_reproj, hint_depth, hint_valid, grad_disp_hint, 0};
    return photo_scale_launch("dmh_photo_scale_dh", target, src_host, T_host, F, disp, disp_h, disp_w, K, inv_K, ident,
                              noise, B, H, W, min_depth, max_depth, flags, 1.0f, sums_partial, grad_disp, grad_P_partial,
                              sel, nullptr, &dh, (cudaStream_t)stream);
}

}  // extern "C"
