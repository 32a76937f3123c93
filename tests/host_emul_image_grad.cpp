// TEST INFRASTRUCTURE ONLY -- never linked into or loaded by the product.
//
// The colour-frame gradients of one scale of the fused objective (csrc/photo_image_grad.cu), computed with the
// per-pixel helpers of dmh_math.cuh (candidate gates, coefficient form of the SSIM backward, reflection
// multiplicities, border-clamped bilinear taps) over whole images with plain loops, so that the maths can be
// checked against the oracle's autograd on a machine without a GPU.  The tiling of the kernels is exercised by the
// `-m gpu` tests.
//
// Build: g++ -O1 -ffp-contract=off -shared -fPIC -o tests/_build/libdmh_hostemu_ig.so tests/host_emul_image_grad.cpp
#include <cstdint>
#include <vector>

#include "../depthmodelhardening_b200/csrc/dmh_math.cuh"

using namespace dmh;

namespace {

// gated coefficient planes k[4][3][H*W] (ax, b, c, ay) of R(x, y) at every window centre with a non-zero gate
void coef_planes(const float* x, const float* y, const float* gate, int H, int W, float w_ssim, std::vector<float>& k) {
    const size_t N = (size_t)H * W;
    k.assign(12 * N, 0.0f);
    for (int qy = 0; qy < H; ++qy)
        for (int qx = 0; qx < W; ++qx) {
            const size_t q = (size_t)qy * W + qx;
            if (gate[q] == 0.0f) continue;
            for (int ch = 0; ch < 3; ++ch) {
                const float* xc = x + ch * N;
                const float* yc = y + ch * N;
                Row5 rows[3];
                for (int dy = 0; dy < 3; ++dy) {
                    const size_t r = (size_t)ext_to_img(qy - 1 + dy, H) * W;
                    const int c0 = ext_to_img(qx - 1, W), c1 = qx, c2 = ext_to_img(qx + 1, W);
                    rows[dy] = row5(xc[r + c0], xc[r + c1], xc[r + c2], yc[r + c0], yc[r + c1], yc[r + c2]);
                }
                float pass;
                SsimCoef kk;
                ssim_value_coef(ssim_stats_rows(rows[0], rows[1], rows[2]), pass, kk);
                const float g = gate[q] * w_ssim * pass;
                k[(0 * 3 + ch) * N + q] = g * kk.ax;
                k[(1 * 3 + ch) * N + q] = g * kk.b;
                k[(2 * 3 + ch) * N + q] = g * kk.c;
                k[(3 * 3 + ch) * N + q] = g * kk.ay;
            }
        }
}

// d/dx (into gx, written) and d/dy (added into gy) of sum_q gate(q) * R(x, y)(q)
void pixel_grads(const float* x, const float* y, const float* gate, const std::vector<float>& k, int H, int W,
                 bool ssim, float w_l1, float* gx, float* gy) {
    const size_t N = (size_t)H * W;
    for (int py = 0; py < H; ++py)
        for (int px = 0; px < W; ++px) {
            const size_t p = (size_t)py * W + px;
            for (int ch = 0; ch < 3; ++ch) {
                float sa = 0.f, sb = 0.f, sc = 0.f, sd = 0.f;
                for (int qy = py - 1; ssim && qy <= py + 1; ++qy)
                    for (int qx = px - 1; qx <= px + 1; ++qx) {
                        if (qy < 0 || qy >= H || qx < 0 || qx >= W) continue;
                        const float w = reflect_mult(py, qy, H) * reflect_mult(px, qx, W);
                        const size_t o = ch * N + (size_t)qy * W + qx;
                        sa = fmaf(w, k[o], sa);
                        sb = fmaf(w, k[3 * N + o], sb);
                        sc = fmaf(w, k[6 * N + o], sc);
                        sd = fmaf(w, k[9 * N + o], sd);
                    }
                float a, b;
                reproj_pixel_grad(sa, sb, sc, sd, x[ch * N + p], y[ch * N + p], gate[p] * w_l1, a, b);
                gx[ch * N + p] = a;
                gy[ch * N + p] += b;
            }
        }
}

}  // namespace

extern "C" {

// Gradients of weight * sum_p m(p) for one scale, m = the candidate `sel` picked (cat order), w.r.t. the target and
// every source frame.  disp_full: (B,1,H,W) disparity at the target's size.  Outputs (B,3,H,W) are overwritten.
void emu_image_grad(const float* target, const float* const* srcs, const float* const* Ts, int F,
                    const float* disp_full, const float* K, const float* inv_K, const uint8_t* sel, int B, int H, int W,
                    float min_depth, float max_depth, int flags, int automask, float weight, float* grad_target,
                    float* const* grad_src) {
    const size_t N = (size_t)H * W;
    const bool no_ssim = (flags & 1) != 0, avg = (flags & 2) != 0;
    const int n_ident = automask ? (avg ? 1 : F) : 0;
    const float w_ssim = no_ssim ? 0.0f : 0.85f / 3.0f;
    const float w_l1 = no_ssim ? 1.0f / 3.0f : 0.15f / 3.0f;
    DepthScale ds;
    ds.min_disp = (float)(1.0 / (double)max_depth);
    ds.range = (float)(1.0 / (double)min_depth - 1.0 / (double)max_depth);
    std::vector<float> gate(N), k, pred(3 * N), gx(3 * N);
    std::vector<Bilinear> bl(N);
    for (int b = 0; b < B; ++b) {
        const float* tg = target + (size_t)b * 3 * N;
        float* gt = grad_target + (size_t)b * 3 * N;
        for (size_t i = 0; i < 3 * N; ++i) gt[i] = 0.0f;
        for (int f = 0; f < F; ++f) {
            const float* sp = srcs[f] + (size_t)b * 3 * N;
            float* gs = grad_src[f] + (size_t)b * 3 * N;
            // identity candidate: the un-warped pair (src_f, target)
            for (size_t q = 0; q < N; ++q) gate[q] = weight * ident_gate(sel[(size_t)b * N + q], f, n_ident, F, avg);
            if (!no_ssim) coef_planes(sp, tg, gate.data(), H, W, w_ssim, k);
            pixel_grads(sp, tg, gate.data(), k, H, W, !no_ssim, w_l1, gs, gt);
            // reprojection candidate: src_f warped into the target view, d/d(warped) scattered to the taps
            Camera cam;
            compose_camera(K + b * 16, Ts[f] + b * 16, inv_K + b * 16, cam);
            for (int py = 0; py < H; ++py)
                for (int px = 0; px < W; ++px) {
                    const size_t p = (size_t)py * W + px;
                    const WarpCoord wc = warp_coord(cam, (float)px, (float)py,
                                                    disp_to_depth(disp_full[(size_t)b * N + p], ds), W, H, 1e-7f);
                    bl[p] = bilinear_setup(wc.ix, wc.iy);
                    const Taps t = make_taps(bl[p], H, W);
                    for (int ch = 0; ch < 3; ++ch) {
                        const float* s = sp + ch * N;
                        float acc = 0.0f;
                        if (t.nw) acc = fmaf(s[t.o00], bl[p].wnw, acc);
                        if (t.ne) acc = fmaf(s[t.o00 + 1], bl[p].wne, acc);
                        if (t.sw) acc = fmaf(s[t.o00 + W], bl[p].wsw, acc);
                        if (t.se) acc = fmaf(s[t.o00 + W + 1], bl[p].wse, acc);
                        pred[ch * N + p] = acc;
                    }
                }
            for (size_t q = 0; q < N; ++q) gate[q] = weight * reproj_gate(sel[(size_t)b * N + q], f, n_ident, F, avg);
            if (!no_ssim) coef_planes(pred.data(), tg, gate.data(), H, W, w_ssim, k);
            pixel_grads(pred.data(), tg, gate.data(), k, H, W, !no_ssim, w_l1, gx.data(), gt);
            for (size_t p = 0; p < N; ++p) {
                const Taps t = make_taps(bl[p], H, W);
                for (int ch = 0; ch < 3; ++ch) {
                    float* g = gs + ch * N;
                    const float go = gx[ch * N + p];
                    if (t.nw) g[t.o00] += bl[p].wnw * go;
                    if (t.ne) g[t.o00 + 1] += bl[p].wne * go;
                    if (t.sw) g[t.o00 + W] += bl[p].wsw * go;
                    if (t.se) g[t.o00 + W + 1] += bl[p].wse * go;
                }
            }
        }
    }
}

}  // extern "C"
