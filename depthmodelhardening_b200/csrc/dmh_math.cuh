// Per-pixel math of the hot path, shared by every kernel.
//
// Everything here is `DMH_HD` (__host__ __device__) and free of CUDA-only
// constructs so that tests/host_emul.cpp can compile the SAME formulas with g++
// and check them against the oracle on a machine without a GPU.  The host build
// is test infrastructure; the product only ever runs the device instantiation.
//
// Reference lines restated (paths under /root/reference/DepthNetworks/monodepth2):
//   disp_to_depth            layers.py:16-25
//   BackprojectDepth.forward layers.py:163-168
//   Project3D.forward        layers.py:182-198
//   F.grid_sample(border, align_corners=True)  trainer.py:515-519 (ATen GridSampler.cuh)
//   SSIM.forward             layers.py:239-253
//   compute_reprojection_loss trainer.py:525-537
#pragma once

#if defined(__CUDACC__)
#define DMH_HD __host__ __device__ __forceinline__
#else
#define DMH_HD inline
#endif

#include <math.h>

namespace dmh {

// Rounded-once primitives: the coordinate chain of the reference is a sequence
// of separate elementwise torch ops, each rounded to fp32.  Forbid FMA
// contraction there so floor() lands on the same side as ATen's.
#if defined(__CUDA_ARCH__)
DMH_HD float mul_rn(float a, float b) { return __fmul_rn(a, b); }
DMH_HD float add_rn(float a, float b) { return __fadd_rn(a, b); }
DMH_HD float sub_rn(float a, float b) { return __fsub_rn(a, b); }
DMH_HD float div_rn(float a, float b) { return __fdiv_rn(a, b); }
// 1/x correctly rounded == div_rn(1.0f, x) bit for bit, without the generic division's slow-path call site
DMH_HD float rcp_rn(float x) { return __frcp_rn(x); }
#else
DMH_HD float rcp_rn(float x) { volatile float r = 1.0f / x; return r; }
DMH_HD float mul_rn(float a, float b) { volatile float r = a * b; return r; }
DMH_HD float add_rn(float a, float b) { volatile float r = a + b; return r; }
DMH_HD float sub_rn(float a, float b) { volatile float r = a - b; return r; }
DMH_HD float div_rn(float a, float b) { volatile float r = a / b; return r; }
#endif

// MUFU.RCP (1 ulp) on the device, IEEE division on the host emulation.  Used only where ~1e-7 relative error is
// irrelevant: the SSIM denominator d = B1*B2 >= C1*C2 > 0 (value tolerance 1e-5) and the 1/z of the BACKWARD
// chain (gradient tolerance 1e-5); never in the forward coordinate chain, whose floor() picks the taps.
#if defined(__CUDA_ARCH__)
DMH_HD float fast_rcp(float x) { float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
#else
DMH_HD float fast_rcp(float x) { return 1.0f / x; }
#endif

// ---------------------------------------------------------------------------
// Camera model for one batch item: P = (K @ T)[:3,:] and inv_K[:3,:3].
struct Camera {
    float P[12];    // row-major 3x4
    float iK[9];    // row-major 3x3
};

// (K @ T)[:3,:], fp32 accumulate in k order (layers.py:188).
DMH_HD void compose_camera(const float* K, const float* T, const float* inv_K, Camera& cam) {
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 4; ++j) {
            float acc = K[i * 4 + 0] * T[0 * 4 + j];
            acc = fmaf(K[i * 4 + 1], T[1 * 4 + j], acc);
            acc = fmaf(K[i * 4 + 2], T[2 * 4 + j], acc);
            acc = fmaf(K[i * 4 + 3], T[3 * 4 + j], acc);
            cam.P[i * 4 + j] = acc;
        }
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) cam.iK[i * 3 + j] = inv_K[i * 4 + j];
}

struct DepthScale {      // disp_to_depth constants, computed in double on the host
    float min_disp;      // 1/max_depth
    float range;         // 1/min_depth - 1/max_depth
};

DMH_HD float disp_to_depth(float disp, const DepthScale& ds) {
    const float scaled = add_rn(ds.min_disp, mul_rn(ds.range, disp));
    return rcp_rn(scaled);
}
// d depth / d disp = -range * depth^2
DMH_HD float ddepth_ddisp(float depth, const DepthScale& ds) { return -ds.range * depth * depth; }

// inv_K[:3,:3] @ (x, y, 1)
DMH_HD void pixel_ray(const Camera& cam, float x, float y, float ray[3]) {
    for (int i = 0; i < 3; ++i) {
        float acc = cam.iK[i * 3 + 0] * x;
        acc = fmaf(cam.iK[i * 3 + 1], y, acc);
        acc = add_rn(acc, cam.iK[i * 3 + 2]);
        ray[i] = acc;
    }
}

// P @ (X, Y, Z, 1)
DMH_HD void project_point(const Camera& cam, const float pt[3], float p[3]) {
    for (int i = 0; i < 3; ++i) {
        float acc = cam.P[i * 4 + 0] * pt[0];
        acc = fmaf(cam.P[i * 4 + 1], pt[1], acc);
        acc = fmaf(cam.P[i * 4 + 2], pt[2], acc);
        acc = add_rn(acc, cam.P[i * 4 + 3]);
        p[i] = acc;
    }
}

// Normalised sampling coordinate as Project3D returns it (layers.py:192-197).
DMH_HD float normalise_coord(float num, float den_eps, int size) {
    const float raw = div_rn(num, den_eps);
    const float n = div_rn(raw, (float)(size - 1));
    return mul_rn(sub_rn(n, 0.5f), 2.0f);
}

// ATen grid_sampler_unnormalize (align_corners True / False)
DMH_HD float unnormalise_coord(float g, int size, bool align_corners) {
    // "/ 2" is exact in binary floating point: x * 0.5f rounds identically and is one instruction
    if (align_corners) return mul_rn(mul_rn(add_rn(g, 1.0f), 0.5f), (float)(size - 1));
    return mul_rn(sub_rn(mul_rn(add_rn(g, 1.0f), (float)size), 1.0f), 0.5f);
}
DMH_HD float unnormalise_mult(int size, bool align_corners) {
    return align_corners ? (float)(size - 1) / 2.0f : (float)size / 2.0f;
}

// ATen clip_coordinates_set_grad: borders count as out of bounds for the gradient.
DMH_HD float clip_coord(float in, int size, float& grad_mult) {
    if (in <= 0.0f) { grad_mult = 0.0f; return 0.0f; }
    const float mx = (float)(size - 1);
    if (in >= mx) { grad_mult = 0.0f; return mx; }
    grad_mult = 1.0f;
    return in;
}
// forward-only clip: min(size-1, max(in, 0)) with fmin/fmax NaN semantics (NaN -> 0)
DMH_HD float clip_coord_fwd(float in, int size) { return fminf((float)(size - 1), fmaxf(in, 0.0f)); }

// ATen safe_downgrade_to_int_range
DMH_HD float safe_coord(float x) {
    if (x > 2147483646.0f || x < -2147483648.0f || !isfinite(x)) return -100.0f;
    return x;
}

struct Bilinear {
    int x0, y0;            // north-west tap (may be out of bounds)
    float wnw, wne, wsw, wse;
    float tx1, tx0, ty1, ty0;   // (ix_se-ix), (ix-ix_nw), (iy_se-iy), (iy-iy_nw)
};

DMH_HD Bilinear bilinear_setup(float ix, float iy) {
    Bilinear b;
    const float fx = floorf(ix), fy = floorf(iy);
    b.x0 = (int)fx;
    b.y0 = (int)fy;
    b.tx1 = (fx + 1.0f) - ix;
    b.tx0 = ix - fx;
    b.ty1 = (fy + 1.0f) - iy;
    b.ty0 = iy - fy;
    b.wnw = b.tx1 * b.ty1;
    b.wne = b.tx0 * b.ty1;
    b.wsw = b.tx1 * b.ty0;
    b.wse = b.tx0 * b.ty0;
    return b;
}

// a / c for a launch constant c (W-1, H-1) in three instructions: q0 = a*rc, r = a - q0*c (exact, FMA),
// q = q0 + r*rc.  Correctly rounded -- i.e. bit-identical to IEEE division -- for the constants the library has
// verified EXHAUSTIVELY on the device (all 2^24 significands of two binades; for normal quotients the result depends
// only on the significand of a: valid for 2^-100 <= |a| <= FLT_MAX), see dmh::const_div_exact() in core.cu; other
// constants take div_rn.  +-inf / NaN pass through.
DMH_HD float div_const(float a, float c, float rc) {
    const float q0 = mul_rn(a, rc);
    const float r = fmaf(-q0, c, a);
    const float q = fmaf(r, rc, q0);
    return (fabsf(a) <= 3.402823466e+38f) ? q : a;
}

// Full forward coordinate chain of A9-A12 for target pixel (x,y) with depth d.
struct WarpCoord {
    float ix, iy;          // clipped source coordinates
    float mx, my;          // d(ix)/d(gx) incl. clip gate; d(iy)/d(gy)
    float inv_z;           // 1/(p2+eps)
    float u_raw, v_raw;    // p0/(p2+eps), p1/(p2+eps)
    float ray[3];
};

template <bool FASTDIV = false>
DMH_HD WarpCoord warp_coord(const Camera& cam, float x, float y, float depth, int W, int H, float eps,
                            float rcw = 0.0f, float rch = 0.0f) {
    WarpCoord wc;
    pixel_ray(cam, x, y, wc.ray);
    float pt[3] = {mul_rn(depth, wc.ray[0]), mul_rn(depth, wc.ray[1]), mul_rn(depth, wc.ray[2])};
    float p[3];
    project_point(cam, pt, p);
    const float z = add_rn(p[2], eps);
    wc.inv_z = fast_rcp(z);          // backward chain only
    wc.u_raw = div_rn(p[0], z);
    wc.v_raw = div_rn(p[1], z);
    const float nu = FASTDIV ? div_const(wc.u_raw, (float)(W - 1), rcw) : div_rn(wc.u_raw, (float)(W - 1));
    const float nv = FASTDIV ? div_const(wc.v_raw, (float)(H - 1), rch) : div_rn(wc.v_raw, (float)(H - 1));
    const float gx = mul_rn(sub_rn(nu, 0.5f), 2.0f);
    const float gy = mul_rn(sub_rn(nv, 0.5f), 2.0f);
    float cgx = 0.0f, cgy = 0.0f;
    const float ux = unnormalise_coord(gx, W, true);
    const float uy = unnormalise_coord(gy, H, true);
    // NaN: ATen's forward clip is fmin/fmax, which maps NaN to 0
    // (after the border clip the coordinate is in [0, size-1] -- +-inf included -- so ATen's
    //  safe_downgrade_to_int_range is the identity here)
    wc.ix = (ux == ux) ? clip_coord(ux, W, cgx) : 0.0f;
    wc.iy = (uy == uy) ? clip_coord(uy, H, cgy) : 0.0f;
    wc.mx = cgx * unnormalise_mult(W, true);
    wc.my = cgy * unnormalise_mult(H, true);
    return wc;
}

// Back-propagate d(loss)/d(ix,iy) to d(loss)/d(depth) through A12..A10.
//   gx = 2*(u_raw/(W-1) - .5): d gx/d u_raw = 2/(W-1);  u_raw = p0/z
// Also returns d(loss)/d(p) (for the pose gradient) in dp[3].
DMH_HD float warp_coord_bwd(const Camera& cam, const WarpCoord& wc, float g_ix, float g_iy, int W, int H,
                            float dp[3]) {
    const float g_u = g_ix * wc.mx * (2.0f / (float)(W - 1));
    const float g_v = g_iy * wc.my * (2.0f / (float)(H - 1));
    dp[0] = g_u * wc.inv_z;
    dp[1] = g_v * wc.inv_z;
    dp[2] = -(g_u * wc.u_raw + g_v * wc.v_raw) * wc.inv_z;
    float g_depth = 0.0f;
    for (int j = 0; j < 3; ++j) {
        const float g_pt = cam.P[0 * 4 + j] * dp[0] + cam.P[1 * 4 + j] * dp[1] + cam.P[2 * 4 + j] * dp[2];
        g_depth = fmaf(g_pt, wc.ray[j], g_depth);
    }
    return g_depth;
}

// ---------------------------------------------------------------------------
// SSIM at one pixel from the five 3x3 SUMS (not means) of x, y, x^2, y^2, xy.
struct SsimStats {
    float mu_x, mu_y, A1, A2, B1, B2, n, d;
};
#define DMH_SSIM_C1 0.0001f
#define DMH_SSIM_C2 0.0009f

DMH_HD SsimStats ssim_stats(float sx, float sy, float sxx, float syy, float sxy) {
    SsimStats s;
    s.mu_x = div_rn(sx, 9.0f);
    s.mu_y = div_rn(sy, 9.0f);
    const float sig_x = sub_rn(div_rn(sxx, 9.0f), mul_rn(s.mu_x, s.mu_x));
    const float sig_y = sub_rn(div_rn(syy, 9.0f), mul_rn(s.mu_y, s.mu_y));
    const float sig_xy = sub_rn(div_rn(sxy, 9.0f), mul_rn(s.mu_x, s.mu_y));
    s.A1 = add_rn(mul_rn(mul_rn(2.0f, s.mu_x), s.mu_y), DMH_SSIM_C1);
    s.A2 = add_rn(mul_rn(2.0f, sig_xy), DMH_SSIM_C2);
    s.B1 = add_rn(add_rn(mul_rn(s.mu_x, s.mu_x), mul_rn(s.mu_y, s.mu_y)), DMH_SSIM_C1);
    s.B2 = add_rn(add_rn(sig_x, sig_y), DMH_SSIM_C2);
    s.n = mul_rn(s.A1, s.A2);
    s.d = mul_rn(s.B1, s.B2);
    return s;
}

// clamp((1 - n/d)/2, 0, 1); `pass` = 1 where the clamp passes gradient (inclusive).
DMH_HD float ssim_value(const SsimStats& s, float& pass) {
    const float v = div_rn(sub_rn(1.0f, div_rn(s.n, s.d)), 2.0f);
    pass = (v >= 0.0f && v <= 1.0f) ? 1.0f : 0.0f;
    return fminf(fmaxf(v, 0.0f), 1.0f);
}

// dS/dx_k = ax + bx*x_k + cx*y_k   and   dS/dy_k = ay + bx*y_k + cx*x_k
// for every tap k of the (reflect-padded) 3x3 window -- see DESIGN.md "SSIM backward".
struct SsimCoef { float ax, ay, b, c; };

DMH_HD SsimCoef ssim_coef(const SsimStats& s) {
    const float r = 1.0f / s.d;
    const float nr2 = s.n * r * r;
    const float inv9 = 1.0f / 9.0f;
    SsimCoef k;
    k.ax = -inv9 * (s.mu_y * (s.A2 - s.A1) * r - nr2 * s.mu_x * (s.B2 - s.B1));
    k.ay = -inv9 * (s.mu_x * (s.A2 - s.A1) * r - nr2 * s.mu_y * (s.B2 - s.B1));
    k.b = inv9 * nr2 * s.B1;
    k.c = -inv9 * s.A1 * r;
    return k;
}

// reflect index for ReflectionPad2d(1): -1 -> 1, n -> n-2 (n >= 2)
DMH_HD int reflect1(int i, int n) { return i < 0 ? -i : (i >= n ? 2 * n - 2 - i : i); }

// image index of a position of a tile's 2-px halo: the 1-px reflection ring, clamped beyond it
DMH_HD int ext_to_img(int e, int n) {
    e = e < -1 ? -1 : (e > n ? n : e);
    return reflect1(e, n);
}
// multiplicity with which window centre q (valid pixel) touches pixel p along one axis
DMH_HD float reflect_mult(int p, int q, int n) {
    float m = 1.0f;
    if (p == 1 && q == 0) m += 1.0f;
    if (p == n - 2 && q == n - 1) m += 1.0f;
    return m;
}

// The in-image taps of one border-clamped bilinear sample (the others contribute nothing)
struct Taps {
    long long o00;
    bool nw, ne, sw, se;
};
DMH_HD Taps make_taps(const Bilinear& bl, int H, int W) {
    Taps t;
    const bool x0in = bl.x0 >= 0 && bl.x0 < W, x1in = bl.x0 + 1 >= 0 && bl.x0 + 1 < W;
    const bool y0in = bl.y0 >= 0 && bl.y0 < H, y1in = bl.y0 + 1 >= 0 && bl.y0 + 1 < H;
    t.o00 = (long long)bl.y0 * W + bl.x0;
    t.nw = y0in && x0in; t.ne = y0in && x1in; t.sw = y1in && x0in; t.se = y1in && x1in;
    return t;
}

// ---------------------------------------------------------------------------
// Colour-frame gradients of the min-reprojection objective.  `sel` is the candidate the forward picked, in the
// reference's cat order: n_ident identity candidates (F, 1 under avg_reprojection, 0 without automask), then the
// reprojections (F, or 1 under avg_reprojection).  Each returns the share of d(loss)/d(candidate) that source
// frame f's reprojection / identity candidate receives at that pixel.
DMH_HD float reproj_gate(int sel, int f, int n_ident, int F, bool avg) {
    if (avg) return sel == n_ident ? 1.0f / (float)F : 0.0f;
    return sel == n_ident + f ? 1.0f : 0.0f;
}
// Depth-hints objective: `sel` = argmin over [reprojection, identity, hint] in bits 0-1 and the source frame whose
// reprojection is the minimum over the frames in bits 2-3 (dmh_photo_scale_dh with DMH_PHOTO_SEL_SOURCE).  The
// reprojection term counts wherever the identity did not win; it is the mean over the frames under avg_reprojection.
DMH_HD float reproj_gate_dh(int sel, int f, int F, bool avg) {
    if ((sel & 3) == 1) return 0.0f;
    if (avg) return 1.0f / (float)F;
    return (sel >> 2) == f ? 1.0f : 0.0f;
}
DMH_HD float ident_gate(int sel, int f, int n_ident, int F, bool avg) {
    if (n_ident == 0) return 0.0f;
    if (avg) return sel == 0 ? 1.0f / (float)F : 0.0f;
    return sel == f ? 1.0f : 0.0f;
}

// d(gated loss)/d(x_p) and d/d(y_p) for one channel of R(x, y) = w_ssim*SSIM + w_l1*|y - x| at pixel p, from the
// window sums over every centre q whose window reaches p (reflection multiplicities included) of the gated
// coefficients: sa = sum ax, sd = sum ay, sb = sum b, sc = sum c (see SsimCoef), and the gate times w_l1 at p.
// The sign of x - y is 0 at a tie, as torch's abs backward.
DMH_HD void reproj_pixel_grad(float sa, float sb, float sc, float sd, float x, float y, float gl1, float& gx,
                              float& gy) {
    const float d = x - y;
    const float sg = d > 0.f ? gl1 : (d < 0.f ? -gl1 : 0.f);
    gx = sa + sb * x + sc * y + sg;
    gy = sd + sb * y + sc * x - sg;
}

// d/d(I_c(a)) of |dn_a - dn_b| * exp(-mean_c |I_c(a) - I_c(b)|) for one edge (a, b) of the smoothness term,
// given the edge's |dn_a - dn_b| * exp(...) = de and the channel count C; d/d(I_c(b)) is its negative.
DMH_HD float smooth_edge_img_grad(float de, float ia, float ib, int C) {
    const float d = ia - ib;
    const float sg = d > 0.f ? 1.f : (d < 0.f ? -1.f : 0.f);
    return -de * sg / (float)C;
}


// ---------------------------------------------------------------------------
// Fast-path SSIM used by the fused kernels (photo_fast.cu, photo_objective.cu, identity loss): separable
// 3x3 sums (row sums of 3, then 3 rows), mean = sum*(1/9).  Same mathematics as ssim_stats(); rounding differs
// at the 1e-7 level.  Written once over a lane type T with an EXPLICIT op sequence (no compiler contraction):
//   T = float   one pixel / channel per lane (host emulation and every kernel)
//   T = float2  two channels per lane on Blackwell's packed fp32 pipe (FADD2 / FMUL2 / FFMA2: one issue slot
//               for two results -- these kernels are issue-bound, not FMA-pipe bound); each half is
//               rounded exactly like the scalar instantiation, so both give bit-identical values.
DMH_HD float vadd(float a, float b) { return add_rn(a, b); }
DMH_HD float vsub(float a, float b) { return sub_rn(a, b); }
DMH_HD float vmul(float a, float b) { return mul_rn(a, b); }
DMH_HD float vfma(float a, float b, float c) { return fmaf(a, b, c); }
DMH_HD float vclamp01(float v) { return fminf(fmaxf(v, 0.0f), 1.0f); }
DMH_HD float vpass01(float v) { return (v >= 0.0f && v <= 1.0f) ? 1.0f : 0.0f; }
DMH_HD float vrcp(float x) { return fast_rcp(x); }
template <class T> struct Lane;
template <> struct Lane<float> { static DMH_HD float splat(float v) { return v; } };
#if defined(__CUDACC__)
// Packed fp32 through inline PTX with explicit .rn: nvcc contracts the __fmul2_rn / __fadd2_rn INTRINSICS into
// FFMA2 (measured: exx*(1/9) - mu^2 came out fused, 97 % of SSIM windows differed in the last bits from the
// scalar instantiation); explicitly rounded PTX instructions are never fused, so each half is bit-identical to
// the scalar __fmul_rn / __fadd_rn / fmaf sequence (profiles/probes/packed_check.cu).
#if defined(__CUDA_ARCH__)
#define DMH_F2_BINOP(name, ptx)                                                                                  \
    __device__ __forceinline__ float2 name(float2 a, float2 b) {                                                \
        float2 r;                                                                                                \
        asm("{ .reg .b64 ra, rb, rr; mov.b64 ra, {%2, %3}; mov.b64 rb, {%4, %5}; " ptx " rr, ra, rb; "            \
            "mov.b64 {%0, %1}, rr; }"                                                                            \
            : "=f"(r.x), "=f"(r.y)                                                                               \
            : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));                                                           \
        return r;                                                                                                \
    }
DMH_F2_BINOP(vadd, "add.rn.f32x2")
DMH_F2_BINOP(vmul, "mul.rn.f32x2")
#undef DMH_F2_BINOP
__device__ __forceinline__ float2 vfma(float2 a, float2 b, float2 c) {
    float2 r;
    asm("{ .reg .b64 ra, rb, rc, rr; mov.b64 ra, {%2, %3}; mov.b64 rb, {%4, %5}; mov.b64 rc, {%6, %7}; "
        "fma.rn.f32x2 rr, ra, rb, rc; mov.b64 {%0, %1}, rr; }"
        : "=f"(r.x), "=f"(r.y)
        : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y), "f"(c.x), "f"(c.y));
    return r;
}
// a - b as fma(b, -1, a): one rounding of the exact difference, i.e. identical to the subtraction
__device__ __forceinline__ float2 vsub(float2 a, float2 b) { return vfma(b, make_float2(-1.0f, -1.0f), a); }
#else
DMH_HD float2 vadd(float2 a, float2 b) { return make_float2(a.x + b.x, a.y + b.y); }
DMH_HD float2 vsub(float2 a, float2 b) { return make_float2(a.x - b.x, a.y - b.y); }
DMH_HD float2 vmul(float2 a, float2 b) { return make_float2(a.x * b.x, a.y * b.y); }
DMH_HD float2 vfma(float2 a, float2 b, float2 c) { return make_float2(fmaf(a.x, b.x, c.x), fmaf(a.y, b.y, c.y)); }
#endif
DMH_HD float2 vclamp01(float2 v) { return make_float2(vclamp01(v.x), vclamp01(v.y)); }
DMH_HD float2 vpass01(float2 v) { return make_float2(vpass01(v.x), vpass01(v.y)); }
DMH_HD float2 vrcp(float2 x) { return make_float2(fast_rcp(x.x), fast_rcp(x.y)); }
template <> struct Lane<float2> { static DMH_HD float2 splat(float v) { return make_float2(v, v); } };
#endif

template <class T> struct Row5T { T x, y, xx, yy, xy; };
typedef Row5T<float> Row5;

template <class T>
DMH_HD Row5T<T> row5(T x0, T x1, T x2, T y0, T y1, T y2) {
    Row5T<T> r;
    r.x = vadd(vadd(x0, x1), x2);
    r.y = vadd(vadd(y0, y1), y2);
    r.xx = vfma(x2, x2, vfma(x1, x1, vmul(x0, x0)));
    r.yy = vfma(y2, y2, vfma(y1, y1, vmul(y0, y0)));
    r.xy = vfma(x2, y2, vfma(x1, y1, vmul(x0, y0)));
    return r;
}

// Window statistics in SUM form: with X = sum x, XY = sum x*y, ... over the 3x3 window (mu_x = X/9,
// sigma_xy = XY/9 - X*Y/81) every factor of SSIM is carried multiplied by 81,
//   A1 = 2*X*Y + 81*C1            B1 = X^2 + Y^2 + 81*C1
//   A2 = 18*XY - 2*X*Y + 81*C2    B2 = 9*(XX + YY) - (X^2 + Y^2) + 81*C2
// n/d = (A1*A2)/(B1*B2) is unchanged (the 81^2 cancel) and the five divisions by 9 disappear; the cancellation
// in the variances is the same as in the mean form (same relative rounding, ~1e-7).
template <class T> struct SsimStatsT { T X, Y, A1, A2, B1, B2, n, d; };

template <class T>
DMH_HD SsimStatsT<T> ssim_stats_rows_t(const Row5T<T>& a, const Row5T<T>& b, const Row5T<T>& c) {
    const T c1 = Lane<T>::splat(81.0f * DMH_SSIM_C1), c2 = Lane<T>::splat(81.0f * DMH_SSIM_C2);
    const T two = Lane<T>::splat(2.0f), mtwo = Lane<T>::splat(-2.0f), nine = Lane<T>::splat(9.0f),
            eighteen = Lane<T>::splat(18.0f);
    SsimStatsT<T> s;
    s.X = vadd(vadd(a.x, b.x), c.x);
    s.Y = vadd(vadd(a.y, b.y), c.y);
    const T sxx = vadd(vadd(a.xx, b.xx), c.xx), syy = vadd(vadd(a.yy, b.yy), c.yy), sxy = vadd(vadd(a.xy, b.xy), c.xy);
    const T pxy = vmul(s.X, s.Y), pxx = vmul(s.X, s.X), pyy = vmul(s.Y, s.Y);
    const T p2 = vadd(pxx, pyy);
    s.A1 = vfma(two, pxy, c1);
    s.A2 = vfma(eighteen, sxy, vfma(mtwo, pxy, c2));
    s.B1 = vadd(p2, c1);
    s.B2 = vfma(nine, vadd(sxx, syy), vsub(c2, p2));
    s.n = vmul(s.A1, s.A2);
    s.d = vmul(s.B1, s.B2);
    return s;
}

// clamp((1 - n/d)/2, 0, 1); also returns r = 1/d and nr = n/d for the coefficients, `pass` = 1 where the
// clamp passes gradient (inclusive)
template <class T>
DMH_HD T ssim_value_t(const SsimStatsT<T>& s, T& pass, T& r, T& nr) {
    r = vrcp(s.d);
    nr = vmul(s.n, r);
    const T v = vfma(nr, Lane<T>::splat(-0.5f), Lane<T>::splat(0.5f));
    pass = vpass01(v);
    return vclamp01(v);
}

// g * dS/dx_k = ka + kb*x_k + kc*y_k for every tap k of the (reflect-padded) 3x3 window (see ssim_coef above;
// in sum form  ka = g*[X*(B2-B1)*n/d^2 - Y*(A2-A1)/d],  kb = 9*g*n*B1/d^2,  kc = -9*g*A1/d)
template <class T>
DMH_HD void ssim_coef_gated_t(const SsimStatsT<T>& s, T r, T nr, T g, T& ka, T& kb, T& kc) {
    const T gr = vmul(g, r);
    const T gnr2 = vmul(gr, nr);
    kc = vmul(vmul(gr, Lane<T>::splat(-9.0f)), s.A1);
    kb = vmul(vmul(gnr2, Lane<T>::splat(9.0f)), s.B1);
    const T e1 = vmul(gnr2, vsub(s.B2, s.B1)), e2 = vmul(gr, vsub(s.A2, s.A1));
    ka = vsub(vmul(s.X, e1), vmul(s.Y, e2));
}

// dS/dx_k = ax + b*x_k + c*y_k   and   dS/dy_k = ay + b*y_k + c*x_k  (see ssim_coef above)
template <class T> struct SsimCoefT { T ax, ay, b, c; };

// value + un-gated coefficients sharing one reciprocal of d; `pass` = 1 where the clamp passes gradient
template <class T>
DMH_HD T ssim_value_coef_t(const SsimStatsT<T>& s, T& pass, SsimCoefT<T>& k) {
    T r, nr;
    const T v = ssim_value_t(s, pass, r, nr);
    ssim_coef_gated_t(s, r, nr, Lane<T>::splat(1.0f), k.ax, k.b, k.c);
    const T nr2 = vmul(nr, r);
    k.ay = vsub(vmul(s.Y, vmul(nr2, vsub(s.B2, s.B1))), vmul(s.X, vmul(r, vsub(s.A2, s.A1))));
    return v;
}

// scalar entry points (names used by the kernels and by tests/host_emul.cpp)
typedef SsimStatsT<float> SsimStatsRows;
DMH_HD SsimStatsRows ssim_stats_rows(const Row5& a, const Row5& b, const Row5& c) { return ssim_stats_rows_t<float>(a, b, c); }
DMH_HD float ssim_value_coef(const SsimStatsRows& s, float& pass, SsimCoef& k) {
    SsimCoefT<float> kt;
    const float v = ssim_value_coef_t<float>(s, pass, kt);
    k.ax = kt.ax; k.ay = kt.ay; k.b = kt.b; k.c = kt.c;
    return v;
}

// d(grad_disp)/d(g_ix, g_iy): warp_coord_bwd collapsed to two scalars
//   g_depth = g_ix * ax + g_iy * ay
DMH_HD void warp_chain_factors(const Camera& cam, const WarpCoord& wc, int W, int H, float& ax, float& ay) {
    float pr[3];
    for (int i = 0; i < 3; ++i)
        pr[i] = cam.P[i * 4 + 0] * wc.ray[0] + cam.P[i * 4 + 1] * wc.ray[1] + cam.P[i * 4 + 2] * wc.ray[2];
    // d(ix)/d(u_raw) = mx * 2/(W-1) with mx = gate * (W-1)/2: the two constants cancel, only the clip gate is left
    (void)W; (void)H;
    const float gx = wc.mx != 0.0f ? wc.inv_z : 0.0f, gy = wc.my != 0.0f ? wc.inv_z : 0.0f;
    ax = gx * (pr[0] - wc.u_raw * pr[2]);
    ay = gy * (pr[1] - wc.v_raw * pr[2]);
}

}  // namespace dmh
