// Tile machinery shared by the single-source photometric kernels (photo_fast.cu: one launch per scale;
// photo_ms.cu: all scales in one launch): TMA / mbarrier primitives, tile geometry, the bilinear tap gather,
// phase B (sliding-window SSIM + decision + gated coefficients) and phase C (box sums -> gradient).
// Everything sits in an anonymous namespace: each translation unit gets its own copy.
#pragma once
#include "photo_launch.cuh"

namespace {


// ---- TMA / mbarrier primitives (sm_90+ PTX; sm_100a here)
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t done = 0;
    while (!done) {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n"
            : "=r"(done)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
    }
}
__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2,
                                            int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}

#define FT_T 32
#define FT_R2 36                 // tile + 2-px halo
#define FT_R1 34                 // tile + 1-px ring
#define FT_N2 (FT_R2 * FT_R2)
#define FT_TP 40                 // row pitch of the target tile: TMA needs a 16-byte aligned start column (x0-4)
#define FT_TO 2                  // column of the target tile that holds halo column 0 (image column x0-2)
#define FT_NT (FT_R2 * FT_TP)
#define FT_N1 (FT_R1 * FT_R1)
#define FT_THREADS 256
#define FT_STRIPS 7
#define FT_ROWS 5                // 7 strips x 5 rows >= 34 ring rows

// ReflectionPad2d(1) at the image border of the target tile tgt [3][36][40] of the tile at (x0, y0): the TMA load
// zero-fills out-of-image elements; a border tile patches them from the in-image rows / columns of the same tile (and
// ends with a barrier).  Uniform across the CTA.
__device__ __forceinline__ void patch_target_border(float* tgt, int tid, int x0, int y0, int H, int W) {
    if (x0 < 2 || y0 < 2 || x0 + FT_T + 2 > W || y0 + FT_T + 2 > H) {
        for (int i = tid; i < FT_N2; i += FT_THREADS) {
            const int r = i / FT_R2, c = i - r * FT_R2;
            const int ey = y0 - 2 + r, ex = x0 - 2 + c;
            if (ey < 0 || ey >= H || ex < 0 || ex >= W) {
                const int sr = ext_to_img(ey, H) - (y0 - 2), sc = ext_to_img(ex, W) - (x0 - 2);
#pragma unroll
                for (int ch = 0; ch < 3; ++ch)
                    tgt[ch * FT_NT + r * FT_TP + c + FT_TO] = tgt[ch * FT_NT + sr * FT_TP + sc + FT_TO];
            }
        }
        __syncthreads();
    }
}

// dynamic shared memory of photo_fast_kernel and photo_ms_kernel: target tile, warped tile, the 9 coefficient planes,
// camera (24 floats), reduction slots (32 floats) and the gate bytes
size_t tile_smem_bytes() { return sizeof(float) * (3 * FT_NT + 3 * FT_N2 + 9 * FT_N1 + 24 + 32) + FT_N1; }

struct FastParams {
    const float* target;
    const float* src;
    const float* T;
    DispSrc disp;
    const float* K;
    const float* inv_K;
    const float* ident;
    const float* noise;
    float* loss_partial;
    float* grad_disp;
    uint8_t* sel;
    float* warped;               // (unused by the fast kernel; kept for the launcher)
    // depth-hints objective (DH/trainer.py:541-590, 666-713), DH instantiation only
    const float* hint_reproj;    // (B,1,H,W) hint reprojection loss + 1000*(1-valid); NULL: no hints
    const float* hint_depth;     // (B,1,H,W)
    const float* hint_valid;     // (B,1,H,W)
    float* grad_hint;            // (B,1,H,W) d(sum proxy*mask_h)/d(up-sampled disp)
    int dh_nblk;                 // stride between the four partial-sum arrays
    int B, H, W, flags;
    DepthScale ds;
    float grad_scale;
    float rcw, rch;              // 1/(W-1), 1/(H-1) for the verified 3-instruction division
};

struct Gathered { float v[3]; float dix[3], diy[3]; };

// The four bilinear taps of one sampling position.  With border padding the clipped coordinate lies in
// [0, W-1] x [0, H-1].  The north-west tap is CLAMPED to (W-2, H-2), so the east / south taps are always
// +1 / +W: every load is unconditional, in bounds, and at a fixed offset from one base address.  The clamp
// only acts when the coordinate sits exactly on the last column / row (ix == W-1): the weights become
// (tx1, tx0) = (0, 1) instead of (1, 0) on the duplicated tap -- the same interpolated value bit for bit --
// and ATen's gradient gate (clip_coordinates_set_grad: borders count as out of bounds) zeroes d/d(ix) there.
struct Tap {
    int o;                       // pixel index of the north-west tap
    float tx0, tx1, ty0, ty1;    // (ix - ix_nw), (ix_se - ix), (iy - iy_nw), (iy_se - iy)
};

__device__ __forceinline__ Tap make_tap(const WarpCoord& wc, int H, int W) {
    const float fx = fminf(floorf(wc.ix), (float)(W - 2)), fy = fminf(floorf(wc.iy), (float)(H - 2));
    Tap t;
    t.o = (int)fy * W + (int)fx;
    t.tx1 = (fx + 1.0f) - wc.ix; t.tx0 = wc.ix - fx;
    t.ty1 = (fy + 1.0f) - wc.iy; t.ty0 = wc.iy - fy;
    return t;
}

// bilinear gather of 3 channels + d(value)/d(ix,iy), split into the loads and their combination so that the
// loads of several pixels can be in flight together.  PK: the source is pixel-packed (B,H,W,4) -- one 128-bit
// load per tap (dmh_identity_loss_pack writes that layout); otherwise planar (B,3,H,W), 12 scalar loads.
template <bool PK>
__device__ __forceinline__ void load_taps(const float* __restrict__ sp, size_t N, int W, const Tap& t, float v[3][4]) {
    if (PK) {
        const float4* s = reinterpret_cast<const float4*>(sp) + t.o;
        const float4 a = __ldg(s), b = __ldg(s + 1), c = __ldg(s + W), d = __ldg(s + W + 1);
        v[0][0] = a.x; v[1][0] = a.y; v[2][0] = a.z;
        v[0][1] = b.x; v[1][1] = b.y; v[2][1] = b.z;
        v[0][2] = c.x; v[1][2] = c.y; v[2][2] = c.z;
        v[0][3] = d.x; v[1][3] = d.y; v[2][3] = d.z;
    } else {
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) {
            const float* s = sp + ch * N + t.o;
            v[ch][0] = __ldg(s); v[ch][1] = __ldg(s + 1); v[ch][2] = __ldg(s + W); v[ch][3] = __ldg(s + W + 1);
        }
    }
}
__device__ __forceinline__ Gathered combine_taps(const float v[3][4], const Tap& t, bool want_grad) {
    const float wnw = t.tx1 * t.ty1, wne = t.tx0 * t.ty1, wsw = t.tx1 * t.ty0, wse = t.tx0 * t.ty0;
    Gathered g;
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) {
        const float nw = v[ch][0], ne = v[ch][1], sw = v[ch][2], se = v[ch][3];
        float acc = nw * wnw;
        acc = fmaf(ne, wne, acc);
        acc = fmaf(sw, wsw, acc);
        acc = fmaf(se, wse, acc);
        g.v[ch] = acc;
        if (want_grad) {
            g.dix[ch] = (ne - nw) * t.ty1 + (se - sw) * t.ty0;
            g.diy[ch] = (sw - nw) * t.tx1 + (se - ne) * t.tx0;
        }
    }
    return g;
}

// position (r, c) in the 36 x 36 frame of halo-ring pixel h < 272: 2 top rows, 2 bottom rows, 2 left / right columns
__device__ __forceinline__ void halo_rc(int h, int& r, int& c) {
    if (h < 72) { r = h / FT_R2; c = h - r * FT_R2; }
    else if (h < 144) { const int t = h - 72; r = FT_R2 - 2 + t / FT_R2; c = t % FT_R2; }
    else if (h < 208) { const int t = h - 144; r = 2 + (t >> 1); c = t & 1; }
    else { const int t = h - 208; r = 2 + (t >> 1); c = FT_R2 - 2 + (t & 1); }
}

// image index of tile coordinate e >= 0 (a pixel of the tile proper): in-image, or the ReflectionPad2d(1) mirror
// of the first row / column past the border (n -> n-2); anything further out is clamped onto that (unused values)
__device__ __forceinline__ int tile_to_img(int e, int n) {
    e = min(e, n);
    return e == n ? n - 2 : e;
}

// F.interpolate(disp, [H, W], bilinear, align_corners=False) at one pixel from its row / column taps
__device__ __forceinline__ float up_sample(const float* __restrict__ dp, int dw, const UpTap& ty, const UpTap& tx) {
    const float* r0 = dp + ty.i0 * dw;
    const float* r1 = dp + ty.i1 * dw;
    // explicit rounding sequence (no compiler-chosen contraction): every kernel that up-samples gets the same bits
    const float a = fmaf(tx.l1, __ldg(r0 + tx.i1), mul_rn(tx.l0, __ldg(r0 + tx.i0)));
    const float c = fmaf(tx.l1, __ldg(r1 + tx.i1), mul_rn(tx.l0, __ldg(r1 + tx.i0)));
    return fmaf(ty.l1, c, mul_rn(ty.l0, a));
}

// One pixel of the warp: depth -> exact coordinate chain -> taps (+ the two backward factors when wanted)
template <bool FASTDIV, class P>
__device__ __forceinline__ Tap pixel_tap(const Camera& cam, const P& p, int ix, int iy, float dv,
                                         bool want_grad, float& gax, float& gay) {
    const float depth = disp_to_depth(dv, p.ds);
    const WarpCoord wc = warp_coord<FASTDIV>(cam, (float)ix, (float)iy, depth, p.W, p.H, 1e-7f, p.rcw, p.rch);
    if (want_grad) {
        float ax, ay;
        warp_chain_factors(cam, wc, p.W, p.H, ax, ay);
        const float dd = ddepth_ddisp(depth, p.ds) * p.grad_scale;
        gax = ax * dd; gay = ay * dd;
    }
    return make_tap(wc, p.H, p.W);
}

// ---- phase B of the tile kernels: SSIM statistics by sliding windows down a ring column; decision; gated
// coefficients.  Channels 0 and 1 ride in the two halves of packed fp32 registers (FADD2 / FMUL2 / FFMA2), channel 2
// is scalar.  Straight-line: rows past the tile are clamped (their results are discarded by the predicated stores),
// out-of-image ring pixels are gated through the NaN identity marker.  `tid` < 256: index among the 256 threads that
// run the phase (threads >= 238 idle); returns this thread's share of the tile's loss sum.
struct TileSmem {
    float* tgt;      // [3][36][40]
    float* pred;     // [3][36][36]
    float4* q1;      // [N1] (a0, a1, b0, b1)
    float4* q2;      // [N1] (c0, c1, a2, b2)
    float* q3;       // [N1] c2
    uint8_t* gate;   // [N1]
};

// DH: the value kept is min(identity + noise, hint loss) -- the hint wins only when strictly smaller -- and bit k of
// `hflags` says that it was the hint (argmin order of the depth-hints objective: reprojection, identity, hint).
template <bool DH = false, class P>
__device__ __forceinline__ void prefetch_ident(const P& p, int tid, int b, int x0, int y0,
                                               float (&idv_pre)[FT_ROWS], unsigned& hflags) {
    hflags = 0u;
    const int H = p.H, W = p.W, N = H * W;
    const int bc = tid % FT_R1, bstrip = tid / FT_R1;
    const bool has_ident = p.ident != nullptr;
    const int qx = x0 - 1 + bc;
    const bool col_ok = qx >= 0 && qx < W && tid < FT_R1 * FT_STRIPS;
    const float* idp = p.ident + (size_t)b * N + qx;
    const float* nzp = p.noise + (size_t)b * N + qx;
#pragma unroll
    for (int k = 0; k < FT_ROWS; ++k) {
        const int qr = bstrip * FT_ROWS + k, qy = y0 - 1 + qr;
        const bool ok = col_ok && qr < FT_R1 && qy >= 0 && qy < H;
        float v = ok ? __int_as_float(0x7f800000) : __int_as_float(0x7fc00000);     // +inf: always loses to rp
        if (ok && has_ident) {
            v = __ldg(idp + qy * W);
            if (p.noise) v = add_rn(v, __ldg(nzp + qy * W));
        }
        if (DH && ok && p.hint_reproj) {
            const float hv = __ldg(p.hint_reproj + (size_t)b * N + qy * W + qx);
            if (hv < v) { v = hv; hflags |= 1u << k; }
        }
        idv_pre[k] = v;
    }
}

// DH: the depth-hints decision -- argmin over [reprojection, identity + noise, hint] with the reprojection first
// (ties go to it), reprojection mask = argmin != identity, hint mask = argmin == hint; four masked sums in acc
// (reproj*mask_r, mask_r, log(|hint - depth| + 1)*valid*mask_h, mask_h) and the proxy-loss gradient map.
template <bool DH, bool UP, class P>
__device__ __forceinline__ float phase_b(const P& p, const TileSmem& sm, int tid, int b, int x0, int y0,
                                         const float (&idv_pre)[FT_ROWS], unsigned hflags, float (&acc)[4]) {
    const int W = p.W, N = p.H * p.W;
    const float w_ssim = 0.85f / 3.0f;
    const int bc = tid % FT_R1, bstrip = tid / FT_R1;
    const bool has_ident = p.ident != nullptr;
    const float* tgt = sm.tgt;
    const float* pred = sm.pred;
    float4* coefQ1 = sm.q1;
    float4* coefQ2 = sm.q2;
    float* coefQ3 = sm.q3;
    uint8_t* gate = sm.gate;
    float loss_local = 0.0f;
    if (tid < FT_R1 * FT_STRIPS) {
        const int r0 = bstrip * FT_ROWS;                // first ring row of this strip == first R2 row of its window
        const bool col_in = bc >= 1 && bc <= FT_T;
        Row5T<float2> histP[2];                         // channels (0,1): [older, newer] row sums
        Row5T<float> histS[2];                          // channel 2
        float2 cenxP, cenyP;                            // centre values of the previous row
        float cenxS, cenyS;
#pragma unroll
        for (int rr = 0; rr < FT_ROWS + 2; ++rr) {
            const int r2 = min(r0 + rr, FT_R2 - 1);     // R2 row being added
            const float* xs = pred + r2 * FT_R2 + bc;
            const float* ys = tgt + r2 * FT_TP + bc + FT_TO;
            const float2 xa = make_float2(xs[0], xs[FT_N2]), xb = make_float2(xs[1], xs[FT_N2 + 1]),
                         xc = make_float2(xs[2], xs[FT_N2 + 2]);
            const float2 ya = make_float2(ys[0], ys[FT_NT]), yb = make_float2(ys[1], ys[FT_NT + 1]),
                         yc = make_float2(ys[2], ys[FT_NT + 2]);
            const Row5T<float2> curP = row5(xa, xb, xc, ya, yb, yc);
            const float* x2 = xs + 2 * FT_N2;
            const float* y2 = ys + 2 * FT_NT;
            const float x2m = x2[1], y2m = y2[1];
            const Row5T<float> curS = row5(x2[0], x2m, x2[2], y2[0], y2m, y2[2]);
            if (rr >= 2) {
                const int qr = r0 + rr - 2;             // ring row of the window centre
                float l1 = fabsf(cenyP.x - cenxP.x);
                l1 += fabsf(cenyP.y - cenxP.y);
                l1 += fabsf(cenyS - cenxS);
                const SsimStatsT<float2> stP = ssim_stats_rows_t(histP[0], histP[1], curP);
                const SsimStatsT<float> stS = ssim_stats_rows_t(histS[0], histS[1], curS);
                float2 passP, rP, nrP;
                const float2 vP = ssim_value_t(stP, passP, rP, nrP);
                float passS, rS, nrS;
                const float vS = ssim_value_t(stS, passS, rS, nrS);
                const float ss = (vP.x + vP.y) + vS;
                l1 *= (1.0f / 3.0f);
                const float rp = fmaf(0.85f, ss * (1.0f / 3.0f), 0.15f * l1);
                const float idv = idv_pre[rr - 2];
                bool win = rp < idv;                    // torch.min: first minimum wins, identity is first
                int dh_idx = 0;
                const bool in_img = idv == idv;         // (NaN marks ring pixels outside the image)
                if (DH) {
                    // idv = min(identity, hint) with the hint flagged: argmin over [reprojection, identity, hint]
                    if (idv < rp) dh_idx = ((hflags >> (rr - 2)) & 1u) ? 2 : 1;
                    win = in_img && dh_idx != 1;        // the reprojection term is optimised unless the identity wins
                }
                const float gw = win ? w_ssim : 0.0f;
                float2 kaP, kbP, kcP;
                ssim_coef_gated_t(stP, rP, nrP, vmul(make_float2(gw, gw), passP), kaP, kbP, kcP);
                float kaS, kbS, kcS;
                ssim_coef_gated_t(stS, rS, nrS, gw * passS, kaS, kbS, kcS);
                if (qr < FT_R1) {
                    const int qi = qr * FT_R1 + bc;
                    coefQ1[qi] = make_float4(kaP.x, kaP.y, kbP.x, kbP.y);
                    coefQ2[qi] = make_float4(kcP.x, kcP.y, kaS, kbS);
                    coefQ3[qi] = kcS;
                    gate[qi] = (uint8_t)((win ? 1 : 0) | ((DH && dh_idx == 2) ? 2 : 0));
                }
                if (col_in && qr >= 1 && qr <= FT_T && in_img) {         // a pixel of the tile proper, inside the image
                    const int qo = (y0 - 1 + qr) * W + x0 - 1 + bc;
                    if (!DH) {
                        loss_local += win ? rp : idv;
                        if (p.sel) p.sel[(size_t)b * N + qo] = (uint8_t)((win && has_ident) ? 1 : 0);
                    } else {
                        if (dh_idx != 1) { acc[0] += rp; acc[1] += 1.0f; }
                        if (p.sel) p.sel[(size_t)b * N + qo] = (uint8_t)dh_idx;
                    }
                }
            }
            histP[0] = histP[1]; histP[1] = curP;
            histS[0] = histS[1]; histS[1] = curS;
            cenxP = xb; cenyP = yb; cenxS = x2m; cenyS = y2m;
        }
    }
    return loss_local;
}

// ---- phase C of the tile kernels: separable weighted box sums of the coefficient planes -> d/d(pred) -> d/d(disp).
// `tid` < 256 owns column tid%32, rows 4*(tid/32)+k of the tile; D = d(pred_ch)/d(disp) of those 4 pixels.
// DH: the proxy loss of the depth hints, log(|hint - depth| + 1) * valid where the hint won (bit 1 of the gate byte),
// its masked sums (acc[2], acc[3]) and its gradient map, for the same 4 pixels.
template <bool DH, bool UP, class P>
__device__ __forceinline__ void phase_c(const P& p, const TileSmem& sm, int tid, int b, int x0, int y0,
                                        const float (&D)[4][3], float (&acc)[4], float (*gp_out)[3] = nullptr,
                                        float* g_acc = nullptr, const float (*xv_in)[3] = nullptr) {
    const int H = p.H, W = p.W, N = H * W;
    const float w_l1 = 0.15f / 3.0f;
    const int oc = tid & 31, os = tid >> 5;
    const float* tgt = sm.tgt;
    const float* pred = sm.pred;
    const float4* coefQ1 = sm.q1;
    const float4* coefQ2 = sm.q2;
    const float* coefQ3 = sm.q3;
    const uint8_t* gate = sm.gate;
    float h_dv[4], h_hd[4], h_va[4];
    if (DH && p.hint_reproj) {
        // only where the hint won (bit 1 of the gate byte); requested up front: the latency hides behind the box sums
        const float* dp = p.disp.ptr + (size_t)b * (p.disp.h * p.disp.w);
        const int hx = min(x0 + oc, W - 1);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int hy = min(y0 + 4 * os + k, H - 1);
            h_dv[k] = 0.f; h_hd[k] = 0.f; h_va[k] = 0.f;
            if (gate[(4 * os + k + 1) * FT_R1 + oc + 1] & 2) {
                h_dv[k] = UP ? up_sample(dp, p.disp.w, up_tap(hy, p.disp.sh, p.disp.h), up_tap(hx, p.disp.sw, p.disp.w))
                             : __ldg(dp + hy * W + hx);
                h_hd[k] = __ldg(p.hint_depth + (size_t)b * N + hy * W + hx);
                h_va[k] = __ldg(p.hint_valid + (size_t)b * N + hy * W + hx);
            }
        }
    }
    {
        const int px = x0 + oc;
        const float wl = (px == 1) ? 2.0f : 1.0f;           // ring column 0 reaches pixel 1 twice (reflection)
        const float wr = (px == W - 2) ? 2.0f : 1.0f;
        const float2 wl2 = make_float2(wl, wl), wr2 = make_float2(wr, wr);
        // packed quantities: 0 = (a0,a1), 1 = (b0,b1), 2 = (c0,c1), 3 = (a2,b2); scalar: c2
        float2 hprev[2][4];
        float hprevC[2];
        float* gout = p.grad_disp + (size_t)b * N + px;
#pragma unroll
        for (int rr = 0; rr < 6; ++rr) {
            const int r1 = 4 * os + rr;                      // ring row
            float2 hc[4];
            float hcC;
            {
                const float4* q1 = coefQ1 + r1 * FT_R1 + oc;
                const float4* q2 = coefQ2 + r1 * FT_R1 + oc;
                const float* q3 = coefQ3 + r1 * FT_R1 + oc;
                const float4 l1 = q1[0], m1 = q1[1], e1 = q1[2];
                const float4 l2 = q2[0], m2 = q2[1], e2 = q2[2];
                hc[0] = vfma(wl2, make_float2(l1.x, l1.y), vfma(wr2, make_float2(e1.x, e1.y), make_float2(m1.x, m1.y)));
                hc[1] = vfma(wl2, make_float2(l1.z, l1.w), vfma(wr2, make_float2(e1.z, e1.w), make_float2(m1.z, m1.w)));
                hc[2] = vfma(wl2, make_float2(l2.x, l2.y), vfma(wr2, make_float2(e2.x, e2.y), make_float2(m2.x, m2.y)));
                hc[3] = vfma(wl2, make_float2(l2.z, l2.w), vfma(wr2, make_float2(e2.z, e2.w), make_float2(m2.z, m2.w)));
                hcC = fmaf(wl, q3[0], fmaf(wr, q3[2], q3[1]));
            }
            if (rr >= 2) {
                const int k = rr - 2;
                const int r = 4 * os + k;
                const int py = y0 + r;
                const float wu = (py == 1) ? 2.0f : 1.0f;
                const float wd = (py == H - 2) ? 2.0f : 1.0f;
                const float2 wu2 = make_float2(wu, wu), wd2 = make_float2(wd, wd);
                const int i2 = (r + 2) * FT_R2 + oc + 2;
                const int it = (r + 2) * FT_TP + oc + 2 + FT_TO;
                const float gl1 = (gate[(r + 1) * FT_R1 + oc + 1] & 1) ? w_l1 : 0.0f;
                const float2 saP = vfma(wu2, hprev[0][0], vfma(wd2, hc[0], hprev[1][0]));
                const float2 sbP = vfma(wu2, hprev[0][1], vfma(wd2, hc[1], hprev[1][1]));
                const float2 scP = vfma(wu2, hprev[0][2], vfma(wd2, hc[2], hprev[1][2]));
                const float2 sab2 = vfma(wu2, hprev[0][3], vfma(wd2, hc[3], hprev[1][3]));
                const float scS = fmaf(wu, hprevC[0], fmaf(wd, hcC, hprevC[1]));
                // (multi-source kernel: the warped values of an earlier source come back from its scratch, xv_in)
                const float2 xvP = xv_in ? make_float2(xv_in[k][0], xv_in[k][1]) : make_float2(pred[i2], pred[FT_N2 + i2]);
                const float2 yvP = make_float2(tgt[it], tgt[FT_NT + it]);
                const float xvS = xv_in ? xv_in[k][2] : pred[2 * FT_N2 + i2], yvS = tgt[2 * FT_NT + it];
                const float2 dP = vsub(xvP, yvP);
                const float dS = xvS - yvS;
                const float2 sgP = make_float2(dP.x > 0.f ? gl1 : (dP.x < 0.f ? -gl1 : 0.f),
                                               dP.y > 0.f ? gl1 : (dP.y < 0.f ? -gl1 : 0.f));
                const float sgS = dS > 0.f ? gl1 : (dS < 0.f ? -gl1 : 0.f);
                const float2 gpP = vadd(vfma(sbP, xvP, vfma(scP, yvP, saP)), sgP);
                const float gpS = fmaf(sab2.y, xvS, fmaf(scS, yvS, sab2.x)) + sgS;
                float g = gpP.x * D[k][0];
                g = fmaf(gpP.y, D[k][1], g);
                g = fmaf(gpS, D[k][2], g);
                // multi-source kernel (photo_mf.cu): d(loss)/d(pred) of this source for the pose-gradient epilogue
                // (gp_out), and the disparity gradient accumulated over the sources in registers (g_acc) instead of
                // stored per source
                if (gp_out) { gp_out[k][0] = gpP.x; gp_out[k][1] = gpP.y; gp_out[k][2] = gpS; }
                if (g_acc) g_acc[k] += g;
                else if (py < H && px < W) gout[py * W] = g;
                if (DH && p.hint_reproj && py < H && px < W) {
                    float gh = 0.0f;
                    if (gate[(r + 1) * FT_R1 + oc + 1] & 2) {            // the hint won here
                        const float depth = disp_to_depth(h_dv[k], p.ds);
                        const float diff = sub_rn(h_hd[k], depth);
                        const float a1 = add_rn(fabsf(diff), 1.0f);
                        acc[2] += mul_rn(logf(a1), h_va[k]);
                        acc[3] += 1.0f;
                        const float sg = diff > 0.f ? -1.f : (diff < 0.f ? 1.f : 0.f);
                        gh = h_va[k] * sg / a1 * ddepth_ddisp(depth, p.ds);
                    }
                    p.grad_hint[(size_t)b * N + py * W + px] = gh;
                }
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) { hprev[0][j] = hprev[1][j]; hprev[1][j] = hc[j]; }
            hprevC[0] = hprevC[1]; hprevC[1] = hcC;
        }
    }
}

}  // namespace
