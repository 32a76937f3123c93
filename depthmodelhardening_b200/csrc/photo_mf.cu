// The photometric objective with SEVERAL source frames (and / or pose gradients), all scales, in ONE launch
// (dmh_photo_multisource) -- the tile machinery of the single-source kernels (photo_tile.cuh, photo_ms_common.cuh:
// TMA target tile, packed 128-bit gather with the exact branch-free coordinate chain, sliding-window SSIM in packed
// fp32, separable box sums) brought to mono / mono+stereo / multi-frame training.
//
// Reference: DepthNetworks/monodepth2/trainer.py:476-523 (generate_images_pred: every frame id of every scale is
// warped), :589-660 (compute_losses: reprojection loss of every source, identity loss of every source + noise,
// torch.cat -> torch.min over [identities, reprojections], mean) and the pose branch of the autograd graph
// (Project3D's T, layers.py:182-198).  One work item = (32 x 32 target tile, scale); a persistent grid of
// 2 CTAs per SM walks over the items.
//
// The per-pixel minimum needs the reprojection loss of EVERY source before any SSIM coefficient can be gated, and the
// backward needs the coefficient planes of each source separately.  Nine planes per source do not fit the shared
// memory of two CTAs per SM, and recomputing the window statistics would cost a second SSIM pass per source.  So:
//   pass 1, per source:  gather (phase A) -> sliding-window statistics, values AND un-gated coefficients (phase B).
//       The LAST source knows the final decision at once: its coefficients are gated and written to the shared-memory
//       planes as in the single-source kernel, its backward factors stay in registers.  Every EARLIER source parks its
//       un-gated coefficients (9 floats per ring pixel), its backward factors and warped centre values (6 floats per
//       pixel) in a per-CTA scratch in global memory -- written and read back by the SAME thread within one work item,
//       so it lives in L2 (2 x 148 CTAs x 80-112 KB per parked source) and needs no fence;
//   decision: running first-minimum over the identities and over the reprojections in torch.cat order, kept in
//       registers by the thread that owns the ring pixel;
//   pass 2, per source (last first): gated planes -> box sums (phase C) -> d/d(disp) accumulated over the sources in
//       registers, and -- when pose gradients are wanted -- d(loss)/d(P) of the source from d(loss)/d(pred) and the
//       gather derivatives parked by phase A.  A source that wins nowhere in the tile is skipped (uniform branch).
// With F == 1 and no pose gradient the kernel evaluates exactly the operations of photo_ms_kernel: same bits
// (tests/test_gpu_photometric.py::test_multisource_kernel_*).
#include "photo_ms_common.cuh"

namespace {

#define MF_MAXF DMH_PHOTO_MAX_FRAMES
#define MF_MAX_SCALES 4
// scratch of one (CTA, source), in floats: Q1 / Q2 [5][256] float4, Q3 [5][256] float, AUX [4 pixels][4][256] float4
//   AUX slots of interior pixel k: 0 = (D0, D1, D2, depth)   1 = (pred0, pred1, pred2, -)
//                                  2 = (gz_x * d(pred_ch)/d(ix), u)   3 = (gz_y * d(pred_ch)/d(iy), v)
#define MF_Q1_OFF 0
#define MF_Q2_OFF (5 * FT_THREADS * 4)
#define MF_Q3_OFF (2 * 5 * FT_THREADS * 4)
#define MF_AUX_OFF (MF_Q3_OFF + 5 * FT_THREADS)
#define MF_SRC_STRIDE (MF_AUX_OFF + 16 * FT_THREADS * 4)

struct MfScale {
    const float* disp;           // (B,1,dh,dw)
    const float* noise;          // (B,F,H,W) tie-break noise of this scale (reference layout); nullable
    float* loss_partial;         // [B * tiles32]
    float* grad_disp;            // (B,1,H,W)
    float* grad_P;               // (F,B,tiles32,12) pose-gradient partials; nullable
    uint8_t* sel;                // (B,H,W) argmin in torch.cat order; nullable
    int dh, dw;
    float sh, sw;
};

struct MfParams {
    const float* src[MF_MAXF];   // pixel-packed sources (B,H,W,4)
    const float* T[MF_MAXF];
    const float* ident[MF_MAXF]; // (B,1,H,W) identity loss of each source; all NULL: automask off
    const float* K;
    const float* inv_K;
    MfScale sc[MF_MAX_SCALES];
    float* scratch;
    int* next_item;              // work counter (zeroed by the launcher): items beyond the first of a CTA are taken dynamically
    int F, S, B, H, W;
    DepthScale ds;
    float grad_scale, rcw, rch;
    // work items: [0, n_full) = one tile walking all S scales; the remaining tiles are split into S single-scale items
    // each (the partial last round of the persistent grid)
    int gx, gy, n_items, n_full;
};

__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// scratch accessors: `base` already points at this thread's column (float4 index tid), idx4 = multiple of 256
// The scratch is re-written every work item and must stay in L2 while the frames stream through it: its accesses carry
// an evict_last cache policy (ncu, first version without it: 1.65 GB of DRAM writes per launch for 0.1 GB of outputs).
__device__ __forceinline__ uint64_t scratch_policy() {
    uint64_t pol;
    asm("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
#if defined(MF_NO_HINT)
__device__ __forceinline__ void st4(float4* base, int idx4, float a, float b, float c, float d) {
    base[idx4] = make_float4(a, b, c, d);
}
__device__ __forceinline__ float4 ld4(const float4* base, int idx4) { return base[idx4]; }
__device__ __forceinline__ void st1(float* ptr, float a) { *ptr = a; }
__device__ __forceinline__ float ld1s(const float* ptr) { return *ptr; }
#else
__device__ __forceinline__ void st4(float4* base, int idx4, float a, float b, float c, float d) {
    asm volatile("st.global.L2::cache_hint.v4.f32 [%0], {%1, %2, %3, %4}, %5;" ::"l"(base + idx4), "f"(a), "f"(b), "f"(c),
                 "f"(d), "l"(scratch_policy()) : "memory");
}
__device__ __forceinline__ float4 ld4(const float4* base, int idx4) {
    float4 v;
    asm volatile("ld.global.L2::cache_hint.v4.f32 {%0, %1, %2, %3}, [%4], %5;"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(base + idx4), "l"(scratch_policy()) : "memory");
    return v;
}
__device__ __forceinline__ void st1(float* ptr, float a) {
    asm volatile("st.global.L2::cache_hint.f32 [%0], %1, %2;" ::"l"(ptr), "f"(a), "l"(scratch_policy()) : "memory");
}
__device__ __forceinline__ float ld1s(const float* ptr) {
    float v;
    asm volatile("ld.global.L2::cache_hint.f32 %0, [%1], %2;" : "=f"(v) : "l"(ptr), "l"(scratch_policy()) : "memory");
    return v;
}
#endif
// one (CTA, source) scratch as seen by one thread
struct Scr {
    float4* q;       // + tid: Q1 at [k*256], Q2 at [(5+k)*256]
    float* q3;       // + tid: [k*256]
    float4* aux;     // + tid: [(pixel*4+slot)*256]
};
__device__ __forceinline__ Scr scr_of(float* cta_base, int f, int tid) {
    float* b = cta_base + (size_t)f * MF_SRC_STRIDE;
    Scr s;
    s.q = reinterpret_cast<float4*>(b) + tid;
    s.q3 = b + MF_Q3_OFF + tid;
    s.aux = reinterpret_cast<float4*>(b + MF_AUX_OFF) + tid;
    return s;
}

// The cold path of a tile whose reciprocal operands left the exponent range of the branch-free chain: generic IEEE
// divisions (warp_coord), same pixel ownership; fills pred and hands the interior pixels' factors back.
template <bool FASTDIV>
__device__ __noinline__ void gather_generic_mf(const MsView& v, const float* cams, const float* sp, float* pred, int b,
                                               int x0, int y0, float* Dout, float* aux_out) {
    const int tid = threadIdx.x;
    const int H = v.H, W = v.W, N = H * W;
    const int oc = tid & 31, os = tid >> 5;
    Camera cam;
    for (int i = 0; i < 12; ++i) cam.P[i] = cams[i];
    for (int i = 0; i < 9; ++i) cam.iK[i] = cams[12 + i];
    const float* dp = v.disp.ptr + (size_t)b * (v.disp.h * v.disp.w);
    const bool up = !(v.disp.h == H && v.disp.w == W);
    for (int k = 0; k < 6; ++k) {
        int r, c;
        if (k < 4) { r = 4 * os + k + 2; c = oc + 2; }
        else if (k == 4) halo_rc(tid, r, c);
        else { if (tid >= 272 - FT_THREADS) break; halo_rc(tid + FT_THREADS, r, c); }
        const int iy = k < 4 ? tile_to_img(y0 + 4 * os + k, H) : ext_to_img(y0 - 2 + r, H);
        const int ix = k < 4 ? tile_to_img(x0 + oc, W) : ext_to_img(x0 - 2 + c, W);
        const float dv = up ? up_sample(dp, v.disp.w, up_tap(iy, v.disp.sh, v.disp.h), up_tap(ix, v.disp.sw, v.disp.w))
                            : __ldg(dp + iy * W + ix);
        const float depth = disp_to_depth(dv, v.ds);
        const WarpCoord wc = warp_coord<FASTDIV>(cam, (float)ix, (float)iy, depth, W, H, 1e-7f, v.rcw, v.rch);
        const Tap t = make_tap(wc, H, W);
        float tv[3][4];
        load_taps<true>(sp, N, W, t, tv);
        const Gathered g = combine_taps(tv, t, k < 4);
        for (int ch = 0; ch < 3; ++ch) pred[ch * FT_N2 + r * FT_R2 + c] = g.v[ch];
        if (k < 4) {
            float ax, ay;
            warp_chain_factors(cam, wc, W, H, ax, ay);
            const float dd = ddepth_ddisp(depth, v.ds) * v.grad_scale;
            const float gzx = wc.mx != 0.0f ? wc.inv_z : 0.0f, gzy = wc.my != 0.0f ? wc.inv_z : 0.0f;
            for (int ch = 0; ch < 3; ++ch) {
                Dout[k * 3 + ch] = g.dix[ch] * (ax * dd) + g.diy[ch] * (ay * dd);
                aux_out[k * 12 + ch] = g.v[ch];
                aux_out[k * 12 + 3 + ch] = gzx * g.dix[ch];
                aux_out[k * 12 + 6 + ch] = gzy * g.diy[ch];
            }
            aux_out[k * 12 + 9] = wc.u_raw; aux_out[k * 12 + 10] = wc.v_raw; aux_out[k * 12 + 11] = depth;
        }
    }
}

// Phase A of one (item, source): the register tap pipeline of photo_ms_common.cuh gather_tile_regs, with what the
// later passes need of the interior pixels parked in the scratch at retire time (nothing extra stays in registers):
//   KEEP_D   the backward factors stay in registers (last source); otherwise AUX slots 0 / 1 receive them together
//            with the warped centre values
//   POSE     AUX slots 2 / 3 (and the depth in slot 0) for the pose-gradient epilogue
template <bool FASTDIV, bool KEEP_D, bool POSE>
__device__ __forceinline__ void gather_tile_mf(const MsView& v, const float* cams, const float* src_packed, int tid, int b,
                                               int x0, int y0, float* pred, float4* aux, float (&D)[4][3], float& lo,
                                               float& hi) {
    const int H = v.H, W = v.W;
    const size_t N = (size_t)H * W;
    const int oc = tid & 31, os = tid >> 5;
    int hr, hc;
    halo_rc(tid, hr, hc);
    const int ixo = tile_to_img(x0 + oc, W);
    const int hy = ext_to_img(y0 - 2 + hr, H), hx = ext_to_img(x0 - 2 + hc, W);
    const bool extra = tid < 272 - FT_THREADS;
    int er = 0, ec = 0;
    if (extra) halo_rc(tid + FT_THREADS, er, ec);
    const float4* sp4 = reinterpret_cast<const float4*>(src_packed) + (size_t)b * N;
    const float* dp = v.disp.ptr + (size_t)b * (v.disp.h * v.disp.w);
    const bool up = !(v.disp.h == H && v.disp.w == W);
    const Camera& cam = *reinterpret_cast<const Camera*>(cams);
    int py[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) py[k] = tile_to_img(y0 + 4 * os + k, H);
    float dv[5];
    if (!up) {
#pragma unroll
        for (int k = 0; k < 4; ++k) dv[k] = __ldg(dp + (unsigned)(py[k] * W + ixo));
        dv[4] = __ldg(dp + (unsigned)(hy * W + hx));
    } else {
        const UpTap txo = up_tap(ixo, v.disp.sw, v.disp.w);
#pragma unroll
        for (int k = 0; k < 4; ++k) dv[k] = up_sample_at(dp, v.disp.w, up_tap(py[k], v.disp.sh, v.disp.h), txo);
        dv[4] = up_sample_at(dp, v.disp.w, up_tap(hy, v.disp.sh, v.disp.h), up_tap(hx, v.disp.sw, v.disp.w));
    }
    Tap tq;
    float gxq = 0.f, gyq = 0.f;
    TapAux axq;
    float4 tvq[4];
#pragma unroll
    for (int k = 0; k < 7; ++k) {
        const bool live = k < 5 || (k == 5 && extra);
        Tap tn;
        float gxn = 0.f, gyn = 0.f;
        TapAux axn;
        if (k < 4) tn = pixel_tap_nb<FASTDIV, true, POSE>(cam, v, ixo, py[k], dv[k], gxn, gyn, lo, hi, &axn);
        else if (k == 4) tn = pixel_tap_nb<FASTDIV, false>(cam, v, hx, hy, dv[4], gxn, gyn, lo, hi);
        else if (k == 5 && extra) {
            const int iy = ext_to_img(y0 - 2 + er, H), ix = ext_to_img(x0 - 2 + ec, W);
            const float dvh = up ? up_sample_at(dp, v.disp.w, up_tap(iy, v.disp.sh, v.disp.h), up_tap(ix, v.disp.sw, v.disp.w))
                                 : __ldg(dp + (unsigned)(iy * W + ix));
            tn = pixel_tap_nb<FASTDIV, false>(cam, v, ix, iy, dvh, gxn, gyn, lo, hi);
        }
        const int j = k - 1;                                // pixel to retire: its taps were requested one chain ago
        if (j >= 0 && (j < 5 || extra)) {
            const Gathered g = combine_taps4(tvq, tq, j < 4);
            const int i2 = j < 4 ? (4 * os + j + 2) * FT_R2 + oc + 2 : (j == 4 ? hr * FT_R2 + hc : er * FT_R2 + ec);
#pragma unroll
            for (int ch = 0; ch < 3; ++ch) pred[ch * FT_N2 + i2] = g.v[ch];
            if (j < 4) {
                float d[3];
#pragma unroll
                for (int ch = 0; ch < 3; ++ch) d[ch] = g.dix[ch] * gxq + g.diy[ch] * gyq;
                if (KEEP_D) {
#pragma unroll
                    for (int ch = 0; ch < 3; ++ch) D[j][ch] = d[ch];
                    if (POSE) st4(aux, (j * 4 + 0) * FT_THREADS, 0.f, 0.f, 0.f, axq.depth);
                } else {
                    st4(aux, (j * 4 + 0) * FT_THREADS, d[0], d[1], d[2], POSE ? axq.depth : 0.f);
                    st4(aux, (j * 4 + 1) * FT_THREADS, g.v[0], g.v[1], g.v[2], 0.f);
                }
                if (POSE) {
                    st4(aux, (j * 4 + 2) * FT_THREADS, axq.gzx * g.dix[0], axq.gzx * g.dix[1], axq.gzx * g.dix[2], axq.u);
                    st4(aux, (j * 4 + 3) * FT_THREADS, axq.gzy * g.diy[0], axq.gzy * g.diy[1], axq.gzy * g.diy[2], axq.v);
                }
            }
        }
        if (live) {
            load_taps4(sp4, W, tn, tvq);
            tq = tn; gxq = gxn; gyq = gyn;
            if (POSE && k < 4) axq = axn;
        }
    }
}

// Phase B of one (item, source): photo_tile.cuh phase_b's sliding windows -- the same operations in the same order,
// the same bits -- with the decision taken out: the reprojection loss updates the running first-minimum (br, idx_r),
// the coefficients are computed un-gated (weight 0.85/3 * clamp gate).  !LAST: they go to the scratch.  LAST: every
// candidate is known now, the coefficients of the pixels this source wins are written to the shared-memory planes.
template <bool LAST>
__device__ __forceinline__ void phase_b_multi(const TileSmem& sm, int tid, int f, bool has_ident, unsigned okbits,
                                              const float (&bi)[FT_ROWS], float (&br)[FT_ROWS], unsigned& idx_r,
                                              const Scr& scr) {
    const float w_ssim = 0.85f / 3.0f;
    const int bc = tid % FT_R1, bstrip = tid / FT_R1;
    const float* tgt = sm.tgt;
    const float* pred = sm.pred;
    if (tid < FT_R1 * FT_STRIPS) {
        const int r0 = bstrip * FT_ROWS;
        Row5T<float2> histP[2];
        Row5T<float> histS[2];
        float2 cenxP, cenyP;
        float cenxS, cenyS;
#pragma unroll
        for (int rr = 0; rr < FT_ROWS + 2; ++rr) {
            const int r2 = min(r0 + rr, FT_R2 - 1);
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
                const int k = rr - 2;
                const int qr = r0 + k;
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
                // torch.min over the reprojections in cat order: the first minimum wins
                if (f == 0 || rp < br[k]) { br[k] = rp; idx_r = (idx_r & ~(3u << (2 * k))) | ((unsigned)f << (2 * k)); }
                float2 kaP, kbP, kcP;
                ssim_coef_gated_t(stP, rP, nrP, vmul(make_float2(w_ssim, w_ssim), passP), kaP, kbP, kcP);
                float kaS, kbS, kcS;
                ssim_coef_gated_t(stS, rS, nrS, w_ssim * passS, kaS, kbS, kcS);
                if (!LAST) {
                    st4(scr.q, k * FT_THREADS, kaP.x, kaP.y, kbP.x, kbP.y);
                    st4(scr.q, (FT_ROWS + k) * FT_THREADS, kcP.x, kcP.y, kaS, kbS);
                    st1(scr.q3 + k * FT_THREADS, kcS);
                } else if (qr < FT_R1) {
                    // identities come first in the cat: a reprojection wins only when strictly smaller
                    const bool win = ((okbits >> k) & 1u) && (!has_ident || br[k] < bi[k]) &&
                                     ((idx_r >> (2 * k)) & 3u) == (unsigned)f;
                    const int qi = qr * FT_R1 + bc;
                    const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
                    sm.q1[qi] = win ? make_float4(kaP.x, kaP.y, kbP.x, kbP.y) : z4;
                    sm.q2[qi] = win ? make_float4(kcP.x, kcP.y, kaS, kbS) : z4;
                    sm.q3[qi] = win ? kcS : 0.f;
                    sm.gate[qi] = (uint8_t)(win ? 1 : 0);
                }
            }
            histP[0] = histP[1]; histP[1] = curP;
            histS[0] = histS[1]; histS[1] = curS;
            cenxP = xb; cenyP = yb; cenxS = x2m; cenyS = y2m;
        }
    }
}

// d(loss)/d(P) of one source over this thread's 4 interior pixels from d(loss)/d(pred) (phase C) and the parked
// gather derivatives; block-reduced to 12 floats (Project3D backward: dp = d(loss)/d(P @ point), dP = dp x point^T).
__device__ __forceinline__ void pose_epilogue(const MfParams& p, const float* cams, const float4* aux, const float (&gp)[4][3],
                                              int tid, int b, int x0, int y0, float* red2, float* out) {
    const int H = p.H, W = p.W;
    const int oc = tid & 31, os = tid >> 5;
    const Camera& cam = *reinterpret_cast<const Camera*>(cams);
    float acc[12];
#pragma unroll
    for (int i = 0; i < 12; ++i) acc[i] = 0.f;
    const int px = x0 + oc;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int py = y0 + 4 * os + k;
        const float4 a0 = ld4(aux, (k * 4 + 0) * FT_THREADS);
        const float4 ex = ld4(aux, (k * 4 + 2) * FT_THREADS);
        const float4 ey = ld4(aux, (k * 4 + 3) * FT_THREADS);
        float dp0 = gp[k][0] * ex.x + gp[k][1] * ex.y + gp[k][2] * ex.z;
        float dp1 = gp[k][0] * ey.x + gp[k][1] * ey.y + gp[k][2] * ey.z;
        if (!(py < H && px < W)) { dp0 = 0.f; dp1 = 0.f; }
        const float dp2 = -(ex.w * dp0 + ey.w * dp1);
        float ray[3];
        pixel_ray(cam, (float)px, (float)py, ray);
        const float dp[3] = {dp0, dp1, dp2};
#pragma unroll
        for (int a = 0; a < 3; ++a) {
#pragma unroll
            for (int j = 0; j < 3; ++j) acc[a * 4 + j] = fmaf(dp[a], a0.w * ray[j], acc[a * 4 + j]);
            acc[a * 4 + 3] += dp[a];
        }
    }
    // warp reduction of the 12 sums as a reduce-scatter: every step halves the number of values a lane carries
    // (12 -> 6 -> 3 -> 2 -> 1: 13 shuffles instead of 60); lane L ends with the warp total of value vi(L)
    {
        const int lane = tid & 31;
        const bool b4 = lane & 16, b3 = lane & 8, b2 = lane & 4, b1 = lane & 2;
        float v6[6], v3[3], v2[2];
#pragma unroll
        for (int i = 0; i < 6; ++i) {
            const float keep = b4 ? acc[6 + i] : acc[i], send = b4 ? acc[i] : acc[6 + i];
            v6[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
        }
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            const float keep = b3 ? v6[3 + i] : v6[i], send = b3 ? v6[i] : v6[3 + i];
            v3[i] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
        }
        {   // 3 values padded to 4: (v3[0], v3[1]) | (v3[2], 0)
            const float k0 = b2 ? v3[2] : v3[0], s0 = b2 ? v3[0] : v3[2];
            const float k1 = b2 ? 0.0f : v3[1], s1 = b2 ? v3[1] : 0.0f;
            v2[0] = k0 + __shfl_xor_sync(0xffffffffu, s0, 4);
            v2[1] = k1 + __shfl_xor_sync(0xffffffffu, s1, 4);
        }
        const float k = b1 ? v2[1] : v2[0], sd = b1 ? v2[0] : v2[1];
        float v1 = k + __shfl_xor_sync(0xffffffffu, sd, 2);
        v1 += __shfl_xor_sync(0xffffffffu, v1, 1);
        // index of the value this lane holds: 6*b4 + 3*b3 + (b2 ? 2 : b1); the slot (b2 && b1) is the zero padding
        const int vi = (b4 ? 6 : 0) + (b3 ? 3 : 0) + (b2 ? 2 : (b1 ? 1 : 0));
        if (!(lane & 1) && !(b2 && b1)) red2[(tid >> 5) * 12 + vi] = v1;
    }
    __syncthreads();
    if (tid < 12) {
        float t = 0.f;
#pragma unroll
        for (int w = 0; w < FT_THREADS / 32; ++w) t += red2[w * 12 + tid];
        out[tid] = t * p.grad_scale;
    }
}

// Pass 1 of one (item, source): identity candidate, gather, fallback check, [target tile wait], phase B.
template <bool FASTDIV, bool POSE, bool LAST>
__device__ __forceinline__ void source_pass(const MfParams& p, const MsView& v, const TileSmem& sm, float* cams, const int* geo,
                                            uint64_t* tgt_bar, unsigned it, bool first_scale, int s, int f, const Scr scr, bool has_ident,
                                            unsigned& okbits, float (&bi)[FT_ROWS], float (&br)[FT_ROWS], unsigned& idx_i,
                                            unsigned& idx_r, float (&D)[4][3]) {
    const int H = p.H, W = p.W, N = H * W, F = p.F;
    float* tgt = sm.tgt;
    float* pred = sm.pred;
    // ---- identity loss + noise of source f: loads requested before the gather, folded in after it
    float ia[FT_ROWS], na[FT_ROWS];
    {
        int tidI = threadIdx.x, bI = geo[0], x0I = geo[1], y0I = geo[2];
        asm volatile("" : "+r"(tidI), "+r"(bI), "+r"(x0I), "+r"(y0I));
        const int bc = tidI % FT_R1, bstrip = tidI / FT_R1;
        const int qx = x0I - 1 + bc;
        const bool col_ok = qx >= 0 && qx < W && tidI < FT_R1 * FT_STRIPS;
        const float* idp = p.ident[f] + (size_t)bI * N + qx;
        const float* nzp = p.sc[s].noise + ((size_t)bI * F + f) * N + qx;
        okbits = 0u;
#pragma unroll
        for (int k = 0; k < FT_ROWS; ++k) {
            const int qr = bstrip * FT_ROWS + k, qy = y0I - 1 + qr;
            const bool ok = col_ok && qr < FT_R1 && qy >= 0 && qy < H;
            okbits |= ok ? (1u << k) : 0u;
            ia[k] = 0.f; na[k] = 0.f;
            if (ok && has_ident) {
                ia[k] = __ldg(idp + qy * W);
                if (p.sc[s].noise) na[k] = __ldg(nzp + qy * W);
            }
        }
    }
    // ---- phase A
    float lo = 1.0f, hi = 1.0f;
    {
        int tidA = threadIdx.x, bA = geo[0], x0A = geo[1], y0A = geo[2];
        asm volatile("" : "+r"(tidA), "+r"(bA), "+r"(x0A), "+r"(y0A));
        gather_tile_mf<FASTDIV, LAST, POSE>(v, cams + f * 24, p.src[f], tidA, bA, x0A, y0A, pred, scr.aux, D, lo, hi);
    }
    if (has_ident) {
#pragma unroll
        for (int k = 0; k < FT_ROWS; ++k) {
            const float c = add_rn(ia[k], na[k]);
            // torch.min over the identities in cat order: the first minimum wins
            if (f == 0 || c < bi[k]) { bi[k] = c; idx_i = (idx_i & ~(3u << (2 * k))) | ((unsigned)f << (2 * k)); }
        }
    }
    int tidB = threadIdx.x, bB = geo[0], x0B = geo[1], y0B = geo[2];
    asm volatile("" : "+r"(tidB), "+r"(bB), "+r"(x0B), "+r"(y0B));
    if (__syncthreads_or((lo >= 8.6736173798840355e-19f && hi <= 1.152921504606846976e18f) ? 0 : 1)) {
        // a pixel of this tile left the exponent range of the branch-free reciprocals: redo the gather with
        // the generic IEEE divisions (uniform branch; results identical wherever the fast form was valid)
        float Dl[12], al[48];
        gather_generic_mf<FASTDIV>(v, cams + f * 24, p.src[f] + (size_t)bB * 4 * N, pred, bB, x0B, y0B, Dl, al);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if (LAST) {
#pragma unroll
                for (int ch = 0; ch < 3; ++ch) D[k][ch] = Dl[k * 3 + ch];
                if (POSE) st4(scr.aux, (k * 4 + 0) * FT_THREADS, 0.f, 0.f, 0.f, al[k * 12 + 11]);
            } else {
                st4(scr.aux, (k * 4 + 0) * FT_THREADS, Dl[k * 3], Dl[k * 3 + 1], Dl[k * 3 + 2], al[k * 12 + 11]);
                st4(scr.aux, (k * 4 + 1) * FT_THREADS, al[k * 12], al[k * 12 + 1], al[k * 12 + 2], 0.f);
            }
            if (POSE) {
                st4(scr.aux, (k * 4 + 2) * FT_THREADS, al[k * 12 + 3], al[k * 12 + 4], al[k * 12 + 5], al[k * 12 + 9]);
                st4(scr.aux, (k * 4 + 3) * FT_THREADS, al[k * 12 + 6], al[k * 12 + 7], al[k * 12 + 8], al[k * 12 + 10]);
            }
        }
        __syncthreads();
    }
    if (f == 0 && first_scale) {
        mbar_wait(tgt_bar, it & 1u);
        // ReflectionPad2d(1) at the image border: TMA zero-fills out-of-image elements; patch them from the
        // in-image rows / columns of the same tile
        if (x0B < 2 || y0B < 2 || x0B + FT_T + 2 > W || y0B + FT_T + 2 > H) {
            for (int i = tidB; i < FT_N2; i += FT_THREADS) {
                const int r = i / FT_R2, c = i - r * FT_R2;
                const int ey = y0B - 2 + r, ex = x0B - 2 + c;
                if (ey < 0 || ey >= H || ex < 0 || ex >= W) {
                    const int sr = ext_to_img(ey, H) - (y0B - 2), sc = ext_to_img(ex, W) - (x0B - 2);
#pragma unroll
                    for (int ch = 0; ch < 3; ++ch)
                        tgt[ch * FT_NT + r * FT_TP + c + FT_TO] = tgt[ch * FT_NT + sr * FT_TP + sc + FT_TO];
                }
            }
            __syncthreads();
        }
    }
    // ---- phase B
    phase_b_multi<LAST>(sm, tidB, f, has_ident, okbits, bi, br, idx_r, scr);
    if (!LAST) __syncthreads();              // pred is free for the next source
}

template <bool FASTDIV, bool POSE>
__global__ void __launch_bounds__(FT_THREADS, 2)
photo_mf_kernel(const MfParams p, const __grid_constant__ CUtensorMap tgt_map) {
    extern __shared__ __align__(128) float smem[];
    __shared__ __align__(8) uint64_t tgt_bar;
    __shared__ int geo2[2][6];               // b, x0, y0, first / end scale, index of the current item (double-buffered over the items)
    float* tgt = smem;                       // [3][36][40] (TMA destination: 128-byte aligned)
    float* pred = tgt + 3 * FT_NT;           // [3][N2]
    float4* coefQ1 = reinterpret_cast<float4*>(pred + 3 * FT_N2);   // [N1]
    float4* coefQ2 = coefQ1 + FT_N1;                                // [N1]
    float* coefQ3 = reinterpret_cast<float*>(coefQ2 + FT_N1);       // [N1]
    float* cams = coefQ3 + FT_N1;            // [MF_MAXF][24]
    float* red = cams + MF_MAXF * 24;        // [8] per-warp loss sums
    float* red2 = red + 8;                   // [8][12] per-warp pose sums
    uint8_t* gate = reinterpret_cast<uint8_t*>(red2 + 96);          // [N1]

    const int H = p.H, W = p.W, N = H * W, F = p.F;
    const bool has_ident = p.ident[0] != nullptr;
    if (threadIdx.x == 0) mbar_init(&tgt_bar, 1);
    float* scr_cta = p.scratch + (size_t)blockIdx.x * F * MF_SRC_STRIDE;
    TileSmem sm;
    sm.tgt = tgt; sm.pred = pred; sm.q1 = coefQ1; sm.q2 = coefQ2; sm.q3 = coefQ3; sm.gate = gate;
    const int per_img = p.gx * p.gy;
    unsigned it = 0;
    int cam_b = -1;

#pragma unroll 1
    for (;; ++it) {
        const int tid0 = threadIdx.x;
        // the item: the first one is the CTA's own index, the following ones come from a global counter (dynamic
        // balance: tiles differ -- border patches, flagged tiles, skipped sources); its geometry is written by one
        // thread into the buffer the previous item does not read
        int* geo = geo2[it & 1u];
        if (tid0 == 32) {
            const int item = it == 0u ? (int)blockIdx.x : (int)gridDim.x + atomicAdd(p.next_item, 1);
            int tile = item, sb = 0, se = p.S;
            if (item >= p.n_full) { const int r = item - p.n_full; tile = p.n_full + r / p.S; sb = r % p.S; se = sb + 1; }
            const int b0 = tile / per_img, trem = tile - b0 * per_img;
            geo[0] = b0; geo[1] = (trem % p.gx) * FT_T; geo[2] = (trem / p.gx) * FT_T; geo[3] = sb; geo[4] = se;
            geo[5] = item;
        }
        __syncthreads();                     // the previous item is done with every shared buffer
        if (geo[5] >= p.n_items) break;      // (uniform)
        const int b0 = geo[0];
        if (tid0 == 0) {
            // target tile by TMA, in flight during the gather of the first source (the reflection patch of the
            // previous item wrote this buffer through the generic proxy)
            fence_proxy_async();
            mbar_expect_tx(&tgt_bar, 3 * FT_NT * sizeof(float));
            tma_load_4d(tgt, &tgt_map, &tgt_bar, geo[1] - 2 - FT_TO, geo[2] - 2, 0, b0);
        }
        if (b0 != cam_b) {                   // (uniform) the cameras stay in shared memory while the batch item does
            cam_b = b0;
            if (tid0 < F * 21) {
                const int f = tid0 / 21, t = tid0 % 21;
                if (t < 12) {
                    const int i = t / 4, j = t % 4;
                    const float* k = p.K + b0 * 16 + i * 4;
                    const float* tt = p.T[f] + b0 * 16 + j;
                    float acc = __ldg(k) * __ldg(tt);
                    acc = fmaf(__ldg(k + 1), __ldg(tt + 4), acc);
                    acc = fmaf(__ldg(k + 2), __ldg(tt + 8), acc);
                    acc = fmaf(__ldg(k + 3), __ldg(tt + 12), acc);
                    cams[f * 24 + t] = acc;
                } else {
                    const int i = (t - 12) / 3, j = (t - 12) % 3;
                    cams[f * 24 + t] = __ldg(p.inv_K + b0 * 16 + i * 4 + j);
                }
            }
            __syncthreads();
        }

        // the scales of the tile one after the other: the taps of scale s + 1 find the source lines of scale s in L1
        // (one (tile, scale) item per CTA round instead: 27 % slower, L1 hit rate 33 % against 49 %)
#pragma unroll 1
        for (int s = geo[3]; s < geo[4]; ++s) {
        const bool first_scale = s == geo[3];
        if (!first_scale) __syncthreads();   // phase C of the previous scale is done with pred / the planes
        MsView v;
        v.ident = nullptr; v.noise = nullptr; v.sel = nullptr; v.grad_disp = p.sc[s].grad_disp;
        v.hint_reproj = nullptr; v.hint_depth = nullptr; v.hint_valid = nullptr; v.grad_hint = nullptr;
        v.disp.ptr = p.sc[s].disp; v.disp.h = p.sc[s].dh; v.disp.w = p.sc[s].dw;
        v.disp.sh = p.sc[s].sh; v.disp.sw = p.sc[s].sw;
        v.ds = p.ds; v.H = H; v.W = W; v.dh_nblk = 0;
        v.grad_scale = p.grad_scale; v.rcw = p.rcw; v.rch = p.rch;

        // running first-minimum of this thread's 5 ring pixels: identities (bi, idx_i) and reprojections (br, idx_r)
        float bi[FT_ROWS], br[FT_ROWS];
        unsigned idx_i = 0u, idx_r = 0u, okbits = 0u;
#pragma unroll
        for (int k = 0; k < FT_ROWS; ++k) { bi[k] = __int_as_float(0x7f800000); br[k] = __int_as_float(0x7f800000); }
        float D[4][3];

#pragma unroll 1
        for (int f = 0; f < F - 1; ++f)
            source_pass<FASTDIV, POSE, false>(p, v, sm, cams, geo, &tgt_bar, it, first_scale, s, f, scr_of(scr_cta, f, threadIdx.x),
                                              has_ident, okbits, bi, br, idx_i, idx_r, D);
        source_pass<FASTDIV, POSE, true>(p, v, sm, cams, geo, &tgt_bar, it, first_scale, s, F - 1, scr_of(scr_cta, F - 1, threadIdx.x),
                                         has_ident, okbits, bi, br, idx_i, idx_r, D);

        // ---- decision: loss, argmin, the ring pixels a reprojection wins
        unsigned winbits = 0u;
        {
            int tidB = threadIdx.x, bB = geo[0], x0B = geo[1], y0B = geo[2];
            asm volatile("" : "+r"(tidB), "+r"(bB), "+r"(x0B), "+r"(y0B));
            const int bc = tidB % FT_R1, bstrip = tidB / FT_R1;
            const bool col_in = bc >= 1 && bc <= FT_T;
            float loss_local = 0.0f;
#pragma unroll
            for (int k = 0; k < FT_ROWS; ++k) {
                const int qr = bstrip * FT_ROWS + k;
                const bool ok = (okbits >> k) & 1u;
                const bool win = ok && (!has_ident || br[k] < bi[k]);
                winbits |= win ? (1u << k) : 0u;
                if (col_in && qr >= 1 && qr <= FT_T && ok) {
                    loss_local += win ? br[k] : bi[k];
                    if (p.sc[s].sel) {
                        const int qo = (y0B - 1 + qr) * W + x0B - 1 + bc;
                        const unsigned ir = (idx_r >> (2 * k)) & 3u, ii = (idx_i >> (2 * k)) & 3u;
                        p.sc[s].sel[(size_t)bB * N + qo] = (uint8_t)(win ? (has_ident ? F : 0) + ir : ii);
                    }
                }
            }
            const float ws = warp_sum(loss_local);
            if ((tidB & 31) == 0) red[tidB >> 5] = ws;
        }

        // ---- pass 2: the last source from shared memory / registers, the earlier ones from the scratch
        float g_acc[4] = {0.f, 0.f, 0.f, 0.f};
        float acc4[4] = {0.f, 0.f, 0.f, 0.f};
        {
            const int f = F - 1;
            unsigned gm = 0u;
#pragma unroll
            for (int k = 0; k < FT_ROWS; ++k)
                gm |= (((winbits >> k) & 1u) && ((idx_r >> (2 * k)) & 3u) == (unsigned)f) ? (1u << k) : 0u;
            // barrier: the planes of the last source are complete
            const int any = __syncthreads_or(gm != 0u);
            int tidC = threadIdx.x, bC = geo[0], x0C = geo[1], y0C = geo[2];
            asm volatile("" : "+r"(tidC), "+r"(bC), "+r"(x0C), "+r"(y0C));
            float* gp_dst = nullptr;
            if (POSE && p.sc[s].grad_P) {
                const int blk = (y0C / FT_T) * p.gx + x0C / FT_T;
                gp_dst = p.sc[s].grad_P + (((size_t)f * p.B + bC) * per_img + blk) * 12;
            }
            if (any) {
                float gp[4][3];
                phase_c<false, false>(v, sm, tidC, bC, x0C, y0C, D, acc4, POSE ? gp : nullptr, g_acc);
                if (POSE && gp_dst)
                    pose_epilogue(p, cams + f * 24, scr_of(scr_cta, f, tidC).aux, gp, tidC, bC, x0C, y0C, red2, gp_dst);
            } else if (gp_dst && tidC < 12) gp_dst[tidC] = 0.f;     // wins nowhere in the tile: no gradient through it
        }
#pragma unroll 1
        for (int f = F - 2; f >= 0; --f) {
            const Scr scr = scr_of(scr_cta, f, threadIdx.x);
            unsigned gm = 0u;
#pragma unroll
            for (int k = 0; k < FT_ROWS; ++k)
                gm |= (((winbits >> k) & 1u) && ((idx_r >> (2 * k)) & 3u) == (unsigned)f) ? (1u << k) : 0u;
            // the parked coefficients / factors are requested BEFORE the barrier (they are this thread's own data) and
            // consumed after it
            float4 qa[FT_ROWS], qc[FT_ROWS], a0[4], a1[4];
            float qe[FT_ROWS];
#pragma unroll
            for (int k = 0; k < FT_ROWS; ++k) {
                qa[k] = ld4(scr.q, k * FT_THREADS); qc[k] = ld4(scr.q, (FT_ROWS + k) * FT_THREADS);
                qe[k] = ld1s(scr.q3 + k * FT_THREADS);
            }
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                a0[k] = ld4(scr.aux, (k * 4 + 0) * FT_THREADS); a1[k] = ld4(scr.aux, (k * 4 + 1) * FT_THREADS);
            }
            // barrier: phase C of the previous source is done with the planes
            const int any = __syncthreads_or(gm != 0u);
            int tidC = threadIdx.x, bC = geo[0], x0C = geo[1], y0C = geo[2];
            asm volatile("" : "+r"(tidC), "+r"(bC), "+r"(x0C), "+r"(y0C));
            float* gp_dst = nullptr;
            if (POSE && p.sc[s].grad_P) {
                const int blk = (y0C / FT_T) * p.gx + x0C / FT_T;
                gp_dst = p.sc[s].grad_P + (((size_t)f * p.B + bC) * per_img + blk) * 12;
            }
            if (!any) {                      // this source wins nowhere in the tile: no gradient through it
                if (gp_dst && tidC < 12) gp_dst[tidC] = 0.f;
                continue;
            }
            const int bc = tidC % FT_R1, bstrip = tidC / FT_R1;
            if (tidC < FT_R1 * FT_STRIPS) {
#pragma unroll
                for (int k = 0; k < FT_ROWS; ++k) {
                    const int qr = bstrip * FT_ROWS + k;
                    if (qr < FT_R1) {
                        const bool w = (gm >> k) & 1u;
                        const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
                        const int qi = qr * FT_R1 + bc;
                        coefQ1[qi] = w ? qa[k] : z4;
                        coefQ2[qi] = w ? qc[k] : z4;
                        coefQ3[qi] = w ? qe[k] : 0.f;
                        gate[qi] = (uint8_t)(w ? 1 : 0);
                    }
                }
            }
            float Dl[4][3], xv[4][3];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                Dl[k][0] = a0[k].x; Dl[k][1] = a0[k].y; Dl[k][2] = a0[k].z;
                xv[k][0] = a1[k].x; xv[k][1] = a1[k].y; xv[k][2] = a1[k].z;
            }
            __syncthreads();
            float gp[4][3];
            phase_c<false, false>(v, sm, tidC, bC, x0C, y0C, Dl, acc4, POSE ? gp : nullptr, g_acc, xv);
            if (POSE && gp_dst) pose_epilogue(p, cams + f * 24, scr.aux, gp, tidC, bC, x0C, y0C, red2, gp_dst);
        }

        // ---- outputs of the item
        {
            int tidO = threadIdx.x, bO = geo[0], x0O = geo[1], y0O = geo[2];
            asm volatile("" : "+r"(tidO), "+r"(bO), "+r"(x0O), "+r"(y0O));
            const int oc = tidO & 31, os = tidO >> 5;
            const int px = x0O + oc;
            float* gout = p.sc[s].grad_disp + (size_t)bO * N + px;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int py = y0O + 4 * os + k;
                if (py < H && px < W) gout[py * W] = g_acc[k];
            }
            if (tidO < 32) {
                // the 8 per-warp sums in block_sum's order (same bits as the single-source kernels)
                float t = tidO < FT_THREADS / 32 ? red[tidO] : 0.0f;
                t = warp_sum(t);
                const int blk = bO * per_img + (y0O / FT_T) * p.gx + x0O / FT_T;
                if (tidO == 0) p.sc[s].loss_partial[blk] = t;
            }
        }
        }   // scales of the item
    }
}

}  // namespace

/* Scratch of dmh_photo_multisource in floats (current device): 2 CTAs per SM x F sources.  */
extern "C" long long dmh_photo_multisource_workspace_floats(int F) {
    int dev = 0, sms = 0;
    if (cudaGetDevice(&dev) != cudaSuccess ||
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0)
        sms = 148;
    if (F < 1) F = 1;
    return (long long)2 * sms * F * MF_SRC_STRIDE + 4;      // + the work counter
}

extern "C" int dmh_photo_multisource(const float* target, const float* const* src_packed_host, const float* const* T_host,
                                     int F, int S, const float* const* disp_host, const int* disp_h, const int* disp_w,
                                     const float* K, const float* inv_K, const float* const* ident_host,
                                     const float* const* noise_host, int B, int H, int W, float min_depth, float max_depth,
                                     float grad_scale, float* workspace, float* const* loss_partial_host,
                                     float* const* grad_disp_host, float* const* grad_P_partial_host,
                                     uint8_t* const* sel_host, dmh_stream_t stream) {
    DMH_REQUIRE(target && src_packed_host && T_host && K && inv_K && disp_host && disp_h && disp_w && workspace &&
                loss_partial_host && grad_disp_host, "dmh_photo_multisource: null argument");
    DMH_REQUIRE(F >= 1 && F <= MF_MAXF, "dmh_photo_multisource: F=%d outside [1,%d]", F, MF_MAXF);
    DMH_REQUIRE(S >= 1 && S <= MF_MAX_SCALES, "dmh_photo_multisource: 1 <= S <= %d (got %d)", MF_MAX_SCALES, S);
    DMH_REQUIRE(B >= 1 && B <= 65535 && H >= 2 && W >= 2, "dmh_photo_multisource: bad sizes B=%d H=%d W=%d", B, H, W);
    DMH_REQUIRE((long long)H * W < (1ll << 27), "dmh_photo_multisource: frame too large for 32-bit tap offsets");
    DMH_REQUIRE(min_depth > 0.f && max_depth > min_depth, "dmh_photo_multisource: bad depth range");
    DMH_REQUIRE((uintptr_t)workspace % 16 == 0, "dmh_photo_multisource: workspace must be 16-byte aligned");
    CUtensorMap map;
    if (!encode_frames_map(&map, target, B, H, W, FT_TP, FT_R2)) {
        set_error("dmh_photo_multisource: needs W %% 4 == 0 and 16-byte aligned frames (TMA); use dmh_photo_scale");
        return DMH_ERR_UNSUPPORTED;
    }
    MfParams p;
    memset(&p, 0, sizeof(p));
    bool any_ident = false, all_ident = true;
    for (int f = 0; f < F; ++f) {
        DMH_REQUIRE(src_packed_host[f] && T_host[f], "dmh_photo_multisource: null src / T for source %d", f);
        DMH_REQUIRE((uintptr_t)src_packed_host[f] % 16 == 0, "dmh_photo_multisource: packed source %d not 16-byte aligned", f);
        p.src[f] = src_packed_host[f]; p.T[f] = T_host[f];
        p.ident[f] = ident_host ? ident_host[f] : nullptr;
        any_ident = any_ident || p.ident[f];
        all_ident = all_ident && p.ident[f];
    }
    DMH_REQUIRE(!any_ident || all_ident, "dmh_photo_multisource: identity losses for some sources only");
    p.K = K; p.inv_K = inv_K; p.next_item = reinterpret_cast<int*>(workspace); p.scratch = workspace + 4;
    p.F = F; p.S = S; p.B = B; p.H = H; p.W = W;
    p.ds = depth_scale(min_depth, max_depth, false);
    p.grad_scale = grad_scale;
    bool pose = false;
    for (int s = 0; s < S; ++s) {
        DMH_REQUIRE(disp_host[s] && loss_partial_host[s] && grad_disp_host[s] && disp_h[s] >= 1 && disp_w[s] >= 1,
                    "dmh_photo_multisource: scale %d: null buffer or empty disparity", s);
        p.sc[s].disp = disp_host[s]; p.sc[s].dh = disp_h[s]; p.sc[s].dw = disp_w[s];
        p.sc[s].sh = (float)disp_h[s] / (float)H; p.sc[s].sw = (float)disp_w[s] / (float)W;
        p.sc[s].noise = (noise_host && any_ident) ? noise_host[s] : nullptr;
        p.sc[s].loss_partial = loss_partial_host[s];
        p.sc[s].grad_disp = grad_disp_host[s];
        p.sc[s].grad_P = grad_P_partial_host ? grad_P_partial_host[s] : nullptr;
        p.sc[s].sel = sel_host ? sel_host[s] : nullptr;
        pose = pose || p.sc[s].grad_P;
    }
    const size_t smem = sizeof(float) * (3 * FT_NT + 3 * FT_N2 + 9 * FT_N1 + MF_MAXF * 24 + 8 + 96) + FT_N1;
    static KernelSetup setup;
    const void* kernels[4] = {(const void*)photo_mf_kernel<true, false>, (const void*)photo_mf_kernel<true, true>,
                              (const void*)photo_mf_kernel<false, false>, (const void*)photo_mf_kernel<false, true>};
    const int sms = setup.sms("dmh_photo_multisource", kernels, 4, smem);
    if (sms == 0) return DMH_ERR_CUDA;
    const bool fastdiv = const_div_exact(W - 1, &p.rcw, (cudaStream_t)stream) &&
                         const_div_exact(H - 1, &p.rch, (cudaStream_t)stream);
    p.gx = ceil_div(W, FT_T); p.gy = ceil_div(H, FT_T);
    cudaStream_t st = (cudaStream_t)stream;
    {
        // loss_partial holds B * dmh_photo_tiles floats (the generic kernel's smaller tiles); this kernel writes one
        // float per 32 x 32 tile: the tail reads as zero
        const int used = B * p.gx * p.gy, total = B * dmh_photo_tiles(H, W);
        for (int s = 0; s < S && total > used; ++s) {
            cudaError_t e = cudaMemsetAsync(loss_partial_host[s] + used, 0, sizeof(float) * (size_t)(total - used), st);
            if (e != cudaSuccess) {
                set_error("dmh_photo_multisource: cudaMemsetAsync failed: %s", cudaGetErrorString(e));
                return DMH_ERR_CUDA;
            }
        }
    }
    // persistent grid of 2 CTAs per SM; the tiles of the partial last round become S single-scale items each
    const int slots = 2 * sms, n_tiles = p.gx * p.gy * B;
    p.n_full = split_last_wave(n_tiles, S, slots);
    p.n_items = p.n_full + (n_tiles - p.n_full) * S;
    const int n_ctas = p.n_items < slots ? p.n_items : slots;
    {
        cudaError_t e = cudaMemsetAsync(workspace, 0, 16, st);
        if (e != cudaSuccess) {
            set_error("dmh_photo_multisource: cudaMemsetAsync failed: %s", cudaGetErrorString(e));
            return DMH_ERR_CUDA;
        }
    }
    if (fastdiv) {
        if (pose) DMH_LAUNCH((photo_mf_kernel<true, true>), n_ctas, FT_THREADS, smem, st)(p, map);
        else DMH_LAUNCH((photo_mf_kernel<true, false>), n_ctas, FT_THREADS, smem, st)(p, map);
    } else {
        if (pose) DMH_LAUNCH((photo_mf_kernel<false, true>), n_ctas, FT_THREADS, smem, st)(p, map);
        else DMH_LAUNCH((photo_mf_kernel<false, false>), n_ctas, FT_THREADS, smem, st)(p, map);
    }
    DMH_CHECK_LAUNCH("dmh_photo_multisource");
    return DMH_OK;
}
