// Fast path of dmh_photo_scale for ONE source frame (the headline stereo
// configuration, frame_ids [0,'s']; also mono with a single source when no pose
// gradient is requested).  Same contract and results as photo_scale_kernel<1>
// in photo_objective.cu, ~3.4x fewer instructions:
//
//   * 32x32 tile, 256 threads; every thread OWNS 4 interior pixels of one
//     column (rows 4s..4s+3) in the warp phase and in the gradient phase, so
//     the whole backward chain of the gather (bilinear taps -> coordinates ->
//     projection -> depth -> disparity) collapses into 3 scalars per pixel
//     held in registers (no second gather, no coordinate recompute);
//   * SSIM statistics by separable sliding windows: a thread walks down a
//     column of the 34x34 ring and reuses the 3-wide row sums across the 3
//     windows they belong to; value and backward coefficients share one
//     reciprocal; the automask decision gates the coefficients in the same pass
//     (single source frame -> the winner is known immediately);
//   * the 3x3 box sums of the 9 coefficient planes are separable sliding
//     windows too; reflection multiplicities are folded into the edge weights.
//
//   * the source is gathered from a pixel-packed (B,H,W,4) copy written once per step by the identity-loss
//     kernel below: one 128-bit load per bilinear tap, the north-west tap clamped so that the other three sit
//     at fixed offsets (bit-identical to the planar gather);
//   * SSIM in sum form (no divisions by 9), branch-free, channels (0,1) in packed fp32 (explicitly rounded
//     add/mul/fma.rn.f32x2), coefficient planes laid out for 128-bit shared-memory accesses.
//
// Shared memory: tgt 3x36x40 + pred 3x36x36 + coef 9x34x34 floats + gate bytes = 75.8 KB -> 3 CTAs / SM.
// Roofline: HBM by traffic (40 B per target pixel, 419 MB per launch at B=32 -- ncu measures exactly that), but
// instruction-issue bound in practice: ~745 lane-instructions / pixel at ~57 % issue utilisation (profiles/).
//
// Also here: ident_fast_kernel (identity reprojection loss + the packed copy, both tiles by TMA).
//
// Target tile staging: ONE elected thread issues a 4-D TMA load
// (cp.async.bulk.tensor, box 40 x 36 x 3 x 1 at (x0-4, y0-2, 0, b) -- the innermost
// start coordinate must be 16-byte aligned, measured: x0-2 raises an illegal
// instruction -- out-of-image elements zero-filled) that lands on an mbarrier while all warps run the gather
// phase; the 1-px reflection (ReflectionPad2d) of border tiles is patched in
// shared memory afterwards.  Rows that are not 16-byte aligned (W % 4 != 0 or a
// misaligned base) take the plain-load instantiation of the same kernel.
#include <array>
#include <utility>

#include "photo_tile.cuh"

namespace {

// TMA: target tile by cp.async.bulk.tensor; FASTDIV: verified 3-instruction division by W-1 / H-1;
// PK: pixel-packed source (128-bit taps); UP: the disparity map is smaller than the frame (scales 1..3).
// SSIM is always on and the input is a disparity here (no_ssim, depth inputs and the materialised warped images
// take the general kernel).
template <bool TMA, bool FASTDIV, bool PK, bool UP, bool DH = false>
__global__ void __launch_bounds__(FT_THREADS, 3)
photo_fast_kernel(const FastParams p, const __grid_constant__ CUtensorMap tgt_map) {
    extern __shared__ __align__(128) float smem[];
    __shared__ __align__(8) uint64_t tgt_bar;
    float* tgt = smem;                       // [3][36][40] (TMA destination: 128-byte aligned)
    float* pred = tgt + 3 * FT_NT;           // [3][N2]
    // gated SSIM coefficients of a ring pixel, laid out for 128-bit accesses: Q1 = (a0, a1, b0, b1),
    // Q2 = (c0, c1, a2, b2), Q3 = c2  (a, b, c of channels 0, 1, 2)
    float4* coefQ1 = reinterpret_cast<float4*>(pred + 3 * FT_N2);  // [N1]
    float4* coefQ2 = coefQ1 + FT_N1;                                // [N1]
    float* coefQ3 = reinterpret_cast<float*>(coefQ2 + FT_N1);       // [N1]
    float* cams = coefQ3 + FT_N1;            // [24]
    float* red = cams + 24;                  // [32]
    uint8_t* gate = reinterpret_cast<uint8_t*>(red + 32);   // [N1]

    const int tid = threadIdx.x;
    const int H = p.H, W = p.W;
    const int b = blockIdx.z;
    const int x0 = blockIdx.x * FT_T, y0 = blockIdx.y * FT_T;
    const int N = H * W;                      // per-item offsets fit 32 bits (checked by the launcher)
    const float w_ssim = 0.85f / 3.0f, w_l1 = 0.15f / 3.0f;

    load_camera(cams, p, b, tid);
    if (TMA) {
        // ---- target tile by TMA: in flight during the whole gather phase
        if (tid == 0) {
            mbar_init(&tgt_bar, 1);
            mbar_expect_tx(&tgt_bar, 3 * FT_NT * sizeof(float));
            tma_load_4d(tgt, &tgt_map, &tgt_bar, x0 - 2 - FT_TO, y0 - 2, 0, b);
        }
    } else if (tid < FT_R2 * 7) {
        // ---- target tile, 2-px reflect halo: 36 columns x 7 row groups = 252 threads, column index maths once
        const int c = tid % FT_R2, rg = tid / FT_R2;
        const float* tp = p.target + (size_t)b * 3 * N + ext_to_img(x0 - 2 + c, W);
        for (int r = rg; r < FT_R2; r += 7) {
            const int o = ext_to_img(y0 - 2 + r, H) * W;
#pragma unroll
            for (int ch = 0; ch < 3; ++ch) tgt[ch * FT_NT + r * FT_TP + c + FT_TO] = __ldg(tp + ch * N + o);
        }
    }
    __syncthreads();
    const int oc = tid & 31, os = tid >> 5;
    float D[4][3];
    Camera cam;
#pragma unroll
    for (int i = 0; i < 12; ++i) cam.P[i] = cams[i];
#pragma unroll
    for (int i = 0; i < 9; ++i) cam.iK[i] = cams[12 + i];
    const float* sp = p.src + (size_t)b * (PK ? 4 : 3) * N;
    const float* dp = p.disp.ptr + (size_t)b * (p.disp.h * p.disp.w);

    // ---- phase A: warp.  A thread owns the interior pixels of column tid%32, rows 4*(tid/32)+k, plus one pixel
    // of the halo ring.  Software-pipelined over those 5 pixels: all disparity loads, then the coordinate chains,
    // then the gathers -- the memory latency is paid once per stage instead of once per pixel.
    {
        int hr, hc;
        halo_rc(tid, hr, hc);
        int py[5], pxx[5];
        const int ixo = tile_to_img(x0 + oc, W);
#pragma unroll
        for (int k = 0; k < 4; ++k) { py[k] = tile_to_img(y0 + 4 * os + k, H); pxx[k] = ixo; }
        py[4] = ext_to_img(y0 - 2 + hr, H);
        pxx[4] = ext_to_img(x0 - 2 + hc, W);
        float dv[5];
        if (!UP) {
#pragma unroll
            for (int k = 0; k < 5; ++k) dv[k] = __ldg(dp + py[k] * W + pxx[k]);
        } else {
            const UpTap txo = up_tap(ixo, p.disp.sw, p.disp.w);        // shared by the 4 owned pixels
#pragma unroll
            for (int k = 0; k < 4; ++k) dv[k] = up_sample(dp, p.disp.w, up_tap(py[k], p.disp.sh, p.disp.h), txo);
            dv[4] = up_sample(dp, p.disp.w, up_tap(py[4], p.disp.sh, p.disp.h), up_tap(pxx[4], p.disp.sw, p.disp.w));
        }
        Tap tp[5];
        float gax[5], gay[5];
#pragma unroll
        for (int k = 0; k < 5; ++k) tp[k] = pixel_tap<FASTDIV>(cam, p, pxx[k], py[k], dv[k], k < 4, gax[k], gay[k]);
        // gathers: the taps of TWO pixels are requested before either is consumed
#pragma unroll
        for (int k0 = 0; k0 < 5; k0 += 2) {
            float tv[2][3][4];
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                if (k0 + j < 5) load_taps<PK>(sp, N, W, tp[k0 + j], tv[j]);
            }
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const int k = k0 + j;
                if (k >= 5) continue;
                const Gathered g = combine_taps(tv[j], tp[k], k < 4);
                const int r = 4 * os + k;
                const int i2 = (k < 4) ? (r + 2) * FT_R2 + oc + 2 : hr * FT_R2 + hc;
#pragma unroll
                for (int ch = 0; ch < 3; ++ch) pred[ch * FT_N2 + i2] = g.v[ch];
                if (k < 4) {
#pragma unroll
                    for (int ch = 0; ch < 3; ++ch) D[k][ch] = g.dix[ch] * gax[k] + g.diy[ch] * gay[k];
                }
            }
        }
    }
    // the remaining 16 pixels of the halo ring
    if (tid < 272 - FT_THREADS) {
        int r, c;
        halo_rc(tid + FT_THREADS, r, c);
        const int iy = ext_to_img(y0 - 2 + r, H), ix = ext_to_img(x0 - 2 + c, W);
        const float dvh = UP ? up_sample(dp, p.disp.w, up_tap(iy, p.disp.sh, p.disp.h), up_tap(ix, p.disp.sw, p.disp.w))
                             : __ldg(dp + iy * W + ix);
        float u0, u1;
        const Tap th = pixel_tap<FASTDIV>(cam, p, ix, iy, dvh, false, u0, u1);
        float tvh[3][4];
        load_taps<PK>(sp, N, W, th, tvh);
        const Gathered g = combine_taps(tvh, th, false);
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) pred[ch * FT_N2 + r * FT_R2 + c] = g.v[ch];
    }
    // identity losses (+ tie-break noise) of this thread's phase-B pixels: requested before the barrier so
    // that their latency overlaps the other warps' gather.  Ring pixels outside the image are marked by a NaN
    // (rp < NaN is false: they never win, their coefficients are gated to 0 and they add nothing to the loss).
    float idv_pre[FT_ROWS];
    unsigned hflags;
    prefetch_ident<DH>(p, tid, b, x0, y0, idv_pre, hflags);
    __syncthreads();
    if (TMA) {
        mbar_wait(&tgt_bar, 0);
        patch_target_border(tgt, tid, x0, y0, H, W);       // (sources are never patched themselves)
    }

    TileSmem sm;
    sm.tgt = tgt; sm.pred = pred; sm.q1 = coefQ1; sm.q2 = coefQ2; sm.q3 = coefQ3; sm.gate = gate;
    float acc4[4] = {0.f, 0.f, 0.f, 0.f};
    const float loss_local = phase_b<DH, UP>(p, sm, tid, b, x0, y0, idv_pre, hflags, acc4);
    __syncthreads();
    phase_c<DH, UP>(p, sm, tid, b, x0, y0, D, acc4);
    const int blk = (b * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x;
    if (DH) {
        // [4][dh_nblk]: sum reproj*mask_r, sum mask_r, sum proxy*mask_h, sum mask_h
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const float s = block_sum(acc4[q], red);
            if (tid == 0) p.loss_partial[q * p.dh_nblk + blk] = s;
        }
    } else {
        const float s = block_sum(loss_local, red);
        if (tid == 0) p.loss_partial[blk] = s;
    }
}


// ---------------------------------------------------------------------------
// Identity reprojection loss (M2/trainer.py:608-615): compute_reprojection_loss of the UN-warped
// source against the target.  Scale independent -> computed once per batch (the reference recomputes it
// for every scale).  32x32 tile, 1-px reflect halo, sliding-window SSIM down each column.
#define ID_R 34
#define ID_N (ID_R * ID_R)
struct IdentParams {
    const float* target;
    const float* src[DMH_PHOTO_MAX_FRAMES];
    float* out;                 // (B,F,H,W); nullable when only the packed copy is wanted
    float4* packed;             // nullable (F == 1): source frame 0 re-laid out as (B,H,W,4) for the 128-bit tap gather
    int B, F, H, W, no_ssim;
};

// TMA: both tiles arrive by cp.async.bulk.tensor (box 40 x 34 x 3 at (x0-4, y0-1): 16-byte aligned start column,
// zero fill outside the image, reflection patched in shared memory on border tiles) -- no per-thread load / index
// instructions at all; otherwise plain loads with the same shared-memory layout.
#define ID_P 40                  // row pitch of the tiles
#define ID_O 3                   // column of the tile that holds halo column 0 (image column x0-1)
#define ID_PL (ID_R * ID_P)      // plane stride
struct IdentMaps { CUtensorMap tgt; CUtensorMap src[DMH_PHOTO_MAX_FRAMES]; };

// Shared tail of the identity-loss kernels: packed copy of the source tile (+ optional fp32 copy of the target tile,
// bf16 inputs) and the identity reprojection loss of the tile from the two staged 34 x 34 x 3 tiles.
__device__ __forceinline__ void ident_tile_tail(const IdentParams& p, const float* xs, const float* ys, int tid, int b,
                                                int f, int x0, int y0, float* tgt_f32) {
    const int H = p.H, W = p.W;
    const size_t N = (size_t)H * W;
    __syncthreads();
    const int c = tid & 31, strip = tid >> 5;           // 8 strips of 4 rows
    const int px = x0 + c;
    if (p.packed && px < W) {     // pixel-packed copy of the source tile: a warp writes 512 contiguous bytes per row
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int r = 4 * strip + k, py = y0 + r;
            if (py < H) {
                const int i = (r + 1) * ID_P + c + 1 + ID_O;
                p.packed[(size_t)b * N + (size_t)py * W + px] = make_float4(xs[i], xs[ID_PL + i], xs[2 * ID_PL + i], 0.0f);
            }
        }
    }
    if (tgt_f32 && x0 + c < W) {   // bf16 inputs: the fp32 target the photometric kernels stage by TMA
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int r = 4 * strip + k, py = y0 + r;
            if (py < H) {
                const int i = (r + 1) * ID_P + c + 1 + ID_O;
#pragma unroll
                for (int ch = 0; ch < 3; ++ch) tgt_f32[((size_t)b * 3 + ch) * N + (size_t)py * W + x0 + c] = ys[ch * ID_PL + i];
            }
        }
    }
    if (!p.out) return;
    // same lane-typed SSIM arithmetic as the fused kernels (channels 0,1 packed, channel 2 scalar): the
    // identity loss and the reprojection loss must come out of identical arithmetic (automask ties)
    Row5T<float2> histP[2];
    Row5T<float> histS[2];
    float2 cenxP = make_float2(0.f, 0.f), cenyP = cenxP;
    float cenxS = 0.f, cenyS = 0.f;
#pragma unroll
    for (int rr = 0; rr < 6; ++rr) {
        const int r2 = 4 * strip + rr;                   // halo-tile row
        const float* x0p = xs + r2 * ID_P + c + ID_O;
        const float* y0p = ys + r2 * ID_P + c + ID_O;
        const float2 xa = make_float2(x0p[0], x0p[ID_PL]), xb = make_float2(x0p[1], x0p[ID_PL + 1]),
                     xc = make_float2(x0p[2], x0p[ID_PL + 2]);
        const float2 ya = make_float2(y0p[0], y0p[ID_PL]), yb = make_float2(y0p[1], y0p[ID_PL + 1]),
                     yc = make_float2(y0p[2], y0p[ID_PL + 2]);
        const Row5T<float2> curP = row5(xa, xb, xc, ya, yb, yc);
        const float* x2p = x0p + 2 * ID_PL;
        const float* y2p = y0p + 2 * ID_PL;
        const Row5T<float> curS = row5(x2p[0], x2p[1], x2p[2], y2p[0], y2p[1], y2p[2]);
        if (rr >= 2) {
            const int py = y0 + 4 * strip + rr - 2;
            if (py < H && px < W) {
                float l1 = fabsf(cenyP.x - cenxP.x);
                l1 += fabsf(cenyP.y - cenxP.y);
                l1 += fabsf(cenyS - cenxS);
                float ss = 0.f;
                if (!p.no_ssim) {
                    float2 passP, rP, nrP;
                    const float2 vP = ssim_value_t(ssim_stats_rows_t(histP[0], histP[1], curP), passP, rP, nrP);
                    float passS, rS, nrS;
                    const float vS = ssim_value_t(ssim_stats_rows_t(histS[0], histS[1], curS), passS, rS, nrS);
                    ss = (vP.x + vP.y) + vS;
                }
                l1 *= (1.0f / 3.0f);
                const float rp = p.no_ssim ? l1 : fmaf(0.85f, ss * (1.0f / 3.0f), 0.15f * l1);
                p.out[((size_t)b * p.F + f) * N + (size_t)py * W + px] = rp;
            }
        }
        histP[0] = histP[1]; histP[1] = curP;
        histS[0] = histS[1]; histS[1] = curS;
        cenxP = xb; cenyP = yb; cenxS = x2p[1]; cenyS = y2p[1];
    }
}

template <bool TMA>
__global__ void __launch_bounds__(256, 4)
ident_fast_kernel(const IdentParams p, const __grid_constant__ IdentMaps maps) {
    __shared__ __align__(128) float xs[3 * ID_PL];
    __shared__ __align__(128) float ys[3 * ID_PL];
    __shared__ __align__(8) uint64_t bar;
    const int tid = threadIdx.x;
    const int H = p.H, W = p.W;
    const int b = blockIdx.z / p.F, f = blockIdx.z % p.F;
    const int x0 = blockIdx.x * FT_T, y0 = blockIdx.y * FT_T;
    const size_t N = (size_t)H * W;
    if (TMA) {
        if (tid == 0) {
            mbar_init(&bar, 1);
            mbar_expect_tx(&bar, 2 * 3 * ID_PL * sizeof(float));
            tma_load_4d(xs, &maps.src[f], &bar, x0 - 1 - ID_O, y0 - 1, 0, b);
            tma_load_4d(ys, &maps.tgt, &bar, x0 - 1 - ID_O, y0 - 1, 0, b);
        }
        __syncthreads();                                  // barrier initialised before anyone polls it
        mbar_wait(&bar, 0);
        if (x0 < 1 || y0 < 1 || x0 + FT_T + 1 > W || y0 + FT_T + 1 > H) {
            for (int i = tid; i < ID_N; i += 256) {
                const int r = i / ID_R, c = i - r * ID_R;
                const int ey = y0 - 1 + r, ex = x0 - 1 + c;
                if (ey < 0 || ey >= H || ex < 0 || ex >= W) {
                    const int sr = ext_to_img(ey, H) - (y0 - 1), sc = ext_to_img(ex, W) - (x0 - 1);
                    // a reflected source may itself lie outside the tile when the image is narrower than the halo
                    if (sr >= 0 && sr < ID_R && sc >= 0 && sc < ID_R) {
#pragma unroll
                        for (int ch = 0; ch < 3; ++ch) {
                            xs[ch * ID_PL + r * ID_P + c + ID_O] = xs[ch * ID_PL + sr * ID_P + sc + ID_O];
                            ys[ch * ID_PL + r * ID_P + c + ID_O] = ys[ch * ID_PL + sr * ID_P + sc + ID_O];
                        }
                    }
                }
            }
        }
    } else {
        // tile + 1-px reflect halo: a warp takes a row (index maths once per row / per lane), 6 loads in flight
        const float* sp = p.src[f] + (size_t)b * 3 * N;
        const float* tp = p.target + (size_t)b * 3 * N;
        const int lane = tid & 31, wid = tid >> 5;
        const int ixa = ext_to_img(x0 - 1 + lane, W);
        const int ixb = ext_to_img(x0 - 1 + 32 + (lane & 1), W);          // columns 32, 33 (lanes 0, 1)
        for (int r = wid; r < ID_R; r += 8) {
            const size_t ro = (size_t)ext_to_img(y0 - 1 + r, H) * W;
#pragma unroll
            for (int ch = 0; ch < 3; ++ch) {
                xs[ch * ID_PL + r * ID_P + lane + ID_O] = __ldg(sp + ch * N + ro + ixa);
                ys[ch * ID_PL + r * ID_P + lane + ID_O] = __ldg(tp + ch * N + ro + ixa);
            }
            if (lane < 2) {
#pragma unroll
                for (int ch = 0; ch < 3; ++ch) {
                    xs[ch * ID_PL + r * ID_P + 32 + lane + ID_O] = __ldg(sp + ch * N + ro + ixb);
                    ys[ch * ID_PL + r * ID_P + 32 + lane + ID_O] = __ldg(tp + ch * N + ro + ixb);
                }
            }
        }
    }
    ident_tile_tail(p, xs, ys, tid, b, f, x0, y0, nullptr);
}

// bf16 frames (north_star: "bf16x8 coalesced loads"): the tiles are filled by 128-bit loads of 8 bf16 each -- aligned
// chunks [x0-8, x0+40) of every tile row, zero outside the image like a TMA box, then the same reflection patch --
// and widened to fp32 in shared memory; everything downstream is the fp32 code.  Needs W % 8 == 0 and 16-byte
// aligned frames.  tgt_f32 (B,3,H,W) receives the widened target (what the per-scale kernels read).
__global__ void __launch_bounds__(256, 4)
ident_bf16_kernel(const IdentParams p, const uint16_t* __restrict__ tgt16, const uint16_t* __restrict__ src16,
                  float* __restrict__ tgt_f32) {
    __shared__ __align__(128) float xs[3 * ID_PL];
    __shared__ __align__(128) float ys[3 * ID_PL];
    const int tid = threadIdx.x;
    const int H = p.H, W = p.W;
    const int b = blockIdx.z;
    const int x0 = blockIdx.x * FT_T, y0 = blockIdx.y * FT_T;
    // items: (frame, channel, tile row, chunk of 8 columns); tile column j holds image column x0 - 4 + j
    for (int it = tid; it < 2 * 3 * ID_R * 6; it += 256) {
        const int ck = it % 6, r = (it / 6) % ID_R, ch = (it / (6 * ID_R)) % 3, fr = it / (6 * ID_R * 3);
        const int y = y0 - 1 + r, xc = x0 - 8 + 8 * ck;
        uint4 v = make_uint4(0u, 0u, 0u, 0u);
        if (y >= 0 && y < H && xc >= 0 && xc < W) {
            const uint16_t* base = (fr ? tgt16 : src16) + (((size_t)b * 3 + ch) * H + y) * W + xc;
            v = __ldg(reinterpret_cast<const uint4*>(base));
        }
        float* dst = (fr ? ys : xs) + ch * ID_PL + r * ID_P;
        const unsigned w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const int j = 8 * ck - 4 + e;                 // tile column
            if (j >= 0 && j < ID_P) dst[j] = __uint_as_float((e & 1) ? (w[e >> 1] & 0xffff0000u) : (w[e >> 1] << 16));
        }
    }
    __syncthreads();
    if (x0 < 1 || y0 < 1 || x0 + FT_T + 1 > W || y0 + FT_T + 1 > H) {
        for (int i = tid; i < ID_N; i += 256) {
            const int r = i / ID_R, c = i - r * ID_R;
            const int ey = y0 - 1 + r, ex = x0 - 1 + c;
            if (ey < 0 || ey >= H || ex < 0 || ex >= W) {
                const int sr = ext_to_img(ey, H) - (y0 - 1), sc = ext_to_img(ex, W) - (x0 - 1);
                if (sr >= 0 && sr < ID_R && sc >= 0 && sc < ID_R) {
#pragma unroll
                    for (int ch = 0; ch < 3; ++ch) {
                        xs[ch * ID_PL + r * ID_P + c + ID_O] = xs[ch * ID_PL + sr * ID_P + sc + ID_O];
                        ys[ch * ID_PL + r * ID_P + c + ID_O] = ys[ch * ID_PL + sr * ID_P + sc + ID_O];
                    }
                }
            }
        }
    }
    ident_tile_tail(p, xs, ys, tid, b, 0, x0, y0, tgt_f32);
}

using FastKernel = void (*)(const FastParams, const CUtensorMap);

// every instantiation of photo_fast_kernel, at index TMA + 2 FASTDIV + 4 PK + 8 UP + 16 DH
template <int... I>
std::array<FastKernel, sizeof...(I)> fast_kernel_table(std::integer_sequence<int, I...>) {
    return {photo_fast_kernel<(I & 1) != 0, (I & 2) != 0, (I & 4) != 0, (I & 8) != 0, (I & 16) != 0>...};
}

}  // namespace

namespace dmh {

int photo_fast_tiles(int H, int W) { return ceil_div(W, FT_T) * ceil_div(H, FT_T); }

// Called by dmh_photo_scale and dmh_photo_scale_dh when F == 1 and no pose gradient is requested.
int launch_photo_fast(const float* target, const float* src, const float* T, const float* disp, int disp_h,
                      int disp_w, const float* K, const float* inv_K, const float* ident, const float* noise, int B, int H, int W, float min_depth,
                      float max_depth, int flags, float grad_scale, float* loss_partial, float* grad_disp,
                      uint8_t* sel, float* warped, const FastDhArgs* dh, cudaStream_t st) {
    FastParams p;
    p.target = target; p.src = src; p.T = T; p.K = K;
    p.disp.ptr = disp; p.disp.h = disp_h; p.disp.w = disp_w; p.disp.sh = (float)disp_h / (float)H; p.disp.sw = (float)disp_w / (float)W; p.inv_K = inv_K; p.ident = ident;
    p.noise = noise; p.loss_partial = loss_partial; p.grad_disp = grad_disp; p.sel = sel; p.warped = warped;
    p.B = B; p.H = H; p.W = W; p.flags = flags;
    p.ds = depth_scale(min_depth, max_depth, (flags & DMH_PHOTO_INPUT_IS_DEPTH) != 0);
    p.grad_scale = grad_scale;
    p.hint_reproj = dh ? dh->hint_reproj : nullptr; p.hint_depth = dh ? dh->hint_depth : nullptr;
    p.hint_valid = dh ? dh->hint_valid : nullptr; p.grad_hint = dh ? dh->grad_hint : nullptr;
    p.dh_nblk = dh ? dh->nblk : 0;
    const size_t smem = tile_smem_bytes();
    static const std::array<FastKernel, 32> kernels = fast_kernel_table(std::make_integer_sequence<int, 32>());
    static KernelSetup setup;
    if (setup.sms("dmh_photo_scale(fast)", kernels.data(), (int)kernels.size(), smem) == 0) return DMH_ERR_CUDA;
    dim3 grid(ceil_div(W, FT_T), ceil_div(H, FT_T), B);
    CUtensorMap map;
    const bool use_tma = encode_frames_map(&map, target, B, H, W, FT_TP, FT_R2);
    // division by W-1 / H-1 in the coordinate chain: the 3-instruction form where it is proven bit-exact
    const bool fastdiv = W > 1 && H > 1 && const_div_exact(W - 1, &p.rcw, st) && const_div_exact(H - 1, &p.rch, st);
    const bool packed = (flags & DMH_PHOTO_SRC_PACKED) != 0;
    const bool up = !(disp_h == H && disp_w == W);
    const FastKernel kernel = kernels[use_tma + 2 * fastdiv + 4 * packed + 8 * up + 16 * (dh != nullptr)];
    DMH_LAUNCH(kernel, grid, FT_THREADS, smem, st)(p, map);
    return DMH_OK;
}


int launch_ident_fast(const float* target, const float* const* src_host, int F, int B, int H, int W, int no_ssim,
                      float* out, float* packed, cudaStream_t st) {
    IdentParams p;
    p.target = target;
    p.packed = reinterpret_cast<float4*>(packed);
    for (int f = 0; f < DMH_PHOTO_MAX_FRAMES; ++f) p.src[f] = f < F ? src_host[f] : nullptr;
    p.out = out; p.B = B; p.F = F; p.H = H; p.W = W; p.no_ssim = no_ssim;
    dim3 grid(ceil_div(W, FT_T), ceil_div(H, FT_T), B * F);
    IdentMaps maps;
    memset(&maps, 0, sizeof(maps));
    bool use_tma = encode_frames_map(&maps.tgt, target, B, H, W, ID_P, ID_R);
    for (int f = 0; f < F && use_tma; ++f) use_tma = encode_frames_map(&maps.src[f], src_host[f], B, H, W, ID_P, ID_R);
    if (use_tma) DMH_LAUNCH(ident_fast_kernel<true>, grid, 256, 0, st)(p, maps);
    else DMH_LAUNCH(ident_fast_kernel<false>, grid, 256, 0, st)(p, maps);
    return DMH_OK;
}

// bf16 frames: identity loss + packed fp32 source + fp32 target in one pass over the bf16 inputs
int launch_ident_bf16(const uint16_t* target, const uint16_t* src, int B, int H, int W, int no_ssim, float* out,
                      float* packed, float* tgt_f32, cudaStream_t st) {
    IdentParams p;
    p.target = nullptr;
    p.packed = reinterpret_cast<float4*>(packed);
    for (int f = 0; f < DMH_PHOTO_MAX_FRAMES; ++f) p.src[f] = nullptr;
    p.out = out; p.B = B; p.F = 1; p.H = H; p.W = W; p.no_ssim = no_ssim;
    dim3 grid(ceil_div(W, FT_T), ceil_div(H, FT_T), B);
    DMH_LAUNCH(ident_bf16_kernel, grid, 256, 0, st)(p, target, src, tgt_f32);
    return DMH_OK;
}

}  // namespace dmh
