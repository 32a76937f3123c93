// Stage 1 -- physical patch attack kernels.
//
//   dmh_perspective_fwd/bwd   PhysicalTrans.project / project_w_trans
//                             (physicalTrans.py:130-196): Pad -> torchvision
//                             perspective (bilinear, zeros, align_corners=False)
//                             for the whole batch in one launch.
//   dmh_patch_apply_fwd/bwd   the attack inner loop fused
//                             (phy_obj_atk.py:86-90, phy_obj_atk_l0.py:115-119):
//                             perspective warp of patch+mask, composite
//                             scene*(1-m)+obj*m, anti-aliased bilinear Resize of
//                             scene and mask to 320x1024 -- canvas-resolution
//                             intermediates never touch HBM.
//
// Roofline: HBM.  Algorithmic bytes per attack-batch item (fp32):
//   fwd  read scene 12*375*1242 + write adv 12*320*1024 + mask 4*320*1024 = 10.83 MB
//   bwd  read upstream 12*320*1024 = 3.93 MB (+ patch/mask/grad 3.7 MB once)
//
// torchvision arithmetic restated (installed 0.26; SURVEY.md 8(c)):
//   grid  : _functional_tensor.py:672-698 (_perspective_grid, pixel centres +0.5)
//   sample: grid_sample(bilinear, zeros, align_corners=False) (:545-561)
//   resize: F.interpolate(bilinear, antialias=True, align_corners=False)
//           (ATen UpSample.cuh upsample_antialias::_compute_weights*)
#include <mutex>
#include <vector>

#include "../../include/dmh_b200.h"
#include "dmh_common.cuh"

using namespace dmh;

namespace {

// ---------------------------------------------------------------------------
struct Homography {           // per item, rescaled as torchvision does
    float ax, bx, cx;         // theta1 row 0 / (0.5*ow)
    float ay, by, cy;         // theta1 row 1 / (0.5*oh)
    float g, h;               // theta2
};

__device__ __forceinline__ Homography load_homography(const float* __restrict__ coeffs, int b, int ow, int oh) {
    const float* c = coeffs + b * 8;
    Homography hm;
    const float hx = 0.5f * (float)ow, hy = 0.5f * (float)oh;
    hm.ax = div_rn(__ldg(c + 0), hx); hm.bx = div_rn(__ldg(c + 1), hx); hm.cx = div_rn(__ldg(c + 2), hx);
    hm.ay = div_rn(__ldg(c + 3), hy); hm.by = div_rn(__ldg(c + 4), hy); hm.cy = div_rn(__ldg(c + 5), hy);
    hm.g = __ldg(c + 6); hm.h = __ldg(c + 7);
    return hm;
}

// source coordinates (in canvas pixels) sampled by output canvas pixel (px,py)
__device__ __forceinline__ void perspective_src(const Homography& hm, int px, int py, int ow, int oh, float& ix,
                                                float& iy) {
    const float x = (float)px + 0.5f, y = (float)py + 0.5f;
    float n1 = x * hm.ax; n1 = fmaf(y, hm.bx, n1); n1 = add_rn(n1, hm.cx);
    float n2 = x * hm.ay; n2 = fmaf(y, hm.by, n2); n2 = add_rn(n2, hm.cy);
    float d = x * hm.g;   d = fmaf(y, hm.h, d);    d = add_rn(d, 1.0f);
    const float gx = sub_rn(div_rn(n1, d), 1.0f);
    const float gy = sub_rn(div_rn(n2, d), 1.0f);
    ix = safe_coord(unnormalise_coord(gx, ow, false));
    iy = safe_coord(unnormalise_coord(gy, oh, false));
}

// bilinear taps of the zero-PADDED patch canvas: a tap contributes iff it lies
// inside the canvas (zeros padding) and inside the patch rectangle (pad value 0)
struct PatchTaps {
    int px0, py0;             // north-west tap in PATCH coordinates
    float w[4];               // nw, ne, sw, se (0 where the tap is invalid)
    bool any;
};

__device__ __forceinline__ PatchTaps patch_taps(float ix, float iy, int ow, int oh, int l_pad, int t_pad, int pw,
                                                int ph) {
    const Bilinear bl = bilinear_setup(ix, iy);
    PatchTaps t;
    t.px0 = bl.x0 - l_pad;
    t.py0 = bl.y0 - t_pad;
    const bool x0 = bl.x0 >= 0 && bl.x0 < ow && t.px0 >= 0 && t.px0 < pw;
    const bool x1 = bl.x0 + 1 >= 0 && bl.x0 + 1 < ow && t.px0 + 1 >= 0 && t.px0 + 1 < pw;
    const bool y0 = bl.y0 >= 0 && bl.y0 < oh && t.py0 >= 0 && t.py0 < ph;
    const bool y1 = bl.y0 + 1 >= 0 && bl.y0 + 1 < oh && t.py0 + 1 >= 0 && t.py0 + 1 < ph;
    t.w[0] = (x0 && y0) ? bl.wnw : 0.f;
    t.w[1] = (x1 && y0) ? bl.wne : 0.f;
    t.w[2] = (x0 && y1) ? bl.wsw : 0.f;
    t.w[3] = (x1 && y1) ? bl.wse : 0.f;
    t.any = (x0 || x1) && (y0 || y1);
    return t;
}

__device__ __forceinline__ float sample_plane(const float* __restrict__ p, const PatchTaps& t, int pw) {
    const long long o = (long long)t.py0 * pw + t.px0;
    float acc = 0.f;
    if (t.w[0] != 0.f) acc = fmaf(__ldg(p + o), t.w[0], acc);
    if (t.w[1] != 0.f) acc = fmaf(__ldg(p + o + 1), t.w[1], acc);
    if (t.w[2] != 0.f) acc = fmaf(__ldg(p + o + pw), t.w[2], acc);
    if (t.w[3] != 0.f) acc = fmaf(__ldg(p + o + pw + 1), t.w[3], acc);
    return acc;
}

// --------------------------------------------------------------------------- perspective (canvas resolution)
__global__ void perspective_fwd_kernel(const float* __restrict__ img, const float* __restrict__ coeffs, int C, int ph,
                                       int pw, int oh, int ow, int l_pad, int t_pad, float* __restrict__ out) {
    const int px = blockIdx.x * blockDim.x + threadIdx.x;
    const int py = blockIdx.y * blockDim.y + threadIdx.y;
    if (px >= ow || py >= oh) return;
    const int b = blockIdx.z;
    const Homography hm = load_homography(coeffs, b, ow, oh);
    float ix, iy;
    perspective_src(hm, px, py, ow, oh, ix, iy);
    const PatchTaps t = patch_taps(ix, iy, ow, oh, l_pad, t_pad, pw, ph);
    const size_t N = (size_t)oh * ow;
    for (int c = 0; c < C; ++c)
        out[((size_t)b * C + c) * N + (size_t)py * ow + px] = t.any ? sample_plane(img + (size_t)c * ph * pw, t, pw) : 0.f;
}

__global__ void perspective_bwd_kernel(const float* __restrict__ gout, const float* __restrict__ coeffs, int C, int ph,
                                       int pw, int oh, int ow, int l_pad, int t_pad, float* __restrict__ gimg) {
    const int px = blockIdx.x * blockDim.x + threadIdx.x;
    const int py = blockIdx.y * blockDim.y + threadIdx.y;
    if (px >= ow || py >= oh) return;
    const int b = blockIdx.z;
    const Homography hm = load_homography(coeffs, b, ow, oh);
    float ix, iy;
    perspective_src(hm, px, py, ow, oh, ix, iy);
    const PatchTaps t = patch_taps(ix, iy, ow, oh, l_pad, t_pad, pw, ph);
    if (!t.any) return;
    const size_t N = (size_t)oh * ow;
    const long long o = (long long)t.py0 * pw + t.px0;
    for (int c = 0; c < C; ++c) {
        const float g = gout[((size_t)b * C + c) * N + (size_t)py * ow + px];
        if (g == 0.f) continue;
        float* gp = gimg + (size_t)c * ph * pw;
        if (t.w[0] != 0.f) atomicAdd(gp + o, t.w[0] * g);
        if (t.w[1] != 0.f) atomicAdd(gp + o + 1, t.w[1] * g);
        if (t.w[2] != 0.f) atomicAdd(gp + o + pw, t.w[2] * g);
        if (t.w[3] != 0.f) atomicAdd(gp + o + pw + 1, t.w[3] * g);
    }
}

// --------------------------------------------------------------------------- anti-aliased bilinear weights
#define AA_MAXT 8
struct AaSpan { int lo, n; float w[AA_MAXT]; };

__device__ __forceinline__ float aa_filter(float x) { x = fabsf(x); return x < 1.0f ? 1.0f - x : 0.0f; }

__device__ __forceinline__ AaSpan aa_span(int i, int in_size, float scale) {
    AaSpan s;
    const float support = scale >= 1.0f ? scale : 1.0f;
    const float invscale = scale >= 1.0f ? 1.0f / scale : 1.0f;
    // rounded before use: a bare product here would be contracted into the FMAs of `center - support` and
    // `lo - center`, which moves the weights by up to ~3e-5 and can move the span start (ATen rounds it too)
    const float center = mul_rn(scale, add_rn((float)i, 0.5f));
    s.lo = max((int)(center - support + 0.5f), 0);
    s.n = min((int)(center + support + 0.5f), in_size) - s.lo;
    s.n = min(s.n, AA_MAXT);
    float total = 0.f;
#pragma unroll
    for (int j = 0; j < AA_MAXT; ++j) {
        float w = 0.f;
        if (j < s.n) w = aa_filter(((float)j + ((float)s.lo - center) + 0.5f) * invscale);
        s.w[j] = w;
        total += w;
    }
    if (total != 0.f) {
#pragma unroll
        for (int j = 0; j < AA_MAXT; ++j) s.w[j] = s.w[j] / total;
    }
    return s;
}

// --------------------------------------------------------------------------- fused apply: forward
#define PA_TW 64            // output tile width
#define PA_TH 16            // output tile height
#define PA_THREADS 256

// NT: compile-time bound on the anti-aliasing taps per axis: a span holds at most ceil(2 * support) pixels, i.e. 3
// when both scale factors are < 1.5 (the 1242x375 -> 1024x320 case), else AA_MAXT.  Fixed trip counts, fully
// unrolled; taps beyond a span carry weight 0 and are clamped onto the tile.
template <int NT>
__global__ void __launch_bounds__(PA_THREADS)
patch_apply_fwd_kernel(const float* __restrict__ patch, const float* __restrict__ pmask,
                       const float* __restrict__ scenes, const float* __restrict__ coeffs,
                       const int* __restrict__ bbox, int ph, int pw, int ih, int iw, int oh, int ow, int l_pad,
                       int t_pad, float sy, float sx, int cw_max, int ch_max, float* __restrict__ adv,
                       float* __restrict__ mask_out) {
    extern __shared__ float smem[];
    float* comp = smem;                                   // [4][ch_max][cw_max] : 3 colour planes + mask
    __shared__ int x_lo[PA_TW], x_n[PA_TW], y_lo[PA_TH], y_n[PA_TH];
    __shared__ float x_w[PA_TW][AA_MAXT], y_w[PA_TH][AA_MAXT];
    const int tid = threadIdx.x;
    const int b = blockIdx.z;
    const int ox0 = blockIdx.x * PA_TW, oy0 = blockIdx.y * PA_TH;
    if (tid < PA_TW) {
        const int ox = min(ox0 + tid, ow - 1);
        const AaSpan s = aa_span(ox, iw, sx);
        x_lo[tid] = s.lo; x_n[tid] = s.n;
#pragma unroll
        for (int j = 0; j < AA_MAXT; ++j) x_w[tid][j] = s.w[j];
    } else if (tid < PA_TW + PA_TH) {
        const int k = tid - PA_TW;
        const int oy = min(oy0 + k, oh - 1);
        const AaSpan s = aa_span(oy, ih, sy);
        y_lo[k] = s.lo; y_n[k] = s.n;
#pragma unroll
        for (int j = 0; j < AA_MAXT; ++j) y_w[k][j] = s.w[j];
    }
    __syncthreads();
    const int cx0 = x_lo[0], cy0 = y_lo[0];
    const int last_x = min(PA_TW, ow - ox0) - 1, last_y = min(PA_TH, oh - oy0) - 1;
    const int cw = min(x_lo[last_x] + x_n[last_x] - cx0, cw_max);
    const int ch = min(y_lo[last_y] + y_n[last_y] - cy0, ch_max);
    const Homography hm = load_homography(coeffs, b, iw, ih);
    const size_t IN = (size_t)ih * iw;
    const float* sc = scenes + (size_t)b * 3 * IN;
    const size_t plane = (size_t)ch_max * cw_max;
    const size_t PN = (size_t)ph * pw;
    // canvas pixels outside the item's bounding box cannot sample the patch: skip the perspective maths there
    bool tile_hits = true;
    int bx0 = 0, by0 = 0, bx1 = iw - 1, by1 = ih - 1;
    if (bbox) {
        bx0 = __ldg(bbox + b * 4); by0 = __ldg(bbox + b * 4 + 1); bx1 = __ldg(bbox + b * 4 + 2); by1 = __ldg(bbox + b * 4 + 3);
        tile_hits = !(cx0 > bx1 || cx0 + cw - 1 < bx0 || cy0 > by1 || cy0 + ch - 1 < by0);
    }
    // a warp takes a tile row, its lanes the columns (no index division); a tile narrower than NT columns is
    // zero-filled up to NT so that the fixed-count loops below never read uninitialised shared memory
    const int lane = tid & 31, wid = tid >> 5;
    const int cwz = max(cw, NT);
    for (int r = wid; r < ch; r += PA_THREADS / 32) {
        const int cy = cy0 + r;
        const bool row_in = true;
        for (int c0 = 0; c0 < cwz; c0 += 96) {
            float sv[3][3];
            bool in[3];
#pragma unroll
            for (int u = 0; u < 3; ++u) {                 // up to 9 scene loads in flight per lane
                const int c = c0 + 32 * u + lane;
                in[u] = row_in && c < cw;
                const size_t so = (size_t)cy * iw + cx0 + c;
#pragma unroll
                for (int k = 0; k < 3; ++k) sv[u][k] = in[u] ? __ldg(sc + k * IN + so) : 0.f;
            }
#pragma unroll
            for (int u = 0; u < 3; ++u) {
                const int c = c0 + 32 * u + lane;
                if (c >= cwz) continue;
                const int cx = cx0 + c;
                float m = 0.f, o0 = 0.f, o1 = 0.f, o2 = 0.f;
                if (in[u] && tile_hits && cx >= bx0 && cx <= bx1 && cy >= by0 && cy <= by1) {
                    float ix, iy;
                    perspective_src(hm, cx, cy, iw, ih, ix, iy);
                    const PatchTaps t = patch_taps(ix, iy, iw, ih, l_pad, t_pad, pw, ph);
                    if (t.any) {
                        m = sample_plane(pmask, t, pw);
                        o0 = sample_plane(patch, t, pw);
                        o1 = sample_plane(patch + PN, t, pw);
                        o2 = sample_plane(patch + 2 * PN, t, pw);
                    }
                }
                const float om = sub_rn(1.0f, m);
                const size_t o = (size_t)r * cw_max + c;
                comp[o] = add_rn(mul_rn(sv[u][0], om), mul_rn(o0, m));
                comp[plane + o] = add_rn(mul_rn(sv[u][1], om), mul_rn(o1, m));
                comp[2 * plane + o] = add_rn(mul_rn(sv[u][2], om), mul_rn(o2, m));
                comp[3 * plane + o] = m;
            }
        }
    }
    __syncthreads();
    const int tx = tid % PA_TW;
    const int ox = ox0 + tx;
    if (ox >= ow) return;
    const int xl = max(min(x_lo[tx] - cx0, cw - NT), 0);  // (the span itself never exceeds the tile)
    const int xshift = (x_lo[tx] - cx0) - xl;             // > 0 only if the clamp moved the window: shift the weights
    float wxr[NT];
#pragma unroll
    for (int i = 0; i < NT; ++i) wxr[i] = (i - xshift >= 0 && i - xshift < AA_MAXT) ? x_w[tx][i - xshift] : 0.f;
    const size_t ON = (size_t)oh * ow;
#pragma unroll
    for (int k = 0; k < PA_TH / (PA_THREADS / PA_TW); ++k) {
        const int ty = tid / PA_TW + k * (PA_THREADS / PA_TW);
        const int oy = oy0 + ty;
        if (oy >= oh) continue;
        const int yl = y_lo[ty] - cy0;
        float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int j = 0; j < NT; ++j) {
            const float wy = y_w[ty][j];                  // 0 beyond the span
            const float* row = comp + (size_t)min(yl + j, ch - 1) * cw_max + xl;
            float h[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
            for (int i = 0; i < NT; ++i) {
                const float wx = wxr[i];
#pragma unroll
                for (int p = 0; p < 4; ++p) h[p] = fmaf(row[p * plane + i], wx, h[p]);
            }
#pragma unroll
            for (int p = 0; p < 4; ++p) acc[p] = fmaf(h[p], wy, acc[p]);
        }
        const size_t oo = (size_t)oy * ow + ox;
        adv[((size_t)b * 3 + 0) * ON + oo] = acc[0];
        adv[((size_t)b * 3 + 1) * ON + oo] = acc[1];
        adv[((size_t)b * 3 + 2) * ON + oo] = acc[2];
        if (mask_out) mask_out[(size_t)b * ON + oo] = acc[3];
    }
}

// --------------------------------------------------------------------------- fused apply: forward, 3-tap windows
// The hot instantiation (both scale factors < 1.5, e.g. 1242x375 -> 1024x320): an anti-aliasing span holds at
// most 3 pixels per axis.  Same arithmetic as the general kernel above, re-organised for the issue slots:
//   * compile-time tile pitch / plane stride: every shared-memory access is base + immediate;
//   * tiles that cannot see the patch (the placement bounding box misses them: ~85 % of the tiles) copy the
//     scene straight into the tile -- scene*(1-0) + 0*0 is the scene bit for bit -- skip the mask plane and
//     write mask 0;
//   * only the 3 live weights per axis are computed (ATen's normalisation included).
struct AaSpan3 { int lo; float w[3]; };
// first input index of the anti-aliasing span of output index i; explicitly rounded op by op so that every caller
// (the per-thread tile geometry and the weight table) gets the same integer
__device__ __forceinline__ int aa_span_lo(int i, float scale) {
    const float support = scale >= 1.0f ? scale : 1.0f;
    const float center = mul_rn(scale, add_rn((float)i, 0.5f));
    return max((int)add_rn(sub_rn(center, support), 0.5f), 0);
}
__device__ __forceinline__ AaSpan3 aa_span3(int i, int in_size, float scale) {
    AaSpan3 s;
    const float support = scale >= 1.0f ? scale : 1.0f;
    const float invscale = scale >= 1.0f ? 1.0f / scale : 1.0f;
    const float center = mul_rn(scale, add_rn((float)i, 0.5f));
    s.lo = aa_span_lo(i, scale);
    const int n = min(min((int)(center + support + 0.5f), in_size) - s.lo, 3);
    float total = 0.f;
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        float w = 0.f;
        if (j < n) w = aa_filter(((float)j + ((float)s.lo - center) + 0.5f) * invscale);
        s.w[j] = w;
        total += w;
    }
    if (total != 0.f) {
#pragma unroll
        for (int j = 0; j < 3; ++j) s.w[j] = s.w[j] / total;
    }
    return s;
}

// The anti-aliasing spans of every output column and row, evaluated ONCE per (sizes, device) instead of by every CTA:
// tab[ox] (ox < ow) and tab[ow + oy] = (span start as an int bit pattern, w0, w1, w2) = aa_span3 of that index.
__global__ void aa_table_kernel(int ih, int iw, int oh, int ow, float sy, float sx, float4* __restrict__ tab) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= ow + oh) return;
    const AaSpan3 s = i < ow ? aa_span3(i, iw, sx) : aa_span3(i - ow, ih, sy);
    tab[i] = make_float4(__int_as_float(s.lo), s.w[0], s.w[1], s.w[2]);
}

// TAB: the weight tables of the tile are read from `aa_tab` (aa_table_kernel) instead of computed -- the same values
// (Staging two adjacent scene columns per lane with 64-bit loads / stores from an even tile start was built and measured
// too: 112 us against 99 us -- the wider accesses leave a third of the lanes idle in the second column group; removed.)
template <int PITCH, int ROWS, bool TAB = false>
__global__ void __launch_bounds__(PA_THREADS, (PITCH <= 84 ? 4 : 3))
patch_apply_fwd3_kernel(const float* __restrict__ patch, const float* __restrict__ pmask,
                        const float* __restrict__ scenes, const float* __restrict__ coeffs,
                        const int* __restrict__ bbox, int ph, int pw, int ih, int iw, int oh, int ow, int l_pad,
                        int t_pad, float sy, float sx, float* __restrict__ adv, float* __restrict__ mask_out,
                        const float4* __restrict__ aa_tab) {
    extern __shared__ float smem[];
    constexpr int PLANE = PITCH * ROWS;
    constexpr int NCU = (PITCH + 31) / 32, NRU = (ROWS + 7) / 8;
    float* comp = smem;                                   // [4][ROWS][PITCH] : 3 colour planes + mask
    __shared__ int x_lo[PA_TW], y_lo[PA_TH];
    __shared__ float x_w[PA_TW][3];
    // vertical weights of a thread's 4 CONSECUTIVE output rows against the (<= 8) input rows their spans cover:
    // wy4[q][i] = weights of input row y_lo[4q] + i in output rows 4q .. 4q+3 (0 outside a row's span)
    __shared__ float4 wy4[PA_TH / 4][8];
    const int tid = threadIdx.x;
    const int b = blockIdx.z;
    const int ox0 = blockIdx.x * PA_TW, oy0 = blockIdx.y * PA_TH;
    // tile geometry from the span starts alone (every thread, no shared memory): the scene loads are issued
    // BEFORE the weights are tabulated, so their latency overlaps that phase
    const int last_x = min(PA_TW, ow - ox0) - 1, last_y = min(PA_TH, oh - oy0) - 1;
    const int cx0 = aa_span_lo(ox0, sx), cy0 = aa_span_lo(oy0, sy);
    const int cw = min(min(aa_span_lo(ox0 + last_x, sx) + 3, iw) - cx0, PITCH);
    const int ch = min(min(aa_span_lo(oy0 + last_y, sy) + 3, ih) - cy0, ROWS);
    const int IN = ih * iw;
    const float* sc = scenes + (size_t)b * 3 * IN + cx0;
    // a warp takes tile rows wid, wid+8, ..., its lanes the columns lane, lane+32, ...: all loads in flight at once
    const int lane = tid & 31, wid = tid >> 5;
    float sv[NRU][NCU][3];
#pragma unroll
    for (int ru = 0; ru < NRU; ++ru) {
        const int r = wid + 8 * ru;
        const float* srow = sc + (cy0 + min(r, ch - 1)) * iw;
#pragma unroll
        for (int u = 0; u < NCU; ++u) {
            const int c = 32 * u + lane;
#pragma unroll
            for (int k = 0; k < 3; ++k) sv[ru][u][k] = (r < ch && c < cw) ? __ldg(srow + k * IN + c) : 0.f;
        }
    }
    if (TAB) {
        if (tid < PA_TW) {
            const float4 t = __ldg(aa_tab + min(ox0 + tid, ow - 1));
            x_lo[tid] = __float_as_int(t.x);
            x_w[tid][0] = t.y; x_w[tid][1] = t.z; x_w[tid][2] = t.w;
        } else if (tid < PA_TW + PA_TH) {
            const int k = tid - PA_TW;
            y_lo[k] = __float_as_int(__ldg(aa_tab + ow + min(oy0 + k, oh - 1)).x);
        } else if (tid < PA_TW + PA_TH + 32 * (PA_TH / 4)) {
            const int t = tid - (PA_TW + PA_TH);
            const int q = t >> 5, i = (t & 31) >> 2, k = t & 3;
            const float4 e = __ldg(aa_tab + ow + min(oy0 + 4 * q + k, oh - 1));
            const int lo0 = __float_as_int(__ldg(aa_tab + ow + min(oy0 + 4 * q, oh - 1)).x);
            const int d = i - (__float_as_int(e.x) - lo0);
            reinterpret_cast<float*>(&wy4[q][i])[k] = d == 0 ? e.y : (d == 1 ? e.z : (d == 2 ? e.w : 0.0f));
        }
    } else if (tid < PA_TW) {
        const AaSpan3 s = aa_span3(min(ox0 + tid, ow - 1), iw, sx);
        x_lo[tid] = s.lo;
#pragma unroll
        for (int j = 0; j < 3; ++j) x_w[tid][j] = s.w[j];
    } else if (tid < PA_TW + PA_TH) {
        const int k = tid - PA_TW;
        y_lo[k] = aa_span_lo(min(oy0 + k, oh - 1), sy);
    } else if (tid < PA_TW + PA_TH + 32 * (PA_TH / 4)) {
        const int t = tid - (PA_TW + PA_TH);
        const int q = t >> 5, i = (t & 31) >> 2, k = t & 3;
        const AaSpan3 s = aa_span3(min(oy0 + 4 * q + k, oh - 1), ih, sy);
        const int d = i - (s.lo - aa_span_lo(min(oy0 + 4 * q, oh - 1), sy));
        reinterpret_cast<float*>(&wy4[q][i])[k] = (d >= 0 && d < 3) ? s.w[d] : 0.0f;
    }
    bool tile_hits = true;
    int bx0 = 0, by0 = 0, bx1 = iw - 1, by1 = ih - 1;
    if (bbox) {
        bx0 = __ldg(bbox + b * 4); by0 = __ldg(bbox + b * 4 + 1); bx1 = __ldg(bbox + b * 4 + 2); by1 = __ldg(bbox + b * 4 + 3);
        tile_hits = !(cx0 > bx1 || cx0 + cw - 1 < bx0 || cy0 > by1 || cy0 + ch - 1 < by0);
    }
    // a tile narrower than 3 columns is zero-filled up to 3 so that the fixed-count loops below never read
    // uninitialised shared memory
    const int cwz = max(cw, 3);
    if (!tile_hits) {
#pragma unroll
        for (int ru = 0; ru < NRU; ++ru) {
            const int r = wid + 8 * ru;
            if (r >= ch) continue;
            float* crow = comp + r * PITCH;
#pragma unroll
            for (int u = 0; u < NCU; ++u) {
                const int c = 32 * u + lane;
                if (c < cwz) {
#pragma unroll
                    for (int k = 0; k < 3; ++k) crow[k * PLANE + c] = sv[ru][u][k];
                }
            }
        }
    } else {
        const Homography hm = load_homography(coeffs, b, iw, ih);
        const int PN = ph * pw;
#pragma unroll
        for (int ru = 0; ru < NRU; ++ru) {
            const int r = wid + 8 * ru;
            if (r >= ch) continue;
            const int cy = cy0 + r;
            float* crow = comp + r * PITCH;
#pragma unroll
            for (int u = 0; u < NCU; ++u) {
                const int c = 32 * u + lane;
                if (c >= cwz) continue;
                const int cx = cx0 + c;
                float m = 0.f, o0 = 0.f, o1 = 0.f, o2 = 0.f;
                if (c < cw && cx >= bx0 && cx <= bx1 && cy >= by0 && cy <= by1) {
                    float ix, iy;
                    perspective_src(hm, cx, cy, iw, ih, ix, iy);
                    const PatchTaps t = patch_taps(ix, iy, iw, ih, l_pad, t_pad, pw, ph);
                    if (t.any) {
                        m = sample_plane(pmask, t, pw);
                        o0 = sample_plane(patch, t, pw);
                        o1 = sample_plane(patch + PN, t, pw);
                        o2 = sample_plane(patch + 2 * PN, t, pw);
                    }
                }
                const float om = sub_rn(1.0f, m);
                crow[c] = add_rn(mul_rn(sv[ru][u][0], om), mul_rn(o0, m));
                crow[PLANE + c] = add_rn(mul_rn(sv[ru][u][1], om), mul_rn(o1, m));
                crow[2 * PLANE + c] = add_rn(mul_rn(sv[ru][u][2], om), mul_rn(o2, m));
                crow[3 * PLANE + c] = m;
            }
        }
    }
    __syncthreads();
    const int tx = tid % PA_TW;
    const int ox = ox0 + tx;
    if (ox >= ow) return;
    const int xl = max(min(x_lo[tx] - cx0, cw - 3), 0);   // (the span itself never exceeds the tile)
    const int xshift = (x_lo[tx] - cx0) - xl;             // > 0 only if the clamp moved the window: shift the weights
    const float xw0 = x_w[tx][0], xw1 = x_w[tx][1], xw2 = x_w[tx][2];
    const float wx0 = xshift == 0 ? xw0 : 0.f;
    const float wx1 = xshift == 0 ? xw1 : (xshift == 1 ? xw0 : 0.f);
    const float wx2 = xshift == 0 ? xw2 : (xshift == 1 ? xw1 : (xshift == 2 ? xw0 : 0.f));
    const int ON = oh * ow;
    // A thread owns 4 consecutive output rows of its column: the horizontal 3-tap sum of an input row is formed once
    // and feeds every output row whose span holds it (7 input rows instead of 12 at 375 -> 320: 70 shared-memory
    // loads per thread instead of 120 -- the kernel was shared-memory bound).  Same products, same order of the
    // non-zero terms, i.e. the same bits as one output at a time.
    const int q = tid / PA_TW;
    const int yb = y_lo[4 * q] - cy0;                                       // first input row (tile coordinates)
    const int last = min(4 * q + 3, last_y);
    const int nrows = min(y_lo[last] - cy0 - yb + 3, 8);                    // warp-uniform (a warp shares q)
    float* aout = adv + (size_t)b * 3 * ON + (oy0 + 4 * q) * ow + ox;
    float* mout = mask_out ? mask_out + (size_t)b * ON + (oy0 + 4 * q) * ow + ox : nullptr;
    const float* cbase = comp + xl;
    if (tile_hits) {
        float acc[4][4];
#pragma unroll
        for (int k = 0; k < 4; ++k)
#pragma unroll
            for (int p = 0; p < 4; ++p) acc[k][p] = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            if (i < nrows) {
                const float4 w = wy4[q][i];
                const float* row = cbase + min(yb + i, ch - 1) * PITCH;
#pragma unroll
                for (int p = 0; p < 4; ++p) {
                    float h = row[p * PLANE] * wx0;
                    h = fmaf(row[p * PLANE + 1], wx1, h);
                    h = fmaf(row[p * PLANE + 2], wx2, h);
                    acc[0][p] = fmaf(h, w.x, acc[0][p]);
                    acc[1][p] = fmaf(h, w.y, acc[1][p]);
                    acc[2][p] = fmaf(h, w.z, acc[2][p]);
                    acc[3][p] = fmaf(h, w.w, acc[3][p]);
                }
            }
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if (oy0 + 4 * q + k >= oh) break;
            aout[k * ow] = acc[k][0];
            aout[ON + k * ow] = acc[k][1];
            aout[2 * ON + k * ow] = acc[k][2];
            if (mout) mout[k * ow] = acc[k][3];
        }
    } else {
        float acc[4][3];
#pragma unroll
        for (int k = 0; k < 4; ++k)
#pragma unroll
            for (int p = 0; p < 3; ++p) acc[k][p] = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            if (i < nrows) {
                const float4 w = wy4[q][i];
                const float* row = cbase + min(yb + i, ch - 1) * PITCH;
#pragma unroll
                for (int p = 0; p < 3; ++p) {
                    float h = row[p * PLANE] * wx0;
                    h = fmaf(row[p * PLANE + 1], wx1, h);
                    h = fmaf(row[p * PLANE + 2], wx2, h);
                    acc[0][p] = fmaf(h, w.x, acc[0][p]);
                    acc[1][p] = fmaf(h, w.y, acc[1][p]);
                    acc[2][p] = fmaf(h, w.z, acc[2][p]);
                    acc[3][p] = fmaf(h, w.w, acc[3][p]);
                }
            }
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if (oy0 + 4 * q + k >= oh) break;
            aout[k * ow] = acc[k][0];
            aout[ON + k * ow] = acc[k][1];
            aout[2 * ON + k * ow] = acc[k][2];
            if (mout) mout[k * ow] = 0.f;
        }
    }
}

// --------------------------------------------------------------------------- fused apply: backward (to the patch)
// One thread per canvas pixel: exits unless the pixel samples the patch; gathers
// the transposed anti-aliased resize of the upstream gradient, multiplies by the
// warped mask, scatters to the <=4 patch taps (RED.ADD; all batch items share
// the one patch, which is why this is a scatter).
__device__ __forceinline__ float aa_weight_of(int o, int in_size, float scale, int ci) {
    // weight with which output index o reads input index ci (0 if outside its span)
    const float support = scale >= 1.0f ? scale : 1.0f;
    const float invscale = scale >= 1.0f ? 1.0f / scale : 1.0f;
    const float center = mul_rn(scale, add_rn((float)o, 0.5f));     // rounded as in aa_span / aa_span3
    const int lo = max((int)(center - support + 0.5f), 0);
    int n = min((int)(center + support + 0.5f), in_size) - lo;
    n = min(n, AA_MAXT);
    if (ci < lo || ci >= lo + n) return 0.f;
    float total = 0.f, mine = 0.f;
    for (int j = 0; j < n; ++j) {
        const float w = aa_filter(((float)j + ((float)lo - center) + 0.5f) * invscale);
        total += w;
        if (lo + j == ci) mine = w;
    }
    return total != 0.f ? mine / total : mine;
}

// weight with which output index o reads input index ci, from the span table (aa_table_kernel: 3-tap spans, both
// scale factors < 1.5): the value aa_weight_of computes, bit for bit
__device__ __forceinline__ float aa_weight_tab(const float4* __restrict__ tab, int o, int ci) {
    const float4 e = __ldg(tab + o);
    const int d = ci - __float_as_int(e.x);
    return d == 0 ? e.y : (d == 1 ? e.z : (d == 2 ? e.w : 0.f));
}

// TAB: resize weights from the span table (aa_tab: columns, then rows) instead of ~12 evaluations of aa_weight_of per
// pixel -- three quarters of this kernel's instructions
template <bool TAB>
__global__ void __launch_bounds__(256)
patch_apply_bwd_kernel(const float* __restrict__ gadv, const float* __restrict__ pmask,
                       const float* __restrict__ coeffs, const int* __restrict__ bbox, int ph, int pw, int ih, int iw,
                       int oh, int ow, int l_pad, int t_pad, float sy, float sx, float* __restrict__ gpatch,
                       const float4* __restrict__ aa_tab) {
    const int b = blockIdx.z;
    int cx = blockIdx.x * blockDim.x + threadIdx.x;
    int cy = blockIdx.y * blockDim.y + threadIdx.y;
    if (bbox) {                                           // grid covers the largest bounding box of the batch
        cx += __ldg(bbox + b * 4);
        cy += __ldg(bbox + b * 4 + 1);
        if (cx > __ldg(bbox + b * 4 + 2) || cy > __ldg(bbox + b * 4 + 3)) return;
    }
    if (cx >= iw || cy >= ih) return;
    const Homography hm = load_homography(coeffs, b, iw, ih);
    float ix, iy;
    perspective_src(hm, cx, cy, iw, ih, ix, iy);
    const PatchTaps t = patch_taps(ix, iy, iw, ih, l_pad, t_pad, pw, ph);
    if (!t.any) return;
    const float m = sample_plane(pmask, t, pw);
    if (m == 0.f) return;
    // outputs whose anti-aliasing window covers this canvas pixel
    const float supx = sx >= 1.0f ? sx : 1.0f, supy = sy >= 1.0f ? sy : 1.0f;
    const int ox_a = max(0, (int)floorf(((float)cx - supx - 0.5f) / sx) - 1);
    const int ox_b = min(ow - 1, (int)ceilf(((float)cx + supx + 0.5f) / sx) + 1);
    const int oy_a = max(0, (int)floorf(((float)cy - supy - 0.5f) / sy) - 1);
    const int oy_b = min(oh - 1, (int)ceilf(((float)cy + supy + 0.5f) / sy) + 1);
    const size_t ON = (size_t)oh * ow;
    const float* g = gadv + (size_t)b * 3 * ON;
    float gc[3] = {0.f, 0.f, 0.f};
    // the column weights do not depend on the row: evaluate them once (the candidate window holds at most
    // 2*support/scale + 4 <= 8 outputs for scale factors in [1, 3))
    constexpr int MAXO = 8;
    float wxv[MAXO];
#pragma unroll
    for (int i = 0; i < MAXO; ++i)
        wxv[i] = (ox_a + i <= ox_b) ? (TAB ? aa_weight_tab(aa_tab, ox_a + i, cx) : aa_weight_of(ox_a + i, iw, sx, cx)) : 0.f;
    for (int oy = oy_a; oy <= oy_b; ++oy) {
        const float wy = TAB ? aa_weight_tab(aa_tab + ow, oy, cy) : aa_weight_of(oy, ih, sy, cy);
        if (wy == 0.f) continue;
        const float* grow = g + (size_t)oy * ow + ox_a;
#pragma unroll
        for (int i = 0; i < MAXO; ++i) {
            const float w = wy * wxv[i];
            if (w == 0.f) continue;
            gc[0] = fmaf(w, __ldg(grow + i), gc[0]);
            gc[1] = fmaf(w, __ldg(grow + ON + i), gc[1]);
            gc[2] = fmaf(w, __ldg(grow + 2 * ON + i), gc[2]);
        }
    }
    // windows wider than MAXO (up-scaling by more than ~1.3x): the remaining columns, weight by weight
    for (int ox = ox_a + MAXO; ox <= ox_b; ++ox) {
        const float wx = TAB ? aa_weight_tab(aa_tab, ox, cx) : aa_weight_of(ox, iw, sx, cx);
        if (wx == 0.f) continue;
        for (int oy = oy_a; oy <= oy_b; ++oy) {
            const float w = (TAB ? aa_weight_tab(aa_tab + ow, oy, cy) : aa_weight_of(oy, ih, sy, cy)) * wx;
            if (w == 0.f) continue;
            const size_t oo = (size_t)oy * ow + ox;
            gc[0] = fmaf(w, __ldg(g + oo), gc[0]);
            gc[1] = fmaf(w, __ldg(g + ON + oo), gc[1]);
            gc[2] = fmaf(w, __ldg(g + 2 * ON + oo), gc[2]);
        }
    }
    const size_t PN = (size_t)ph * pw;
    const long long o = (long long)t.py0 * pw + t.px0;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const float gv = gc[c] * m;                       // d comp / d obj_warp = m
        if (gv == 0.f) continue;
        float* gp = gpatch + c * PN;
        if (t.w[0] != 0.f) atomicAdd(gp + o, t.w[0] * gv);
        if (t.w[1] != 0.f) atomicAdd(gp + o + 1, t.w[1] * gv);
        if (t.w[2] != 0.f) atomicAdd(gp + o + pw, t.w[2] * gv);
        if (t.w[3] != 0.f) atomicAdd(gp + o + pw + 1, t.w[3] * gv);
    }
}

// --------------------------------------------------------------------------- loader-side composite, 8-bit (next-2)
// MonoDataset.prep_adv_data (mono_dataset.py:193-251) for one frame of every item: to_tensor(scene), the perspective
// warp of up to two patches that share one placement and one mask (the adversarial and the benign patch on frame 0),
// optional mirror of the warped patch / mask, scene*(1-m) + obj*m, to_pilimage (`.mul(255).byte()`).  The warped
// canvases (B,3,375,1242 fp32 each) never exist: a pixel samples the patch itself, with exactly the arithmetic of
// perspective_fwd_kernel.  One thread per canvas pixel; HBM-bound by bytes (3 in, 3..7 out per pixel).
__device__ __forceinline__ uint8_t to_byte(float v) {
    const float q = mul_rn(v, 255.0f);
    return (uint8_t)min(max((int)q, 0), 255);             // `.byte()` truncates; images in [0,1] never saturate
}

// PX pixels per thread (2 when rows are 2-byte aligned: 16-bit loads / stores halve the byte-wide memory instructions)
template <int PX>
__global__ void __launch_bounds__(256)
compose_patch_u8_kernel(const uint8_t* __restrict__ scene, const float* __restrict__ patch_a,
                        const float* __restrict__ patch_b, const float* __restrict__ pmask,
                        const float* __restrict__ coeffs, const int* __restrict__ bbox, const int* __restrict__ flip,
                        const int* __restrict__ active, int ph, int pw, int H, int W, int l_pad, int t_pad,
                        uint8_t* __restrict__ out_a,
                        uint8_t* __restrict__ out_b, uint8_t* __restrict__ mask_out) {
    const int x0 = (blockIdx.x * blockDim.x + threadIdx.x) * PX;
    const int y = blockIdx.y, b = blockIdx.z;
    if (x0 >= W) return;
    const bool fl = flip && __ldg(flip + b) != 0;
    // items without synthesis (half_no_synthesis, mono_dataset.py:321-328) keep the raw frame: with m = 0 the
    // composite is to_pilimage(to_tensor(scene)), which returns every byte unchanged (k/255*255 == k in fp32)
    const bool on = !(active && __ldg(active + b) == 0);
    int bx0 = 0, by0 = 0, bx1 = W - 1, by1 = H - 1;
    if (on && bbox) {
        const int4 bb = __ldg(reinterpret_cast<const int4*>(bbox) + b);
        bx0 = bb.x; by0 = bb.y; bx1 = bb.z; by1 = bb.w;
    }
    float m[PX], oa[PX][3], ob[PX][3];
#pragma unroll
    for (int i = 0; i < PX; ++i) {
        m[i] = 0.f;
#pragma unroll
        for (int c = 0; c < 3; ++c) oa[i][c] = ob[i][c] = 0.f;
        const int x = x0 + i;
        const int xs = fl ? W - 1 - x : x;                // torch.flip(warped, [3])
        if (on && x < W && xs >= bx0 && xs <= bx1 && y >= by0 && y <= by1) {
            const Homography hm = load_homography(coeffs, b, W, H);
            float ix, iy;
            perspective_src(hm, xs, y, W, H, ix, iy);
            const PatchTaps t = patch_taps(ix, iy, W, H, l_pad, t_pad, pw, ph);
            if (t.any) {
                const int PN = ph * pw;
                m[i] = sample_plane(pmask, t, pw);
#pragma unroll
                for (int c = 0; c < 3; ++c) {
                    oa[i][c] = sample_plane(patch_a + c * PN, t, pw);
                    if (patch_b) ob[i][c] = sample_plane(patch_b + c * PN, t, pw);
                }
            }
        }
    }
    const size_t N = (size_t)H * W, po = (size_t)y * W + x0;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const size_t o = ((size_t)b * 3 + c) * N + po;
        unsigned sv;
        if (PX == 2) sv = __ldg(reinterpret_cast<const unsigned short*>(scene + o));       // (W even: x0 + 1 < W)
        else sv = __ldg(scene + o);
        unsigned ra = 0u, rb = 0u;
#pragma unroll
        for (int i = 0; i < PX; ++i) {
            const float s = mul_rn(div_rn((float)((sv >> (8 * i)) & 0xffu), 255.0f), sub_rn(1.0f, m[i]));
            ra |= (unsigned)to_byte(add_rn(s, mul_rn(oa[i][c], m[i]))) << (8 * i);
            if (out_b) rb |= (unsigned)to_byte(add_rn(s, mul_rn(ob[i][c], m[i]))) << (8 * i);
        }
        if (PX == 2) {
            *reinterpret_cast<unsigned short*>(out_a + o) = (unsigned short)ra;
            if (out_b) *reinterpret_cast<unsigned short*>(out_b + o) = (unsigned short)rb;
        } else {
            out_a[o] = (uint8_t)ra;
            if (out_b) out_b[o] = (uint8_t)rb;
        }
    }
    if (mask_out) {
        if (PX == 2)
            *reinterpret_cast<unsigned short*>(mask_out + (size_t)b * N + po) =
                (unsigned short)((unsigned)to_byte(m[0]) | ((unsigned)to_byte(m[PX - 1]) << 8));
        else
            mask_out[(size_t)b * N + po] = to_byte(m[0]);
    }
}

}  // namespace

extern "C" {

int dmh_compose_patch_u8(const uint8_t* scene, const float* patch_a, const float* patch_b, const float* patch_mask,
                         const float* coeffs, const int* bbox, const int* flip, const int* active, int B, int ph, int pw,
                         int H, int W, uint8_t* out_a, uint8_t* out_b, uint8_t* mask_out, dmh_stream_t stream) {
    DMH_REQUIRE(scene && patch_a && patch_mask && coeffs && out_a, "dmh_compose_patch_u8: null pointer");
    DMH_REQUIRE((patch_b != nullptr) == (out_b != nullptr), "dmh_compose_patch_u8: patch_b and out_b go together");
    DMH_REQUIRE(B > 0 && B <= 65535 && ph > 0 && pw > 0 && H >= ph && H <= 65535 && W >= pw,
                "dmh_compose_patch_u8: bad shape (patch %dx%d, canvas %dx%d)", ph, pw, H, W);
    const int l_pad = (W - pw) / 2, t_pad = (H - ph) / 2;
    DMH_REQUIRE(!bbox || ((uintptr_t)bbox & 15) == 0, "dmh_compose_patch_u8: bbox must be 16-byte aligned");
    const uintptr_t al = (uintptr_t)scene | (uintptr_t)out_a | (uintptr_t)out_b | (uintptr_t)mask_out;
    if (W % 2 == 0 && (al & 1) == 0) {
        dim3 grid(ceil_div(W, 512), H, B);
        DMH_LAUNCH(compose_patch_u8_kernel<2>, grid, 256, 0, (cudaStream_t)stream)(
            scene, patch_a, patch_b, patch_mask, coeffs, bbox, flip, active, ph, pw, H, W, l_pad, t_pad, out_a, out_b, mask_out);
    } else {
        dim3 grid(ceil_div(W, 256), H, B);
        DMH_LAUNCH(compose_patch_u8_kernel<1>, grid, 256, 0, (cudaStream_t)stream)(
            scene, patch_a, patch_b, patch_mask, coeffs, bbox, flip, active, ph, pw, H, W, l_pad, t_pad, out_a, out_b, mask_out);
    }
    DMH_CHECK_LAUNCH("dmh_compose_patch_u8");
    return DMH_OK;
}

int dmh_perspective_fwd(const float* img, const float* coeffs, int B, int C, int ph, int pw, int oh, int ow,
                        float* out, dmh_stream_t stream) {
    DMH_REQUIRE(img && coeffs && out, "dmh_perspective_fwd: null pointer");
    DMH_REQUIRE(B > 0 && B <= 65535 && C > 0 && ph > 0 && pw > 0 && oh >= ph && ow >= pw,
                "dmh_perspective_fwd: bad shape (patch %dx%d, canvas %dx%d)", ph, pw, oh, ow);
    const int l_pad = (ow - pw) / 2, t_pad = (oh - ph) / 2;
    dim3 block(32, 8), grid(ceil_div(ow, 32), ceil_div(oh, 8), B);
    DMH_LAUNCH(perspective_fwd_kernel, grid, block, 0, (cudaStream_t)stream)(img, coeffs, C, ph, pw, oh, ow, l_pad, t_pad, out);
    DMH_CHECK_LAUNCH("dmh_perspective_fwd");
    return DMH_OK;
}

int dmh_perspective_bwd(const float* grad_out, const float* coeffs, int B, int C, int ph, int pw, int oh, int ow,
                        float* grad_img, dmh_stream_t stream) {
    DMH_REQUIRE(grad_out && coeffs && grad_img, "dmh_perspective_bwd: null pointer");
    DMH_REQUIRE(B > 0 && B <= 65535 && C > 0 && ph > 0 && pw > 0 && oh >= ph && ow >= pw, "dmh_perspective_bwd: bad shape");
    const int l_pad = (ow - pw) / 2, t_pad = (oh - ph) / 2;
    dim3 block(32, 8), grid(ceil_div(ow, 32), ceil_div(oh, 8), B);
    DMH_LAUNCH(perspective_bwd_kernel, grid, block, 0, (cudaStream_t)stream)(grad_out, coeffs, C, ph, pw, oh, ow, l_pad, t_pad,
                                                                          grad_img);
    DMH_CHECK_LAUNCH("dmh_perspective_bwd");
    return DMH_OK;
}

static int aa_tile_extent(int tile, float scale) {
    const float support = scale >= 1.0f ? scale : 1.0f;
    return (int)(scale * tile + 2.0f * support + 3.0f);
}

}  // extern "C"

namespace {
// Weight tables of the 3-tap forward kernel, one per (device, sizes), built on first use: a 20 KB allocation and one
// small launch on a private stream, waited for once.  Never built while the caller's stream is being captured (an
// allocation would invalidate the capture): the kernel then computes its weights itself, as it does when the table
// cannot be built -- same values either way.
struct AaTabEntry { int dev, ih, iw, oh, ow; float4* tab; };
std::mutex g_aa_mu;
std::vector<AaTabEntry> g_aa_tabs;

const float4* aa_table_get(int ih, int iw, int oh, int ow, float sy, float sx, cudaStream_t st) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return nullptr;
    std::lock_guard<std::mutex> lk(g_aa_mu);
    for (const AaTabEntry& e : g_aa_tabs)
        if (e.dev == dev && e.ih == ih && e.iw == iw && e.oh == oh && e.ow == ow) return e.tab;
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(st, &cs) != cudaSuccess || cs != cudaStreamCaptureStatusNone) {
        cudaGetLastError();
        return nullptr;
    }
    float4* tab = nullptr;
    cudaStream_t priv = nullptr;
    bool ok = cudaMalloc(&tab, sizeof(float4) * (size_t)(ow + oh)) == cudaSuccess &&
              cudaStreamCreateWithFlags(&priv, cudaStreamNonBlocking) == cudaSuccess;
    if (ok) {
        count_launches(1);
        aa_table_kernel<<<ceil_div(ow + oh, 256), 256, 0, priv>>>(ih, iw, oh, ow, sy, sx, tab);
        ok = cudaGetLastError() == cudaSuccess && cudaStreamSynchronize(priv) == cudaSuccess;
    }
    if (priv) cudaStreamDestroy(priv);
    if (!ok) {
        if (tab) cudaFree(tab);
        cudaGetLastError();
        return nullptr;
    }
    g_aa_tabs.push_back(AaTabEntry{dev, ih, iw, oh, ow, tab});
    return tab;
}
}  // namespace

extern "C" {

int dmh_patch_apply_fwd(const float* patch, const float* patch_mask, const float* scenes, const float* coeffs,
                        const int* bbox, int B, int ph, int pw, int ih, int iw, int oh, int ow, float* adv,
                        float* mask_out, dmh_stream_t stream) {
    DMH_REQUIRE(patch && patch_mask && scenes && coeffs && adv, "dmh_patch_apply_fwd: null pointer");
    DMH_REQUIRE(B > 0 && B <= 65535 && ph > 0 && pw > 0 && ih >= ph && iw >= pw && oh > 0 && ow > 0,
                "dmh_patch_apply_fwd: bad shape");
    const float sy = (float)ih / (float)oh, sx = (float)iw / (float)ow;
    DMH_REQUIRE(sy < 3.0f && sx < 3.0f, "dmh_patch_apply_fwd: down-scale factor >= 3 unsupported (AA window > %d taps)", AA_MAXT);
    const int l_pad = (iw - pw) / 2, t_pad = (ih - ph) / 2;
    const int cw_max = aa_tile_extent(PA_TW, sx), ch_max = aa_tile_extent(PA_TH, sy);
    const size_t smem = sizeof(float) * 4 * (size_t)cw_max * ch_max;
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(patch_apply_fwd_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e == cudaSuccess)
            e = cudaFuncSetAttribute(patch_apply_fwd_kernel<AA_MAXT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) {
            set_error("dmh_patch_apply_fwd: %zu B shared memory unavailable: %s", smem, cudaGetErrorString(e));
            return DMH_ERR_CUDA;
        }
    }
    dim3 grid(ceil_div(ow, PA_TW), ceil_div(oh, PA_TH), B);
    if (sy < 1.5f && sx < 1.5f && (long long)ih * iw * 3 < (1ll << 31) && (long long)oh * ow * 3 < (1ll << 31)) {
        // 3-tap windows: tile extents are compile-time (84 x 24 covers scale factors up to ~1.23, else 104 x 30)
        const bool small = cw_max <= 84 && ch_max <= 24;
        const size_t smem3 = sizeof(float) * 4 * (small ? 84 * 24 : 104 * 30);
        static bool configured[64] = {false};
        int dev = 0;
        cudaGetDevice(&dev);
        if (!configured[dev & 63]) {
            cudaError_t e = cudaFuncSetAttribute(patch_apply_fwd3_kernel<104, 30>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                 (int)(sizeof(float) * 4 * 104 * 30));
            if (e != cudaSuccess) {
                set_error("dmh_patch_apply_fwd: shared memory unavailable: %s", cudaGetErrorString(e));
                return DMH_ERR_CUDA;
            }
            configured[dev & 63] = true;
        }
        const float4* tab = small ? aa_table_get(ih, iw, oh, ow, sy, sx, (cudaStream_t)stream) : nullptr;
        if (small && tab)
            DMH_LAUNCH((patch_apply_fwd3_kernel<84, 24, true>), grid, PA_THREADS, smem3, (cudaStream_t)stream)(
                patch, patch_mask, scenes, coeffs, bbox, ph, pw, ih, iw, oh, ow, l_pad, t_pad, sy, sx, adv, mask_out, tab);
        else if (small)
            DMH_LAUNCH((patch_apply_fwd3_kernel<84, 24>), grid, PA_THREADS, smem3, (cudaStream_t)stream)(
                patch, patch_mask, scenes, coeffs, bbox, ph, pw, ih, iw, oh, ow, l_pad, t_pad, sy, sx, adv, mask_out,
                nullptr);
        else
            DMH_LAUNCH((patch_apply_fwd3_kernel<104, 30>), grid, PA_THREADS, smem3, (cudaStream_t)stream)(
                patch, patch_mask, scenes, coeffs, bbox, ph, pw, ih, iw, oh, ow, l_pad, t_pad, sy, sx, adv, mask_out,
                nullptr);
    } else if (sy < 1.5f && sx < 1.5f)
        DMH_LAUNCH(patch_apply_fwd_kernel<3>, grid, PA_THREADS, smem, (cudaStream_t)stream)(
            patch, patch_mask, scenes, coeffs, bbox, ph, pw, ih, iw, oh, ow, l_pad, t_pad, sy, sx, cw_max, ch_max, adv,
            mask_out);
    else
        DMH_LAUNCH(patch_apply_fwd_kernel<AA_MAXT>, grid, PA_THREADS, smem, (cudaStream_t)stream)(
            patch, patch_mask, scenes, coeffs, bbox, ph, pw, ih, iw, oh, ow, l_pad, t_pad, sy, sx, cw_max, ch_max, adv,
            mask_out);
    DMH_CHECK_LAUNCH("dmh_patch_apply_fwd");
    return DMH_OK;
}

int dmh_patch_apply_bwd(const float* grad_adv, const float* patch_mask, const float* coeffs, const int* bbox,
                        int bbox_max_w, int bbox_max_h, int B, int ph, int pw, int ih, int iw, int oh, int ow,
                        float* grad_patch, dmh_stream_t stream) {
    DMH_REQUIRE(grad_adv && patch_mask && coeffs && grad_patch, "dmh_patch_apply_bwd: null pointer");
    DMH_REQUIRE(B > 0 && B <= 65535 && ph > 0 && pw > 0 && ih >= ph && iw >= pw && oh > 0 && ow > 0,
                "dmh_patch_apply_bwd: bad shape");
    const float sy = (float)ih / (float)oh, sx = (float)iw / (float)ow;
    DMH_REQUIRE(sy < 3.0f && sx < 3.0f, "dmh_patch_apply_bwd: down-scale factor >= 3 unsupported");
    const int l_pad = (iw - pw) / 2, t_pad = (ih - ph) / 2;
    DMH_REQUIRE(!bbox || (bbox_max_w > 0 && bbox_max_h > 0), "dmh_patch_apply_bwd: bbox given without its max extent");
    const int gw = bbox ? (bbox_max_w < iw ? bbox_max_w : iw) : iw, gh = bbox ? (bbox_max_h < ih ? bbox_max_h : ih) : ih;
    dim3 block(32, 8), grid(ceil_div(gw, 32), ceil_div(gh, 8), B);
    // the span table of the 3-tap forward kernel serves the backward too (same cache; nullptr: weights computed in place)
    const float4* tab = (sy < 1.5f && sx < 1.5f) ? aa_table_get(ih, iw, oh, ow, sy, sx, (cudaStream_t)stream) : nullptr;
    if (tab)
        DMH_LAUNCH(patch_apply_bwd_kernel<true>, grid, block, 0, (cudaStream_t)stream)(
            grad_adv, patch_mask, coeffs, bbox, ph, pw, ih, iw, oh, ow, l_pad, t_pad, sy, sx, grad_patch, tab);
    else
        DMH_LAUNCH(patch_apply_bwd_kernel<false>, grid, block, 0, (cudaStream_t)stream)(
            grad_adv, patch_mask, coeffs, bbox, ph, pw, ih, iw, oh, ow, l_pad, t_pad, sy, sx, grad_patch, nullptr);
    DMH_CHECK_LAUNCH("dmh_patch_apply_bwd");
    return DMH_OK;
}

}  // extern "C"
