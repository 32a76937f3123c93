/* dmh_b200 -- C ABI of the B200-native hot path of DepthModelHardening.
 *
 * The reference has no FFI / plugin layer (it is 100 % Python; SURVEY.md 8(b)):
 * the boundary it exposes for this path is a set of Python symbols.  Each entry
 * point below names the reference symbol(s) it replaces (paths relative to
 * /root/reference; M2 = DepthNetworks/monodepth2, TA = torchattacks).
 * INTEGRATION.md shows the ctypes binding and the rebinding of those symbols.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer to caller-owned fp32 memory (NCHW,
 *     contiguous) unless the name ends in `_host`; the library never allocates,
 *     frees or synchronises -- work is enqueued on `stream` and returns;
 *   - return value: DMH_OK (0) or an error code; `dmh_last_error()` returns a
 *     thread-local message.  Wrappers raise RuntimeError on non-zero;
 *   - "nullable" outputs may be NULL to skip that result;
 *   - buffers marked "accumulated" must be zeroed by the caller (atomics add);
 *   - re-entrant: no global state except the thread-local error string.
 */
#ifndef DMH_B200_H
#define DMH_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default) /* the library is built with -fvisibility=hidden */
#endif

typedef struct CUstream_st* dmh_stream_t; /* == cudaStream_t */

#define DMH_OK 0
#define DMH_ERR_INVALID 1
#define DMH_ERR_CUDA 2
#define DMH_ERR_UNSUPPORTED 3

#define DMH_PAD_ZEROS 0
#define DMH_PAD_BORDER 1

/* -- library ------------------------------------------------------------- */
const char* dmh_last_error(void);
int dmh_version(void);    /* 100*major + minor */
int dmh_build_arch(void); /* 100 == compiled for sm_100a */
long long dmh_launch_count(void); /* kernels launched by this library in this process so far */

/* -- A9  disp_to_depth (M2/layers.py:16-25) ------------------------------ */
int dmh_disp_to_depth(const float* disp, long long n, float min_depth, float max_depth, float* scaled_disp,
                      float* depth, dmh_stream_t stream);

/* -- A10 BackprojectDepth.forward (M2/layers.py:163-168) ------------------
 * depth (B,1,H,W), inv_K (B,4,4) -> points (B,4,H*W) [x,y,z,1 planes]
 * bwd: grad_depth (B,1,H,W) (nullable); grad_inv_K_partial (B, nblk, 9) per-block partial sums of
 * d/d(inv_K[:3,:3]) with nblk = dmh_backproject_bwd_blocks(H,W) (nullable; needs depth).          */
int dmh_backproject_fwd(const float* depth, const float* inv_K, int B, int H, int W, float* points,
                        dmh_stream_t stream);
int dmh_backproject_bwd_blocks(int H, int W);
int dmh_backproject_bwd(const float* grad_points, const float* depth, const float* inv_K, int B, int H, int W,
                        float* grad_depth, float* grad_inv_K_partial, dmh_stream_t stream);

/* -- A11 Project3D.forward (M2/layers.py:182-198) -------------------------
 * points (B,4,N), K,T (B,4,4) -> grid (B,H,W,2) in [-1,1] (unclamped)
 * bwd: grad_points (B,4,N); grad_P_partial (B, nblk, 12) per-block partial sums
 * of d/d((K@T)[:3,:]) with nblk = dmh_project3d_bwd_blocks(H,W) (nullable).      */
int dmh_project3d_fwd(const float* points, const float* K, const float* T, int B, int H, int W, float eps,
                      float* grid, dmh_stream_t stream);
int dmh_project3d_bwd_blocks(int H, int W);
int dmh_project3d_bwd(const float* grad_grid, const float* points, const float* K, const float* T, int B, int H,
                      int W, float eps, float* grad_points, float* grad_P_partial, dmh_stream_t stream);

/* -- A12 F.grid_sample bilinear (M2/trainer.py:515-519; DH/trainer.py:523) --
 * src (B,C,Hs,Ws), grid (B,Ho,Wo,2) -> out (B,C,Ho,Wo)
 * bwd: grad_src (accumulated, nullable), grad_grid (nullable)                  */
int dmh_grid_sample_fwd(const float* src, const float* grid, int B, int C, int Hs, int Ws, int Ho, int Wo,
                        int padding_mode, int align_corners, float* out, dmh_stream_t stream);
int dmh_grid_sample_bwd(const float* grad_out, const float* src, const float* grid, int B, int C, int Hs, int Ws,
                        int Ho, int Wo, int padding_mode, int align_corners, float* grad_src, float* grad_grid,
                        dmh_stream_t stream);

/* -- A13 SSIM.forward (M2/layers.py:239-253) ------------------------------
 * x,y (B,C,H,W) -> out (B,C,H,W); bwd gives grad_x / grad_y (each nullable)   */
int dmh_ssim_fwd(const float* x, const float* y, int B, int C, int H, int W, float* out, dmh_stream_t stream);
int dmh_ssim_bwd(const float* grad_out, const float* x, const float* y, int B, int C, int H, int W, float* grad_x,
                 float* grad_y, dmh_stream_t stream);

/* -- A14 Trainer.compute_reprojection_loss (M2/trainer.py:525-537) --------
 * pred,target (B,C,H,W) -> out (B,1,H,W) = 0.85*mean_c SSIM + 0.15*mean_c|t-p|
 * (L1 only when no_ssim)                                                      */
int dmh_reproj_loss_fwd(const float* pred, const float* target, int B, int C, int H, int W, int no_ssim,
                        float* out, dmh_stream_t stream);
int dmh_reproj_loss_bwd(const float* grad_out, const float* pred, const float* target, int B, int C, int H, int W,
                        int no_ssim, float* grad_pred, float* grad_target, dmh_stream_t stream);

/* -- A16 get_smooth_loss (M2/layers.py:207-220) + mean-normalisation
 *        (M2/trainer.py:662-664) -------------------------------------------
 * disp (B,1,h,w), img (B,C,h,w).  normalise != 0 divides disp by its per-image
 * mean + 1e-7 first.  Two-phase, deterministic:
 *   fwd : loss_out[0] = loss (device scalar); ws = workspace of
 *         dmh_smooth_workspace_floats(B,h,w) floats
 *   bwd : grad_disp (B,1,h,w) and optional grad_img (B,C,h,w), both scaled by
 *         the device scalar *grad_loss (nullable -> 1) times `weight`.          */
long long dmh_smooth_workspace_floats(int B, int h, int w);
int dmh_smooth_fwd(const float* disp, const float* img, int B, int C, int h, int w, int normalise, float* ws,
                   float* loss_out, dmh_stream_t stream);
int dmh_smooth_bwd(const float* disp, const float* img, int B, int C, int h, int w, int normalise,
                   const float* grad_loss, float weight, float* ws, float* grad_disp, float* grad_img,
                   dmh_stream_t stream);

/* -- F.interpolate(disp, [H,W], "bilinear", align_corners=False) (M2/trainer.py:481-482)
 * in (planes,h,w) -> out (planes,H,W).  bwd is a deterministic gather (ATen's CUDA
 * backward uses atomics): grad_in = (*grad_scale, nullable -> 1) * dOut/dIn^T grad_out */
int dmh_upsample_bilinear_fwd(const float* in, int planes, int h, int w, int H, int W, float* out,
                              dmh_stream_t stream);
int dmh_upsample_bilinear_bwd(const float* grad_out, int planes, int h, int w, int H, int W, const float* grad_scale,
                              float* grad_in, dmh_stream_t stream);

/* -- A9-A12 fused gather: disp -> depth -> backproject -> project -> bilinear
 *    border warp in ONE kernel (M2/trainer.py:485-519 for one (scale, frame)).
 * disp (B,1,H,W) full resolution (or depth when input_is_depth), src (B,C,H,W),
 * K,inv_K,T (B,4,4) -> warped (B,C,H,W); optional grid (B,H,W,2), depth (B,1,H,W)
 * fwd: input_is_depth bit 0 = the input is a depth map, bit 1 = sample with align_corners=False (the depth-hints
 *      warp, DH/trainer.py:523-525; forward only).
 * bwd: grad_disp (B,1,H,W) [d/d(disp) or d/d(depth)], grad_src (accumulated,
 * nullable), grad_P_partial (B, nblk, 12) nullable, nblk = dmh_warp_bwd_blocks.  */
int dmh_warp_fwd(const float* disp, int input_is_depth, float min_depth, float max_depth, const float* src,
                 const float* K, const float* inv_K, const float* T, int B, int C, int H, int W, float* warped,
                 float* grid_out, float* depth_out, dmh_stream_t stream);
int dmh_warp_bwd_blocks(int H, int W);
int dmh_warp_bwd(const float* grad_warped, const float* disp, int input_is_depth, float min_depth, float max_depth,
                 const float* src, const float* K, const float* inv_K, const float* T, int B, int C, int H, int W,
                 float* grad_disp, float* grad_src, float* grad_P_partial, dmh_stream_t stream);

/* -- A9-A15 fused objective for ONE scale, forward AND backward in one pass
 *    (M2/trainer.py:472-523 + 589-660 for one value of `scale`).
 *
 * target (B,3,H,W); src_host[f] device pointers to (B,3,H,W), f < F <= 4;
 * T_host[f] device pointers to (B,4,4); disp (B,1,disp_h,disp_w): the network's
 * disparity at its native scale -- the bilinear F.interpolate to (H,W) of
 * trainer.py:481-482 is fused into the read (disp_h==H: direct); ident (B,F,H,W) identity reprojection losses WITHOUT noise
 * (dmh_reproj_loss_fwd of the un-warped sources; scale independent) or NULL when
 * automasking is disabled; noise (B,Fi,H,W) tie-break noise already scaled
 * (nullable == zeros), Fi = avg_reprojection ? 1 : F.
 * flags: DMH_PHOTO_*.
 * Outputs:
 *   loss_partial : B * dmh_photo_tiles(H,W) floats, per-CTA sums of to_optimise
 *   grad_disp    : (B,1,H,W) = grad_scale * d(sum to_optimise)/d(up-sampled disp); push it
 *                  through dmh_upsample_bilinear_bwd / dmh_disp_grad to reach (disp_h,disp_w)
 *   grad_P_partial (nullable): (F, B, tiles, 12) per-CTA partial sums of
 *                  grad_scale * d(sum)/d((K@T_f)[:3,:])
 *   sel (nullable): (B,H,W) uint8 argmin index over [ident..., reproj...]
 *   warped_host (nullable): F device pointers (nullable each) to (B,3,H,W)      */
/* identity reprojection losses of the automask (M2/trainer.py:608-615): ident (B,F,H,W),
 * ident[:,f] = compute_reprojection_loss(src_f, target); scale independent, computed once. */
int dmh_identity_loss(const float* target, const float* const* src_host, int F, int B, int H, int W, int no_ssim,
                      float* ident, dmh_stream_t stream);
/* Single-source variant that ALSO writes the source frame pixel-packed, src_packed (B,H,W,4) fp32 (RGB + one pad
 * float, 16-byte aligned): with DMH_PHOTO_SRC_PACKED the per-scale kernel gathers each bilinear tap with one
 * 128-bit load instead of three scalar ones (the gather of F.grid_sample, M2/trainer.py:515-519, is repeated for
 * every scale, the re-layout is done once).  ident nullable: re-layout only (automasking disabled).            */
int dmh_identity_loss_pack(const float* target, const float* src, int B, int H, int W, int no_ssim, float* ident,
                           float* src_packed, dmh_stream_t stream);
/* bf16 frames (BASELINE north_star: bf16 inputs at 2e-3, "bf16x8 coalesced loads"): the same pass reading the two
 * frames as bf16 (B,3,H,W) with 128-bit loads of 8 elements and ALSO writing target_f32 (B,3,H,W), the widened
 * target every later kernel of the step stages by TMA -- no separate up-cast pass over the frames.  The identity
 * loss is computed on the widened values, i.e. equals dmh_identity_loss_pack on target.float(), src.float() bit for
 * bit.  Needs W % 8 == 0 and 16-byte aligned frames.                                                          */
int dmh_identity_loss_pack_bf16(const uint16_t* target_bf16, const uint16_t* src_bf16, int B, int H, int W, int no_ssim,
                                float* ident, float* src_packed, float* target_f32, dmh_stream_t stream);
#define DMH_PHOTO_NO_SSIM 1
#define DMH_PHOTO_AVG_REPROJECTION 2
#define DMH_PHOTO_INPUT_IS_DEPTH 4
#define DMH_PHOTO_SEL_SOURCE 8  /* dmh_photo_scale_dh only: sel = argmin | (winning source frame << 2), see there */
#define DMH_PHOTO_SRC_PACKED 16 /* src_host[0] is the (B,H,W,4) layout of dmh_identity_loss_pack; F == 1, no pose grad */
#define DMH_PHOTO_PIXEL_SUM 32  /* dmh_photo_image_grad only: the loss is the sum of the per-pixel losses, see there */
#define DMH_PHOTO_MAX_FRAMES 4
int dmh_photo_tiles(int H, int W);           /* CTAs per batch item */
int dmh_photo_scale(const float* target, const float* const* src_host, const float* const* T_host, int F,
                    const float* disp, int disp_h, int disp_w, const float* K, const float* inv_K, const float* ident,
                    const float* noise, int B, int H, int W, float min_depth, float max_depth, int flags, float grad_scale,
                    float* loss_partial, float* grad_disp, float* grad_P_partial, uint8_t* sel,
                    float* const* warped_host, dmh_stream_t stream);

/* ALL scales of the single-source objective in one launch (DepthNetworks/monodepth2/trainer.py:476-523 and
 * :589-660 -- the `for scale in self.opt.scales` loops of generate_images_pred and compute_losses run inside the
 * kernel: a CTA owns one 32 x 32 target tile and walks over the S <= 4 scales).  Same contract and the same bits as
 * S calls of dmh_photo_scale with F == 1, DMH_PHOTO_SRC_PACKED, SSIM on, disparity input, no pose gradient:
 * src_packed = the (B,H,W,4) copy written by dmh_identity_loss_pack; disp_host[s] (B,1,disp_h[s],disp_w[s]);
 * noise_host[s] (B,1,H,W) or NULL; loss_partial_host[s] receives B*dmh_photo_tiles(H,W) floats (the first
 * B*ceil(H/32)*ceil(W/32) are written); grad_disp_host[s] (B,1,H,W); sel_host (nullable) / sel_host[s] (B,H,W).
 * The *_host arguments are HOST arrays of device pointers.  Returns DMH_ERR_UNSUPPORTED when the frames cannot be
 * staged by TMA (W % 4 != 0 or unaligned bases): the caller then uses dmh_photo_scale per scale.               */
int dmh_photo_multiscale(const float* target, const float* src_packed, const float* T, int S,
                         const float* const* disp_host, const int* disp_h, const int* disp_w, const float* K,
                         const float* inv_K, const float* ident, const float* const* noise_host, int B, int H, int W,
                         float min_depth, float max_depth, float grad_scale, float* const* loss_partial_host,
                         float* const* grad_disp_host, uint8_t* const* sel_host, dmh_stream_t stream);

/* The objective with SEVERAL source frames and / or pose gradients, ALL scales, in one launch
 * (DepthNetworks/monodepth2/trainer.py:476-523 -- every frame id of every scale is warped -- and :589-660 --
 * torch.cat([identity losses + noise, reprojection losses]) -> torch.min, the first minimum in cat order wins --;
 * pose branch: Project3D's T, layers.py:182-198).  The tile kernel of dmh_photo_multiscale for F <= 4 sources:
 * min-reprojection, SSIM on, disparity input (avg_reprojection / no_ssim / depth input / depth hints stay with
 * dmh_photo_scale).  src_packed_host[f] = (B,H,W,4) copy of source f and ident_host[f] = its (B,1,H,W) identity loss,
 * both from dmh_identity_loss_pack (ident_host NULL or all NULL: automask off); noise_host[s] (B,F,H,W), the
 * reference's layout, or NULL; workspace: dmh_photo_multisource_workspace_floats(F) floats, 16-byte aligned, contents
 * irrelevant before and after (per-CTA scratch that lives in L2).  Outputs per scale: loss_partial_host[s]
 * (B*dmh_photo_tiles floats; the first B*ceil(H/32)*ceil(W/32) are written, the rest zeroed), grad_disp_host[s]
 * (B,1,H,W) = grad_scale * d(sum loss)/d(up-sampled disparity), grad_P_partial_host (nullable) /
 * grad_P_partial_host[s] (F, B, ceil(H/32)*ceil(W/32), 12) = grad_scale * per-tile d(sum loss)/d((K@T)[:3,:]),
 * sel_host (nullable) / sel_host[s] (B,H,W) argmin in cat order.  With F == 1 and no pose gradient the results are
 * bit-identical to dmh_photo_multiscale.  Returns DMH_ERR_UNSUPPORTED when the frames cannot be staged by TMA.    */
long long dmh_photo_multisource_workspace_floats(int F);
int dmh_photo_multisource(const float* target, const float* const* src_packed_host, const float* const* T_host, int F,
                          int S, const float* const* disp_host, const int* disp_h, const int* disp_w, const float* K,
                          const float* inv_K, const float* const* ident_host, const float* const* noise_host, int B,
                          int H, int W, float min_depth, float max_depth, float grad_scale, float* workspace,
                          float* const* loss_partial_host, float* const* grad_disp_host,
                          float* const* grad_P_partial_host, uint8_t* const* sel_host, dmh_stream_t stream);

/* Test hook of dmh_photo_multiscale's branch-free IEEE reciprocals (the instruction sequence of the hardware fast
 * path of 1/x and a/z, valid for operands in [2^-60, 2^60]; operands outside raise a per-tile flag and take the
 * generic division): counts the mismatches against __frcp_rn over EVERY float of that range and against
 * __fdiv_rn over 2^32 pseudo-random pairs.  mismatches: 2 device counters (uint64); both must read 0.           */
int dmh_selftest_reciprocals(unsigned long long* mismatches, unsigned int seed, dmh_stream_t stream);

/* Depth-hints variant of dmh_photo_scale (A18; DepthNetworks/depth-hints/trainer.py:476-525, 541-590, 629-727),
 * one scale: same fused warp + SSIM/L1 + backward, but the per-pixel decision is the depth-hints one -- min (or
 * mean) over the source frames first, ONE tie-break noise plane noise (B,1,H,W) added to the identity minimum,
 * argmin over [reprojection, identity, hint_reproj]; reprojection mask = argmin != identity, hint mask =
 * argmin == hint.  hint_reproj (B,1,H,W) = reprojection loss of the depth-hint warp + 1000*(1-hint_valid)
 * (NULL: use_depth_hints off), hint_depth / hint_valid (B,1,H,W).
 * Outputs: sums_partial = 4 x B*dmh_photo_tiles floats, per-CTA partial sums of [reproj*mask_r, mask_r,
 * log(|hint-depth|+1)*valid*mask_h, mask_h]; grad_disp = d(sum reproj*mask_r)/d(up-sampled disp) and
 * grad_disp_hint = d(sum proxy*mask_h)/d(up-sampled disp), both UN-normalised (the masked-mean denominators are
 * known only after the pass: the caller divides); grad_P_partial as in dmh_photo_scale; sel = argmin index.
 * With DMH_PHOTO_SEL_SOURCE in flags, sel also records the source frame whose reprojection is the (first) minimum
 * over the frames: sel = argmin | (frame << 2), so sel & 3 is the argmin index as without the flag.  It is the
 * decision dmh_photo_image_grad_dh routes the reprojection gradient by.  On the single-source fast path (F == 1) the
 * flag is accepted and the upper bits are 0; under DMH_PHOTO_AVG_REPROJECTION they are 0 as well (no minimum is
 * taken).  dmh_photo_scale ignores the flag.                                                                      */
int dmh_photo_scale_dh(const float* target, const float* const* src_host, const float* const* T_host, int F,
                       const float* disp, int disp_h, int disp_w, const float* K, const float* inv_K,
                       const float* ident, const float* noise, const float* hint_reproj, const float* hint_depth,
                       const float* hint_valid, int B, int H, int W, float min_depth, float max_depth, int flags,
                       float* sums_partial, float* grad_disp, float* grad_disp_hint, float* grad_P_partial,
                       uint8_t* sel, dmh_stream_t stream);

/* -- fused multi-scale objective glue (M2/trainer.py:589-674) -------------------
 * dmh_smooth_fused: A16 forward + gradient w.r.t. the mean-normalised disparity in
 *   one pass: gN (B,1,h,w) = d(smooth loss)/d(norm disp); ws (workspace of
 *   dmh_smooth_fused_workspace_floats floats) receives the per-block partial sums.
 * dmh_objective_finish: ONE launch for all S scales: img_scalars (S,B,2) = per image
 *   {1/(mean+1e-7), correction term of the normalisation backward}; losses (S+1) =
 *   per-scale losses [photo_sum/photo_den + smooth_weight*smooth] and their mean.
 *   *_host arrays are host arrays of length S (device pointers / ints / floats);
 *   workspace: dmh_objective_finish_workspace_bytes(S,B) bytes, 16-byte aligned.
 * dmh_disp_grad: backward, one launch per scale:
 *   grad_disp (B,1,h,w) = u * [ interpolate^T(G_full (B,1,H,W)) + smooth_weight *
 *   (gN*inv_mean - corr) ],  u = *g_total * inv_S + *g_scale (device scalars, either
 *   nullable); gN nullable (no smoothness term); img_scalars = the (B,2) slice of
 *   this scale.  g_smooth (nullable device scalar): separate upstream weight of the
 *   smoothness term: grad = u * interpolate^T(G_full) + *g_smooth * smooth_weight * (...)
 *   (depth-hints objective, whose photometric gradients carry their own weights).  */
long long dmh_smooth_fused_workspace_floats(int B, int h, int w);
int dmh_smooth_fused(const float* disp, const float* img, int B, int C, int h, int w, float* ws, float* gN,
                     dmh_stream_t stream);
long long dmh_objective_finish_workspace_bytes(int S, int B);
int dmh_objective_finish(int S, int B, const float* const* smooth_ws_host, const int* h_host, const int* w_host,
                         const float* const* photo_part_host, const int* photo_n_host,
                         const float* smooth_weight_host, double photo_den, void* workspace, float* img_scalars,
                         float* losses, dmh_stream_t stream);
int dmh_disp_grad(const float* G_full, const float* gN, const float* img_scalars, float smooth_weight,
                  const float* g_total, const float* g_scale, const float* g_smooth, float inv_S, int B, int h, int w,
                  int H, int W, float* grad_disp, dmh_stream_t stream);

/* -- colour-frame gradients of the fused objective (backward of ops.objective w.r.t. the frames) ----------------
 * Recomputed from the frames, the disparities and the forward's selections sel_s (B,H,W) (argmin in cat order, as
 * dmh_photo_scale / dmh_photo_multiscale / dmh_photo_multisource emit it).  Upstream weight of scale s:
 * u_s = *g_total / S + g_scales[s] (device scalars, either nullable), read on the device.  flags: DMH_PHOTO_NO_SSIM,
 * DMH_PHOTO_AVG_REPROJECTION; automask: identity candidates present.  grad_target (B,3,H,W) and grad_src_host[f]
 * (B,3,H,W) are nullable (that frame's gradient is not computed).
 * dmh_identity_image_grad: ONE launch for all S scales: the identity candidates' terms (un-warped source f vs
 *   target, gated by sum_s u_s [sel_s picked f's identity]).  INITIALISES grad_target and every grad_src[f].
 * dmh_photo_image_grad: one launch per scale `scale`: the reprojection candidates' terms; ADDS into grad_target and
 *   (atomically: the last bits depend on the order) into grad_src[f] through the bilinear taps of the warp.  It also
 *   takes DMH_PHOTO_INPUT_IS_DEPTH (disp is a depth map, used as it is; min_depth / max_depth are ignored) and
 *   DMH_PHOTO_PIXEL_SUM (the loss is the sum of the per-pixel losses, as dmh_photo_scale computes it with
 *   inv_den = 1: the per-pixel weight is u_s, not u_s / (B*H*W)).
 * dmh_smooth_image_grad: u_s * smooth_weight * d(smoothness of scale s)/d(img) for img = colour(0, s) (B,3,h,w),
 *   disp (B,1,h,w), img_scalars the (B,2) slice of dmh_objective_finish for scale s; accumulate: add into grad_img
 *   instead of writing it.                                                                                         */
int dmh_identity_image_grad(const float* target, const float* const* src_host, int F, const uint8_t* const* sel_host,
                            int S, const float* g_total, const float* g_scales, int B, int H, int W, int flags,
                            int automask, float* grad_target, float* const* grad_src_host, dmh_stream_t stream);
int dmh_photo_image_grad(const float* target, const float* const* src_host, const float* const* T_host, int F,
                         const float* disp, int disp_h, int disp_w, const float* K, const float* inv_K,
                         const uint8_t* sel, int scale, int S, const float* g_total, const float* g_scales, int B,
                         int H, int W, float min_depth, float max_depth, int flags, int automask, float* grad_target,
                         float* const* grad_src_host, dmh_stream_t stream);
int dmh_smooth_image_grad(const float* disp, const float* img, int B, int h, int w, const float* img_scalars,
                          float smooth_weight, int scale, int S, const float* g_total, const float* g_scales,
                          int accumulate, float* grad_img, dmh_stream_t stream);
/* dmh_photo_image_grad_dh: the reprojection terms of ONE scale of the depth-hints objective (backward of
 * depth_hints.depth_hint_losses w.r.t. the frames), the contract of dmh_photo_image_grad otherwise.  sel (B,H,W) as
 * dmh_photo_scale_dh writes it with DMH_PHOTO_SEL_SOURCE (needed when F > 1 without DMH_PHOTO_AVG_REPROJECTION):
 * pixels whose argmin (sel & 3) is the identity get nothing, the others send their reprojection term's gradient to
 * source frame sel >> 2 (to every frame with weight 1/F under DMH_PHOTO_AVG_REPROJECTION).  u: device scalar, the
 * upstream weight of the term's per-pixel losses, (d loss / d reproj_loss_s) / (sum(mask_r) + 1e-7).  The identity
 * and hint candidates only decide the mask: there is no identity launch, so the caller zeroes grad_target and every
 * grad_src[f] before the first scale.  ADDS into grad_target, and atomically into grad_src[f].                   */
int dmh_photo_image_grad_dh(const float* target, const float* const* src_host, const float* const* T_host, int F,
                            const float* disp, int disp_h, int disp_w, const float* K, const float* inv_K,
                            const uint8_t* sel, const float* u, int B, int H, int W, float min_depth, float max_depth,
                            int flags, float* grad_target, float* const* grad_src_host, dmh_stream_t stream);

/* ======================= stage 1: physical patch attack ======================= */

/* -- A2+A3 PhysicalTrans.project / project_w_trans (physicalTrans.py:130-196):
 * zero-pad the (C,ph,pw) image to the (oh,ow) canvas (centred, :107-122) and apply
 * torchvision.perspective (bilinear, zeros, align_corners=False) with coeffs[b]
 * (8 fp32 homography coefficients per item, output pixel -> input pixel, solved on
 * the host in fp64 like torchvision functional.py:674-704) for all B items at once.
 * img (C,ph,pw) shared by the batch -> out (B,C,oh,ow); bwd: grad_img accumulated. */
int dmh_perspective_fwd(const float* img, const float* coeffs, int B, int C, int ph, int pw, int oh, int ow,
                        float* out, dmh_stream_t stream);
int dmh_perspective_bwd(const float* grad_out, const float* coeffs, int B, int C, int ph, int pw, int oh, int ow,
                        float* grad_img, dmh_stream_t stream);

/* -- A2-A5 fused attack forward (TA/attacks/phy_obj_atk.py:86-90, phy_obj_atk_l0.py:115-119):
 * perspective(patch), perspective(mask), scene*(1-m)+obj*m, Resize([oh,ow]) (bilinear,
 * antialias) of the composite and of the mask.
 * patch (3,ph,pw), patch_mask (1,ph,pw), scenes (B,3,ih,iw), coeffs (B,8)
 * -> adv (B,3,oh,ow), mask_out (B,1,oh,ow) (nullable)
 * bwd: grad_adv (B,3,oh,ow) -> grad_patch (3,ph,pw) accumulated (sum over the batch).
 * bbox (nullable): (B,4) int32 device array {x0,y0,x1,y1} (inclusive canvas pixels) outside of which item b
 * cannot sample the patch (host-computed from the projected corners; an optimisation hint that must be
 * conservative); bwd launches only max-bbox-sized grids (bbox_max_w/h = largest extent over the batch).
 * State: the first forward call for a new (device, ih, iw, oh, ow) outside a stream capture builds a small table of
 * resize weights (one 16 (oh+ow)-byte allocation kept for the life of the process, one launch on a private stream that
 * is waited for); inside a capture, or if that fails, the kernel computes the same weights itself.               */
int dmh_patch_apply_fwd(const float* patch, const float* patch_mask, const float* scenes, const float* coeffs,
                        const int* bbox, int B, int ph, int pw, int ih, int iw, int oh, int ow, float* adv,
                        float* mask_out, dmh_stream_t stream);
int dmh_patch_apply_bwd(const float* grad_adv, const float* patch_mask, const float* coeffs, const int* bbox,
                        int bbox_max_w, int bbox_max_h, int B, int ph, int pw, int ih, int iw, int oh, int ow,
                        float* grad_patch, dmh_stream_t stream);

/* -- A6 L-inf PGD update (phy_obj_atk.py:98-100; pgd_depth.py:76-78; pgd.py:73-75):
 * out = clamp(clean + clamp(adv + alpha*sign(grad) - clean, -eps, eps), 0, 1)          */
int dmh_pgd_linf_step(const float* adv, const float* grad, const float* clean, long long n, float alpha, float eps,
                      float* out, dmh_stream_t stream);

/* -- APGD L-inf step with momentum (next-4; torchattacks/attacks/phy_obj_atk_apgd.py:214-222), one launch:
 * z = clamp(proj_eps(x_adv + step*sign(grad)), 0, 1); out = clamp(proj_eps(x_adv + (z - x_adv)*a +
 * (x_adv - x_adv_old)*(1-a)), 0, 1), proj_eps = min(max(., x0-eps), x0+eps).  out may alias x_adv.            */
int dmh_apgd_linf_step(const float* x_adv, const float* x_adv_old, const float* grad, const float* x0, long long n,
                       float step, float a, float eps, float* out, dmh_stream_t stream);

/* -- black-box patch searches (next-4): candidates and acceptance on the device ---------------------------------
 * Tube-light candidate (torchattacks/attacks/light_simulation.py:132-170 tube_light_generation_by_func, then
 * phy_obj_atk_light.py:118-122 / light_simulation.py:23-28): per pixel d = |k*x - y + b| / norm in float64;
 * light = ca[c] for d <= full_end, ca[c] * beta / d^2 for d <= light_end, else 0; lit = uint8(clip(base +
 * float32(light * 255), 0, 255)); patch = float(lit) / 255 (ToTensor).  base_u8 / lit_u8 (optional): planar (3,h,w)
 * bytes; patch: (3,h,w) floats.  The scalars are formed on the host as the reference forms them: k = round(tan, 2),
 * norm = sqrt(1 + k*k), full_end = int(sqrt(beta) + .5), light_end = int(sqrt(20 beta) + .5), ca = rgb * alpha.   */
int dmh_tube_light_patch(const uint8_t* base_u8, int h, int w, double k, double b, double norm, double beta,
                         int full_end, int light_end, double ca0, double ca1, double ca2, float* patch, uint8_t* lit_u8,
                         dmh_stream_t stream);
/* Square-attack L-inf candidate (torchattacks/attacks/phy_obj_atk_square.py:263-274): x_new = clamp(min(max(x_best +
 * delta, x - eps), x + eps), 0, 1), delta = d[c] inside the window [vh,vh+s) x [vw,vw+s), 0 outside; (3,H,W).   */
int dmh_square_linf_candidate(const float* x_best, const float* x, int H, int W, int vh, int vw, int s, float d0,
                              float d1, float d2, float eps, float* x_new, dmh_stream_t stream);
/* `if cost < best_cost: best_cost, best = cost, cand` without a host round trip (phy_obj_atk_light.py:148-150,
 * phy_obj_atk_square.py:281-297): best_cost_out[0] = min-select of cost[0] / best_cost_in[0] (strict <, NaN never
 * accepted), best[0..n) = cand where accepted.  best_cost_in != best_cost_out (the caller ping-pongs them).     */
int dmh_keep_best(const float* cost, const float* best_cost_in, float* best_cost_out, const float* cand, float* best,
                  long long n, dmh_stream_t stream);

/* -- evaluation metrics of the attack harness (next-4; DepthNetworks/monodepth2/evaluate_depth.py:193-196 and
 * compute_errors :57-99), one launch per batch: depth = clamp(disp_to_depth(|disp|, min_disp_depth, max_disp_depth)[1]
 * * scale_factor, min_depth, max_depth) for both maps, then out[9] (double, zeroed here) = [sum mask, sum |d|*m,
 * sum |d|/gt*m, sum d^2/gt*m, sum d^2*m, sum (log gt - log pred)^2*m, sum [thr<1.25]*m, [thr<1.25^2], [thr<1.25^3]],
 * thr = max(gt/pred, pred/gt); mask NULL = all ones.  The caller divides by out[0] and takes the two roots.    */
int dmh_depth_errors(const float* disp_gt, const float* disp_pred, const float* mask, long long n, float min_disp_depth,
                     float max_disp_depth, float scale_factor, float min_depth, float max_depth, double* out,
                     dmh_stream_t stream);

/* -- L2 PGD update of the shared patch (next-4; torchattacks/attacks/phy_obj_atk_l2.py:108-120):
 * g = grad / (||grad||_2 + eps_div); x = adv + alpha*g; d = x - clean;
 * out = clamp(clean + d * min(eps / ||d||_2, 1), 0, 1).  One launch; out may alias adv.                      */
int dmh_pgd_l2_step(const float* adv, const float* grad, const float* clean, long long n, float alpha, float eps,
                    float eps_div, float* out, dmh_stream_t stream);

/* -- A7 L0 compose + cal_l0 (phy_obj_atk_l0.py:94-99, 43-52): adv (nullable) =
 * clamp(obj + clamp(P+) - clamp(P-)); *count = #pixels whose thresholded pattern is
 * non-zero in any channel (device uint64, overwritten).                              */
int dmh_l0_compose_count(const float* obj, const float* pattern_pos, const float* pattern_neg, int C, int H, int W,
                         float clip_max, float threshold, float* adv, unsigned long long* count,
                         dmh_stream_t stream);

/* -- A8 mask-cost gradient + Adam (phy_obj_atk_l0.py:130-138, torch.optim.Adam):
 * grad_adv = d(adv_cost)/d(adv patch) (nullable); counts (nullable) = {l0 now, l0 at
 * step 0} on the device: mask_weight becomes 0 when their ratio <= l0_thresh (:105-108)
 * without a host sync.  P+/P-, m, v updated in place; `step` is 1-based.                */
int dmh_l0_adam_step(const float* obj, const float* grad_adv, float* pattern_pos, float* pattern_neg, float* m_pos,
                     float* v_pos, float* m_neg, float* v_neg, int C, int H, int W, float clip_max,
                     const unsigned long long* counts, float l0_thresh, float mask_weight, float lr, float beta1,
                     float beta2, float adam_eps, int step, dmh_stream_t stream);

/* The same step with the step index kept ON THE DEVICE, so that a whole attack iteration (compose, patch apply,
 * network, this update) can be captured once into a CUDA graph and replayed: a host-side `step` argument would be
 * frozen into the capture.  bias_table: table_len x 2 device floats, entry t-1 = {lr / (1 - beta1^t),
 * sqrt(1 - beta2^t)} -- the two scalars dmh_l0_adam_step forms from `step`, filled on the host by
 * dmh_l0_adam_bias_table with the same double arithmetic (bit-identical updates); steps past the table read its last
 * entry (both factors have converged in fp32 long before: t > 25 / 160 for torch's betas (0.5, 0.9)).
 * step_state: 2 uint32 of device memory, zeroed before the first step: {steps done, CTA arrival ticket}; the last
 * CTA of a launch advances the step, after every CTA has read it.                                            */
int dmh_l0_adam_bias_table(float lr, float beta1, float beta2, int table_len, float* table_host);
int dmh_l0_adam_step_dev(const float* obj, const float* grad_adv, float* pattern_pos, float* pattern_neg, float* m_pos,
                         float* v_pos, float* m_neg, float* v_neg, int C, int H, int W, float clip_max,
                         const unsigned long long* counts, float l0_thresh, float mask_weight, float beta1, float beta2,
                         float adam_eps, const float* bias_table, int table_len, unsigned* step_state,
                         dmh_stream_t stream);

/* -- phy_obj_atk_l0.py:143-150: hard threshold at `threshold`, compose; pattern nullable */
int dmh_l0_finalize(const float* obj, const float* pattern_pos, const float* pattern_neg, long long n, float clip_max,
                    float threshold, float* adv, float* pattern, dmh_stream_t stream);

/* -- EXTENSION (not reference behaviour, SURVEY.md fact 3): exact top-k L0 projection by
 * radix select: keep the k pixels with the largest channel-max pattern magnitude (ties ->
 * lower index), zero P+/P- elsewhere.  keep (H*W bytes) and kth_key nullable.          */
int dmh_topk_select(float* pattern_pos, float* pattern_neg, int C, int H, int W, int k, unsigned char* keep,
                    unsigned* kth_key, dmh_stream_t stream);

/* -- A18 depth-hints objective, per scale (DepthNetworks/depth-hints/trainer.py:541-590
 * compute_loss_masks, :525-539 compute_proxy_supervised_loss, :666-713):
 * reproj_host[f] (B,1,H,W) per-frame reprojection losses, f < F <= 4; ident (B,F,H,W)
 * identity losses WITHOUT noise (NULL: automasking disabled); noise (B,1,H,W) nullable;
 * hint_reproj (B,1,H,W) = reprojection loss of the depth-hint warp + 1000*(1-hint_valid)
 * (NULL: no depth hints); depth = predicted depth, hint_depth, hint_valid (B,1,H,W).
 * Outputs: part = 4 x dmh_hint_select_blocks floats: per-CTA partial sums of
 *   [reproj*mask_r, mask_r, proxy*mask_h, mask_h]  (mask_r = argmin != identity,
 *   mask_h = argmin == hint); g_reproj_host[f] (B,1,H,W) = d(sum reproj*mask_r)/d reproj_f;
 *   g_depth (B,1,H,W) = d(sum proxy*mask_h)/d depth; sel (B,H,W) argmin index (nullable). */
int dmh_hint_select_blocks(int B, int H, int W);
int dmh_hint_select(const float* const* reproj_host, int F, const float* ident, const float* noise,
                    const float* hint_reproj, const float* depth, const float* hint_depth, const float* hint_valid,
                    int avg_reprojection, int B, int H, int W, float* part, float* const* g_reproj_host,
                    float* g_depth, unsigned char* sel, dmh_stream_t stream);

/* -- next-3: ManyDepth cost volume (DepthNetworks/manydepth2/networks/resnet_encoder.py:157-236,
 * ResnetEncoderMatching.match_features), no gradient (the reference builds it under no_grad):
 * current_feats (B,C,h,w), lookup_feats (B,L,C,h,w), poses (B,L,4,4) (an all-zero pose marks a missing
 * lookup frame), K, inv_K (B,4,4) at the matching resolution, depth_bins (D) on the device.
 * -> cost_volume (B,D,h,w) = mean over contributing lookups of mean_c |warp(lookup) - current| with the
 * 2-px edge masks, empty cells filled with the per-pixel max over the bins when set_missing_to_max;
 * missing_mask (B,D,h,w) = 1 where the cell was empty.  C must be 16, L <= 4.
 * workspace: dmh_cost_volume_workspace_floats floats, 16-byte aligned (channel-last copy of the lookups). */
long long dmh_cost_volume_workspace_floats(int B, int L, int C, int h, int w);
int dmh_cost_volume(const float* current_feats, const float* lookup_feats, const float* poses, const float* K,
                    const float* inv_K, const float* depth_bins, int B, int L, int C, int D, int h, int w,
                    int set_missing_to_max, float* workspace, float* cost_volume, float* missing_mask,
                    dmh_stream_t stream);

/* Diagnostics: 1 iff the library's 3-instruction division by the constant c (used for the /(W-1), /(H-1) of
 * Project3D, layers.py:195-196, in the fused kernel) has been verified bit-identical to IEEE division for
 * every float numerator on the current device (exhaustive over all significands; first call per constant
 * launches a small kernel and synchronises, then cached).  0: the kernels use IEEE division for that size. */
int dmh_const_div_exact(int c);

/* -- training-batch compositing on the device (SURVEY.md 8(f) next-2) ------------------------------------------
 * The byte work of MonoDataset.prep_adv_data + preprocess (DepthNetworks/monodepth2/datasets/mono_dataset.py:
 * 186-265, 119-144), which the reference runs per item inside DataLoader workers on the CPU.
 *
 * dmh_compose_u8: out = (uint8) trunc(255 * (scene/255 * (1 - mask) + obj * mask)) -- to_tensor, the composite
 * (:227-228, 246-249) and to_pilimage (`.mul(255).byte()`, :235-236, 251) in one pass; every fp32 operation
 * rounded as torch's CPU kernels round it.  scene (B,C,H,W) u8, obj (B,C,H,W) f32 (the warped patch, from
 * dmh_perspective_fwd), mask (B,1,H,W) f32, flip (B) int32 or NULL: items whose warped patch / mask are mirrored
 * horizontally first (torch.flip(..., [3]), :222-225).  scene == NULL: out = trunc(255 * obj) (the `color_objmask`
 * image, :254; mask may be NULL). */
int dmh_compose_u8(const uint8_t* scene, const float* obj, const float* mask, const int* flip, int B, int C, int H,
                   int W, uint8_t* out, dmh_stream_t stream);

/* dmh_compose_patch_u8: the same composite with the perspective warp inside (PhysicalTrans.project /
 * project_w_trans, physicalTrans.py:130-196, with the arithmetic of dmh_perspective_fwd): the (B,3,H,W) fp32 warped
 * canvases are never materialised.  patch_a / patch_b (1,3,ph,pw): up to two patches that share the placement
 * `coeffs` (B,8) and the mask (1,1,ph,pw) -- the adversarial and the benign patch on frame 0 (mono_dataset.py:
 * 207-251); patch_b / out_b may both be NULL.  bbox (B,4) int32 or NULL: conservative placement boxes (optimisation
 * hint only).  active (B) int32 or NULL: items with 0 get no patch (`half_no_synthesis`, :321-328: the raw frame
 * goes through unchanged).  out_a / out_b (B,3,H,W) u8; mask_out (B,1,H,W) u8 or NULL = to_pilimage of the warped
 * mask (:254). */
int dmh_compose_patch_u8(const uint8_t* scene, const float* patch_a, const float* patch_b, const float* patch_mask,
                         const float* coeffs, const int* bbox, const int* flip, const int* active, int B, int ph, int pw,
                         int H, int W, uint8_t* out_a, uint8_t* out_b, uint8_t* mask_out, dmh_stream_t stream);

/* dmh_lanczos_u8: `transforms.Resize((h, w), interpolation=Image.ANTIALIAS)` on 8-bit PIL images (:71, 100-104,
 * 126-131) == Pillow's fixed-point Lanczos resampling (libImaging/Resample.c), bit-exact: horizontal pass, then
 * vertical pass, each with 22-bit integer weights, rounded and clipped to 8 bits.  in (planes, in_h, in_w) ->
 * out (planes, out_h, out_w).  bounds_* (out, 2) int32 = (first input index, tap count), kk_* (ksize, out) int32
 * weights (tap-major, so that neighbouring outputs read neighbouring weights): host-computed in double precision as Pillow does (depthmodelhardening_b200/loader.py
 * lanczos_coefficients); an axis that keeps its size is skipped and needs no tables.  tmp: (planes, in_h, out_w)
 * bytes, needed when both axes change.  out_f32 (nullable, 16-byte aligned): additionally out / 255 in fp32 --
 * `to_tensor` of the resized image (:137-144), written by the last pass instead of a separate dmh_unpack_u8. */
int dmh_lanczos_u8(const uint8_t* in, int planes, int in_h, int in_w, int out_h, int out_w, const int* bounds_x,
                   const int* kk_x, int ksize_x, const int* bounds_y, const int* kk_y, int ksize_y, uint8_t* tmp,
                   uint8_t* out, float* out_f32, dmh_stream_t stream);

/* Colour jitter on 8-bit frames (next-2; DepthNetworks/monodepth2/datasets/mono_dataset.py:297, 344-350, applied to
 * every pyramid level in preprocess :140-144; torchvision ColorJitter.forward -> functional_pil -> PIL.ImageEnhance /
 * convert("HSV")): in (B,3,H,W) uint8; per item order (B,4) int32 = the drawn fn_idx (0 brightness, 1 contrast,
 * 2 saturation, 3 hue; < 0: step off), factors (B,3) = brightness / contrast / saturation factors, hue_shift (B)
 * int32 = uint8(hue_factor * 255) -- all DEVICE arrays; sums (B) uint64 workspace (per-image grey-level sums of the
 * contrast step).  out_u8 (B,3,H,W) and / or out_f32 = byte / 255 (to_tensor).  Pillow's integer / single-precision
 * arithmetic, bit-exact.  Two launches.                                                                        */
int dmh_color_jitter_u8(const uint8_t* in, int B, int H, int W, const int* order, const float* factors,
                        const int* hue_shift, unsigned long long* sums, uint8_t* out_u8, float* out_f32,
                        dmh_stream_t stream);

/* 8-bit frame transport (data format either side of the path): out[i] = (float)in[i] / 255 with IEEE division --
 * torchvision's `to_tensor` (`pic.to(float32).div(255)`), the conversion every colour frame of the reference goes
 * through in its loaders (DepthNetworks/monodepth2/datasets/mono_dataset.py:79, 133-144; composited frames are
 * re-quantised by to_pilimage first, :235-236) -- done on the device, so that a batch
 * can cross PCIe as bytes (a quarter of the fp32 volume) and still arrive bit-identical.  in/out 16-byte aligned. */
int dmh_unpack_u8(const uint8_t* in, long long n, float* out, dmh_stream_t stream);

/* out[i] = a[0] * x[i] + b[0] * y[i] with DEVICE scalars a, b (no host sync); out may alias x or y. */
int dmh_axpby_dev(const float* a, const float* x, const float* b, const float* y, long long n, float* out,
                  dmh_stream_t stream);

/* deterministic fixed-order sum of n floats into out[0] (double accumulate),
 * out[0] = scale * sum (+ out[0] if accumulate)                                */
int dmh_reduce_sum(const float* in, long long n, float scale, int accumulate, float* out, dmh_stream_t stream);
/* the same for every row of a (rows, n) array in one launch: out[r] = scale * sum(in[r, :])  (the four masked sums
 * of the depth-hints objective, DH/trainer.py:699-713) */
int dmh_reduce_rows(const float* in, int rows, long long n, float scale, float* out, dmh_stream_t stream);

/* -- SURVEY.md 8(e): the ONE collective of stage 1, as one kernel over NVLink peer memory -----------------------
 * all-reduce(sum) of the shared patch gradient (the scalar attack loss rides in its tail), scaled by `scale`
 * (1 / world: dist.allreduce_patch_grad's average), optionally fused with the L-inf PGD update that consumes it
 * (TA/attacks/phy_obj_atk.py:98-100) -- replaces torch.distributed.all_reduce (NCCL) + div_ [+ dmh_pgd_linf_step].
 * peer_bufs_host[r]  = rank r's n-float gradient buffer AS MAPPED IN THIS PROCESS (a symmetric allocation: CUDA VMM
 *                      handles exchanged by the host, e.g. torch.distributed._symmetric_memory), 16-byte aligned;
 * peer_flags_host[r] = rank r's flag block, 2 * world uint32 (zeroed once before the first call), same mapping rule;
 * state              = 2 uint32 of LOCAL device memory (zeroed once): step counter, CTA arrival counter;
 * out                = n LOCAL floats: sum over ranks in rank order (the same bits on every rank) * scale;
 * adv / clean / adv_out (all NULL: no update; else n_update <= n floats each): adv_out = clamp(clean +
 *                      clamp(adv + alpha * sign(out) - clean, +-eps), 0, 1).
 * Every rank of the group must enqueue the call for the same step (like a collective).  The kernel synchronises the
 * ranks through the flag blocks (system-scope release / acquire) at its start and at its end: when it retires, the
 * rank's buffer may be overwritten by the next step.  The step counter lives on the device: CUDA-graph capturable. */
int dmh_peer_allreduce(const float* const* peer_bufs_host, unsigned* const* peer_flags_host, int rank, int world,
                       long long n, float scale, float* out, unsigned* state, const float* adv, const float* clean,
                       long long n_update, float alpha, float eps, float* adv_out, dmh_stream_t stream);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* DMH_B200_H */
