"""torch.autograd.Function wrappers around the C-ABI kernels (stage 2).

PyTorch is plumbing here: it owns the buffers (caching allocator) and the
stream; every numeric result comes from libdmh_b200.so.  Backward passes
recompute from the saved *inputs* -- no intermediate is kept (SURVEY.md 8(b)).
"""
from __future__ import annotations

from typing import List, Optional, Sequence

import torch

from . import _lib
from ._lib import check, f32c, ptr, ptr_array, stream

PAD_MODES = {"zeros": 0, "border": 1}

# bench.py sets this to a list to collect (name, start_event, end_event) around
# selected kernel launches on the launching stream; None = no instrumentation.
KERNEL_EVENTS = None


class _timed:
    def __init__(self, name):
        self.name = name

    def __enter__(self):
        if KERNEL_EVENTS is not None:
            self.a = torch.cuda.Event(enable_timing=True)
            self.b = torch.cuda.Event(enable_timing=True)
            self.a.record()

    def __exit__(self, *exc):
        if KERNEL_EVENTS is not None:
            self.b.record()
            KERNEL_EVENTS.append((self.name, self.a, self.b))
        return False


def _lib_():
    return _lib.load()


def _mat_batch(m: torch.Tensor, B: int, name: str) -> torch.Tensor:
    """(B,4,4) camera matrix for a kernel that indexes `m + b*16`.  The reference relies on broadcasting -- ManyDepth's
    `match_features` hands (1,4,4) matrices to `BackprojectDepth(batch_size=96)` / `Project3D`
    (MD/networks/resnet_encoder.py:182,194) -- so a batch-1 matrix is expanded; anything else raises (torch.matmul
    would raise for it too) instead of reading past the end of the buffer.  The gradient of an expanded matrix is
    summed back over the batch by autograd's expand."""
    if m.dim() == 2:
        m = m.unsqueeze(0)
    if m.dim() != 3 or tuple(m.shape[1:]) != (4, 4):
        raise RuntimeError("%s must be (B,4,4) or (1,4,4), got %s" % (name, tuple(m.shape)))
    if m.shape[0] == B:
        return m
    if m.shape[0] == 1:
        return m.expand(B, 4, 4)
    raise RuntimeError("%s holds %d matrices but the batch is %d (only a batch of 1 broadcasts)" % (name, m.shape[0], B))


def _same_shape(op, a, b, an, bn):
    """Raise (as torch would) when two inputs that a kernel indexes with one set of dimensions disagree in shape."""
    if a.shape != b.shape:
        raise RuntimeError("%s: %s and %s must have the same shape, got %s and %s" %
                           (op, an, bn, tuple(a.shape), tuple(b.shape)))


def _disp_matches(op, disp, img, img_name):
    """A (B,1,H,W) disparity / depth map and the (B,C,H,W) image it belongs to."""
    if disp.dim() != 4 or img.dim() != 4 or disp.shape[1] != 1 or disp.shape[0] != img.shape[0] \
            or disp.shape[2:] != img.shape[2:]:
        raise RuntimeError("%s: expected disp of shape (B,1,H,W) matching %s (B,C,H,W), got disp %s and %s %s" %
                           (op, img_name, tuple(disp.shape), img_name, tuple(img.shape)))


# ----------------------------------------------------------------------------- A9
def disp_to_depth_cuda(disp: torch.Tensor, min_depth: float, max_depth: float):
    d = f32c(disp)
    scaled = torch.empty_like(d)
    depth = torch.empty_like(d)
    check(_lib_().dmh_disp_to_depth(ptr(d), d.numel(), min_depth, max_depth, ptr(scaled), ptr(depth), stream()),
          "disp_to_depth")
    return scaled, depth


class _DispToDepth(torch.autograd.Function):
    @staticmethod
    def forward(ctx, disp, min_depth, max_depth):
        scaled, depth = disp_to_depth_cuda(disp, min_depth, max_depth)
        ctx.save_for_backward(depth)
        ctx.range = 1.0 / min_depth - 1.0 / max_depth
        return scaled, depth

    @staticmethod
    def backward(ctx, g_scaled, g_depth):
        (depth,) = ctx.saved_tensors
        g = None
        if g_scaled is not None:
            g = g_scaled * ctx.range
        if g_depth is not None:
            gd = g_depth * (-ctx.range) * depth * depth
            g = gd if g is None else g + gd
        return g, None, None


# ----------------------------------------------------------------------------- A10
class _Backproject(torch.autograd.Function):
    @staticmethod
    def forward(ctx, depth, inv_K, B, H, W):
        d, ik = f32c(depth), f32c(inv_K)
        pts = torch.empty(B, 4, H * W, device=d.device, dtype=torch.float32)
        check(_lib_().dmh_backproject_fwd(ptr(d), ptr(ik), B, H, W, ptr(pts), stream()), "backproject_fwd")
        ctx.save_for_backward(d if ctx.needs_input_grad[1] else None, ik)     # depth: only for d/d(inv_K)
        ctx.dims = (B, H, W, depth.shape)
        return pts

    @staticmethod
    def backward(ctx, g_pts):
        d, ik = ctx.saved_tensors
        B, H, W, shape = ctx.dims
        g = f32c(g_pts)
        gd = torch.empty(B, 1, H, W, device=g.device, dtype=torch.float32) if ctx.needs_input_grad[0] else None
        nblk = _lib_().dmh_backproject_bwd_blocks(H, W)
        giK_part = torch.empty(B, nblk, 9, device=g.device, dtype=torch.float32) if ctx.needs_input_grad[1] else None
        check(_lib_().dmh_backproject_bwd(ptr(g), ptr(d), ptr(ik), B, H, W, ptr(gd), ptr(giK_part), stream()),
              "backproject_bwd")
        giK = None
        if giK_part is not None:
            # cam = depth * (inv_K[:3,:3] @ pix): only the 3x3 block receives a gradient
            giK = torch.zeros(B, 4, 4, device=g.device, dtype=torch.float32)
            giK[:, :3, :3] = giK_part.sum(1).view(B, 3, 3)
        return (gd.view(shape) if gd is not None else None), giK, None, None, None


# ----------------------------------------------------------------------------- A11
class _Project3D(torch.autograd.Function):
    @staticmethod
    def forward(ctx, points, K, T, B, H, W, eps):
        p, k, t = f32c(points), f32c(K), f32c(T)
        grid = torch.empty(B, H, W, 2, device=p.device, dtype=torch.float32)
        check(_lib_().dmh_project3d_fwd(ptr(p), ptr(k), ptr(t), B, H, W, eps, ptr(grid), stream()), "project3d_fwd")
        ctx.save_for_backward(p, k, t)
        ctx.dims = (B, H, W, eps)
        return grid

    @staticmethod
    def backward(ctx, g_grid):
        p, k, t = ctx.saved_tensors
        B, H, W, eps = ctx.dims
        g = f32c(g_grid)
        need_pts = ctx.needs_input_grad[0]
        need_kt = ctx.needs_input_grad[1] or ctx.needs_input_grad[2]
        g_pts = torch.empty_like(p) if need_pts else None
        nblk = _lib_().dmh_project3d_bwd_blocks(H, W)
        gP_part = torch.empty(B, nblk, 12, device=g.device, dtype=torch.float32) if need_kt else None
        check(_lib_().dmh_project3d_bwd(ptr(g), ptr(p), ptr(k), ptr(t), B, H, W, eps, ptr(g_pts), ptr(gP_part),
                                        stream()), "project3d_bwd")
        gK = gT = None
        if need_kt:
            gK, gT = _grad_KT_from_P(gP_part.sum(1).view(B, 3, 4), k, t, ctx.needs_input_grad[1],
                                     ctx.needs_input_grad[2])
        return g_pts, gK, gT, None, None, None, None


def _grad_KT_from_P(gP, K, T, need_K, need_T):
    """P = (K @ T)[:3,:]  ->  dK[:3,:] = gP @ T^T,  dT = K[:3,:]^T @ gP   (tiny 4x4 algebra)."""
    B = gP.shape[0]
    gK = gT = None
    if need_K:
        gK = torch.zeros(B, 4, 4, device=gP.device, dtype=gP.dtype)
        gK[:, :3, :] = torch.matmul(gP, T.transpose(1, 2))
    if need_T:
        gT = torch.matmul(K[:, :3, :].transpose(1, 2), gP)
    return gK, gT


def _pose_grad_T(gPs, u, f, K, T):
    """d(loss)/d(T) of source f from the per-scale pose-gradient partials gPs[s] (F,B,tiles,12): summed over the tiles,
    weighted by the upstream u[s] and added in scale order."""
    acc = None
    for s, gP in enumerate(gPs):
        t = gP[f].sum(1) * u[s]
        acc = t if acc is None else acc + t
    return _grad_KT_from_P(acc.view(-1, 3, 4), K, T, False, True)[1]


# ----------------------------------------------------------------------------- A12
class _GridSample(torch.autograd.Function):
    @staticmethod
    def forward(ctx, src, grid, padding_mode, align_corners):
        if src.dim() != 4 or grid.dim() != 4:
            raise RuntimeError("grid_sample: expected 4-D input and grid, got input %s and grid %s" %
                               (tuple(src.shape), tuple(grid.shape)))
        if grid.shape[0] != src.shape[0]:
            raise RuntimeError("grid_sample: expected grid and input to have same batch size, but got input with "
                               "sizes %s and grid with sizes %s" % (list(src.shape), list(grid.shape)))
        if grid.shape[3] != 2:
            raise RuntimeError("grid_sample: expected grid to have size 2 in last dimension, but got grid with "
                               "sizes %s" % list(grid.shape))
        s, g = f32c(src), f32c(grid)
        B, Cc, Hs, Ws = s.shape
        _, Ho, Wo, _ = g.shape
        out = torch.empty(B, Cc, Ho, Wo, device=s.device, dtype=torch.float32)
        check(_lib_().dmh_grid_sample_fwd(ptr(s), ptr(g), B, Cc, Hs, Ws, Ho, Wo, padding_mode, int(align_corners),
                                          ptr(out), stream()), "grid_sample_fwd")
        ctx.save_for_backward(s, g)
        ctx.cfg = (padding_mode, int(align_corners))
        return out

    @staticmethod
    def backward(ctx, g_out):
        s, g = ctx.saved_tensors
        pm, ac = ctx.cfg
        B, Cc, Hs, Ws = s.shape
        _, Ho, Wo, _ = g.shape
        go = f32c(g_out)
        g_src = torch.zeros_like(s) if ctx.needs_input_grad[0] else None
        g_grid = torch.empty_like(g) if ctx.needs_input_grad[1] else None
        check(_lib_().dmh_grid_sample_bwd(ptr(go), ptr(s), ptr(g), B, Cc, Hs, Ws, Ho, Wo, pm, ac, ptr(g_src),
                                          ptr(g_grid), stream()), "grid_sample_bwd")
        return g_src, g_grid, None, None


def grid_sample(src, grid, mode="bilinear", padding_mode="zeros", align_corners=False):
    """Bilinear `F.grid_sample` on the CUDA kernels (zeros | border padding)."""
    if mode != "bilinear":
        raise NotImplementedError("dmh_b200.grid_sample: only bilinear is on the hot path")
    if padding_mode not in PAD_MODES:
        raise NotImplementedError("dmh_b200.grid_sample: padding_mode %r unsupported" % padding_mode)
    return _GridSample.apply(src, grid, PAD_MODES[padding_mode], bool(align_corners))


# ----------------------------------------------------------------------------- A13
class _SSIM(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, y):
        _same_shape("SSIM", x, y, "x", "y")
        a, b = f32c(x), f32c(y)
        B, Cc, H, W = a.shape
        out = torch.empty_like(a)
        check(_lib_().dmh_ssim_fwd(ptr(a), ptr(b), B, Cc, H, W, ptr(out), stream()), "ssim_fwd")
        ctx.save_for_backward(a, b)
        return out

    @staticmethod
    def backward(ctx, g_out):
        a, b = ctx.saved_tensors
        B, Cc, H, W = a.shape
        g = f32c(g_out)
        gx = torch.empty_like(a) if ctx.needs_input_grad[0] else None
        gy = torch.empty_like(a) if ctx.needs_input_grad[1] else None
        check(_lib_().dmh_ssim_bwd(ptr(g), ptr(a), ptr(b), B, Cc, H, W, ptr(gx), ptr(gy), stream()), "ssim_bwd")
        return gx, gy


# ----------------------------------------------------------------------------- A14
class _ReprojLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pred, target, no_ssim):
        _same_shape("reprojection_loss", pred, target, "pred", "target")
        a, b = f32c(pred), f32c(target)
        B, Cc, H, W = a.shape
        out = torch.empty(B, 1, H, W, device=a.device, dtype=torch.float32)
        check(_lib_().dmh_reproj_loss_fwd(ptr(a), ptr(b), B, Cc, H, W, int(no_ssim), ptr(out), stream()),
              "reproj_loss_fwd")
        ctx.save_for_backward(a, b)
        ctx.no_ssim = int(no_ssim)
        return out

    @staticmethod
    def backward(ctx, g_out):
        a, b = ctx.saved_tensors
        B, Cc, H, W = a.shape
        g = f32c(g_out)
        gp = torch.empty_like(a) if ctx.needs_input_grad[0] else None
        gt = torch.empty_like(a) if ctx.needs_input_grad[1] else None
        check(_lib_().dmh_reproj_loss_bwd(ptr(g), ptr(a), ptr(b), B, Cc, H, W, ctx.no_ssim, ptr(gp), ptr(gt),
                                          stream()), "reproj_loss_bwd")
        return gp, gt, None


def reprojection_loss(pred, target, no_ssim=False):
    return _ReprojLoss.apply(pred, target, bool(no_ssim))


# ----------------------------------------------------------------------------- A16
class _Smooth(torch.autograd.Function):
    @staticmethod
    def forward(ctx, disp, img, normalise):
        _disp_matches("smooth_loss", disp, img, "img")
        d, im = f32c(disp), f32c(img)
        B, _, h, w = d.shape
        Cc = im.shape[1]
        ws = torch.empty(_lib_().dmh_smooth_workspace_floats(B, h, w), device=d.device, dtype=torch.float32)
        loss = torch.empty((), device=d.device, dtype=torch.float32)
        check(_lib_().dmh_smooth_fwd(ptr(d), ptr(im), B, Cc, h, w, int(normalise), ptr(ws), ptr(loss), stream()),
              "smooth_fwd")
        ctx.save_for_backward(d, im)
        ctx.normalise = int(normalise)
        return loss

    @staticmethod
    def backward(ctx, g_loss):
        d, im = ctx.saved_tensors
        B, _, h, w = d.shape
        Cc = im.shape[1]
        ws = torch.empty(_lib_().dmh_smooth_workspace_floats(B, h, w), device=d.device, dtype=torch.float32)
        gl = f32c(g_loss).reshape(1)
        gd = torch.empty_like(d)
        gi = torch.empty_like(im) if ctx.needs_input_grad[1] else None
        check(_lib_().dmh_smooth_bwd(ptr(d), ptr(im), B, Cc, h, w, ctx.normalise, ptr(gl), 1.0, ptr(ws), ptr(gd),
                                     ptr(gi), stream()), "smooth_bwd")
        return gd, gi, None


def smooth_loss(disp, img, normalise=False):
    return _Smooth.apply(disp, img, bool(normalise))



# ----------------------------------------------------------------------------- F.interpolate (trainer.py:481-482)
class _UpsampleBilinear(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, H, W):
        a = f32c(x)
        B, Cc, h, w = a.shape
        out = torch.empty(B, Cc, H, W, device=a.device, dtype=torch.float32)
        check(_lib_().dmh_upsample_bilinear_fwd(ptr(a), B * Cc, h, w, H, W, ptr(out), stream()), "upsample_fwd")
        ctx.dims = (B, Cc, h, w, H, W)
        return out

    @staticmethod
    def backward(ctx, g_out):
        B, Cc, h, w, H, W = ctx.dims
        g = f32c(g_out)
        gi = torch.empty(B, Cc, h, w, device=g.device, dtype=torch.float32)
        check(_lib_().dmh_upsample_bilinear_bwd(ptr(g), B * Cc, h, w, H, W, None, ptr(gi), stream()), "upsample_bwd")
        return gi, None, None


def upsample_bilinear(x, size):
    """`F.interpolate(x, size, mode="bilinear", align_corners=False)` with a
    deterministic (gather) backward."""
    return _UpsampleBilinear.apply(x, int(size[0]), int(size[1]))

# ----------------------------------------------------------------------------- A9-A12 fused
class _WarpFused(torch.autograd.Function):
    @staticmethod
    def forward(ctx, disp, src, K, inv_K, T, min_depth, max_depth, input_is_depth):
        _disp_matches("warp_reproject", disp, src, "src")
        d, s, k, ik, t = f32c(disp), f32c(src), f32c(K), f32c(inv_K), f32c(T)
        B, Cc, H, W = s.shape
        out = torch.empty_like(s)
        check(_lib_().dmh_warp_fwd(ptr(d), int(input_is_depth), min_depth, max_depth, ptr(s), ptr(k), ptr(ik), ptr(t),
                                   B, Cc, H, W, ptr(out), None, None, stream()), "warp_fwd")
        ctx.save_for_backward(d, s, k, ik, t)
        ctx.cfg = (float(min_depth), float(max_depth), int(input_is_depth), disp.shape)
        return out

    @staticmethod
    def backward(ctx, g_out):
        d, s, k, ik, t = ctx.saved_tensors
        mn, mx, isd, dshape = ctx.cfg
        B, Cc, H, W = s.shape
        g = f32c(g_out)
        need_d, need_s = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        need_kt = ctx.needs_input_grad[2] or ctx.needs_input_grad[4]
        gd = torch.empty_like(d) if need_d else None
        gs = torch.zeros_like(s) if need_s else None
        nblk = _lib_().dmh_warp_bwd_blocks(H, W)
        gP = torch.empty(B, nblk, 12, device=g.device, dtype=torch.float32) if need_kt else None
        check(_lib_().dmh_warp_bwd(ptr(g), ptr(d), isd, mn, mx, ptr(s), ptr(k), ptr(ik), ptr(t), B, Cc, H, W, ptr(gd),
                                   ptr(gs), ptr(gP), stream()), "warp_bwd")
        gK = gT = None
        if need_kt:
            gK, gT = _grad_KT_from_P(gP.sum(1).view(B, 3, 4), k, t, ctx.needs_input_grad[2], ctx.needs_input_grad[4])
        return (gd.view(dshape) if gd is not None else None), gs, gK, None, gT, None, None, None


def warp_reproject(disp, src, K, inv_K, T, min_depth=0.1, max_depth=100.0, input_is_depth=False):
    """disp (B,1,H,W) [or depth] + src (B,C,H,W) -> src warped into the target view.
    One gather kernel for trainer.py:485-519 (disp_to_depth, BackprojectDepth,
    Project3D, grid_sample(border, align_corners=True)).  Differentiable w.r.t. disp, src, K and T, not inv_K: an
    inv_K that requires grad is refused rather than given a zero gradient."""
    if inv_K.requires_grad and torch.is_grad_enabled():
        raise RuntimeError("warp_reproject: no gradient w.r.t. inv_K; detach it (or use BackprojectDepth / Project3D, "
                           "which return one)")
    B = src.shape[0]
    return _WarpFused.apply(disp, src, _mat_batch(K, B, "K"), _mat_batch(inv_K, B, "inv_K"), _mat_batch(T, B, "T"),
                            float(min_depth), float(max_depth), bool(input_is_depth))


def warp_with_aux(disp, src, K, inv_K, T, min_depth=0.1, max_depth=100.0, input_is_depth=False, align_corners=True,
                  want_aux=True):
    """No-grad variant also returning the sampling grid and the depth map
    (the tensors the reference stores in `outputs` for logging).  align_corners=False: the sampling convention of
    the depth-hints warp (`F.grid_sample` default, DH/trainer.py:523-525).  Returns no gradient, so an input that
    requires grad is refused while grad mode is on."""
    if torch.is_grad_enabled() and any(t.requires_grad for t in (disp, src, K, inv_K, T)):
        raise RuntimeError("warp_with_aux returns no gradient; call it under torch.no_grad() or use warp_reproject")
    _disp_matches("warp_with_aux", disp, src, "src")
    B = src.shape[0]
    d, s, k, ik, t = (f32c(disp), f32c(src), f32c(_mat_batch(K, B, "K")), f32c(_mat_batch(inv_K, B, "inv_K")),
                      f32c(_mat_batch(T, B, "T")))
    B, Cc, H, W = s.shape
    out = torch.empty_like(s)
    grid = torch.empty(B, H, W, 2, device=s.device, dtype=torch.float32) if want_aux else None
    depth = torch.empty(B, 1, H, W, device=s.device, dtype=torch.float32) if want_aux else None
    mode = (1 if input_is_depth else 0) | (0 if align_corners else 2)       # dmh_warp_fwd: bit 0 depth input, bit 1 half-pixel
    check(_lib_().dmh_warp_fwd(ptr(d), mode, min_depth, max_depth, ptr(s), ptr(k), ptr(ik), ptr(t),
                               B, Cc, H, W, ptr(out), ptr(grid), ptr(depth), stream()), "warp_fwd")
    return out, grid, depth


# ----------------------------------------------------------------------------- A9-A15 fused
FLAG_NO_SSIM = 1
FLAG_AVG_REPROJECTION = 2
FLAG_INPUT_IS_DEPTH = 4
FLAG_SEL_SOURCE = 8          # dmh_photo_scale_dh: sel also records the winning source frame (sel >> 2)
FLAG_SRC_PACKED = 16
FLAG_PIXEL_SUM = 32          # dmh_photo_image_grad: the loss is the sum over the pixels (photo_scale_sum), not the mean


class _PhotoScale(torch.autograd.Function):
    """sum over (B,H,W) of the per-pixel min-reprojection loss for one scale, with
    its gradient w.r.t. the full-resolution disparity (and poses) produced in the
    same kernel launch.  Gradients for the target, the sources and the identity losses
    are recomputed in the backward from the saved frames and the forward's `sel`."""

    @staticmethod
    def forward(ctx, disp, target, ident, noise, K, inv_K, min_depth, max_depth, flags, want_sel, n_src, *src_and_T):
        srcs = [f32c(t) for t in src_and_T[:n_src]]
        Ts = [f32c(t) for t in src_and_T[n_src:]]
        d, tg, k, ik = f32c(disp), f32c(target), f32c(K), f32c(inv_K)
        idn = f32c(ident) if ident is not None else None
        nz = f32c(noise) if noise is not None else None
        B, _, H, W = tg.shape
        lib = _lib_()
        tiles = lib.dmh_photo_tiles(H, W)
        part = torch.empty(B * tiles, device=d.device, dtype=torch.float32)
        gdisp = torch.empty_like(d)
        need_T = any(ctx.needs_input_grad[11 + n_src + i] for i in range(n_src))
        # gradients for the frames and the identity losses follow the forward's decision, so `sel` is requested
        # internally
        colour_grad = ctx.needs_input_grad[1] or any(ctx.needs_input_grad[11 + i] for i in range(n_src))
        ident_grad = ctx.needs_input_grad[2]
        gP = torch.empty(n_src, B, tiles, 12, device=d.device, dtype=torch.float32) if need_T else None
        want_sels = want_sel or colour_grad or ident_grad
        sel = torch.empty(B, H, W, device=d.device, dtype=torch.uint8) if want_sels else None
        with _timed("photo_scale"):
            check(lib.dmh_photo_scale(ptr(tg), ptr_array(srcs), ptr_array(Ts), n_src, ptr(d), H, W, ptr(k), ptr(ik),
                                      ptr(idn), ptr(nz), B, H, W, min_depth, max_depth, flags, 1.0, ptr(part),
                                      ptr(gdisp), ptr(gP), ptr(sel), None, stream()), "photo_scale")
        total = torch.empty((), device=d.device, dtype=torch.float32)
        check(lib.dmh_reduce_sum(ptr(part), part.numel(), 1.0, 0, ptr(total), stream()), "reduce_sum")
        ctx.n_src = n_src
        ctx.dshape = disp.shape
        ctx.colour = None
        extra = []
        if colour_grad or ident_grad:
            ctx.colour = (float(min_depth), float(max_depth), flags, target.dtype, [t.dtype for t in src_and_T[:n_src]],
                          ident.dtype if ident is not None else None, ident.shape[1] if ident is not None else 0)
            extra = [sel, ik, d, tg, *srcs] if colour_grad else [sel]
        ctx.save_for_backward(gdisp, gP, k, *Ts, *extra)
        if want_sel:
            ctx.mark_non_differentiable(sel)
            return total, sel
        return total, None

    @staticmethod
    def backward(ctx, g_total, _g_sel):
        saved = ctx.saved_tensors
        gdisp, gP, k = saved[0], saved[1], saved[2]
        n_src = ctx.n_src
        Ts = saved[3:3 + n_src]
        g_d = (gdisp * g_total).view(ctx.dshape) if ctx.needs_input_grad[0] else None
        g_T: List[Optional[torch.Tensor]] = [None] * n_src
        if gP is not None:
            gPs = gP.sum(2) * g_total            # (F,B,12)
            for i in range(n_src):
                if ctx.needs_input_grad[11 + n_src + i]:
                    _, g_T[i] = _grad_KT_from_P(gPs[i].view(-1, 3, 4), k, Ts[i], False, True)
        g_tg, g_id, g_src = None, None, [None] * n_src
        if ctx.colour is not None:
            g_tg, g_id, g_src = _PhotoScale._input_grads(ctx, saved[3 + n_src:], k, Ts, f32c(g_total).reshape(1))
        return (g_d, g_tg, g_id, None, None, None, None, None, None, None, None) + tuple(g_src) + tuple(g_T)

    @staticmethod
    def _input_grads(ctx, saved, k, Ts, gt):
        """d(sum)/d(target), d(sum)/d(source f) and d(sum)/d(ident) for the inputs that require them (None for the
        rest), in each input's dtype.  The identity losses are inputs here, so the frames only receive the
        reprojection terms (one dmh_photo_image_grad launch); an identity plane receives g_total where `sel` picked
        it (g_total / F on every plane under avg_reprojection, which compares their mean)."""
        min_depth, max_depth, flags, tg_dtype, src_dtypes, id_dtype, n_planes = ctx.colour
        n_src = ctx.n_src
        sel = saved[0]
        g_tg, g_id, g_src = None, None, [None] * n_src
        if ctx.needs_input_grad[2]:
            if flags & FLAG_AVG_REPROJECTION:
                g_id = ((sel == 0).unsqueeze(1) * (gt / n_planes)).expand(-1, n_planes, -1, -1)
            else:
                planes = torch.arange(n_planes, device=sel.device, dtype=sel.dtype).view(1, -1, 1, 1)
                g_id = (sel.unsqueeze(1) == planes) * gt
            g_id = g_id.to(id_dtype).contiguous()
        need_tg = ctx.needs_input_grad[1]
        need_src = [bool(ctx.needs_input_grad[11 + i]) for i in range(n_src)]
        if need_tg or any(need_src):
            ik, d, tg = saved[1], saved[2], saved[3]
            srcs = saved[4:4 + n_src]
            B, _, H, W = tg.shape
            g_tg = torch.zeros_like(tg) if need_tg else None
            g_src = [torch.zeros_like(srcs[i]) if need_src[i] else None for i in range(n_src)]
            with _timed("photo_image_grad"):
                check(_lib_().dmh_photo_image_grad(ptr(tg), ptr_array(srcs), ptr_array(Ts), n_src, ptr(d), H, W,
                                                   ptr(k), ptr(ik), ptr(sel), 0, 1, ptr(gt), None, B, H, W, min_depth,
                                                   max_depth, (flags & (FLAG_NO_SSIM | FLAG_AVG_REPROJECTION |
                                                                        FLAG_INPUT_IS_DEPTH)) | FLAG_PIXEL_SUM,
                                                   int(n_planes > 0), ptr(g_tg), ptr_array(g_src), stream()),
                      "photo_image_grad")
            g_tg = g_tg if g_tg is None or g_tg.dtype == tg_dtype else g_tg.to(tg_dtype)
            g_src = [g if g is None or g.dtype == dt else g.to(dt) for g, dt in zip(g_src, src_dtypes)]
        return g_tg, g_id, g_src


def photo_scale_sum(disp_full, target, srcs: Sequence[torch.Tensor], Ts: Sequence[torch.Tensor], K, inv_K,
                    ident=None, noise=None, min_depth=0.1, max_depth=100.0, no_ssim=False, avg_reprojection=False,
                    input_is_depth=False, want_sel=False):
    """Sum over (B,H,W) of the per-pixel minimum over [ident (+ noise), reprojection of each source] at full
    resolution.  disp_full (B,1,H,W) [or depth with input_is_depth]; ident (B,F,H,W) identity losses (averaged over
    the frames under avg_reprojection) or None; noise (B,F,H,W) ((B,1,H,W) under avg_reprojection) or None.
    Differentiable w.r.t. disp_full, the poses, the target, the sources and ident (not noise, K or inv_K).
    Returns (total, sel or None)."""
    if tuple(disp_full.shape[-2:]) != tuple(target.shape[-2:]):
        raise ValueError("photo_scale_sum: the disparity (%dx%d) must have the target's resolution (%dx%d)" %
                         (*disp_full.shape[-2:], *target.shape[-2:]))
    flags = (FLAG_NO_SSIM if no_ssim else 0) | (FLAG_AVG_REPROJECTION if avg_reprojection else 0) | \
            (FLAG_INPUT_IS_DEPTH if input_is_depth else 0)
    B = target.shape[0]
    return _PhotoScale.apply(disp_full, target, ident, noise, _mat_batch(K, B, "K"), _mat_batch(inv_K, B, "inv_K"),
                             float(min_depth), float(max_depth), flags, bool(want_sel), len(srcs), *srcs,
                             *[_mat_batch(t, B, "T") for t in Ts])


# ----------------------------------------------------------------------------- whole multi-scale objective
import ctypes as _C
import os as _os

_SIDE_STREAMS = {}
# all scales of the single-source objective in one launch (csrc/photo_ms.cu, bit-identical to the per-scale launches);
# DMH_MULTISCALE=0 keeps one launch per scale
MULTISCALE = _os.environ.get("DMH_MULTISCALE", "1") != "0"
# several source frames and / or pose gradients: all sources and all scales in one launch of the tile kernel
# (csrc/photo_mf.cu); DMH_MULTISOURCE=0 keeps the general per-scale kernel (csrc/photo_objective.cu)
MULTISOURCE = _os.environ.get("DMH_MULTISOURCE", "1") != "0"
# The glue steps stay one launch per scale: those launches run as independent branches (streams / graph nodes) beside
# the photometric kernel.  All-scales launches were measured on B200 and were no faster per step (DESIGN.md section 4).


def _side_stream(dev, which=0):
    """Side streams of a device, created once: 0 = high priority (smoothness launches), 1 = normal priority."""
    idx = torch.device(dev).index if torch.device(dev).index is not None else torch.cuda.current_device()
    key = (idx, which)
    st = _SIDE_STREAMS.get(key)
    if st is None:
        st = _SIDE_STREAMS[key] = torch.cuda.Stream(device=idx, priority=-1 if which == 0 else 0)
    return st


class _Objective(torch.autograd.Function):
    """generate_images_pred + compute_losses (photometric part) for ALL scales as one
    autograd node: forward = ident + S x (photo kernel with fused up-sampling, smooth
    fused) + one finish launch; backward = one dmh_disp_grad launch per scale that
    applies the incoming scalar gradient(s) on the device."""

    @staticmethod
    def forward(ctx, K, inv_K, cfg, *tensors):
        (min_depth, max_depth, flags, smooth_w, want_sel, n_src, S, automask, has_noise) = cfg
        it = iter(tensors)
        colors_in = [next(it) for _ in range(S)]             # color(0, s)
        srcs_in = [next(it) for _ in range(n_src)]
        # bf16 frames (2e-3 tolerance class): the full-resolution target / source are read AS bf16 by the identity
        # kernel (128-bit loads of 8 elements), which also writes the widened target -- no up-cast pass over them
        bf16_frames = (n_src == 1 and colors_in[0].dtype == torch.bfloat16 and srcs_in[0].dtype == torch.bfloat16
                       and colors_in[0].is_cuda and colors_in[0].shape[3] % 8 == 0 and not (flags & FLAG_NO_SSIM))
        if bf16_frames:
            colors = [colors_in[0].contiguous()] + [f32c(c) for c in colors_in[1:]]
            srcs = [srcs_in[0].contiguous()]
        else:
            colors = [f32c(c) for c in colors_in]
            srcs = [f32c(t) for t in srcs_in]
        Ts = [f32c(next(it)) for _ in range(n_src)]
        disps = [f32c(next(it)) for _ in range(S)]
        noises = [f32c(next(it)) for _ in range(S)] if has_noise else [None] * S
        k, ik = f32c(K), f32c(inv_K)
        target = colors[0]
        B, _, H, W = target.shape
        dev = target.device
        lib = _lib_()
        no_ssim = 1 if (flags & FLAG_NO_SSIM) else 0
        # disp grads are needed iff any disparity requires grad; pose grads iff any T does
        base = 3 + S + n_src
        need_T = any(ctx.needs_input_grad[base + i] for i in range(n_src))
        # gradients for the colour frames (target, pyramid, sources): the backward recomputes them from the frames,
        # the disparities and every scale's selection, so `sel` is requested internally
        colour_grad = any(ctx.needs_input_grad[3 + i] for i in range(S + n_src))
        # single source, no pose gradient: the per-scale kernel gathers from a pixel-packed (B,H,W,4) copy of the
        # source (one 128-bit load per bilinear tap), written once by the identity-loss kernel
        packed = n_src == 1 and not need_T and not no_ssim and H * W < (1 << 28)
        if bf16_frames and not (packed and target.data_ptr() % 16 == 0 and srcs[0].data_ptr() % 16 == 0):
            bf16_frames = False                             # general kernels: widen first
            target = colors[0] = f32c(target)
            srcs = [f32c(srcs[0])]
        # mono / mono+stereo / multi-frame (or one source with pose gradients): every source is packed and the
        # tile kernel walks sources and scales in one launch
        multisrc = (MULTISOURCE and not packed and not no_ssim and not (flags & (FLAG_AVG_REPROJECTION | FLAG_INPUT_IS_DEPTH))
                    and 1 <= n_src <= 4 and S <= 4 and W % 4 == 0 and H * W < (1 << 27) and target.data_ptr() % 16 == 0)
        ident = torch.empty(B, n_src, H, W, device=dev, dtype=torch.float32) if (automask and not multisrc) else None
        src_arr = ptr_array(srcs) if not bf16_frames else None
        if multisrc:
            src_pks = [torch.empty(B, H, W, 4, device=dev, dtype=torch.float32) for _ in range(n_src)]
            idents = [torch.empty(B, 1, H, W, device=dev, dtype=torch.float32) if automask else None for _ in range(n_src)]
            for f in range(n_src):
                check(lib.dmh_identity_loss_pack(ptr(target), ptr(srcs[f]), B, H, W, 0, ptr(idents[f]), ptr(src_pks[f]),
                                                 stream()), "identity_loss_pack")
        elif packed:
            src_pk = torch.empty(B, H, W, 4, device=dev, dtype=torch.float32)
            if bf16_frames:
                tgt32 = torch.empty(B, 3, H, W, device=dev, dtype=torch.float32)
                check(lib.dmh_identity_loss_pack_bf16(ptr(target), ptr(srcs[0]), B, H, W, no_ssim, ptr(ident),
                                                      ptr(src_pk), ptr(tgt32), stream()), "identity_loss_pack_bf16")
                target = colors[0] = tgt32
            else:
                check(lib.dmh_identity_loss_pack(ptr(target), ptr(srcs[0]), B, H, W, no_ssim, ptr(ident), ptr(src_pk),
                                                 stream()), "identity_loss_pack")
            src_arr = ptr_array([src_pk])
            flags |= FLAG_SRC_PACKED
        elif automask:
            check(lib.dmh_identity_loss(ptr(target), src_arr, n_src, B, H, W, no_ssim, ptr(ident), stream()),
                  "identity_loss")
        tiles = lib.dmh_photo_tiles(H, W)
        gN, wss = [], []
        T_arr = ptr_array(Ts)
        inv_den = 1.0 / float(B * H * W)
        # the smoothness term (memory-bound, 8 small launches) is independent of the photometric kernels
        # (issue-bound): it runs on a side stream and fills their idle issue / memory slots; joined before `finish`
        cur = torch.cuda.current_stream(dev)
        side = _side_stream(dev)
        for s in range(S):
            d = disps[s]
            h, w = d.shape[2], d.shape[3]
            wss.append(torch.empty(lib.dmh_smooth_fused_workspace_floats(B, h, w), device=dev, dtype=torch.float32))
            gN.append(torch.empty(B, 1, h, w, device=dev, dtype=torch.float32))
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            for s in range(S):
                d = disps[s]
                check(lib.dmh_smooth_fused(ptr(d), ptr(colors[s]), B, 3, d.shape[2], d.shape[3], ptr(wss[s]),
                                           ptr(gN[s]), stream()), "smooth_fused")
        # the per-scale launches are independent of each other: odd scales go to a second stream so that the
        # tail of one launch (10240 CTAs = 23.06 waves of 444) overlaps the head of the next
        multiscale = (packed and MULTISCALE and S <= 4 and W % 4 == 0 and target.data_ptr() % 16 == 0
                      and H * W < (1 << 27))
        parts = [torch.empty(B * tiles, device=dev, dtype=torch.float32) for _ in range(S)]
        G = [torch.empty(B, 1, H, W, device=dev, dtype=torch.float32) for _ in range(S)]
        want_sels = want_sel or colour_grad
        sels = [torch.empty(B, H, W, device=dev, dtype=torch.uint8) if want_sels else None for _ in range(S)]
        if multisrc and need_T:
            tiles32 = ((H + 31) // 32) * ((W + 31) // 32)
            # one buffer for the pose-gradient partials of every scale: the backward reduces it with one einsum
            gP_all = torch.empty(S, n_src, B, tiles32, 12, device=dev, dtype=torch.float32)
            gPs = list(gP_all)
        else:
            gPs = [torch.empty(n_src, B, tiles, 12, device=dev, dtype=torch.float32) if need_T else None
                   for _ in range(S)]
        dh_ = (_C.c_int * S)(*[d.shape[2] for d in disps])
        dw_ = (_C.c_int * S)(*[d.shape[3] for d in disps])
        if multisrc:
            mf_ws = torch.empty(lib.dmh_photo_multisource_workspace_floats(n_src), device=dev, dtype=torch.float32)
            with _timed("photo_mf"):
                check(lib.dmh_photo_multisource(ptr(target), ptr_array(src_pks), ptr_array(Ts), n_src, S, ptr_array(disps),
                                                dh_, dw_, ptr(k), ptr(ik), ptr_array(idents) if automask else None,
                                                ptr_array(noises) if has_noise else None, B, H, W, min_depth, max_depth,
                                                inv_den, ptr(mf_ws), ptr_array(parts), ptr_array(G),
                                                ptr_array(gPs) if need_T else None,
                                                ptr_array(sels) if want_sels else None, stream()), "photo_multisource")
        if multiscale:
            # ONE launch for all scales (csrc/photo_ms.cu): the scale loop of generate_images_pred / compute_losses
            # runs inside the kernel; same bits as the per-scale launches below
            with _timed("photo_ms"):
                check(lib.dmh_photo_multiscale(ptr(target), ptr(src_pk), ptr(Ts[0]), S, ptr_array(disps), dh_, dw_, ptr(k),
                                               ptr(ik), ptr(ident), ptr_array(noises) if has_noise else None, B, H, W,
                                               min_depth, max_depth, inv_den, ptr_array(parts), ptr_array(G),
                                               ptr_array(sels) if want_sels else None, stream()), "photo_multiscale")
        alt = _side_stream(dev, 1)
        alt.wait_stream(cur)
        for s in range(S if not (multiscale or multisrc) else 0):
            with torch.cuda.stream(alt if (s & 1) else cur):
                with _timed("photo_scale"):
                    check(lib.dmh_photo_scale(ptr(target), src_arr, T_arr, n_src, ptr(disps[s]), dh_[s], dw_[s], ptr(k),
                                              ptr(ik), ptr(ident), ptr(noises[s]), B, H, W, min_depth, max_depth, flags,
                                              inv_den, ptr(parts[s]), ptr(G[s]), ptr(gPs[s]), ptr(sels[s]), None,
                                              stream()), "photo_scale")
        cur.wait_stream(alt)
        cur.wait_stream(side)
        img_scalars = torch.empty(S, B, 2, device=dev, dtype=torch.float32)
        losses = torch.empty(S + 1, device=dev, dtype=torch.float32)
        pn = (_C.c_int * S)(*[p_.numel() for p_ in parts])
        sw = (_C.c_float * S)(*[float(x) for x in smooth_w])
        fin_ws = torch.empty(lib.dmh_objective_finish_workspace_bytes(S, B), device=dev, dtype=torch.uint8)
        check(lib.dmh_objective_finish(S, B, ptr_array(wss), dh_, dw_, ptr_array(parts), pn, sw, float(B * H * W),
                                       ptr(fin_ws), ptr(img_scalars), ptr(losses), stream()), "objective_finish")
        ctx.cfg = (S, n_src, B, H, W, tuple(float(x) for x in smooth_w), need_T, [tuple(d.shape) for d in disps],
                   has_noise)
        if multisrc and need_T:
            gPs = [gP_all]                                   # (S, F, B, tiles, 12) as ONE saved tensor
        ctx.gp_stacked = bool(multisrc and need_T)
        gPs = [g for g in gPs if g is not None]
        ctx.n_gP = len(gPs)
        ctx.colour = None
        colour_saved = []
        if colour_grad:
            # the frames as the kernels read them (fp32; a bf16 source is widened in the backward), the disparities
            # and the selections
            ctx.colour = (float(min_depth), float(max_depth), flags & (FLAG_NO_SSIM | FLAG_AVG_REPROJECTION),
                          bool(automask), [c.dtype for c in colors_in], [t.dtype for t in srcs_in])
            colour_saved = [ik, *colors, *srcs, *disps, *sels]
        ctx.save_for_backward(img_scalars, k, *G, *gN, *[t for t in Ts], *gPs, *colour_saved)
        out_sels = tuple(sels) if want_sel else ()
        for t in out_sels:
            ctx.mark_non_differentiable(t)
        return (losses[S], losses[:S]) + out_sels

    @staticmethod
    def backward(ctx, g_total, g_scales, *_unused):
        S, n_src, B, H, W, smooth_w, need_T, dshapes, has_noise = ctx.cfg
        saved = ctx.saved_tensors
        img_scalars, k = saved[0], saved[1]
        G = saved[2:2 + S]
        gN = saved[2 + S:2 + 2 * S]
        Ts = saved[2 + 2 * S:2 + 2 * S + n_src]
        gPs = saved[2 + 2 * S + n_src:2 + 2 * S + n_src + ctx.n_gP]
        lib = _lib_()
        gt = f32c(g_total).reshape(1) if g_total is not None else None
        gs = f32c(g_scales) if g_scales is not None else None
        if gt is None and gs is None:
            gt = torch.zeros(1, device=G[0].device)
        base = 3 + S + n_src
        grads_disp = []
        # four independent, short launches: alternate two streams so that their tails overlap
        dev = G[0].device
        cur, alt = torch.cuda.current_stream(dev), _side_stream(dev, 1)
        want = [bool(ctx.needs_input_grad[base + n_src + s]) for s in range(S)]
        alt.wait_stream(cur)
        for s in range(S):
            if not want[s]:
                grads_disp.append(None)
                continue
            _, _, h, w = dshapes[s]
            gd = torch.empty(B, 1, h, w, device=dev, dtype=torch.float32)
            with torch.cuda.stream(alt if (s & 1) else cur):
                check(lib.dmh_disp_grad(ptr(G[s]), ptr(gN[s]), ptr(img_scalars[s]), smooth_w[s], ptr(gt),
                                        ptr(gs[s:s + 1]) if gs is not None else None, None, 1.0 / S, B, h, w, H, W,
                                        ptr(gd), stream()), "disp_grad")
            grads_disp.append(gd.view(dshapes[s]))
        cur.wait_stream(alt)
        g_T = [None] * n_src
        if need_T and ctx.gp_stacked:
            # multi-source kernel: sum over tiles and weighted sum over scales in one contraction, then the 4x4
            # algebra of all sources in one batched matmul
            u = (gt[0] / S if gt is not None else torch.zeros((), device=dev)) + \
                (gs if gs is not None else torch.zeros(S, device=dev))
            acc = torch.einsum("s,sfbtk->fbk", u.expand(S).to(torch.float32), gPs[0]).view(n_src, B, 3, 4)
            gT_all = torch.matmul(k[:, :3, :].transpose(1, 2).unsqueeze(0), acc)        # (F,B,4,4)
            for f in range(n_src):
                if ctx.needs_input_grad[base + f]:
                    g_T[f] = gT_all[f]
        elif need_T:
            u = [(gt[0] / S if gt is not None else 0.0) + (gs[s] if gs is not None else 0.0) for s in range(S)]
            for f in range(n_src):
                if ctx.needs_input_grad[base + f]:
                    g_T[f] = _pose_grad_T(gPs, u, f, k, Ts[f])
        g_col, g_src = [None] * S, [None] * n_src
        if ctx.colour is not None:
            g_col, g_src = _Objective._colour_grads(ctx, saved[2 + 2 * S + n_src + ctx.n_gP:], img_scalars, k, Ts, gt,
                                                    gs)
        return (None, None, None) + tuple(g_col) + tuple(g_src) + tuple(g_T) + tuple(grads_disp) + \
            ((None,) * S if has_noise else ())

    @staticmethod
    def _colour_grads(ctx, saved, img_scalars, k, Ts, gt, gs):
        """d(loss)/d(colour(0, s)) and d(loss)/d(source f) for the inputs that require them (None for the rest):
        the identity candidates' terms (one launch, initialises the target and source gradients), the reprojection
        terms (one launch per scale) and the smoothness terms (one launch per scale; scale 0 adds into the target's).
        Computed on the fp32 frames; returned in each input's dtype."""
        S, n_src, B, H, W, smooth_w = ctx.cfg[:6]
        min_depth, max_depth, flags, automask, col_dtypes, src_dtypes = ctx.colour
        ik = saved[0]
        colors = [f32c(c) for c in saved[1:1 + S]]
        srcs = [f32c(t) for t in saved[1 + S:1 + S + n_src]]
        disps = saved[1 + S + n_src:1 + 2 * S + n_src]
        sels = saved[1 + 2 * S + n_src:1 + 3 * S + n_src]
        need_col = [bool(ctx.needs_input_grad[3 + s]) for s in range(S)]
        need_src = [bool(ctx.needs_input_grad[3 + S + f]) for f in range(n_src)]
        lib = _lib_()
        g_col = [None] * S
        g_src = [torch.empty_like(srcs[f]) if need_src[f] else None for f in range(n_src)]
        if need_col[0]:
            g_col[0] = torch.empty_like(colors[0])
        if need_col[0] or any(need_src):
            src_arr, gsrc_arr = ptr_array(srcs), ptr_array(g_src)
            with _timed("identity_image_grad"):
                check(lib.dmh_identity_image_grad(ptr(colors[0]), src_arr, n_src, ptr_array(sels), S, ptr(gt), ptr(gs),
                                                  B, H, W, flags, int(automask), ptr(g_col[0]), gsrc_arr, stream()),
                      "identity_image_grad")
            T_arr = ptr_array(Ts)
            for s in range(S):
                d = disps[s]
                with _timed("photo_image_grad"):
                    check(lib.dmh_photo_image_grad(ptr(colors[0]), src_arr, T_arr, n_src, ptr(d), d.shape[2], d.shape[3],
                                                   ptr(k), ptr(ik), ptr(sels[s]), s, S, ptr(gt), ptr(gs), B, H, W,
                                                   min_depth, max_depth, flags, int(automask), ptr(g_col[0]), gsrc_arr,
                                                   stream()), "photo_image_grad")
        for s in range(S):
            if not need_col[s]:
                continue
            d = disps[s]
            if s > 0:
                g_col[s] = torch.empty_like(colors[s])
            check(lib.dmh_smooth_image_grad(ptr(d), ptr(colors[s]), B, d.shape[2], d.shape[3], ptr(img_scalars[s]),
                                            smooth_w[s], s, S, ptr(gt), ptr(gs), int(s == 0), ptr(g_col[s]), stream()),
                  "smooth_image_grad")
        g_col = [g if g is None or g.dtype == dt else g.to(dt) for g, dt in zip(g_col, col_dtypes)]
        g_src = [g if g is None or g.dtype == dt else g.to(dt) for g, dt in zip(g_src, src_dtypes)]
        return g_col, g_src


def objective(colors0, srcs, Ts, disps, K, inv_K, noises=None, min_depth=0.1, max_depth=100.0, no_ssim=False,
              avg_reprojection=False, automask=True, smooth_weights=None, want_sel=False):
    """colors0[s] = colour(0, s) pyramid (scale 0 is the target); srcs/Ts per source frame;
    disps[s] network disparities; noises[s] (B,Fi,H,W) or None.
    Returns (total, per-scale losses (S,), *sel)."""
    S, n_src = len(disps), len(srcs)
    flags = (FLAG_NO_SSIM if no_ssim else 0) | (FLAG_AVG_REPROJECTION if avg_reprojection else 0)
    has_noise = automask and noises is not None and all(n is not None for n in noises)
    cfg = (float(min_depth), float(max_depth), flags, tuple(smooth_weights), bool(want_sel), n_src, S, bool(automask),
           has_noise)
    B = colors0[0].shape[0]
    Ts = [_mat_batch(t, B, "T") for t in Ts]
    tensors = list(colors0) + list(srcs) + list(Ts) + list(disps) + (list(noises) if has_noise else [])
    return _Objective.apply(_mat_batch(K, B, "K"), _mat_batch(inv_K, B, "inv_K"), cfg, *tensors)
