"""Depth-hints objective (SURVEY.md 8(a) row A18): host-side mirror of
`DepthNetworks/depth-hints/trainer.py` -- `generate_images_pred` (:476-525, the
extra depth-hint warp), `compute_loss_masks` (:541-590),
`compute_proxy_supervised_loss` (:525-539) and the per-scale loop of
`compute_losses` (:629-727).

Differences of the depth-hints objective from monodepth2's (`objective.py`):
  * the minimum over the source frames is taken first ("compute mins as we go",
    :670-672, 683-685), ONE tie-break noise plane is added to the identity minimum;
  * the per-pixel argmin runs over [reprojection, identity, depth-hint reprojection];
    the reprojection loss is a MASKED mean  sum(l * m) / (sum(m) + 1e-7), m = argmin != identity;
  * where the hint wins, log(|hint - depth| + 1) is added (masked mean again).

Built from the op-level kernels (fused warp, SSIM+L1 reprojection loss, smoothness,
bilinear up-sampling: `ops.py`) plus `dmh_hint_select`, which does the min / argmin /
masks / both masked-sum numerators / proxy loss and their derivatives in one pass.
CUDA tensors only -- no CPU fallback.
"""
from __future__ import annotations

from typing import Dict, Optional

import torch

import ctypes as _C

from . import _lib, ops
from ._lib import check, f32c, ptr, ptr_array, stream
from .objective import _frame_T, tie_break_noise


def _lib_():
    return _lib.load()


class _HintSelect(torch.autograd.Function):
    """(reprojection loss, proxy loss, argmin) of one scale from the per-frame
    reprojection losses [grad], the predicted depth [grad] and the constant maps."""

    @staticmethod
    def forward(ctx, ident, noise, hint_reproj, depth, hint_depth, hint_valid, avg, want_sel, *reproj):
        rl = [f32c(t) for t in reproj]
        F_ = len(rl)
        B, _, H, W = rl[0].shape
        dev = rl[0].device
        idn = f32c(ident) if ident is not None else None
        nz = f32c(noise) if noise is not None else None
        hr = f32c(hint_reproj) if hint_reproj is not None else None
        dp = f32c(depth) if hr is not None else None
        hd = f32c(hint_depth) if hr is not None else None
        hv = f32c(hint_valid) if hr is not None else None
        lib = _lib_()
        nblk = lib.dmh_hint_select_blocks(B, H, W)
        part = torch.empty(4, nblk, device=dev, dtype=torch.float32)
        g_rl = [torch.empty_like(t) for t in rl]
        g_dp = torch.empty_like(dp) if hr is not None else None
        sel = torch.empty(B, H, W, device=dev, dtype=torch.uint8) if want_sel else None
        check(lib.dmh_hint_select(ptr_array(rl), F_, ptr(idn), ptr(nz), ptr(hr), ptr(dp), ptr(hd), ptr(hv), int(avg),
                                  B, H, W, ptr(part), ptr_array(g_rl), ptr(g_dp), ptr(sel), stream()), "hint_select")
        sums = torch.empty(4, device=dev, dtype=torch.float32)
        for k in range(4 if hr is not None else 2):
            check(lib.dmh_reduce_sum(ptr(part[k]), nblk, 1.0, 0, ptr(sums[k:k + 1]), stream()), "reduce_sum")
        inv_r = 1.0 / (sums[1] + 1e-7)
        loss_r = sums[0] * inv_r
        if hr is not None:
            inv_h = 1.0 / (sums[3] + 1e-7)
            loss_h = sums[2] * inv_h
        else:
            inv_h = torch.zeros((), device=dev)
            loss_h = torch.zeros((), device=dev)
        ctx.save_for_backward(inv_r, inv_h, g_dp, *g_rl)
        ctx.n = F_
        if sel is not None:
            ctx.mark_non_differentiable(sel)
        return loss_r, loss_h, sel

    @staticmethod
    def backward(ctx, g_r, g_h, _g_sel):
        inv_r, inv_h, g_dp, *g_rl = ctx.saved_tensors
        grads = [None] * 8
        if ctx.needs_input_grad[3] and g_dp is not None and g_h is not None:
            grads[3] = g_dp * (g_h * inv_h)
        out = []
        for i in range(ctx.n):
            out.append(g_rl[i] * (g_r * inv_r) if (g_r is not None and ctx.needs_input_grad[8 + i]) else None)
        return tuple(grads) + tuple(out)


def hint_reprojection_loss(target, src, depth_hint, depth_hint_mask, K, inv_K, T, no_ssim=False, fast_math=False):
    """`DH/trainer.py:510-525` + `:629-634`: warp the stereo source with the depth
    hint -- NOTE `F.grid_sample(..., padding_mode="border")` with the DEFAULT
    align_corners (False), unlike the main warp -- then compute_reprojection_loss and
    `+ 1000 * (1 - depth_hint_mask)`.  No gradient (inputs only).
    fast_math: evaluate SSIM with the arithmetic of the fused kernels (`dmh_identity_loss`) so that the argmin
    compares like with like -- a hint equal to the prediction then ties EXACTLY and the reprojection wins the
    tie, as in the reference, where both losses come out of the same code."""
    with torch.no_grad():
        B, _, H, W = target.shape
        # one fused gather (same op sequence as BackprojectDepth -> Project3D -> grid_sample(border, align_corners=False))
        pred, _, _ = ops.warp_with_aux(depth_hint, src, K, inv_K, T, input_is_depth=True, align_corners=False,
                                       want_aux=False)
        if fast_math:
            loss = torch.empty(B, 1, H, W, device=pred.device, dtype=torch.float32)
            check(_lib_().dmh_identity_loss(ptr(f32c(target)), ptr_array([pred]), 1, B, H, W, int(no_ssim), ptr(loss),
                                            stream()), "identity_loss")
        else:
            loss = ops.reprojection_loss(pred, target, no_ssim)
        loss = loss + 1000 * (1 - depth_hint_mask)
    return loss, pred


def depth_hint_losses(colors: Dict, disps: Dict, K, inv_K, Ts: Dict, frame_ids, scales, height, width,
                      depth_hint=None, depth_hint_mask=None, use_depth_hints=True, min_depth=0.1, max_depth=100.0,
                      no_ssim=False, avg_reprojection=False, disable_automasking=False, disparity_smoothness=1e-3,
                      noise: Optional[Dict] = None, noise_mode="reference", want_selection=False, fused=True):
    """Per-scale loop of the depth-hints `compute_losses` (`DH/trainer.py:636-727`).  fused=True (default): one
    `dmh_photo_scale_dh` launch per scale does warp + SSIM/L1 + decision + masked sums + backward (`_ObjectiveDH`);
    fused=False: the op-level composition below (kept as an independent cross-check)."""
    if fused:
        return _depth_hint_losses_fused(colors, disps, K, inv_K, Ts, frame_ids, scales, height, width, depth_hint,
                                        depth_hint_mask, use_depth_hints, min_depth, max_depth, no_ssim,
                                        avg_reprojection, disable_automasking, disparity_smoothness, noise, noise_mode,
                                        want_selection)
    return _depth_hint_losses_oplevel(colors, disps, K, inv_K, Ts, frame_ids, scales, height, width, depth_hint,
                                      depth_hint_mask, use_depth_hints, min_depth, max_depth, no_ssim,
                                      avg_reprojection, disable_automasking, disparity_smoothness, noise, noise_mode,
                                      want_selection)


def _prologue(colors, Ts, frame_ids, height, width, depth_hint, depth_hint_mask, use_depth_hints, no_ssim,
              disable_automasking, K, inv_K, fast_math=True, pack_out=None):
    """Scale-independent, gradient-free parts: the hint reprojection loss and the identity losses."""
    srcs_ids = list(frame_ids[1:])
    target = colors[(0, 0)]
    B = target.shape[0]
    srcs = [colors[(f, 0)] for f in srcs_ids]
    if use_depth_hints:
        if "s" not in srcs_ids:
            raise KeyError(("color_depth_hint", "s", 0))     # the reference only builds the hint warp for 's'
        if disable_automasking:
            # DH/trainer.py:554-555 evaluates `if depth_hint_reprojection_loss:` on a (B,1,H,W) tensor
            raise RuntimeError("Boolean value of Tensor with more than one element is ambiguous")
        hint_rl, hint_pred = hint_reprojection_loss(target, colors[("s", 0)], depth_hint, depth_hint_mask, K, inv_K,
                                                    Ts["s"], no_ssim, fast_math)
    else:
        hint_rl = hint_pred = None
    ident = None
    with torch.no_grad():
        if not disable_automasking:
            ident = torch.empty(B, len(srcs), height, width, device=target.device, dtype=torch.float32)
        # widened frames (a copy for non-fp32 frames) held until the launch: a copy made inside the call's argument
        # list is freed as soon as its pointer is taken, and the next copy may then reuse its memory
        target32, srcs32 = f32c(target), [f32c(s) for s in srcs]
        if pack_out is not None and len(srcs) == 1 and not no_ssim:
            # single source: the identity-loss kernel also writes the pixel-packed copy the fast kernel gathers from
            pk = torch.empty(B, height, width, 4, device=target.device, dtype=torch.float32)
            check(_lib_().dmh_identity_loss_pack(ptr(target32), ptr(srcs32[0]), B, height, width, 0, ptr(ident),
                                                 ptr(pk), stream()), "identity_loss_pack")
            pack_out.append(pk)
        elif ident is not None:
            check(_lib_().dmh_identity_loss(ptr(target32), ptr_array(srcs32), len(srcs), B, height, width,
                                            int(no_ssim), ptr(ident), stream()), "identity_loss")
    return srcs_ids, srcs, target, B, hint_rl, hint_pred, ident


class _ObjectiveDH(torch.autograd.Function):
    """All scales of the depth-hints objective as one autograd node (fused kernels)."""

    @staticmethod
    def forward(ctx, K, inv_K, cfg, ident, hint_rl, hint_depth, hint_valid, *tensors):
        (min_depth, max_depth, flags, smooth_w, want_sel, n_src, S, has_noise, src_pk) = cfg
        it = iter(tensors)
        colors_in = [next(it) for _ in range(S)]
        srcs_in = [next(it) for _ in range(n_src)]
        colors = [f32c(c) for c in colors_in]
        srcs = [f32c(t) for t in srcs_in]
        Ts = [f32c(next(it)) for _ in range(n_src)]
        disps = [f32c(next(it)) for _ in range(S)]
        noises = [f32c(next(it)) for _ in range(S)] if has_noise else [None] * S
        target = colors[0]
        B, _, H, W = target.shape
        k, ik = f32c(ops._mat_batch(K, B, "K")), f32c(ops._mat_batch(inv_K, B, "inv_K"))
        Ts = [f32c(ops._mat_batch(t, B, "T")) for t in Ts]
        dev = target.device
        lib = _lib_()
        idn = f32c(ident) if ident is not None else None
        hr = f32c(hint_rl) if hint_rl is not None else None
        hd = f32c(hint_depth) if hr is not None else None
        hv = f32c(hint_valid) if hr is not None else None
        base = 7 + S + n_src
        need_T = any(ctx.needs_input_grad[base + i] for i in range(n_src))
        # gradients for the colour frames (target, pyramid, sources): the backward recomputes them from the frames,
        # the disparities and every scale's selection, so `sel` is requested internally -- with the winning source
        # frame in its upper bits where several sources compete for the minimum
        colour_grad = any(ctx.needs_input_grad[7 + i] for i in range(S + n_src))
        sel_src = colour_grad and n_src > 1 and not (flags & ops.FLAG_AVG_REPROJECTION)
        want_sels = want_sel or colour_grad
        tiles = lib.dmh_photo_tiles(H, W)
        nblk = B * tiles
        src_arr, T_arr = ptr_array(srcs), ptr_array(Ts)
        if src_pk is not None and not need_T:             # single source, no pose gradient: packed 128-bit gather
            src_arr = ptr_array([src_pk])
            flags |= ops.FLAG_SRC_PACKED
        G_r, G_h, gN, wss, gPs, sels, sums = [], [], [], [], [], [], []
        for s in range(S):
            d = disps[s]
            h, w = d.shape[2], d.shape[3]
            part = torch.empty(4, nblk, device=dev, dtype=torch.float32)
            g_r = torch.empty(B, 1, H, W, device=dev, dtype=torch.float32)
            g_h = torch.empty(B, 1, H, W, device=dev, dtype=torch.float32) if hr is not None else None
            gP = torch.empty(n_src, B, tiles, 12, device=dev, dtype=torch.float32) if need_T else None
            sel = torch.empty(B, H, W, device=dev, dtype=torch.uint8) if want_sels else None
            check(lib.dmh_photo_scale_dh(ptr(target), src_arr, T_arr, n_src, ptr(d), h, w, ptr(k), ptr(ik), ptr(idn),
                                         ptr(noises[s]), ptr(hr), ptr(hd), ptr(hv), B, H, W, min_depth, max_depth,
                                         flags | (ops.FLAG_SEL_SOURCE if sel_src else 0), ptr(part), ptr(g_r), ptr(g_h),
                                         ptr(gP), ptr(sel), stream()), "photo_scale_dh")
            sm = torch.empty(4, device=dev, dtype=torch.float32)
            check(lib.dmh_reduce_rows(ptr(part), 4 if hr is not None else 2, nblk, 1.0, ptr(sm), stream()), "reduce_rows")
            ws = torch.empty(lib.dmh_smooth_fused_workspace_floats(B, h, w), device=dev, dtype=torch.float32)
            gn = torch.empty(B, 1, h, w, device=dev, dtype=torch.float32)
            check(lib.dmh_smooth_fused(ptr(d), ptr(colors[s]), B, 3, h, w, ptr(ws), ptr(gn), stream()), "smooth_fused")
            G_r.append(g_r); G_h.append(g_h); gN.append(gn); wss.append(ws); gPs.append(gP); sels.append(sel)
            sums.append(sm)
        # smoothness losses + per-image normalisation scalars: the shared finish launch with no photometric partials
        img_scalars = torch.empty(S, B, 2, device=dev, dtype=torch.float32)
        sm_losses = torch.empty(S + 1, device=dev, dtype=torch.float32)
        hs = (_C.c_int * S)(*[d.shape[2] for d in disps])
        wsz = (_C.c_int * S)(*[d.shape[3] for d in disps])
        pn = (_C.c_int * S)(*([0] * S))
        sw = (_C.c_float * S)(*[float(x) for x in smooth_w])
        dummy = torch.zeros(1, device=dev, dtype=torch.float32)
        fin_ws = torch.empty(lib.dmh_objective_finish_workspace_bytes(S, B), device=dev, dtype=torch.uint8)
        check(lib.dmh_objective_finish(S, B, ptr_array(wss), hs, wsz, ptr_array([dummy] * S), pn, sw, float(B * H * W),
                                       ptr(fin_ws), ptr(img_scalars), ptr(sm_losses), stream()), "objective_finish")
        sums_t = torch.stack(sums, 0)                                   # (S,4)
        inv_r = 1.0 / (sums_t[:, 1] + 1e-7)                             # DH/trainer.py:699-700
        loss_r = sums_t[:, 0] * inv_r
        if hr is not None:
            inv_h = 1.0 / (sums_t[:, 3] + 1e-7)                         # :712-713
            loss_h = sums_t[:, 2] * inv_h
        else:
            inv_h = torch.zeros(S, device=dev)
            loss_h = torch.zeros(S, device=dev)
        per_scale = loss_r + loss_h + sm_losses[:S]
        total = per_scale.sum() / S
        ctx.cfg = (S, n_src, B, H, W, tuple(float(x) for x in smooth_w), need_T, [tuple(d.shape) for d in disps],
                   has_noise, hr is not None)
        gPs = [g for g in gPs if g is not None]
        ctx.n_gP = len(gPs)
        ctx.colour = None
        colour_saved = []
        if colour_grad:
            ctx.colour = (float(min_depth), float(max_depth), flags & (ops.FLAG_NO_SSIM | ops.FLAG_AVG_REPROJECTION),
                          [c.dtype for c in colors_in], [t.dtype for t in srcs_in])
            colour_saved = [ik, *colors, *srcs, *disps, *sels]
        ctx.save_for_backward(img_scalars, k, inv_r, inv_h, *G_r, *[g for g in G_h if g is not None], *gN, *Ts, *gPs,
                              *colour_saved)
        # the argmin index over [reprojection, identity, hint], as without the source bits
        out_sels = tuple(t & 3 if sel_src else t for t in sels) if want_sel else ()
        for t in out_sels:
            ctx.mark_non_differentiable(t)
        return (total, per_scale, loss_r, loss_h) + out_sels

    @staticmethod
    def backward(ctx, g_total, g_scales, g_lr, g_lh, *_unused):
        S, n_src, B, H, W, smooth_w, need_T, dshapes, has_noise, hints = ctx.cfg
        saved = list(ctx.saved_tensors)
        img_scalars, k, inv_r, inv_h = saved[:4]
        pos = 4
        G_r = saved[pos:pos + S]; pos += S
        G_h = saved[pos:pos + S] if hints else [None] * S
        pos += S if hints else 0
        gN = saved[pos:pos + S]; pos += S
        Ts = saved[pos:pos + n_src]; pos += n_src
        gPs = saved[pos:pos + ctx.n_gP]; pos += ctx.n_gP
        lib = _lib_()
        dev = G_r[0].device
        zero = torch.zeros((), device=dev)
        gt = g_total if g_total is not None else zero
        # upstream weight of every per-scale term (device scalars, no host sync)
        u_all = gt / S + (g_scales if g_scales is not None else torch.zeros(S, device=dev))     # total & loss/s
        u_r = (u_all + (g_lr if g_lr is not None else 0.0)) * inv_r                               # reprojection term
        u_h = (u_all + (g_lh if g_lh is not None else 0.0)) * inv_h                               # proxy term
        base = 7 + S + n_src
        grads_disp = []
        one = torch.ones(1, device=dev)
        for s in range(S):
            if not ctx.needs_input_grad[base + n_src + s]:
                grads_disp.append(None)
                continue
            _, _, h, w = dshapes[s]
            # G = u_r * G_r + u_h * G_h  (one fused pass), then F.interpolate^T + smoothness backward
            if hints:
                comb = torch.empty_like(G_r[s])
                check(lib.dmh_axpby_dev(ptr(f32c(u_r[s:s + 1])), ptr(G_r[s]), ptr(f32c(u_h[s:s + 1])), ptr(G_h[s]),
                                        comb.numel(), ptr(comb), stream()), "axpby")
            else:
                comb = G_r[s] * u_r[s]
            gd = torch.empty(B, 1, h, w, device=dev, dtype=torch.float32)
            # grad = 1 * interpolate^T(comb) + u_all * w * (smoothness backward)
            check(lib.dmh_disp_grad(ptr(comb), ptr(gN[s]), ptr(img_scalars[s]), smooth_w[s], None, ptr(one),
                                    ptr(f32c(u_all[s:s + 1])), 1.0, B, h, w, H, W, ptr(gd), stream()), "disp_grad")
            grads_disp.append(gd.view(dshapes[s]))
        g_T = [None] * n_src
        if need_T:
            for f in range(n_src):
                if ctx.needs_input_grad[base + f]:
                    g_T[f] = ops._pose_grad_T(gPs, u_r, f, k, Ts[f])
        g_col, g_src = [None] * S, [None] * n_src
        if ctx.colour is not None:
            g_col, g_src = _ObjectiveDH._colour_grads(ctx, saved[pos:], img_scalars, k, Ts, u_all, u_r)
        return (None,) * 7 + tuple(g_col) + tuple(g_src) + tuple(g_T) + tuple(grads_disp) + \
            ((None,) * S if has_noise else ())

    @staticmethod
    def _colour_grads(ctx, saved, img_scalars, k, Ts, u_all, u_r):
        """d(loss)/d(colour(0, s)) and d(loss)/d(source f) for the inputs that require them (None for the rest).
        Only the reprojection term (one launch per scale, weight u_r[s]) and the smoothness term (one launch per
        scale, weight u_all[s]; scale 0 adds into the target's) depend on the colours: the identity and the hint
        candidates only decide the masks.  Computed on the fp32 frames; returned in each input's dtype."""
        S, n_src, B, H, W, smooth_w = ctx.cfg[:6]
        min_depth, max_depth, flags, col_dtypes, src_dtypes = ctx.colour
        ik = saved[0]
        colors = saved[1:1 + S]
        srcs = saved[1 + S:1 + S + n_src]
        disps = saved[1 + S + n_src:1 + 2 * S + n_src]
        sels = saved[1 + 2 * S + n_src:1 + 3 * S + n_src]
        need_col = [bool(ctx.needs_input_grad[7 + s]) for s in range(S)]
        need_src = [bool(ctx.needs_input_grad[7 + S + f]) for f in range(n_src)]
        lib = _lib_()
        u_all, u_r = f32c(u_all), f32c(u_r)
        g_col = [None] * S
        g_src = [torch.zeros_like(srcs[f]) if need_src[f] else None for f in range(n_src)]
        if need_col[0]:
            g_col[0] = torch.zeros_like(colors[0])
        if need_col[0] or any(need_src):
            src_arr, T_arr, gsrc_arr = ptr_array(srcs), ptr_array(Ts), ptr_array(g_src)
            for s in range(S):
                d = disps[s]
                with ops._timed("photo_image_grad_dh"):
                    check(lib.dmh_photo_image_grad_dh(ptr(colors[0]), src_arr, T_arr, n_src, ptr(d), d.shape[2],
                                                      d.shape[3], ptr(k), ptr(ik), ptr(sels[s]), ptr(u_r[s:s + 1]), B, H,
                                                      W, min_depth, max_depth, flags, ptr(g_col[0]), gsrc_arr, stream()),
                          "photo_image_grad_dh")
        for s in range(S):
            if not need_col[s]:
                continue
            d = disps[s]
            if s > 0:
                g_col[s] = torch.empty_like(colors[s])
            # upstream u_all[s] = g_total / S + g_scales[s], already formed: passed as the per-scale weights
            check(lib.dmh_smooth_image_grad(ptr(d), ptr(colors[s]), B, d.shape[2], d.shape[3], ptr(img_scalars[s]),
                                            smooth_w[s], s, S, None, ptr(u_all), int(s == 0), ptr(g_col[s]), stream()),
                  "smooth_image_grad")
        g_col = [g if g is None or g.dtype == dt else g.to(dt) for g, dt in zip(g_col, col_dtypes)]
        g_src = [g if g is None or g.dtype == dt else g.to(dt) for g, dt in zip(g_src, src_dtypes)]
        return g_col, g_src


def _depth_hint_losses_fused(colors, disps, K, inv_K, Ts, frame_ids, scales, height, width, depth_hint,
                             depth_hint_mask, use_depth_hints, min_depth, max_depth, no_ssim, avg_reprojection,
                             disable_automasking, disparity_smoothness, noise, noise_mode, want_selection):
    scales = list(scales)
    if scales[0] != 0:
        raise NotImplementedError("the fused objective needs scale 0 first in opt.scales")
    packs = []
    srcs_ids, srcs, target, B, hint_rl, hint_pred, ident = _prologue(
        colors, Ts, frame_ids, height, width, depth_hint, depth_hint_mask, use_depth_hints, no_ssim,
        disable_automasking, K, inv_K, pack_out=None if avg_reprojection else packs)
    nz = None
    if ident is not None:
        nz = [noise[s] if noise is not None else tie_break_noise((B, 1, height, width), target.device, noise_mode)
              for s in scales]
        if any(t is None for t in nz):
            nz = None
    S, n_src = len(scales), len(srcs)
    flags = (ops.FLAG_NO_SSIM if no_ssim else 0) | (ops.FLAG_AVG_REPROJECTION if avg_reprojection else 0)
    cfg = (float(min_depth), float(max_depth), flags, tuple(disparity_smoothness / (2 ** s) for s in scales),
           bool(want_selection), n_src, S, nz is not None, packs[0] if packs else None)
    colors0 = [target] + [colors[(0, s)] for s in scales[1:]]
    tensors = colors0 + srcs + [Ts[f] for f in srcs_ids] + [disps[s] for s in scales] + (nz if nz is not None else [])
    out = _ObjectiveDH.apply(K, inv_K, cfg, ident, hint_rl, depth_hint if use_depth_hints else None,
                             depth_hint_mask if use_depth_hints else None, *tensors)
    total, per_scale, loss_r, loss_h = out[:4]
    losses, aux = {}, {}
    for i, scale in enumerate(scales):
        losses["reproj_loss/{}".format(scale)] = loss_r[i]
        if use_depth_hints:
            losses["depth_hint_loss/{}".format(scale)] = loss_h[i]
        losses["loss/{}".format(scale)] = per_scale[i]
        if want_selection:
            sel = out[4 + i]
            aux[("argmin", scale)] = sel
            aux["identity_selection/{}".format(scale)] = (sel == 1).float().unsqueeze(1)
            if use_depth_hints:
                aux["depth_hint_pixels/{}".format(scale)] = (sel == 2).float().unsqueeze(1)
    losses["loss"] = total
    if hint_pred is not None:
        aux[("color_depth_hint", "s", 0)] = hint_pred
    return losses, aux


def _depth_hint_losses_oplevel(colors: Dict, disps: Dict, K, inv_K, Ts: Dict, frame_ids, scales, height, width,
                               depth_hint=None, depth_hint_mask=None, use_depth_hints=True, min_depth=0.1,
                               max_depth=100.0, no_ssim=False, avg_reprojection=False, disable_automasking=False,
                               disparity_smoothness=1e-3, noise: Optional[Dict] = None, noise_mode="reference",
                               want_selection=False):
    """Op-level composition (fused warp, SSIM+L1, smoothness, up-sampling kernels + `dmh_hint_select`).

    colors / disps / Ts as in `objective.photometric_losses`; noise: optional
    {scale: (B,1,H,W)} tie-break noise already * 1e-5; depth_hint, depth_hint_mask (B,1,H,W).
    Returns (losses, aux) with the reference's keys: 'loss', 'loss/s', 'reproj_loss/s',
    'depth_hint_loss/s'; aux: 'identity_selection/s', 'depth_hint_pixels/s' when requested."""
    srcs_ids = list(frame_ids[1:])
    target = colors[(0, 0)]
    B = target.shape[0]
    srcs = [colors[(f, 0)] for f in srcs_ids]
    if use_depth_hints:
        if "s" not in srcs_ids:
            raise KeyError(("color_depth_hint", "s", 0))     # the reference only builds the hint warp for 's'
        if disable_automasking:
            # DH/trainer.py:554-555 evaluates `if depth_hint_reprojection_loss:` on a (B,1,H,W) tensor
            raise RuntimeError("Boolean value of Tensor with more than one element is ambiguous")
        hint_rl, hint_pred = hint_reprojection_loss(target, colors[("s", 0)], depth_hint, depth_hint_mask, K, inv_K,
                                                    Ts["s"], no_ssim)
    else:
        hint_rl = hint_pred = None
    ident = None
    if not disable_automasking:
        with torch.no_grad():
            ident = torch.empty(B, len(srcs), height, width, device=target.device, dtype=torch.float32)
            target32, srcs32 = f32c(target), [f32c(s) for s in srcs]      # held until the launch (see _prologue)
            check(_lib_().dmh_identity_loss(ptr(target32), ptr_array(srcs32), len(srcs), B, height, width,
                                            int(no_ssim), ptr(ident), stream()), "identity_loss")
    losses, aux = {}, {}
    total = 0
    for scale in scales:
        disp = disps[scale]
        disp_full = ops.upsample_bilinear(disp, (height, width)) if disp.shape[2] != height else disp
        rl = []
        for f, src in zip(srcs_ids, srcs):
            pred = ops.warp_reproject(disp_full, src, K, inv_K, Ts[f], min_depth, max_depth)
            rl.append(ops.reprojection_loss(pred, target, no_ssim))
        _, depth = ops._DispToDepth.apply(disp_full, float(min_depth), float(max_depth))
        nz = None
        if ident is not None:
            nz = noise[scale] if noise is not None else tie_break_noise((B, 1, height, width), target.device, noise_mode)
        loss_r, loss_h, sel = _HintSelect.apply(ident, nz, hint_rl, depth, depth_hint, depth_hint_mask,
                                                bool(avg_reprojection), bool(want_selection), *rl)
        losses["reproj_loss/{}".format(scale)] = loss_r
        loss = loss_r
        if use_depth_hints:
            losses["depth_hint_loss/{}".format(scale)] = loss_h
            loss = loss + loss_h
        if want_selection:
            aux[("argmin", scale)] = sel
            aux["identity_selection/{}".format(scale)] = (sel == 1).float().unsqueeze(1)
            if use_depth_hints:
                aux["depth_hint_pixels/{}".format(scale)] = (sel == 2).float().unsqueeze(1)
        smooth = ops.smooth_loss(disp, colors[(0, scale)], normalise=True)
        loss = loss + disparity_smoothness * smooth / (2 ** scale)
        losses["loss/{}".format(scale)] = loss
        total = total + loss
    total = total / len(scales)
    losses["loss"] = total
    if hint_pred is not None:
        aux[("color_depth_hint", "s", 0)] = hint_pred
    return losses, aux


# ----------------------------------------------------------------------------- Trainer patches (depth-hints trainer)
def dh_generate_images_pred(self, inputs, outputs):
    """Replacement for the depth-hints `Trainer.generate_images_pred`: only the depth
    maps (read by `compute_depth_losses`) are produced; warps happen inside the loss."""
    opt = self.opt
    if opt.v1_multiscale or getattr(opt, "pose_model_type", "") == "posecnn" or opt.predictive_mask:
        return self._dmh_ref_generate_images_pred(inputs, outputs)
    import torch.nn.functional as F
    for scale in opt.scales:
        with torch.no_grad():
            disp_full = F.interpolate(outputs[("disp", scale)], [opt.height, opt.width], mode="bilinear",
                                      align_corners=False)
            _, depth = ops.disp_to_depth_cuda(disp_full, opt.min_depth, opt.max_depth)
        outputs[("depth", 0, scale)] = depth


def dh_compute_losses(self, inputs, outputs):
    """Replacement for the depth-hints `Trainer.compute_losses` (`DH/trainer.py:592-729`)."""
    opt = self.opt
    if opt.v1_multiscale or getattr(opt, "pose_model_type", "") == "posecnn" or opt.predictive_mask:
        return self._dmh_ref_compute_losses(inputs, outputs)
    losses = {}
    total_loss = 0
    if opt.adv_train and opt.supervised_adv:               # network-side terms: stock PyTorch (:597-611)
        with torch.no_grad():
            disp_gt = self.gt_model(inputs[("color_ben", 0, 0)])
        loss_sup = self.sup_loss_creteria(disp_gt, outputs[("disp", 0)])
        losses["sup_loss"] = loss_sup
        total_loss = total_loss + loss_sup
    if opt.adv_train and opt.contrastive_learning:         # (:613-624)
        contras_loss = self.models["contrastive_learning"](outputs["middle_features_aug"],
                                                           outputs["middle_features_ben"]) * 0.1
        losses["contras_loss"] = contras_loss
        total_loss = total_loss + contras_loss
    if opt.adv_train and opt.no_original_train:
        losses["loss"] = total_loss
        return losses
    colors = {(0, s): inputs[("color", 0, s)] for s in opt.scales}
    Ts = {}
    for f in opt.frame_ids[1:]:
        colors[(f, 0)] = inputs[("color", f, 0)]
        Ts[f] = _frame_T(opt, inputs, outputs, f)
    disps = {s: outputs[("disp", s)] for s in opt.scales}
    pl, aux = depth_hint_losses(colors, disps, inputs[("K", 0)], inputs[("inv_K", 0)], Ts, opt.frame_ids, opt.scales,
                                opt.height, opt.width, inputs.get("depth_hint"), inputs.get("depth_hint_mask"),
                                bool(opt.use_depth_hints), opt.min_depth, opt.max_depth, bool(opt.no_ssim),
                                bool(opt.avg_reprojection), bool(opt.disable_automasking), opt.disparity_smoothness,
                                noise=getattr(self, "_dmh_noise", None),
                                noise_mode=getattr(self, "_dmh_noise_mode", "reference"), want_selection=True)
    for k, v in aux.items():
        if isinstance(k, str):
            outputs[k] = v
    for k, v in pl.items():
        if k != "loss":
            losses[k] = v
    losses["loss"] = total_loss + pl["loss"]
    return losses
