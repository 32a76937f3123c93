"""Fused photometric objective: host-side mirror of `Trainer.generate_images_pred`
(`M2/trainer.py:472-523`) and `Trainer.compute_losses` (`:539-674`).

`fused_generate_images_pred` / `fused_compute_losses` are unbound methods with
the reference's signatures; `install.install()` patches them onto the
reference's `Trainer` so `train.py --adv_train` runs unchanged.  One
`dmh_photo_scale` launch per scale replaces ~60 ATen kernels per (scale, frame)
forward and their autograd backward.
"""
from __future__ import annotations

from typing import Dict, Optional

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import ops


def _frame_T(self_opt, inputs, outputs, frame_id):
    if frame_id == "s":
        return inputs["stereo_T"]
    return outputs[("cam_T_cam", 0, frame_id)]


def tie_break_noise(shape, device, mode="reference"):
    """`M2/trainer.py:644-645`: randn * 1e-5.  'reference' draws from the CPU
    generator exactly as the reference does (same RNG stream, one H2D copy);
    'device' draws on the GPU (different stream, no copy)."""
    if mode == "reference":
        return (torch.randn(shape) * 0.00001).to(device, non_blocking=True)
    if mode == "device":
        return torch.randn(shape, device=device) * 0.00001
    if mode == "none":
        return None
    raise ValueError("noise mode %r" % mode)


def photometric_losses(colors: Dict, disps: Dict, K, inv_K, Ts: Dict, frame_ids, scales, height, width,
                       min_depth=0.1, max_depth=100.0, no_ssim=False, avg_reprojection=False,
                       disable_automasking=False, disparity_smoothness=1e-3, noise: Optional[Dict] = None,
                       noise_mode="reference", want_selection=False):
    """Per-scale loop of compute_losses on the fused kernels.

    colors : {(frame_id, scale): (B,3,h,w)} -- sources at scale 0, frame 0 at every scale
    disps  : {scale: (B,1,h_s,w_s)} network outputs (grad flows here)
    Ts     : {frame_id: (B,4,4)} (grad flows here if required)
    noise  : optional {scale: (B,Fi,H,W)} injected tie-break noise (already * 1e-5)
    returns (losses dict like the reference's, aux dict)
    """
    srcs_ids = list(frame_ids[1:])
    scales = list(scales)
    target = colors[(0, 0)]
    B = target.shape[0]
    srcs = [colors[(f, 0)] for f in srcs_ids]
    T_list = [Ts[f] for f in srcs_ids]
    n_src = len(srcs)
    n_ident = 0 if disable_automasking else (1 if avg_reprojection else n_src)
    nz = None
    if n_ident:
        nz = []
        for scale in scales:
            if noise is not None:
                t = noise[scale]
                if t is not None and t.shape[1] != n_ident:
                    t = t[:, :n_ident].contiguous()
            else:
                t = tie_break_noise((B, n_ident, height, width), target.device, noise_mode)
            nz.append(t)
        if any(t is None for t in nz):
            nz = None
    if scales[0] != 0:
        raise NotImplementedError("the fused objective needs scale 0 first in opt.scales (it is the photometric "
                                  "target: source_scale == 0, trainer.py:483)")
    colors0 = [target] + [colors[(0, s)] for s in scales[1:]]
    out = ops.objective(colors0, srcs, T_list, [disps[s] for s in scales], K, inv_K, noises=nz, min_depth=min_depth,
                        max_depth=max_depth, no_ssim=no_ssim, avg_reprojection=avg_reprojection,
                        automask=not disable_automasking,
                        smooth_weights=[disparity_smoothness / (2 ** s) for s in scales], want_sel=want_selection)
    total, per_scale = out[0], out[1]
    losses, aux = {}, {}
    for i, scale in enumerate(scales):
        losses["loss/{}".format(scale)] = per_scale[i]
        if want_selection:
            sel = out[2 + i]
            aux[("argmin", scale)] = sel
            if n_ident:
                aux["identity_selection/{}".format(scale)] = (sel > n_ident - 1).float()
    losses["loss"] = total
    return losses, aux


# ----------------------------------------------------------------------------- Trainer patches
def fused_generate_images_pred(self, inputs, outputs):
    """Replacement for `Trainer.generate_images_pred`.  The warped images are
    not needed by the fused loss; they are only materialised (no-grad) when the
    trainer is about to log them (`self._dmh_materialise` set by the caller) --
    `outputs[("depth", 0, scale)]` is always provided because
    `compute_depth_losses` (`M2/trainer.py:676-704`) reads it."""
    opt = self.opt
    if opt.v1_multiscale or getattr(opt, "pose_model_type", "") == "posecnn" or opt.predictive_mask:
        return self._dmh_ref_generate_images_pred(inputs, outputs)
    materialise = getattr(self, "_dmh_materialise", False)
    for scale in opt.scales:
        disp = outputs[("disp", scale)]
        disp_full = F.interpolate(disp, [opt.height, opt.width], mode="bilinear", align_corners=False)
        with torch.no_grad():
            if not materialise:
                _, depth = ops.disp_to_depth_cuda(disp_full, opt.min_depth, opt.max_depth)
                outputs[("depth", 0, scale)] = depth
                continue
            for frame_id in opt.frame_ids[1:]:
                T = _frame_T(opt, inputs, outputs, frame_id)
                warped, grid, depth = ops.warp_with_aux(disp_full, inputs[("color", frame_id, 0)], inputs[("K", 0)],
                                                        inputs[("inv_K", 0)], T, opt.min_depth, opt.max_depth)
                outputs[("depth", 0, scale)] = depth
                outputs[("sample", frame_id, scale)] = grid
                outputs[("color", frame_id, scale)] = warped
                if not opt.disable_automasking:
                    outputs[("color_identity", frame_id, scale)] = inputs[("color", frame_id, 0)]


def fused_compute_losses(self, inputs, outputs):
    """Replacement for `Trainer.compute_losses` (`M2/trainer.py:539-674`)."""
    opt = self.opt
    if opt.v1_multiscale or getattr(opt, "pose_model_type", "") == "posecnn" or opt.predictive_mask:
        return self._dmh_ref_compute_losses(inputs, outputs)
    losses = {}
    total_loss = 0
    # supervised / contrastive terms: network-side, stock PyTorch (outside the graft); trainer.py:545-575
    if opt.adv_train and opt.supervised_adv:
        disp = outputs[("disp", 0)]
        color_ben = inputs[("color_ben", 0, 0)]
        with torch.no_grad():
            disp_gt = self.gt_model(color_ben)
        if opt.gt_depth:
            from .layers import disp_to_depth
            color_objmask = inputs[("color_objmask", 0, 0)][:, [0], :, :]
            objdepth = inputs[("objdepth", 0, 0)].unsqueeze(3)
            pred_depth = torch.clamp(disp_to_depth(disp, opt.min_depth, opt.max_depth)[1] * 5.4, 1e-3, 80)
            pseudo_depth = torch.clamp(disp_to_depth(disp_gt, opt.min_depth, opt.max_depth)[1] * 5.4, 1e-3, 80)
            gt_depth = color_objmask * objdepth + pseudo_depth * (1 - color_objmask)
            loss_sup = self.sup_loss_creteria(gt_depth, pred_depth)
        else:
            loss_sup = self.sup_loss_creteria(disp_gt, disp)
        losses["sup_loss"] = loss_sup
        total_loss = total_loss + loss_sup
    if opt.adv_train and opt.contrastive_learning:
        contras_loss = self.models["contrastive_learning"](outputs["middle_features_aug"],
                                                           outputs["middle_features_ben"])
        losses["contras_loss"] = contras_loss
        total_loss = total_loss + contras_loss
    if opt.adv_train and opt.no_original_train:
        losses["loss"] = total_loss
        return losses

    colors = {(0, s): inputs[("color", 0, s)] for s in opt.scales}
    colors[(0, 0)] = inputs[("color", 0, 0)]
    Ts = {}
    for f in opt.frame_ids[1:]:
        colors[(f, 0)] = inputs[("color", f, 0)]
        Ts[f] = _frame_T(opt, inputs, outputs, f)
    disps = {s: outputs[("disp", s)] for s in opt.scales}
    pl, aux = photometric_losses(colors, disps, inputs[("K", 0)], inputs[("inv_K", 0)], Ts, opt.frame_ids, opt.scales,
                                 opt.height, opt.width, opt.min_depth, opt.max_depth, bool(opt.no_ssim),
                                 bool(opt.avg_reprojection), bool(opt.disable_automasking),
                                 opt.disparity_smoothness, noise=getattr(self, "_dmh_noise", None),
                                 noise_mode=getattr(self, "_dmh_noise_mode", "reference"),
                                 want_selection=getattr(self, "_dmh_materialise", False))
    for k, v in aux.items():
        if isinstance(k, str):
            outputs[k] = v
    for s in opt.scales:
        losses["loss/{}".format(s)] = pl["loss/{}".format(s)]
    losses["loss"] = total_loss + pl["loss"]
    return losses


# ----------------------------------------------------------------------------- CUDA-graph replay (small batches)
# keyword options of each objective (everything else is fixed by the constructor's arguments)
_OPTS = {"photometric": frozenset({"min_depth", "max_depth", "no_ssim", "avg_reprojection", "disable_automasking",
                                   "disparity_smoothness", "noise_mode", "want_selection"})}
_OPTS["depth_hints"] = _OPTS["photometric"] | {"use_depth_hints"}


class GraphedObjective:
    """Forward + backward of `photometric_losses` (or, given `depth_hint` and `depth_hint_mask`, of the fused
    `depth_hints.depth_hint_losses`) captured once into a CUDA graph and replayed.

    At the reference's CPU-runnable configuration (B=4, 640x192) one step is ~25 short launches and eager
    PyTorch is launch-bound (0.55 ms per step against 0.22 ms of GPU work, measured on B200); replaying a graph
    removes the Python / launch overhead.  Shapes, options and the set of tensors are frozen at construction;
    `__call__` copies new values into the static buffers (device-to-device), replays, and returns the static
    losses and gradients (valid until the next call).

    Gradients: `grads[scale]` is d(loss)/d(disps[scale]), always.  A `colors[(f, s)]` or `Ts[f]` entry that requires
    grad when the object is built is differentiated too: `grads[("color", f, s)]` and `grads[("T", f)]`, in the
    input's dtype.  Only the frames the objective reads (colour(0, s) for every scale, colour(f, 0) for every source)
    and the sources' poses are considered.  With none marked, the capture is the disparity-only one.

    Tie-break noise: a static buffer per scale, (B, Fi, H, W) for `photometric_losses` and (B, 1, H, W) for the
    depth-hints objective, that the caller may refresh through `noise=`; it is NOT redrawn by the replay.  The noise,
    K / inv_K and the depth hint get no gradient."""

    def __init__(self, colors: Dict, disps: Dict, K, inv_K, Ts: Dict, frame_ids, scales, height, width,
                 noise: Optional[Dict] = None, warmup: int = 3, depth_hint=None, depth_hint_mask=None, **opts):
        if (depth_hint is None) != (depth_hint_mask is None):
            raise ValueError("GraphedObjective: depth_hint and depth_hint_mask go together")
        kind = "photometric" if depth_hint is None else "depth_hints"
        unknown = sorted(set(opts) - _OPTS[kind])
        if unknown:
            raise TypeError("GraphedObjective: option(s) %s not accepted by the %s objective" % (", ".join(unknown), kind))
        dev = colors[(0, 0)].device
        self.frame_ids, self.scales, self.hw, self.opts = list(frame_ids), list(scales), (height, width), dict(opts)
        self.colors = {k: v.detach().clone().requires_grad_(v.requires_grad) for k, v in colors.items()}
        self.disps = {s: disps[s].detach().clone().requires_grad_(True) for s in self.scales}
        self.K, self.inv_K = K.detach().clone(), inv_K.detach().clone()
        self.Ts = {k: v.detach().clone().requires_grad_(v.requires_grad) for k, v in Ts.items()}
        self.hint = depth_hint.detach().clone() if depth_hint is not None else None
        self.hint_mask = depth_hint_mask.detach().clone() if depth_hint_mask is not None else None
        srcs = self.frame_ids[1:]
        used = [(0, s) for s in self.scales] + [(f, 0) for f in srcs]
        self.colour_keys = [k for k in used if self.colors[k].requires_grad]
        self.T_keys = [f for f in srcs if self.Ts[f].requires_grad]
        automask = not self.opts.get("disable_automasking", False)
        if self.hint is not None:
            n_ident = 1 if automask else 0
        else:
            n_ident = 0 if not automask else (1 if self.opts.get("avg_reprojection", False) else len(srcs))
        self.noise = None
        if n_ident:
            B = self.colors[(0, 0)].shape[0]
            self.noise = {s: (noise[s][:, :n_ident].detach().clone() if noise is not None else
                              tie_break_noise((B, n_ident, height, width), dev, "device")) for s in self.scales}
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream())
        # warm-up outside the capture, with the gradients the capture takes: lazy one-time set-up (side streams,
        # kernel attributes, division constants) of every path the replay runs
        with torch.cuda.stream(side):
            for _ in range(max(1, warmup)):
                self._run()
        torch.cuda.current_stream().wait_stream(side)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.losses, self.grads = self._run()

    def _run(self):
        if self.hint is None:
            losses, _ = photometric_losses(self.colors, self.disps, self.K, self.inv_K, self.Ts, self.frame_ids,
                                           self.scales, self.hw[0], self.hw[1], noise=self.noise, **self.opts)
        else:
            from . import depth_hints
            losses, _ = depth_hints.depth_hint_losses(self.colors, self.disps, self.K, self.inv_K, self.Ts,
                                                      self.frame_ids, self.scales, self.hw[0], self.hw[1], self.hint,
                                                      self.hint_mask, noise=self.noise, fused=True, **self.opts)
        S, nc = len(self.scales), len(self.colour_keys)
        grads = torch.autograd.grad(losses["loss"], [self.disps[s] for s in self.scales] +
                                    [self.colors[k] for k in self.colour_keys] + [self.Ts[f] for f in self.T_keys])
        out = dict(zip(self.scales, grads[:S]))
        out.update({("color",) + k: g for k, g in zip(self.colour_keys, grads[S:S + nc])})
        out.update({("T", f): g for f, g in zip(self.T_keys, grads[S + nc:])})
        return losses, out

    @torch.no_grad()
    def __call__(self, colors: Optional[Dict] = None, disps: Optional[Dict] = None, K=None, inv_K=None,
                 Ts: Optional[Dict] = None, noise: Optional[Dict] = None, depth_hint=None, depth_hint_mask=None):
        for dst, src in ((self.colors, colors), (self.disps, disps), (self.Ts, Ts), (self.noise, noise)):
            if src is not None and dst is not None:
                for k, v in src.items():
                    if k in dst:
                        dst[k].copy_(v if dst is not self.noise else v[:, :dst[k].shape[1]], non_blocking=True)
        for dst, src in ((self.K, K), (self.inv_K, inv_K), (self.hint, depth_hint), (self.hint_mask, depth_hint_mask)):
            if src is not None:
                if dst is None:
                    raise ValueError("GraphedObjective: built without a depth hint")
                dst.copy_(src, non_blocking=True)
        self.graph.replay()
        return self.losses, self.grads
