"""Drop-in replacements for the hot-path symbols of the reference's `layers.py`
(star-imported by `M2/trainer.py:24`, `DH/trainer.py`, `MD/trainer.py`,
`MD/networks/resnet_encoder.py:19`).  Same names, constructor / forward
signatures, shapes and error behaviour; the arithmetic runs in the sm_100a
kernels of libdmh_b200.so.  CUDA tensors only -- no CPU fallback.
"""
from __future__ import annotations

import torch
import torch.nn as nn

from . import ops


def disp_to_depth(disp, min_depth, max_depth):
    """`layers.py:16-25`: sigmoid disparity -> (scaled_disp, depth)."""
    return ops._DispToDepth.apply(disp, float(min_depth), float(max_depth))


class BackprojectDepth(nn.Module):
    """`layers.py:139-168`: depth image -> homogeneous point cloud (B,4,H*W).

    Unlike the reference no (B,3,N) pixel-grid / ones buffers are kept in HBM
    (168 MB at B=32, 1024x320): the kernel regenerates pixel coordinates.
    The batch size stays baked in, as in the reference (`.view(self.batch_size, ...)`).
    """

    def __init__(self, batch_size, height, width):
        super().__init__()
        self.batch_size = batch_size
        self.height = height
        self.width = width

    def forward(self, depth, inv_K):
        depth = depth.view(self.batch_size, 1, -1)        # same shape error as layers.py:165
        if depth.shape[2] != self.height * self.width:
            raise RuntimeError("shape '[%d, 1, %d]' is invalid for input of size %d" %
                               (self.batch_size, self.height * self.width, depth.numel()))
        return ops._Backproject.apply(depth.view(self.batch_size, 1, self.height, self.width),
                                      ops._mat_batch(inv_K, self.batch_size, "inv_K"),
                                      self.batch_size, self.height, self.width)


class Project3D(nn.Module):
    """`layers.py:171-198`: project points with K @ T, normalise to [-1,1] -> (B,H,W,2)."""

    def __init__(self, batch_size, height, width, eps=1e-7):
        super().__init__()
        self.batch_size = batch_size
        self.height = height
        self.width = width
        self.eps = eps

    def forward(self, points, K, T):
        if points.dim() != 3 or points.shape[1] != 4:
            raise RuntimeError("Project3D: expected homogeneous points of shape (B,4,N), got %s" % (tuple(points.shape),))
        if points.shape[0] != self.batch_size or points.shape[-1] != self.height * self.width:
            raise RuntimeError("shape '[%d, 2, %d, %d]' is invalid for input of size %d" %
                               (self.batch_size, self.height, self.width, points.shape[0] * 2 * points.shape[-1]))
        B = self.batch_size
        return ops._Project3D.apply(points, ops._mat_batch(K, B, "K"), ops._mat_batch(T, B, "T"), B, self.height,
                                    self.width, float(self.eps))


class SSIM(nn.Module):
    """`layers.py:223-253`: clamp((1 - SSIM)/2, 0, 1) with 3x3 reflect-padded boxes."""

    def __init__(self):
        super().__init__()
        self.C1 = 0.01 ** 2
        self.C2 = 0.03 ** 2

    def forward(self, x, y):
        return ops._SSIM.apply(x, y)


def get_smooth_loss(disp, img):
    """`layers.py:207-220`: edge-aware smoothness, 0-dim result."""
    return ops.smooth_loss(disp, img, normalise=False)


def compute_reprojection_loss(self, pred, target):
    """`M2/trainer.py:525-537` as an unbound method: patch onto `Trainer`."""
    return ops.reprojection_loss(pred, target, no_ssim=bool(self.opt.no_ssim))
