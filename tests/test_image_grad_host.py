"""CPU: the colour-frame gradients of the fused objective (csrc/photo_image_grad.cu) -- candidate gates, the
y-side SSIM coefficients, reflection multiplicities, the L1 sign term and the bilinear scatter into the sources --
compiled for the host from dmh_math.cuh by tests/host_emul_image_grad.cpp and compared, for one scale given the
oracle's argmin, with the autograd gradients of the oracle's objective w.r.t. the target and the source frames."""
import ctypes as C
import os
import subprocess

import pytest
import torch

from depthmodelhardening_b200 import synth
from oracle import photometric as OP
from tests.util import assert_grad_close

HERE = os.path.dirname(os.path.abspath(__file__))
BUILD = os.path.join(HERE, "_build")
SO = os.path.join(BUILD, "libdmh_hostemu_ig.so")
SRC = os.path.join(HERE, "host_emul_image_grad.cpp")
HDR = os.path.join(os.path.dirname(HERE), "depthmodelhardening_b200", "csrc", "dmh_math.cuh")

CASES = {
    "mono_stereo_f1": ((0, "s"), {}),
    "f2": ((0, -1, 1), {}),
    "f1_no_automask": ((0, "s"), dict(disable_automasking=True)),
    "f2_no_automask": ((0, -1, 1), dict(disable_automasking=True)),
    "f2_avg": ((0, -1, 1), dict(avg_reprojection=True)),
    "f1_no_ssim": ((0, "s"), dict(no_ssim=True)),
}


@pytest.fixture(scope="module")
def emu():
    os.makedirs(BUILD, exist_ok=True)
    if (not os.path.exists(SO)) or os.path.getmtime(SO) < max(os.path.getmtime(SRC), os.path.getmtime(HDR)):
        subprocess.check_call(["g++", "-O1", "-ffp-contract=off", "-shared", "-fPIC", "-x", "c++", "-o", SO, SRC])
    return C.CDLL(SO)


def _oracle(pb, opts, dtype):
    """Scale-0 objective without smoothness; returns (argmin or None, d/d target, [d/d source f])."""
    ids = pb.frame_ids
    colors = {k: v.detach().to(dtype).requires_grad_(True) for k, v in pb.color.items()}
    disps = {0: pb.disp[0].detach().to(dtype)}
    Ts = {k: v.to(dtype) for k, v in pb.T.items()}
    noise = {k: v.to(dtype) for k, v in pb.noise.items()}
    total, _, aux = OP.photometric_objective(colors, disps, pb.K.to(dtype), pb.inv_K.to(dtype), Ts, ids, noise, opts,
                                             return_aux=True)
    total.backward()
    return aux.get(("argmin", 0)), colors[(0, 0)].grad, [colors[(f, 0)].grad for f in ids[1:]]


@pytest.mark.parametrize("name", sorted(CASES))
def test_image_grad_math_vs_oracle(emu, name):
    ids, over = CASES[name]
    pb = synth.photo_batch(batch=2, height=40, width=66, frame_ids=ids, scales=(0,), seed=7)
    B, H, W = pb.batch, pb.height, pb.width
    opts = OP.default_opts(scales=[0], min_depth=pb.min_depth, max_depth=pb.max_depth, disparity_smoothness=0.0,
                           **over)
    sel, g_tgt32, g_src32 = _oracle(pb, opts, torch.float32)
    _, g_tgt64, g_src64 = _oracle(pb, opts, torch.float64)
    sel = torch.zeros(B, H, W, dtype=torch.uint8) if sel is None else sel.to(torch.uint8).contiguous()
    srcs = [pb.color[(f, 0)].contiguous() for f in ids[1:]]
    Ts = [pb.T[f].contiguous() for f in ids[1:]]
    dfull = torch.nn.functional.interpolate(pb.disp[0], [H, W], mode="bilinear", align_corners=False).contiguous()
    g_tgt = torch.empty(B, 3, H, W)
    g_src = [torch.empty(B, 3, H, W) for _ in srcs]
    arr = lambda ts: (C.c_void_p * len(ts))(*[t.data_ptr() for t in ts])
    flags = (1 if over.get("no_ssim") else 0) | (2 if over.get("avg_reprojection") else 0)
    emu.emu_image_grad(C.c_void_p(pb.color[(0, 0)].contiguous().data_ptr()), arr(srcs), arr(Ts), len(srcs),
                       C.c_void_p(dfull.data_ptr()), C.c_void_p(pb.K.data_ptr()), C.c_void_p(pb.inv_K.data_ptr()),
                       C.c_void_p(sel.data_ptr()), B, H, W, C.c_float(pb.min_depth), C.c_float(pb.max_depth), flags,
                       0 if over.get("disable_automasking") else 1, C.c_float(1.0 / (B * H * W)),
                       C.c_void_p(g_tgt.data_ptr()), arr(g_src))
    assert_grad_close(g_tgt, g_tgt32, g_tgt64, 1e-5, "grad_target", outlier_frac=2e-3)
    for f, g in enumerate(g_src):
        assert_grad_close(g, g_src32[f], g_src64[f], 1e-5, "grad_src[%d]" % f, outlier_frac=2e-3)
