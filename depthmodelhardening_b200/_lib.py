"""ctypes binding of the C-ABI library (include/dmh_b200.h).

There is NO fallback: if `libdmh_b200.so` is missing or a tensor is not on a
CUDA device the call raises.  Build the library with
`python -c "import __graft_entry__ as g; g.build()"` or `make -C
depthmodelhardening_b200/csrc`.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libdmh_b200.so")

_f = C.c_void_p          # device float*
_i = C.c_int
_ll = C.c_longlong
_fl = C.c_float
_d = C.c_double
_st = C.c_void_p         # cudaStream_t

# name -> (restype, argtypes); mirrors include/dmh_b200.h one to one
SIGNATURES = {
    "dmh_last_error": (C.c_char_p, []),
    "dmh_version": (_i, []),
    "dmh_build_arch": (_i, []),
    "dmh_launch_count": (_ll, []),
    "dmh_const_div_exact": (_i, [_i]),
    "dmh_disp_to_depth": (_i, [_f, _ll, _fl, _fl, _f, _f, _st]),
    "dmh_backproject_fwd": (_i, [_f, _f, _i, _i, _i, _f, _st]),
    "dmh_backproject_bwd_blocks": (_i, [_i, _i]),
    "dmh_backproject_bwd": (_i, [_f, _f, _f, _i, _i, _i, _f, _f, _st]),
    "dmh_project3d_fwd": (_i, [_f, _f, _f, _i, _i, _i, _fl, _f, _st]),
    "dmh_project3d_bwd_blocks": (_i, [_i, _i]),
    "dmh_project3d_bwd": (_i, [_f, _f, _f, _f, _i, _i, _i, _fl, _f, _f, _st]),
    "dmh_grid_sample_fwd": (_i, [_f, _f, _i, _i, _i, _i, _i, _i, _i, _i, _f, _st]),
    "dmh_grid_sample_bwd": (_i, [_f, _f, _f, _i, _i, _i, _i, _i, _i, _i, _i, _f, _f, _st]),
    "dmh_ssim_fwd": (_i, [_f, _f, _i, _i, _i, _i, _f, _st]),
    "dmh_ssim_bwd": (_i, [_f, _f, _f, _i, _i, _i, _i, _f, _f, _st]),
    "dmh_reproj_loss_fwd": (_i, [_f, _f, _i, _i, _i, _i, _i, _f, _st]),
    "dmh_reproj_loss_bwd": (_i, [_f, _f, _f, _i, _i, _i, _i, _i, _f, _f, _st]),
    "dmh_smooth_workspace_floats": (_ll, [_i, _i, _i]),
    "dmh_smooth_fwd": (_i, [_f, _f, _i, _i, _i, _i, _i, _f, _f, _st]),
    "dmh_smooth_bwd": (_i, [_f, _f, _i, _i, _i, _i, _i, _f, _fl, _f, _f, _f, _st]),
    "dmh_upsample_bilinear_fwd": (_i, [_f, _i, _i, _i, _i, _i, _f, _st]),
    "dmh_upsample_bilinear_bwd": (_i, [_f, _i, _i, _i, _i, _i, _f, _f, _st]),
    "dmh_warp_fwd": (_i, [_f, _i, _fl, _fl, _f, _f, _f, _f, _i, _i, _i, _i, _f, _f, _f, _st]),
    "dmh_warp_bwd_blocks": (_i, [_i, _i]),
    "dmh_warp_bwd": (_i, [_f, _f, _i, _fl, _fl, _f, _f, _f, _f, _i, _i, _i, _i, _f, _f, _f, _st]),
    "dmh_identity_loss": (_i, [_f, C.POINTER(C.c_void_p), _i, _i, _i, _i, _i, _f, _st]),
    "dmh_identity_loss_pack": (_i, [_f, _f, _i, _i, _i, _i, _f, _f, _st]),
    "dmh_identity_loss_pack_bf16": (_i, [_f, _f, _i, _i, _i, _i, _f, _f, _f, _st]),
    "dmh_photo_tiles": (_i, [_i, _i]),
    "dmh_photo_scale": (_i, [_f, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), _i, _f, _i, _i, _f, _f, _f, _f, _i, _i, _i,
                             _fl, _fl, _i, _fl, _f, _f, _f, _f, C.POINTER(C.c_void_p), _st]),
    "dmh_photo_multiscale": (_i, [_f, _f, _f, _i, C.POINTER(C.c_void_p), C.POINTER(C.c_int), C.POINTER(C.c_int), _f, _f, _f,
                                  C.POINTER(C.c_void_p), _i, _i, _i, _fl, _fl, _fl, C.POINTER(C.c_void_p),
                                  C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), _st]),
    "dmh_photo_multisource_workspace_floats": (_ll, [_i]),
    "dmh_photo_multisource": (_i, [_f, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), _i, _i, C.POINTER(C.c_void_p),
                                   C.POINTER(C.c_int), C.POINTER(C.c_int), _f, _f, C.POINTER(C.c_void_p),
                                   C.POINTER(C.c_void_p), _i, _i, _i, _fl, _fl, _fl, _f, C.POINTER(C.c_void_p),
                                   C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), _st]),
    "dmh_selftest_reciprocals": (_i, [_f, C.c_uint, _st]),
    "dmh_peer_allreduce": (_i, [C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), _i, _i, _ll, _fl, _f, _f, _f, _f, _ll, _fl, _fl,
                                _f, _st]),
    "dmh_photo_scale_dh": (_i, [_f, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), _i, _f, _i, _i, _f, _f, _f, _f, _f, _f,
                                _f, _i, _i, _i, _fl, _fl, _i, _f, _f, _f, _f, _f, _st]),
    "dmh_smooth_fused_workspace_floats": (_ll, [_i, _i, _i]),
    "dmh_smooth_fused": (_i, [_f, _f, _i, _i, _i, _i, _f, _f, _st]),
    "dmh_objective_finish": (_i, [_i, _i, C.POINTER(C.c_void_p), C.POINTER(C.c_int), C.POINTER(C.c_int),
                                  C.POINTER(C.c_void_p), C.POINTER(C.c_int), C.POINTER(C.c_float), C.c_double, _f, _f,
                                  _f, _st]),
    "dmh_objective_finish_workspace_bytes": (_ll, [_i, _i]),
    "dmh_disp_grad": (_i, [_f, _f, _f, _fl, _f, _f, _f, _fl, _i, _i, _i, _i, _i, _f, _st]),
    "dmh_identity_image_grad": (_i, [_f, C.POINTER(C.c_void_p), _i, C.POINTER(C.c_void_p), _i, _f, _f, _i, _i, _i, _i,
                                     _i, _f, C.POINTER(C.c_void_p), _st]),
    "dmh_photo_image_grad": (_i, [_f, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), _i, _f, _i, _i, _f, _f, _f, _i, _i,
                                  _f, _f, _i, _i, _i, _fl, _fl, _i, _i, _f, C.POINTER(C.c_void_p), _st]),
    "dmh_smooth_image_grad": (_i, [_f, _f, _i, _i, _i, _f, _fl, _i, _i, _f, _f, _i, _f, _st]),
    "dmh_photo_image_grad_dh": (_i, [_f, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), _i, _f, _i, _i, _f, _f, _f, _f,
                                     _i, _i, _i, _fl, _fl, _i, _f, C.POINTER(C.c_void_p), _st]),
    "dmh_compose_u8": (_i, [_f, _f, _f, _f, _i, _i, _i, _i, _f, _st]),
    "dmh_compose_patch_u8": (_i, [_f, _f, _f, _f, _f, _f, _f, _f, _i, _i, _i, _i, _i, _f, _f, _f, _st]),
    "dmh_lanczos_u8": (_i, [_f, _i, _i, _i, _i, _i, _f, _f, _i, _f, _f, _i, _f, _f, _f, _st]),
    "dmh_color_jitter_u8": (_i, [_f, _i, _i, _i, _f, _f, _f, _f, _f, _f, _st]),
    "dmh_unpack_u8": (_i, [_f, _ll, _f, _st]),
    "dmh_axpby_dev": (_i, [_f, _f, _f, _f, _ll, _f, _st]),
    "dmh_perspective_fwd": (_i, [_f, _f, _i, _i, _i, _i, _i, _i, _f, _st]),
    "dmh_perspective_bwd": (_i, [_f, _f, _i, _i, _i, _i, _i, _i, _f, _st]),
    "dmh_patch_apply_fwd": (_i, [_f, _f, _f, _f, _f, _i, _i, _i, _i, _i, _i, _i, _f, _f, _st]),
    "dmh_patch_apply_bwd": (_i, [_f, _f, _f, _f, _i, _i, _i, _i, _i, _i, _i, _i, _i, _f, _st]),
    "dmh_pgd_linf_step": (_i, [_f, _f, _f, _ll, _fl, _fl, _f, _st]),
    "dmh_apgd_linf_step": (_i, [_f, _f, _f, _f, _ll, _fl, _fl, _fl, _f, _st]),
    "dmh_tube_light_patch": (_i, [_f, _i, _i, _d, _d, _d, _d, _i, _i, _d, _d, _d, _f, _f, _st]),
    "dmh_square_linf_candidate": (_i, [_f, _f, _i, _i, _i, _i, _i, _fl, _fl, _fl, _fl, _f, _st]),
    "dmh_keep_best": (_i, [_f, _f, _f, _f, _f, _ll, _st]),
    "dmh_depth_errors": (_i, [_f, _f, _f, _ll, _fl, _fl, _fl, _fl, _fl, _f, _st]),
    "dmh_pgd_l2_step": (_i, [_f, _f, _f, _ll, _fl, _fl, _fl, _f, _st]),
    "dmh_l0_compose_count": (_i, [_f, _f, _f, _i, _i, _i, _fl, _fl, _f, _f, _st]),
    "dmh_l0_adam_step": (_i, [_f, _f, _f, _f, _f, _f, _f, _f, _i, _i, _i, _fl, _f, _fl, _fl, _fl, _fl, _fl, _fl, _i,
                              _st]),
    "dmh_l0_adam_bias_table": (_i, [_fl, _fl, _fl, _i, C.POINTER(C.c_float)]),
    "dmh_l0_adam_step_dev": (_i, [_f, _f, _f, _f, _f, _f, _f, _f, _i, _i, _i, _fl, _f, _fl, _fl, _fl, _fl, _fl, _f, _i, _f,
                                  _st]),
    "dmh_l0_finalize": (_i, [_f, _f, _f, _ll, _fl, _fl, _f, _f, _st]),
    "dmh_topk_select": (_i, [_f, _f, _i, _i, _i, _i, _f, _f, _st]),
    "dmh_hint_select_blocks": (_i, [_i, _i, _i]),
    "dmh_hint_select": (_i, [C.POINTER(C.c_void_p), _i, _f, _f, _f, _f, _f, _f, _i, _i, _i, _i, _f,
                             C.POINTER(C.c_void_p), _f, _f, _st]),
    "dmh_cost_volume_workspace_floats": (_ll, [_i, _i, _i, _i, _i]),
    "dmh_cost_volume": (_i, [_f, _f, _f, _f, _f, _f, _i, _i, _i, _i, _i, _i, _i, _f, _f, _f, _st]),
    "dmh_reduce_sum": (_i, [_f, _ll, _fl, _i, _f, _st]),
    "dmh_reduce_rows": (_i, [_f, _i, _ll, _fl, _f, _st]),
}

ERR_UNSUPPORTED = 3      # DMH_ERR_UNSUPPORTED: nothing was launched, the caller takes the general entry point

_lib = None


def load() -> C.CDLL:
    """Load the shared library (once) and declare every prototype."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "depthmodelhardening_b200: %s not found -- the CUDA extension is not built. "
            "Run `python -c 'import __graft_entry__ as g; g.build()'` (no CPU fallback exists)." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)      # AttributeError if the symbol is missing
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error() -> str:
    return load().dmh_last_error().decode("utf-8", "replace")


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        raise RuntimeError("dmh_b200 %s failed (code %d): %s" % (what, rc, last_error()))


def ptr(t):
    """Device pointer of a contiguous fp32 CUDA tensor (None -> NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("dmh_b200: tensor is on %s; the hot path is CUDA-only (no CPU fallback)" % t.device)
    if not t.is_contiguous():
        raise RuntimeError("dmh_b200: tensor must be contiguous")
    if t.dtype not in (torch.float32, torch.float64, torch.uint8, torch.int32, torch.int64, torch.bfloat16):
        raise RuntimeError("dmh_b200: unsupported dtype %s" % t.dtype)
    return C.c_void_p(t.data_ptr())


def stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr_array(tensors):
    """Host array of device pointers (for the `*_host` arguments)."""
    arr = (C.c_void_p * len(tensors))()
    for i, t in enumerate(tensors):
        arr[i] = None if t is None else ptr(t).value
    return arr


def f32c(t: torch.Tensor) -> torch.Tensor:
    """fp32 + contiguous view/copy of a CUDA tensor (the reference's tensors
    on this path are all contiguous NCHW fp32; SURVEY.md 8(b) 'Ownership')."""
    if not t.is_cuda:
        raise RuntimeError("dmh_b200: tensor is on %s; the hot path is CUDA-only (no CPU fallback)" % t.device)
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()
